/* zmconv_b200.h -- C ABI of libzmconv_b200.so: the B200-native (sm_100a CUDA, FP64) drop-in for
 * the five public procedures of module zm_conv in NorESMhub/CAM-Nor-physics
 * (physics/zm_conv.F90:33-37): zm_convi, zm_convr, zm_conv_evap, convtran, momtran.
 *
 * Layout contract (identical to the reference's chunk storage): every field is the Fortran
 * array (pcols, nlev[, ncnst]) of each chunk, chunks back to back:
 *     element (i,k[,m]) of chunk c  ->  base[ ((c*ncnst + (m-1))*nlev + (k-1))*pcols + (i-1) ]
 * nchunks = 1 reproduces the reference's per-chunk call exactly.  All integer index outputs
 * (ideep, jt, maxg, and the real-valued jctop/jcbot) are 1-based like the reference.
 *
 * Gathered outputs (mu, md, du, eu, ed, dp, dsubcld, jt, maxg) are indexed by gathered position
 * 1..lengath(c) inside each chunk, exactly like the reference (zm_conv.F90:926-940); rows
 * lengath(c)+1..pcols are zero-filled (the reference leaves them undefined).
 *
 * Every *_batch entry point takes HOST pointers and does its own H2D/D2H; the *_batch_dev
 * twins take DEVICE pointers and only enqueue work on `stream` (a cudaStream_t cast to void*,
 * NULL = the CUDA default stream) -- callers that keep physics_state resident use those.
 * Return value: 0 on success; >0 = number of Brent non-convergence events (the reference's
 * endrun at zm_conv.F90:5401-5410, 5557-5566; details via zm_last_error); <0 = API/CUDA error.
 * The library is re-entrant across host threads after zm_init (per-thread workspaces).
 */
#ifndef ZMCONV_B200_H
#define ZMCONV_B200_H
#ifdef __cplusplus
extern "C" {
#endif

/* All scalars zm_convi copies into module state (zm_conv.F90:115-227) + ppgrid + physconst. */
typedef struct zm_params {
  int pcols, pver;              /* ppgrid (zm_conv.F90:17) */
  int limcnv, num_cin;          /* zm_convi args (zm_conv.F90:115-120) */
  int zm_org;                   /* organisation tracer branches (zm_conv.F90:793-819, 5066-5074, 1860-1864): see zm_org_fields */
  int microp;                   /* must be 0: zm_microphysics is not part of the reference tree */
  int no_deep_pbl, lparcel_pbl;
  int cam3;                     /* cam_physpkg_is('cam3'), zm_conv.F90:871 -> undilute buoyan */
  int masterproc;               /* zm_conv.F90:213: tentrm=-dmpdz only assigned on masterproc */
  double c0_lnd, c0_ocn, ke, ke_lnd, momcu, momcd;
  double tiedke_add, capelmt, dmpdz, tau;
  /* physconst (zm_conv.F90:19-20) */
  double cpair, epsilo, gravit, latice, latvap, tmelt, rair, cpwv, cpliq, rh2o, cpvir, zvir;
} zm_params_t;

/* CAM6 namelist defaults + shr_const_mod physconst for a grid. */
void zm_params_default(zm_params_t* p, int pcols, int pver, int limcnv);

/* replaces zm_convi (zm_conv.F90:115; call site zm_conv_intr.F90:376-379). */
int zm_init(const zm_params_t* p);
int zm_finalize(void);
/* copies the last error text (Brent failure diagnostics / CUDA error) into buf. */
int zm_last_error(char* buf, int buflen);

/* replaces zm_convr (zm_conv.F90:231-244; call site zm_conv_intr.F90:662-673).
 * Argument order follows the Fortran dummy list; lchnk/org/orgt/org2d/conv/aero dropped. */
int zm_convr_batch(int nchunks, const int* ncol,
                   const double* t, const double* qh, double* prec, double* jctop, double* jcbot,
                   const double* pblh, const double* zm, const double* geos, const double* zi,
                   double* qtnd, double* heat, const double* pap, const double* paph,
                   const double* dpp, double delt, double* mcon, double* cme, double* cape,
                   double* eurt, const double* tpert, double* dlf, double* pflx, double* zdu,
                   double* rprd, double* mu, double* md, double* du, double* eu, double* ed,
                   double* dp, double* dsubcld, int* jt, int* maxg, int* ideep, int* lengath,
                   double* ql, double* rliq, const double* landfrac,
                   double* dif, double* dnlf, double* dnif, double* rice);
int zm_convr_batch_dev(int nchunks, const int* ncol,
                   const double* t, const double* qh, double* prec, double* jctop, double* jcbot,
                   const double* pblh, const double* zm, const double* geos, const double* zi,
                   double* qtnd, double* heat, const double* pap, const double* paph,
                   const double* dpp, double delt, double* mcon, double* cme, double* cape,
                   double* eurt, const double* tpert, double* dlf, double* pflx, double* zdu,
                   double* rprd, double* mu, double* md, double* du, double* eu, double* ed,
                   double* dp, double* dsubcld, int* jt, int* maxg, int* ideep, int* lengath,
                   double* ql, double* rliq, const double* landfrac,
                   double* dif, double* dnlf, double* dnif, double* rice, void* stream);

/* replaces zm_conv_evap (zm_conv.F90:1712-1717; call site zm_conv_intr.F90:764-769);
 * prdsnow absent (old_snow). prec is inout. */
int zm_conv_evap_batch(int nchunks, const int* ncol,
                       const double* t, const double* pmid, const double* pdel, const double* q,
                       const double* landfrac,
                       double* tend_s, double* tend_s_snwprd, double* tend_s_snwevmlt, double* tend_q,
                       const double* prdprec, const double* cldfrc, double deltat,
                       double* prec, double* snow, double* ntprprd, double* ntsnprd,
                       double* flxprec, double* flxsnow);
int zm_conv_evap_batch_dev(int nchunks, const int* ncol,
                       const double* t, const double* pmid, const double* pdel, const double* q,
                       const double* landfrac,
                       double* tend_s, double* tend_s_snwprd, double* tend_s_snwevmlt, double* tend_q,
                       const double* prdprec, const double* cldfrc, double deltat,
                       double* prec, double* snow, double* ntprprd, double* ntsnprd,
                       double* flxprec, double* flxsnow, void* stream);

/* replaces momtran (zm_conv.F90:2315-2319; call site zm_conv_intr.F90:822-826).
 * il1g = 1, il2g = lengath[c].  q/dqdt/pguall/pgdall/icwu/icwd are (pcols,pver,ncnst). */
int zm_momtran_batch(int nchunks, const int* ncol, const int* domomtran, const double* q, int ncnst,
                     const double* mu, const double* md, const double* du, const double* eu,
                     const double* ed, const double* dp, const double* dsubcld,
                     const int* jt, const int* mx, const int* ideep, const int* lengath,
                     double* dqdt, double* pguall, double* pgdall, double* icwu, double* icwd,
                     double dt, double* seten);
int zm_momtran_batch_dev(int nchunks, const int* ncol, const int* domomtran, const double* q, int ncnst,
                     const double* mu, const double* md, const double* du, const double* eu,
                     const double* ed, const double* dp, const double* dsubcld,
                     const int* jt, const int* mx, const int* ideep, const int* lengath,
                     double* dqdt, double* pguall, double* pgdall, double* icwu, double* icwd,
                     double dt, double* seten, void* stream);

/* replaces convtran (zm_conv.F90:1976-1980; call sites zm_conv_intr.F90:875-879, 1020-1024).
 * doconvtran[ncnst] / cnst_is_dry[ncnst] are HOST int flags in both variants
 * (cnst_is_dry replaces the external cnst_get_type_byind(m).eq.'dry', zm_conv.F90:2087).
 * dqdt(:,:,m) is written (zero + scatter) only for active m >= 2, like the reference. */
int zm_convtran_batch(int nchunks, const int* doconvtran, const double* q, int ncnst,
                      const double* mu, const double* md, const double* du, const double* eu,
                      const double* ed, const double* dp, const double* dsubcld,
                      const int* jt, const int* mx, const int* ideep, const int* lengath,
                      const double* fracis, double* dqdt, const double* dpdry, double dt,
                      const int* cnst_is_dry);
int zm_convtran_batch_dev(int nchunks, const int* doconvtran, const double* q, int ncnst,
                      const double* mu, const double* md, const double* du, const double* eu,
                      const double* ed, const double* dp, const double* dsubcld,
                      const int* jt, const int* mx, const int* ideep, const int* lengath,
                      const double* fracis, double* dqdt, const double* dpdry, double dt,
                      const int* cnst_is_dry, void* stream);

/* The reference's driver for this path, zm_conv_tend (zm_conv_intr.F90:390-951), batched and kept on
 * the device end to end: zm_convr (delt = 0.5*ztodt, :666) -> physics_update of state1 (t += s*dt/cpair,
 * q(:,:,1) += qtnd*dt clipped at qmin=1e-12; physics_types.F90:322-329,427) -> zm_conv_evap (:764) ->
 * momtran on (u,v) (:822; skipped when cam3 = 1, :808 -- ptend_u, ptend_v are then 0 and ptend_s carries no KE
 * dissipation term) -> convtran1 (:865-880) when zm_convtran1_fields attached the constituent arrays ->
 * ptend_all = sum of the ptend_loc (:736,803,833,886).  mcon is returned in kg/m2/s (:693).  zm_org goes through
 * zm_org_fields; zmconv_microp is out of scope.
 * State in: t,q(wv),u,v,pmid,pint,pdel,zm,zi,phis + pblh,tpert,landfrac,cld(pbuf 'CLD').
 * Out: ptend_all%s,q(:,:,1),u,v; the dummy outputs mcon,cme,pflx,zdu,rliq,rice,jctop,jcbot; and the
 * pbuf fields the reference fills (prec_dp, snow_dp, icwmrdp=ql, rprddp=rprd, nevapr_dpcu=evapcdp,
 * DP_FLXPRC/SNW, dlfzm, ZM_MU..ZM_IDEEP) + cape + lengath.
 *
 * Execution (environment variables, read per call):
 *   host-pointer variant: the batch is pipelined over sub-batches of whole chunks so that host->device copies,
 *     kernels and device->host copies overlap; results do not depend on it.  Default for >= 1024 chunks: four
 *     equal sub-batches; ZM_TEND_SUBBATCHES=n
 *     (1..8) or ZM_TEND_SCHEDULE=uniform selects equal parts (default 8, never below 128 chunks each);
 *     ZM_TEND_SCHEDULE="1,2,3,4,6" gives explicit sizes in sixteenths; ZM_TEND_DEBUG prints the host-side timing.
 *     Every output array travels whole; zm_conv_tend_batch_gathered returns the (pcols,pver[p]) outputs as the
 *     convective columns' records instead.
 *   _dev variant: from the third call with an identical argument list on, the step is replayed as a CUDA graph on
 *     `stream` (ZM_DEV_GRAPH=0 disables). */
int zm_conv_tend_batch(int nchunks, const int* ncol, const double* t, const double* q, const double* u,
                       const double* v, const double* pmid, const double* pint, const double* pdel,
                       const double* zm, const double* zi, const double* phis, const double* pblh,
                       const double* tpert, const double* landfrac, const double* cld, double ztodt,
                       double* ptend_s, double* ptend_q, double* ptend_u, double* ptend_v, double* mcon,
                       double* cme, double* pflx, double* zdu, double* rliq, double* rice, double* jctop,
                       double* jcbot, double* prec, double* snow, double* ql, double* rprd, double* evapcdp,
                       double* flxprec, double* flxsnow, double* dlf, double* mu, double* md, double* du,
                       double* eu, double* ed, double* dp, double* dsubcld, int* jt, int* maxg, int* ideep,
                       int* lengath, double* cape);
int zm_conv_tend_batch_dev(int nchunks, const int* ncol, const double* t, const double* q, const double* u,
                       const double* v, const double* pmid, const double* pint, const double* pdel,
                       const double* zm, const double* zi, const double* phis, const double* pblh,
                       const double* tpert, const double* landfrac, const double* cld, double ztodt,
                       double* ptend_s, double* ptend_q, double* ptend_u, double* ptend_v, double* mcon,
                       double* cme, double* pflx, double* zdu, double* rliq, double* rice, double* jctop,
                       double* jcbot, double* prec, double* snow, double* ql, double* rprd, double* evapcdp,
                       double* flxprec, double* flxsnow, double* dlf, double* mu, double* md, double* du,
                       double* eu, double* ed, double* dp, double* dsubcld, int* jt, int* maxg, int* ideep,
                       int* lengath, double* cape, void* stream);

/* zm_conv_tend_batch with the (pcols,pver[p]) outputs returned as one record of doubles per convective column, for a
 * caller that scatters them in its own chunk loop (the batched Fortran binding's zm_batch_scatter in gathered mode).
 * Those outputs are zero outside the convective columns -- the reference computes on the gathered columns
 * ideep(1:lengath), zm_conv.F90:926-940 -- so a caller that zeroes its chunk arrays (physics_ptend_init does) and
 * scatters the records gets zm_conv_tend_batch's arrays exactly, from about a third of the device->host bytes.
 *
 * Per-column outputs travel whole as in zm_conv_tend_batch.  ideep and lengath are required (NULL: -9);
 * dsubcld, jt, maxg may be NULL (they then stay in the device pbuf mirror only).
 *
 * Records: chunk after chunk, within a chunk in gathered order (slot j = 1..lengath(c) is column ideep(j) of chunk c);
 * chunk c's first record has the index sum(lengath(1:c-1)).  With L = pver, a record holds, at these offsets in doubles:
 *   column-indexed, the values of column ideep(j), levels 1..L (or 1..L+1):
 *     ptend_s 0, ptend_q L, ptend_u 2L, ptend_v 3L, cme 4L, zdu 5L, ql 6L, rprd 7L, evapcdp 8L, dlf 9L,
 *     mcon 10L (L+1), pflx 11L+1 (L+1), flxprec 12L+2 (L+1), flxsnow 13L+3 (L+1);
 *   pbuf_in_records != 0 only, slot-indexed (gathered row j of the pbuf field, as zm_conv_tend_batch returns it):
 *     mu 14L+4, md 15L+4, du 16L+4, eu 17L+4, ed 18L+4, dp 19L+4.
 * rec_len = 20L+4 with the pbuf fields, 14L+4 without; with pbuf_in_records = 0 mu..dp stay in the device mirror
 * only (zm_conv_tend_2_batch, zm_conv_tend_diag_batch read them there).  In Fortran one chunk's records are
 * g(rec_len, lengath(c)) and one field of one column a contiguous slice g(off+1:off+nlev, j).
 *
 * rec_cap (doubles) must be >= nchunks*pcols*rec_len, checked before anything else (-9, nothing written); only
 * sum(lengath)*rec_len doubles are written and moved; a sub-batch's records leave the device as soon as its kernels
 * end, while later sub-batches compute.  The copies into rec are asynchronous when the caller has registered it once
 * with cudaHostRegister.  Everything else -- sub-batch pipelining (ZM_TEND_SUBBATCHES,
 * ZM_TEND_SCHEDULE), the one-shot attachments (their arrays travel whole), the device pbuf mirror (published on
 * success only), zm_tend_trace, zm_tend_transfer_bytes, the Brent-failure return -- is that of zm_conv_tend_batch. */
int zm_conv_tend_batch_gathered(int nchunks, const int* ncol, const double* t, const double* q, const double* u,
                                const double* v, const double* pmid, const double* pint, const double* pdel,
                                const double* zm, const double* zi, const double* phis, const double* pblh,
                                const double* tpert, const double* landfrac, const double* cld, double ztodt,
                                double* rliq, double* rice, double* jctop, double* jcbot, double* prec, double* snow,
                                double* cape, double* dsubcld, int* jt, int* maxg, int* ideep, int* lengath,
                                int pbuf_in_records, double* rec, long long rec_cap);

/* Per-rank terms of the global water/energy budget check (the quantities check_energy_chng compares
 * after ZM, physpkg.F90:2865-2867); all pointers are device pointers, out6 receives
 * [sum pdel/g*ptend_q, sum 1000*(prec+rliq), sum pdel/g*ptend_s,
 *  sum 1000*(latvap*(prec+rliq)+latice*snow), #convective columns, #columns].
 * Multi-GPU runs all-reduce these six doubles over NCCL; nothing else crosses GPUs. */
int zm_conservation_dev(int nchunks, const int* ncol, const double* pdel, const double* ptend_q,
                        const double* ptend_s, const double* prec, const double* snow, const double* rliq,
                        const int* lengath, double* out6, void* stream);

/* ---- "next" rows (SURVEY.md section 8f, N4): neighbours of the path --------------------------------
 * geopotential_t (physics/geopotential.F90:153-247): zm/zi from t,q,p; dycore_lr != 0 selects the FV
 * ('LR') hydrostatic branch (:218-223), 0 the EUL/SE one (:224-233).  q is q(:,:,1); rair/zvir are
 * (pcols,pver) like the reference's dummy arrays.  The generalized-Tv branch (:248-310) is
 * zm_geopotential_t_gen_batch below. */
int zm_geopotential_t_batch(int nchunks, const int* ncol, int dycore_lr, const double* piln, const double* pmln,
                            const double* pint, const double* pmid, const double* pdel, const double* rpdel,
                            const double* t, const double* q, const double* rair, double gravit,
                            const double* zvir, double* zi, double* zm);
int zm_geopotential_t_batch_dev(int nchunks, const int* ncol, int dycore_lr, const double* piln,
                            const double* pmln, const double* pint, const double* pmid, const double* pdel,
                            const double* rpdel, const double* t, const double* q, const double* rair,
                            double gravit, const double* zvir, double* zi, double* zm, void* stream);
/* geopotential_t, generalized-virtual-temperature branch (physics/geopotential.F90:248-310), the one the reference
 * takes when dycore_is('MPAS') or dycore_is('SE'): tvfac = (1 + (zvir+1)*q(:,:,1)*qfac) * 1/(1 + sum q_s*qfac) with
 * qfac = 1/(1 - sum q_s) over the thermodynamically active species.  q3 is the constituent array q(pcols,pver,ncnst)
 * of each chunk ([chunk][m][k][i]); species_idx[nspecies] are the 1-based constituent indices of
 * air_composition::thermodynamic_active_species_idx (that module is not in the reference tree, hence an argument;
 * a host array for the host-pointer call, a device array for the _dev call).  dycore_lr as above (:283-298). */
int zm_geopotential_t_gen_batch(int nchunks, const int* ncol, int dycore_lr, int ncnst, int nspecies,
                            const int* species_idx, const double* piln, const double* pmln, const double* pint,
                            const double* pmid, const double* pdel, const double* rpdel, const double* t,
                            const double* q3, const double* rair, double gravit, const double* zvir, double* zi,
                            double* zm);
int zm_geopotential_t_gen_batch_dev(int nchunks, const int* ncol, int dycore_lr, int ncnst, int nspecies,
                            const int* species_idx, const double* piln, const double* pmln, const double* pint,
                            const double* pmid, const double* pdel, const double* rpdel, const double* t,
                            const double* q3, const double* rair, double gravit, const double* zvir, double* zi,
                            double* zm, void* stream);
/* convect_diagnostics_calc (physics/convect_diagnostics.F90:115-249) for shallow_scheme='CLUBB_SGS', the
 * only configuration in which its locals cnt2/cnb2 are defined (:187-198): zeroes the shallow-scheme
 * fields, merges them into cmfmc/qc/rliq, merges cloud top/bottom indices and looks up their pressures,
 * rprdtot = rprdsh + rprddp. */
int zm_convect_diagnostics_batch(int nchunks, const int* ncol, double* cmfmc, double* qc, double* qc2,
                            double* rliq, double* rliq2, const double* pmid, const double* rprddp, double* cnt,
                            double* cnb, double* cmfmc2, double* rprdsh, double* rprdtot, double* pcnt,
                            double* pcnb);
int zm_convect_diagnostics_batch_dev(int nchunks, const int* ncol, double* cmfmc, double* qc, double* qc2,
                            double* rliq, double* rliq2, const double* pmid, const double* rprddp, double* cnt,
                            double* cnb, double* cmfmc2, double* rprdsh, double* rprdtot, double* pcnt,
                            double* pcnb, void* stream);

/* In zm_conv_tend_batch (host-pointer variant) the pbuf outputs mu, md, du, eu, ed, dp, dsubcld, jt, maxg,
 * ideep, lengath may be NULL: they are then not copied back but stay in a device-resident mirror owned by
 * the calling thread until its next zm_conv_tend_batch call (the reference keeps them in pbuf between
 * tphysbc and tphysac, zm_conv_intr.F90:113-132).  zm_conv_tend_2_batch replaces zm_conv_tend_2
 * (zm_conv_intr.F90:955-1028): dpdry gather (:1014-1017) + convtran (:1020-1024) using that mirror.
 * q, fracis, ptend_q are (pcols,pver,pcnst); pdeldry is (pcols,pver). */
int zm_conv_tend_2_batch(int nchunks, const int* doconvtran, const double* q, int pcnst, const double* pdeldry,
                         const double* fracis, double* ptend_q, double ztodt, const int* cnst_is_dry);
/* the same on DEVICE arrays, the pbuf fields being the caller's own device arrays (as zm_conv_tend_batch_dev filled
 * them); doconvtran / cnst_is_dry stay HOST flags.  Enqueue on the stream the tend step ran on. */
int zm_conv_tend_2_batch_dev(int nchunks, const int* doconvtran, const double* q, int pcnst, const double* pdeldry,
                         const double* fracis, double* ptend_q, double ztodt, const int* cnst_is_dry,
                         const double* mu, const double* md, const double* du, const double* eu,
                         const double* ed, const double* dp, const double* dsubcld, const int* jt,
                         const int* maxg, const int* ideep, const int* lengath, void* stream);

/* zm_conv_tend_2_batch on the convective columns' records, for a caller that packs and scatters them in its own chunk
 * loops (the batched Fortran binding's gathered mode).  convtran reads and writes only the gathered columns
 * ideep(1:lengath) (zm_conv.F90:2109-2114, 2298-2304; dpdry zm_conv_intr.F90:1014-1017) and the model copies the
 * result into a ptend that physics_ptend_init has just zeroed, so only those columns of the flagged constituents
 * need to cross PCIe and host memory.
 *
 * Active list: m = 2..pcnst (1-based) with doconvtran(m) != 0, ascending, nact of them; entry 1 is ignored as in
 * zm_conv_tend_2_batch.  cnst_is_dry[pcnst] may be NULL (all moist).
 * Layout, with base(c) = sum(lengath(1:c-1)) and n = lengath(c): chunk c's block of q_rec, fracis_rec and dqdt_rec
 * starts at nact*pver*base(c) and is the Fortran array g(n, pver, nact) = q(ideep(1:n), :, iact(1:nact)) of the chunk
 * (C order [a][k][slot]); pdeldry_rec holds pdeldry(ideep(1:n), :) at pver*base(c).  The pack and the scatter of a
 * chunk are each one array section.
 * mu..dp, jt, maxg, ideep, lengath come from the calling thread's device pbuf mirror as in zm_conv_tend_2_batch
 * (none, or another nchunks: -7).  Refused with -9 before anything is written: lengath differing from the mirror's
 * (read back from the device: 4*nchunks bytes), rec_cap (doubles; the size of each of q_rec, fracis_rec, dqdt_rec)
 * below sum(lengath)*pver*nact, pdeldry_rec NULL while a flagged constituent is dry.  nact = 0: returns 0, writes
 * nothing.  Exactly sum(lengath)*pver*nact doubles of dqdt_rec are written; the records are the only data that cross
 * PCIe besides that lengath check.  Device times go to the GPTL name convtran2 (zm_get_timers). */
int zm_conv_tend_2_batch_gathered(int nchunks, const int* lengath, const int* doconvtran, int pcnst,
                                  const int* cnst_is_dry, const double* q_rec, const double* fracis_rec,
                                  const double* pdeldry_rec, double* dqdt_rec, long long rec_cap, double ztodt);
/* bytes the calling thread's last zm_conv_tend_2_batch[_gathered] moved over PCIe in each direction (its data arrays
 * and, in the gathered call, the lengath check; the constituent flag table, uploaded only when the flags change, is
 * not counted) */
int zm_tend_2_transfer_bytes(long long* h2d, long long* d2h);

/* zm_org = 1 (zmconv_org, SURVEY N3): attach the pointer dummies org / orgt / org2d of zm_convr
 * (zm_conv.F90:242, 421-423; zm_conv_intr.F90:656-659) for the NEXT zm_convr_batch / zm_conv_tend_batch [_dev] call
 * of the calling thread: host pointers for the host-pointer entry points, device pointers for *_dev.  All three are
 * (pcols,pver) per chunk.  org: state%q(:,:,ixorg) (in).  org2d: pressure-weighted column mean of org (out,
 * zm_conv.F90:793-819).  orgt: ptend%q(:,:,ixorg) (out) -- zm_convr zeroes it (zm_conv.F90:555-556); zm_conv_tend adds
 * the organisation tendency diagnosed from the evaporation of convective precipitation (zm_conv_intr.F90:773-777).
 * With zm_org = 1 the test-parcel entrainment is divided by (1 + 10 org) and land-weighted (zm_conv.F90:5066-5074) and
 * zm_conv_evap uses ke over ocean / ke_lnd over land (zm_conv.F90:1860-1864).  Calls without attached fields fail (-8). */
int zm_org_fields(const double* org, double* orgt, double* org2d);

/* convtran1 inside zm_conv_tend (zm_conv_intr.F90:865-880: `lq(2:) = cnst_is_convtran1(2:)`, convtran on state1%q with
 * fake_dpdry = 0, result summed into ptend_all%q): attach for the NEXT zm_conv_tend_batch[_dev] call of the calling
 * thread (host pointers for the host-pointer entry point, device pointers for _dev) the constituent arrays
 * q = state%q, fracis (pbuf 'FRACIS') and ptend_q = ptend_all%q, all (pcols,pver,pcnst) per chunk, and the HOST flag
 * arrays doconvtran[pcnst] (= cnst_is_convtran1; entry 0, water vapour, is ignored like the reference's m = 2..pcnst
 * loop, zm_conv.F90:2084) and cnst_is_dry[pcnst] (may be NULL = all moist).  ptend_q(:,:,m) is written (zero + scatter,
 * zm_conv.F90:2298-2304) for the flagged m only; ptend_all%q(:,:,1) stays the separate ptend_q argument of
 * zm_conv_tend_batch.  state1%q(:,:,m >= 2) equals state%q(:,:,m) at that point of zm_conv_tend (only q(:,:,1) -- and the
 * org tracer under zm_org, which is not a convtran1 species -- was updated), so the caller's array is transported
 * as is.  The host-pointer variant moves only the flagged slices over PCIe.  pcnst <= 0 or a NULL pointer detaches. */
int zm_convtran1_fields(int pcnst, const int* doconvtran, const int* cnst_is_dry, const double* q,
                        const double* fracis, double* ptend_q);

/* zm_conv_tend's history fields (zm_conv_intr.F90:676-857): attach for the NEXT zm_conv_tend_batch[_dev] call of the
 * calling thread (host pointers for the host-pointer entry point, device pointers for _dev) the intermediate results
 * the step otherwise keeps to itself -- zm_convr's heat (ptend_loc%s), qtnd (ptend_loc%q(:,:,1)), eurt, dif, dnlf, dnif;
 * zm_conv_evap's (on state1) tend_s, tend_s_snwprd, tend_s_snwevmlt, ntprprd, ntsnprd; momtran's (on state1%u/v) seten,
 * pguall, pgdall, icwu, icwd.  The procedures' own quantities: no /cpair, no unit change (ZMDT = heat/cpair etc. stay
 * with the caller's outfld calls).  pguall, pgdall, icwu, icwd are (pcols,pver,2) per chunk, component 1 = u and 2 = v
 * as momtran returns them; all others (pcols,pver) per chunk.  Any pointer may be NULL: that field is neither
 * materialised nor copied.  Every element of an attached field is defined on return; padding columns (i > ncol) are 0,
 * and with cam3 = 1 (no momtran, zm_conv_intr.F90:808) the five momtran fields are 0.  The regular outputs do not
 * depend on what is attached.  The host-pointer variants copy the attached fields whole, also with the gathered
 * return, and zm_tend_transfer_bytes counts them. */
int zm_conv_tend_hist_fields(double* heat, double* qtnd, double* eurt, double* dif, double* dnlf, double* dnif,
                             double* tend_s, double* tend_s_snwprd, double* tend_s_snwevmlt,
                             double* ntprprd, double* ntsnprd,
                             double* seten, double* pguall, double* pgdall, double* icwu, double* icwd);

/* zm_conv_tend's history diagnostics that involve arithmetic (zm_conv_intr.F90): freqzm (:685-688, 1 where the
 * column convects), mu_out / md_out (:575-576, 700-706: ungathered mass fluxes in kg/m2/s), pcont / pconb (:721-729:
 * pressure at cloud top / base, ps elsewhere).  ps, freqzm, pcont, pconb are (pcols); pmid, mu, md, mu_out, md_out
 * (pcols,pver).  In the host-pointer variant mu, md, jt, maxg, ideep, lengath may all be NULL: they are then taken
 * from the device pbuf mirror of the calling thread's last zm_conv_tend_batch. */
int zm_conv_tend_diag_batch(int nchunks, const int* ncol, const double* ps, const double* pmid, const double* mu,
                            const double* md, const int* jt, const int* maxg, const int* ideep, const int* lengath,
                            double* freqzm, double* mu_out, double* md_out, double* pcont, double* pconb);
int zm_conv_tend_diag_batch_dev(int nchunks, const int* ncol, const double* ps, const double* pmid, const double* mu,
                            const double* md, const int* jt, const int* maxg, const int* ideep, const int* lengath,
                            double* freqzm, double* mu_out, double* md_out, double* pcont, double* pconb,
                            void* stream);

/* Pipeline timeline of the calling thread's last zm_conv_tend_batch[_gathered] (diagnostics): per sub-batch six times
 * in ms (inputs on device, late inputs on device, zm_convr done, all kernels done, zm_convr outputs on host,
 * remaining outputs -- in the gathered call the records -- on host).  Returns the number of sub-batches; fills at most
 * cap doubles. */
int zm_tend_trace(double* ms, int cap);
/* bytes the calling thread's last zm_conv_tend_batch[_gathered] moved over PCIe in each direction */
int zm_tend_transfer_bytes(long long* h2d, long long* d2h);

/* Synchronises `stream` (NULL = the CUDA default stream) and returns the number of
 * Brent non-convergence events of this thread's last zm_convr_batch_dev call (0 = clean). */
int zm_sync_check(void* stream);

/* ---- diagnostics used by tests and bench (not part of the reference surface) ------------ */
/* evaluates the portable math library on the DEVICE: id 0 log,1 log10,2 exp,3 10**x,4 x**y */
int zm_math_eval_dev(int id, int n, const double* x_host, const double* y_host, double* out_host);
/* same functions evaluated by the host build of zm_math.h */
int zm_math_eval_host(int id, int n, const double* x, const double* y, double* out);
/* device scalar thermodynamics, one call per element (host arrays in/out):
 * id 0: entropy(t,p,q)  1: enthalpy(t,p,q,z)  2: ientropy(s,p,q,tfg)->t,qst
 * 3: ienthalpy(s,p,z,q,tfg)->t,qst  4: qsat_hPa(t,p)->es,q  5: table qsat(t,pPa)->es,qs */
int zm_thermo_eval_dev(int id, int n, const double* a, const double* b, const double* c,
                       const double* d, const double* e, double* out0, double* out1);
/* FP64 FMA-chain microbenchmark on the current device: returns achieved FLOP/s (FMA = 2). */
double zm_fp64_peak_flops(int iters);
/* single-warp latency microbenchmark: cycles per dependent call of
 * 0 div,1 log,2 log10,3 10**x,4 exp,5 es(T),6 enthalpy,7 entropy,8 ienthalpy,9 ientropy,10 pow,
 * 11 Goff-Gratch formula,12 DFMA,13 DADD,14 DMUL,15 div_hot,16 log_hot,17 es(T) shared-memory table,
 * 18 compare+select,19 F2I+I2F.  Writes min(cap, ZM_MICROBENCH_N) values, returns that count. */
#define ZM_MICROBENCH_N 20
int zm_microbench(long long* cycles, int cap, int n);
/* per-kernel device time (ms) of the last zm_convr_batch[_dev] call made with profiling on:
 * names/ms arrays of length *n (max 24). */
int zm_set_profiling(int on);
int zm_get_kernel_times(int* n, const char** names, float* ms);
/* the same device times under the reference's GPTL timer names (zm_conv_intr.F90:654-880, 1019-1025):
 * zm_convr, zm_conv_evap, momtran, convtran1, convtran2 (+ physics_update for the glue kernels); *n in = capacity
 * (>= 6), out = count.  Covers the calling thread's last profiled zm_conv_tend_batch_dev and zm_conv_tend_2_batch. */
int zm_get_timers(int* n, const char** names, float* ms);
/* "ZMSRCHASH:<sha256 prefix of the sources and flags the binary was built from> sm_100a" */
const char* zm_build_info(void);
/* number of kernel launches issued by this thread since the last call (bench's gpu_launches) */
long long zm_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif
