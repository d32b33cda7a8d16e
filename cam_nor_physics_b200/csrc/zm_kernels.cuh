// zm_kernels.cuh -- sm_100a CUDA kernels for the CAM-Nor Zhang-McFarlane deep-convection path.
//
// Design (B200-first, not a translation of the chunk-loop Fortran):
//   * one thread per column for the trigger (buoyan_dilute + parcel_dilute): the two parcel
//     loops of the reference (zm_conv.F90:4997-5148 and 5175-5273) are fused into ONE
//     bottom-up sweep with all per-level state carried in registers, the only per-level
//     storage being one buoyancy value in shared memory ([level][thread], conflict free);
//     launches that leave the schedulers mostly idle (second passes, small batches) put the two
//     loops on two warps instead (k_buoyan_dilute_ws);
//   * trigger/gather (zm_conv.F90:905-917, 1095-1111) is an order-preserving warp-ballot
//     compaction per chunk, so ideep/lengath are bit-identical to the serial loop, plus a
//     device-side worklist so that later kernels run only on convective columns and the host
//     never synchronises inside a step;
//   * pass 2 of the dilute CAPE runs only on pass-1 triggered columns (the others are provably
//     unchanged: their dmpdz row is untouched, zm_conv.F90:544,1053,1074); after cam3's undilute first
//     pass it runs on every column of the chunks that have a first-gather column, as the reference does;
//   * both CAPE passes take their columns from a list bucketed by parcel launch level, most levels
//     first (k_order_*): a warp lasts as long as its longest lane, and the level count decides that;
//   * cldprp + closure + q1q2_pjr + scatter + precipitation are one fused per-column kernel;
//   * zm_conv_evap is a thread-per-column level scan, momtran a warp per convective column,
//     convtran a block per chunk (zm_transport.cuh).
// All arithmetic is FP64 with -fmad=false and the portable zm_math.h transcendentals, so
// results are bit-identical to the CPU oracle built with the same math header.
#pragma once
#include "zm_device.cuh"

#define ZM_MAXCIN 5
#define ZM_ORD_KEYS 132                 // launch levels 1..pver <= 128 (+ slack)
#define ZM_ORD_INTS (4 * ZM_ORD_KEYS)   // per CAPE pass: bucket sizes, bucket cursors

// ---- argument blocks ----------------------------------------------------------------------
struct ConvrIn {
  int nchunks;
  const int* ncol;                       // [nchunks]
  const double *t, *qh, *pap, *paph, *dpp, *zm, *zi, *geos, *pblh, *tpert, *landfrac;
  double delt;
  const double* org;                     // zm_org only: state%q(:,:,ixorg), (pcols,pver) per chunk; else NULL
};
struct ConvrOut {
  double *prec, *jctop, *jcbot, *qtnd, *heat, *mcon, *cme, *cape, *eurt, *dlf, *pflx, *zdu, *rprd;
  double *mu, *md, *du, *eu, *ed, *dp, *dsubcld;
  int *jt, *maxg, *ideep, *lengath;
  double *ql, *rliq, *dif, *dnlf, *dnif, *rice;
  int mcon_kgm2s = 0;                    // fused zm_conv_tend step: mcon leaves the plume kernel as mcon*100/gravit
                                         // (the unit conversion of zm_conv_intr.F90:693; zm_convr itself returns mb/s)
};
// per-column scratch (all sized ncolpad = nchunks*pcols; 2-D ones [pver][ncolpad])
struct ConvrWork {
  double *cape, *cin, *tl, *dmpdz;       // [ncolpad]
  int *lcl, *lel, *mx;                   // [ncolpad]
  double *tp, *qstp;                     // [pver][ncolpad]
  double *ab;                            // [3][pver][ncolpad] first-loop parcel handed to the second loop (k_buoyan_dilute_ws)
  int *wl1, *wl2;                        // worklists: pass-1 columns; final (col, slot) pairs
  int *okey;                             // [ncolpad] launch level of the dilute parcel (the CAPE kernels' work key)
  int *ord1, *ord2;                      // [ncolpad] columns of CAPE pass 1 / pass 2, most parcel levels first
  int *count;                            // [0]=n pass-1, [1]=n final, [2]=brent failures, [3]=real columns;
                                         // then ZM_ORD_INTS work-ordering counters (see k_order_*)
  double *errinfo;                       // first failure: rcall, col, p, Tfg, qt, s
  int *n1chunk;                          // [nchunks] pass-1 convective columns per chunk (k_trigger<0>)
  int skip_idle_chunks;                  // CAPE kernel: leave chunks with n1chunk == 0 alone (cam3 second pass)
  int ws_gate;                           // second pass: worklists up to this size go to k_buoyan_dilute_ws, larger ones
                                         // to k_buoyan_dilute (both are launched, the device-side count decides)
};

__device__ __forceinline__ size_t cidx(int c, int k0, int i, int nlev) {
  return ((size_t)c * nlev + k0) * P.pcols + i;      // k0 is 0-based
}

__device__ __forceinline__ void report_fail(const ConvrWork& w, int rcall, int col, double p,
                                            double tfg, double qt, double s) {
  int n = atomicAdd(&w.count[2], 1);
  if (n == 0) {
    w.errinfo[0] = rcall; w.errinfo[1] = col; w.errinfo[2] = p; w.errinfo[3] = tfg;
    w.errinfo[4] = qt; w.errinfo[5] = s;
  }
}

// ---- output initialisation (zm_conv.F90:559-563, 625-650, 771-784, 906) ---------------------
// Per-column outputs, the per-column scratch the CAPE passes read and the worklist counters: on the launching stream.
__global__ void k_convr_init_cols(ConvrIn in, ConvrOut o, ConvrWork w) {
  const int pcols = P.pcols, pver = P.pver;
  const size_t ncolpad = (size_t)in.nchunks * pcols;
  size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t nth = (size_t)gridDim.x * blockDim.x;
  for (size_t e = tid; e < ncolpad; e += nth) {
    o.prec[e] = 0.0; o.rliq[e] = 0.0; o.rice[e] = 0.0; o.cape[e] = 0.0; o.dsubcld[e] = 0.0;
    // jctop = pver, jcbot = 1 for i <= ncol (zm_conv.F90:781-782); padding lanes are zero-filled
    const bool real_col = (int)(e % pcols) < in.ncol[e / pcols];
    o.jctop[e] = real_col ? (double)pver : 0.0; o.jcbot[e] = real_col ? 1.0 : 0.0;
    o.jt[e] = 0; o.maxg[e] = 0; o.ideep[e] = 0;
    w.dmpdz[e] = -P.tentrm;
  }
  for (size_t e = tid; e < (size_t)in.nchunks; e += nth) o.lengath[e] = 0;
  for (size_t e = tid; e < 4 + ZM_ORD_INTS; e += nth) w.count[e] = 0;
}
// The per-level outputs (zero outside the convective columns; nothing reads them before the plume kernel writes the
// convective columns) and whatever else the caller wants zeroed with them (the fused step: ptend_u, ptend_v and the KE
// heating, which momtran writes for convective columns only): 16-byte stores over a list of arrays, scalar ones for
// an array that is not 16-byte aligned or has an odd length.
// Measured and dropped: the same fill on a side stream, either as ONE WARP PER SM with 32 registers -- resident beside
// the single wave of the first CAPE pass, which leaves 1,024 of an SM's 65,536 registers free -- or as an ordinary grid
// beside cldprp / the second CAPE pass, joined before the plume kernel: 2.107 / 2.109 ms against 2.108 ms with the
// fill on the launching stream ahead of everything.
// Capacity: the fused step under cam3 with every history field attached lists 26 arrays -- zm_convr's 13 + 4 per-level
// outputs, mcon and pflx, ptend_u and ptend_v, then pguall, pgdall, seten, icwu and icwd.
#define ZM_FILL_MAX 26
struct FillList {
  double* p[ZM_FILL_MAX];
  unsigned long long n[ZM_FILL_MAX];     // doubles
  int cnt;
};
__global__ void __launch_bounds__(256)
k_zero_fill(FillList f) {
  const double2 z = make_double2(0.0, 0.0);
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
  for (int a = 0; a < f.cnt; ++a) {
    double* p = f.p[a];
    const size_t n = f.n[a];
    if ((((uintptr_t)p) & 15) == 0 && !(n & 1)) {
      double2* q = reinterpret_cast<double2*>(p) + tid;
      double2* const end = reinterpret_cast<double2*>(p) + (n >> 1);
#pragma unroll 4
      for (; q < end; q += nth) *q = z;
    } else {
      for (size_t e = tid; e < n; e += nth) p[e] = 0.0;
    }
  }
}

// ---- launch level of the dilute parcel and the work ordering of the CAPE passes ---------------------
// boundary-layer top level (zm_conv.F90:839-843)
__device__ __forceinline__ int pbl_top_level(const ConvrIn& in, int c, int i, double zs, double pblh) {
  const int pver = P.pver, msg = P.msg;
  int pblt = pver;
  for (int k = pver - 1; k >= msg + 1; --k) {
    const double zk = in.zm[cidx(c, k - 1, i, pver)] + zs;
    const double zfk = in.zi[cidx(c, k - 1, i, pver + 1)] + zs, zfk1 = in.zi[cidx(c, k, i, pver + 1)] + zs;
    if (fabs(zk - zs - pblh) < (zfk - zfk1) * 0.5) pblt = k;
  }
  return pblt;
}
// moist static energy that picks the launch level (zm_conv.F90:4677-4689; same expression at 4650-4652)
__device__ __forceinline__ double hmn_launch(double tk, double qk, double zk) {
  return (P.cpres + qk * P.cpliq) * tk / (1.0 + qk) + (1.0 + qk / P.eps1) / (1.0 + qk) * P.grav * zk +
         (P.rl - (P.cpliq - P.cpwv) * (tk - P.tfreez)) * qk;
}
// level the parcel is launched from: `mx` of buoyan_dilute (zm_conv.F90:4677-4689), or the top level of the
// mixed parcel layer when parcel_pbl is on (zm_conv.F90:4638-4673).  Used only as the work key below; the CAPE
// kernel derives the level itself from the same two functions.
__device__ __forceinline__ int launch_level(const ConvrIn& in, int c, int i) {
  const int pcols = P.pcols, pver = P.pver, msg = P.msg;
  const double zs = in.geos[(size_t)c * pcols + i] * P.rgrav;
  const int pblt = pbl_top_level(in, c, i, zs, in.pblh[(size_t)c * pcols + i]);
  if (P.lparcel_pbl) {
    const double pbl_dz = (in.zm[cidx(c, pblt - 1, i, pver)] + zs) - zs;
    const double parcel_dz = fmax2(in.zi[cidx(c, pver - 1, i, pver + 1)], P.parcel_hscale * pbl_dz);
    int ipar = pver;
    for (int k = pver; k >= msg + 1; --k)
      if (in.zi[cidx(c, k, i, pver + 1)] <= parcel_dz) ipar = k;
    return ipar;
  }
  const int lon = min(pver, pblt + 2);
  int mx = lon;
  double hmax = 0.0;
  for (int k = lon; k >= max(pblt, msg + 1); --k) {
    const double hmn = hmn_launch(in.t[cidx(c, k - 1, i, pver)], in.qh[cidx(c, k - 1, i, pver)],
                                  in.zm[cidx(c, k - 1, i, pver)] + zs);
    if (hmn > hmax) { hmax = hmn; mx = k; }
  }
  return mx;
}

// A column's parcel sweep climbs from its launch level to level msg+1 with three Brent inversions per level, and a
// warp of k_buoyan_dilute lasts as long as its longest lane.  Both CAPE passes therefore take their columns from a
// list bucketed by launch level, most levels first (counting sort): lanes of a warp then climb the same levels (the
// iteration counts of the inversions follow the level closely), and every SM receives long and short blocks.
// The order changes nothing in the results: columns are independent.
//   counters (w.count + 4): [0,K) bucket sizes pass 1, [K,2K) cursors pass 1, [2K,3K) sizes pass 2, [3K,4K) cursors
template <int PASS>
__global__ void __launch_bounds__(256) k_order_count(ConvrIn in, ConvrWork w) {
  __shared__ int s_n[ZM_ORD_KEYS];
  for (int t = threadIdx.x; t < ZM_ORD_KEYS; t += blockDim.x) s_n[t] = 0;
  __syncthreads();
  const int pcols = P.pcols;
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = PASS == 1 ? in.nchunks * pcols : w.count[0];
  if (gid < n) {
    const int col = PASS == 1 ? gid : w.wl1[gid];
    const int c = col / pcols, i = col - c * pcols;
    if (i < in.ncol[c]) {
      int key;
      if (PASS == 1) { key = min(max(launch_level(in, c, i), 0), ZM_ORD_KEYS - 1); w.okey[col] = key; }
      else key = w.okey[col];
      atomicAdd(&s_n[key], 1);
    }
  }
  __syncthreads();
  int* sizes = w.count + 4 + (PASS == 1 ? 0 : 2 * ZM_ORD_KEYS);
  for (int t = threadIdx.x; t < ZM_ORD_KEYS; t += blockDim.x)
    if (s_n[t]) atomicAdd(&sizes[t], s_n[t]);
}
template <int PASS>
__global__ void __launch_bounds__(256) k_order_scatter(ConvrIn in, ConvrWork w) {
  __shared__ int s_size[ZM_ORD_KEYS], s_base[ZM_ORD_KEYS], s_n[ZM_ORD_KEYS], s_off[ZM_ORD_KEYS];
  const int* sizes = w.count + 4 + (PASS == 1 ? 0 : 2 * ZM_ORD_KEYS);
  int* cursors = w.count + 4 + (PASS == 1 ? 1 : 3) * ZM_ORD_KEYS;
  for (int t = threadIdx.x; t < ZM_ORD_KEYS; t += blockDim.x) { s_size[t] = sizes[t]; s_n[t] = 0; }
  __syncthreads();
  for (int t = threadIdx.x; t < ZM_ORD_KEYS; t += blockDim.x) {      // bucket start: everything with a larger key
    int b = 0;
    for (int u = t + 1; u < ZM_ORD_KEYS; ++u) b += s_size[u];
    s_base[t] = b;
    if (PASS == 1 && t == 0 && blockIdx.x == 0) w.count[3] = b + s_size[0];
  }
  const int pcols = P.pcols;
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = PASS == 1 ? in.nchunks * pcols : w.count[0];
  int col = -1, key = 0, r = 0;
  if (gid < n) {
    col = PASS == 1 ? gid : w.wl1[gid];
    const int c = col / pcols, i = col - c * pcols;
    if (i < in.ncol[c]) { key = w.okey[col]; r = atomicAdd(&s_n[key], 1); }
    else col = -1;
  }
  __syncthreads();
  for (int t = threadIdx.x; t < ZM_ORD_KEYS; t += blockDim.x)
    if (s_n[t]) s_off[t] = atomicAdd(&cursors[t], s_n[t]);
  __syncthreads();
  if (col >= 0) (PASS == 1 ? w.ord1 : w.ord2)[s_base[key] + s_off[key] + r] = col;
}

// ---- buoyan_dilute + parcel_dilute, one thread per column ----------------------------------
// zm_conv.F90:4425-4819 and 4824-5277.  PASS 1: every column (list ord1).  PASS 2: worklist wl1 only (as ord2).
// ORG = true adds the zm_org branches of parcel_dilute (zm_conv.F90:5066-5074, 5186-5188, 5255-5257).
// LAT = true: up to 255 registers, for launches with few columns (second passes too large for k_buoyan_dilute_ws);
// LAT = false: 168 registers so that a whole f09 shard is resident in one wave.  (PAIR is a leftover of round 1's
// paired bracket evaluation: both bracket ends are evaluated side by side by Brent::open in either mode now.)
template <int PASS, bool ORG = false, bool LAT = (PASS == 2)>
__global__ void __launch_bounds__(128, LAT ? 2 : 3)
k_buoyan_dilute(ConvrIn in, ConvrWork w) {
  extern __shared__ double sm_buoy[];               // [pver+2][blockDim.x]
  constexpr bool PAIR = LAT;
  // blocks without work leave before the tables are staged (both conditions are uniform over the block)
  if (PASS == 2 && w.count[0] <= w.ws_gate) return;                  // this worklist goes to k_buoyan_dilute_ws
  if ((int)(blockIdx.x * blockDim.x) >= (PASS == 1 ? w.count[3] : w.count[0])) return;
  zmm::hot_tables_load();                            // before any per-thread return (block-wide barrier inside)
  zmm::hot_svp_load();
  const int pcols = P.pcols, pver = P.pver, msg = P.msg;
  const int ncolpad = in.nchunks * pcols;
  const int nthr = blockDim.x;
  int gid = blockIdx.x * blockDim.x + threadIdx.x;
  int col;
  if (PASS == 1) { if (gid >= w.count[3]) return; col = w.ord1[gid]; }     // work-ordered lists (k_order_*)
  else           { if (gid >= w.count[0] || w.count[0] <= w.ws_gate) return; col = w.ord2[gid]; }
  const int c = col / pcols, i = col - c * pcols;
  // zm_convr returns after the first gather when a chunk has no convective column (zm_conv.F90:917): its
  // first-pass results stand
  if (w.skip_idle_chunks && w.n1chunk[c] == 0) return;
#define BUOY(k) sm_buoy[(k) * nthr + threadIdx.x]
#define IN2(a, k) in.a[cidx(c, (k) - 1, i, pver)]
#define IN2P(a, k) in.a[cidx(c, (k) - 1, i, pver + 1)]

  const double eps1 = P.eps1, grav = P.grav, cp = P.cpres, rl = P.rl;
  const double zs = in.geos[(size_t)c * pcols + i] * P.rgrav;
  const double pblh = in.pblh[(size_t)c * pcols + i];
  const double tpert = in.tpert[(size_t)c * pcols + i];
  const double dmpdz = w.dmpdz[col];
  const double landfrac = ORG ? in.landfrac[(size_t)c * pcols + i] : 0.0;
  const double org2rkm = 10.0, org2Tpert = 0.0;     // zm_conv.F90:4948-4951

  const int pblt = pbl_top_level(in, c, i, zs, pblh);
  const int lon = min(pver, pblt + 2);
  int mx = lon;
  double tl, ql, pl, zl = 0.0;
  if (P.lparcel_pbl) {
    // zm_conv.F90:4638-4673, 4698-4708
    double pbl_dz = (IN2(zm, pblt) + zs) - zs;
    double parcel_dz = fmax2(IN2P(zi, pver), P.parcel_hscale * pbl_dz);
    double parcel_ztop = parcel_dz + zs;
    double parcel_hdp = 0.0, parcel_qdp = 0.0, parcel_dp = 0.0;
    int ipar = 0;
    for (int k = pver; k >= msg + 1; --k) {
      if (IN2P(zi, k + 1) <= parcel_dz) {
        ipar = k;
        double dp_zfrac;
        if (k == pver) dp_zfrac = 1.0;
        else dp_zfrac = fmin2(1.0, (parcel_dz - IN2P(zi, k + 1)) / (IN2P(zi, k) - IN2P(zi, k + 1)));
        double qk = IN2(qh, k), tk = IN2(t, k), zk = IN2(zm, k) + zs;
        double hmn_lev = hmn_launch(tk, qk, zk);
        double dp_lev = IN2P(paph, k + 1) * 0.01 - IN2P(paph, k) * 0.01;
        parcel_hdp = parcel_hdp + (hmn_lev * dp_lev) * dp_zfrac;
        parcel_qdp = parcel_qdp + (qk * dp_lev) * dp_zfrac;
        parcel_dp = parcel_dp + dp_lev * dp_zfrac;
      }
    }
    double hpar = parcel_hdp / parcel_dp, qpar = parcel_qdp / parcel_dp;
    mx = ipar;
    tl = (hpar - rl * qpar - grav * parcel_ztop) / cp;
    ql = qpar;
    pl = IN2(pap, mx) * 0.01;
  } else {
    // zm_conv.F90:4677-4689
    double hmax = 0.0;
    for (int k = lon; k >= max(pblt, msg + 1); --k) {
      double qk = IN2(qh, k), tk = IN2(t, k), zk = IN2(zm, k) + zs;
      double hmn = hmn_launch(tk, qk, zk);
      if (hmn > hmax) { hmax = hmn; mx = k; }
    }
    tl = IN2(t, mx);
    ql = IN2(qh, mx);
    pl = IN2(pap, mx) * 0.01;
  }
  int lcl = mx;

  // ---- fused parcel sweep ------------------------------------------------------------------
  double* tp_o = w.tp + col;        // stride ncolpad per level
  double* qstp_o = w.qstp + col;
  // levels outside [msg+1, mx] keep environment values (zm_conv.F90:4597-4598, 4760-4761)
  for (int k = 1; k <= pver; ++k)
    if (k <= msg || k > mx) {
      tp_o[(size_t)(k - 1) * ncolpad] = IN2(t, k);
      qstp_o[(size_t)(k - 1) * ncolpad] = IN2(qh, k);
    }

  double t_p, q_p, p_p, z_p;                 // environment at level k+1
  double tmix1_p, qtmix_p, qsmix1_p, smix_p; // loop-1 parcel at level k+1
  double qsmix2_p, xsh2o_p = 0.0, ds_xsh2o_p = 0.0, ds_freeze_p = 0.0;  // loop-2 parcel at k+1
  double sp = 0.0, qtp = 0.0, mp = 0.0, sp0, qtp0, mp0 = 1.0;
  bool ok = true;
  {
    const int k = mx;                        // launch level (zm_conv.F90:5002-5038, 5180-5200)
    t_p = IN2(t, k); q_p = IN2(qh, k); p_p = IN2(pap, k) * 0.01; z_p = IN2(zm, k) + zs;
    double dum;
    tmix1_p = t_p;
    if (P.lparcel_pbl) {
      qtp0 = ql; sp0 = enthalpy_q(tl, pl, qtp0, zl, dum);
      (void)enthalpy_q(tmix1_p, p_p, qtp0, z_p, qsmix1_p);     // qsmix = qsat_hPa(tmix, p)
    } else {
      // enthalpy(t,p,..) evaluates qsat_hPa(t,p) internally: same arguments as zm_conv.F90:5031
      qtp0 = q_p; sp0 = enthalpy_q(t_p, p_p, qtp0, z_p, qsmix1_p);
    }
    smix_p = sp0; qtmix_p = qtp0;
    qsmix2_p = qsmix1_p;
    double tpk = tmix1_p, qstpk = q_p;
    double tpv;
    if (ORG) tpv = (tpk + (org2Tpert * IN2(org, k) + tpert)) * (1.0 + qstpk / eps1) / (1.0 + qstpk);
    else     tpv = (tpk + tpert) * (1.0 + qstpk / eps1) / (1.0 + qstpk);
    double tv = t_p * (1.0 + q_p / eps1) / (1.0 + q_p);
    BUOY(k) = tpv - tv + P.tiedke_add;
    tp_o[(size_t)(k - 1) * ncolpad] = tpk;
    qstp_o[(size_t)(k - 1) * ncolpad] = qstpk;
  }
  const double lwmax = 1.e-3, tscool = 0.0;
  for (int k = mx - 1; k >= msg + 1; --k) {
    const double t_k = IN2(t, k), q_k = IN2(qh, k), p_k = IN2(pap, k) * 0.01, z_k = IN2(zm, k) + zs;
    const double org_k = ORG ? IN2(org, k) : 0.0;
    // ---- loop 1 body (zm_conv.F90:5042-5144) ----
    double dp = (p_k - p_p);
    double qtenv = 0.5 * (q_k + q_p);
    double tenv = 0.5 * (t_k + t_p);
    double penv = 0.5 * (p_k + p_p);
    double zenv = 0.5 * (z_k + z_p);
    double dum;
    double senv = enthalpy_q(tenv, penv, qtenv, zenv, dum);
    double dpdz = -(penv * grav) / (P.rgas * tenv);
    double dzdp = 1.0 / dpdz;
    double dmpdp;
    if (ORG) {                                   // tht_tweaks: dmpdz_lnd = dmpdz_mask (zm_conv.F90:5072)
      double dmpdz_mask = dmpdz;
      const double dmpdz_lnd = dmpdz_mask;
      dmpdz_mask = landfrac * dmpdz_lnd + (1.0 - landfrac) * dmpdz_mask;
      dmpdp = (dmpdz_mask / (1.0 + org_k * org2rkm)) * dzdp;
    } else {
      dmpdp = dmpdz * dzdp;
    }
    sp = sp - dmpdp * dp * senv;
    qtp = qtp - dmpdp * dp * qtenv;
    mp = mp - dmpdp * dp;
    double smix_k = (sp0 + sp) / (mp0 + mp);
    double qtmix_k = (qtp0 + qtp) / (mp0 + mp);
    double tmix_k, qsmix_k;
    if (!invert<1, PAIR>(smix_k, p_k, z_k, qtmix_k, tmix1_p, tmix_k, qsmix_k)) {
      ok = false; report_fail(w, 2, col, p_k, tmix1_p, qtmix_k, smix_k);
    }
    if (qsmix_k <= qtmix_k && qsmix1_p > qtmix_p) {
      lcl = k;
      double qxsk = qtmix_k - qsmix_k;
      double qxskp1 = qtmix_p - qsmix1_p;
      double dqxsdp = (qxsk - qxskp1) / dp;
      pl = p_p - qxskp1 / dqxsdp;
      zl = z_p - qxskp1 / dqxsdp * dzdp;
      double dsdp = (smix_k - smix_p) / dp;
      double dqtdp = (qtmix_k - qtmix_p) / dp;
      double slcl = smix_p + dsdp * (pl - p_p);
      double qtlcl = qtmix_p + dqtdp * (pl - p_p);
      double qslcl;
      if (!invert<1, PAIR>(slcl, pl, zl, qtlcl, tmix_k, tl, qslcl)) {
        ok = false; report_fail(w, 3, col, pl, tmix_k, qtlcl, slcl);
      }
    }
    // ---- loop 2 body (zm_conv.F90:5202-5269) ----
    double tmix2 = tmix_k, qsmix2 = qsmix_k;
    double smix2 = entropy_q(tmix2, p_k, qtmix_k, dum);
    double xsh2o_k = 0.0, ds_xsh2o_k = 0.0, ds_freeze_k = 0.0, new_s = 0.0, new_q = 0.0;
#pragma unroll 1
    for (int ii = 0; ii < 2; ++ii) {
      xsh2o_k = fmax2(0.0, qtmix_k - qsmix2 - lwmax);
      ds_xsh2o_k = ds_xsh2o_p - P.cpliq * zmm::log_(tmix2 / P.tfreez) * fmax2(0.0, (xsh2o_k - xsh2o_p));
      if (tmix2 <= P.tfreez + tscool && ds_freeze_p == 0.0)
        ds_freeze_k = (P.latice / tmix2) * fmax2(0.0, qtmix_k - qsmix2 - xsh2o_k);
      if (tmix2 <= P.tfreez + tscool && ds_freeze_p != 0.0)
        ds_freeze_k = ds_freeze_p + (P.latice / tmix2) * fmax2(0.0, (qsmix2_p - qsmix2));
      new_s = smix2 + ds_xsh2o_k + ds_freeze_k;
      new_q = qtmix_k - xsh2o_k;
      double tfg = tmix2;
      if (!invert<0, PAIR>(new_s, p_k, 0.0, new_q, tfg, tmix2, qsmix2)) {
        ok = false; report_fail(w, 4, col, p_k, tfg, new_q, new_s);
      }
    }
    double tpk = tmix2;
    double qstpk = (new_q > qsmix2) ? qsmix2 : new_q;
    double tpv;
    if (ORG) tpv = (tpk + (org2Tpert * org_k + tpert)) * (1.0 + qstpk / eps1) / (1.0 + new_q);
    else     tpv = (tpk + tpert) * (1.0 + qstpk / eps1) / (1.0 + new_q);
    double tv = t_k * (1.0 + q_k / eps1) / (1.0 + q_k);
    BUOY(k) = tpv - tv + P.tiedke_add;
    tp_o[(size_t)(k - 1) * ncolpad] = tpk;
    qstp_o[(size_t)(k - 1) * ncolpad] = qstpk;
    // shift level k -> k+1
    t_p = t_k; q_p = q_k; p_p = p_k; z_p = z_k;
    tmix1_p = tmix_k; qtmix_p = qtmix_k; qsmix1_p = qsmix_k; smix_p = smix_k;
    qsmix2_p = qsmix2; xsh2o_p = xsh2o_k; ds_xsh2o_p = ds_xsh2o_k; ds_freeze_p = ds_freeze_k;
  }
  (void)ok;

  // ---- CAPE / CIN (zm_conv.F90:4742-4816) ----------------------------------------------------
  const bool plge600 = pl >= P.plclmin;
  double cape = 0.0, cin = 0.0;
  int lel = pver;
  if (!plge600) {
    for (int k = msg + 1; k <= mx; ++k) {
      tp_o[(size_t)(k - 1) * ncolpad] = IN2(t, k);
      qstp_o[(size_t)(k - 1) * ncolpad] = IN2(qh, k);
    }
  } else {
    int lelten[ZM_MAXCIN];
    double capeten[ZM_MAXCIN], cinten[ZM_MAXCIN];
#pragma unroll
    for (int n = 0; n < ZM_MAXCIN; ++n) { lelten[n] = pver; capeten[n] = 0.0; cinten[n] = 0.0; }
    int knt = 0;
    for (int k = msg + 2; k <= pver; ++k) {
      if (k < lcl) {
        if (BUOY(k + 1) > 0.0 && BUOY(k) <= 0.0) {
          knt = min(P.num_cin, knt + 1);
#pragma unroll
          for (int n = 0; n < ZM_MAXCIN; ++n) if (n == knt - 1) lelten[n] = k;
        }
      }
    }
    // interface pressures are carried from level to level and fetched one level ahead (the loop used to wait
    // for two dependent global loads per level: 5 % of the kernel's stall samples)
    double pf_k = IN2P(paph, msg + 1) * 0.01, pf_n = IN2P(paph, msg + 2) * 0.01;
    for (int k = msg + 1; k <= mx; ++k) {
      const double pf_k1 = pf_n;
      if (k < mx) pf_n = IN2P(paph, k + 2) * 0.01;
      double lg = zmm::log_hot(div_hot(pf_k1, pf_k));        // log(pf(k+1)/pf(k)), zm_conv.F90:4789
      pf_k = pf_k1;
      double b = BUOY(k);
#pragma unroll
      for (int n = 0; n < ZM_MAXCIN; ++n) {
        if (n < P.num_cin && k > lelten[n]) {
          capeten[n] = capeten[n] + P.rgas * b * lg;
          cinten[n] = cinten[n] - P.rgas * fmin2(b, 0.0) * lg;
        }
      }
    }
#pragma unroll
    for (int n = 0; n < ZM_MAXCIN; ++n) {
      if (n < P.num_cin && capeten[n] > cape) { cape = capeten[n]; cin = cinten[n]; lel = lelten[n]; }
    }
    cape = fmax2(cape, 0.0);
  }
  w.cape[col] = cape; w.cin[col] = cin; w.tl[col] = tl;
  w.lcl[col] = lcl; w.lel[col] = lel; w.mx[col] = mx;
#undef BUOY
#undef IN2
#undef IN2P
}

// ---- buoyan_dilute + parcel_dilute with the two parcel loops on two warps -------------------------------------
// Same arithmetic as k_buoyan_dilute, for launches whose columns leave most schedulers idle (the second CAPE pass,
// small batches, a GPU's share of a strongly scaled grid): there the time is the length of one column's dependency
// chain, and a third of that chain -- the first parcel loop (mixing + one enthalpy inversion per level,
// zm_conv.F90:4997-5148) -- does not depend on the second loop (rain-out / freezing, two entropy inversions per
// level, :5175-5273) at all.  A block is two warps over the same 32 columns: warp 0 runs the first loop and hands
// (tmix, qsmix, qtmix) of every level to warp 1 through global scratch, publishing its progress per lane in shared
// memory; warp 1 runs the second loop one or more levels behind, then the CAPE / CIN sums.  Every quantity is
// computed by the same operations as in the one-thread version.
template <int PASS, bool ORG = false>
__global__ void __launch_bounds__(64, 6)
k_buoyan_dilute_ws(ConvrIn in, ConvrWork w) {
  extern __shared__ double sm_buoy[];               // [pver+2][32], then 2*32 ints of handshake state
  // blocks without work leave before the tables are staged (both conditions are uniform over the block)
  if (PASS == 2 && w.count[0] > w.ws_gate) return;                   // this worklist goes to k_buoyan_dilute
  if ((int)(blockIdx.x * 32) >= (PASS == 1 ? w.count[3] : w.count[0])) return;
  zmm::hot_tables_load();
  zmm::hot_svp_load();
  const int pcols = P.pcols, pver = P.pver, msg = P.msg;
  const int ncolpad = in.nchunks * pcols;
  const int lane = threadIdx.x & 31;
  const bool roleA = threadIdx.x < 32;
  volatile int* prog = reinterpret_cast<volatile int*>(sm_buoy + (size_t)(pver + 2) * 32);   // [32] level published
  int* sh_i = const_cast<int*>(prog) + 32;                                                 // [32] lcl of the column
  if (roleA) prog[lane] = 0x7fffffff;
  __syncthreads();
  const int gid = blockIdx.x * 32 + lane;
  int col;
  if (PASS == 1) { if (gid >= w.count[3]) return; col = w.ord1[gid]; }
  else           { if (gid >= w.count[0] || w.count[0] > w.ws_gate) return; col = w.ord2[gid]; }
  const int c = col / pcols, i = col - c * pcols;
  if (w.skip_idle_chunks && w.n1chunk[c] == 0) return;
#define BUOY(k) sm_buoy[(k) * 32 + lane]
#define IN2(a, k) in.a[cidx(c, (k) - 1, i, pver)]
#define IN2P(a, k) in.a[cidx(c, (k) - 1, i, pver + 1)]
  const size_t n2 = (size_t)ncolpad * pver;
  double* ab_t = w.ab + col;                         // stride ncolpad per level
  double* ab_qs = w.ab + n2 + col;
  double* ab_qt = w.ab + 2 * n2 + col;

  const double eps1 = P.eps1, grav = P.grav, cp = P.cpres, rl = P.rl;
  const double zs = in.geos[(size_t)c * pcols + i] * P.rgrav;
  const double pblh = in.pblh[(size_t)c * pcols + i];
  const double tpert = in.tpert[(size_t)c * pcols + i];
  const double org2rkm = 10.0, org2Tpert = 0.0;     // zm_conv.F90:4948-4951
  // launch level: both warps derive it (inputs only)
  const int pblt = pbl_top_level(in, c, i, zs, pblh);
  const int lon = min(pver, pblt + 2);
  int mx = lon;
  double tl, ql, pl, zl = 0.0;
  if (P.lparcel_pbl) {
    double pbl_dz = (IN2(zm, pblt) + zs) - zs;
    double parcel_dz = fmax2(IN2P(zi, pver), P.parcel_hscale * pbl_dz);
    double parcel_ztop = parcel_dz + zs;
    double parcel_hdp = 0.0, parcel_qdp = 0.0, parcel_dp = 0.0;
    int ipar = 0;
    for (int k = pver; k >= msg + 1; --k) {
      if (IN2P(zi, k + 1) <= parcel_dz) {
        ipar = k;
        double dp_zfrac;
        if (k == pver) dp_zfrac = 1.0;
        else dp_zfrac = fmin2(1.0, (parcel_dz - IN2P(zi, k + 1)) / (IN2P(zi, k) - IN2P(zi, k + 1)));
        double qk = IN2(qh, k), tk = IN2(t, k), zk = IN2(zm, k) + zs;
        double hmn_lev = hmn_launch(tk, qk, zk);
        double dp_lev = IN2P(paph, k + 1) * 0.01 - IN2P(paph, k) * 0.01;
        parcel_hdp = parcel_hdp + (hmn_lev * dp_lev) * dp_zfrac;
        parcel_qdp = parcel_qdp + (qk * dp_lev) * dp_zfrac;
        parcel_dp = parcel_dp + dp_lev * dp_zfrac;
      }
    }
    double hpar = parcel_hdp / parcel_dp, qpar = parcel_qdp / parcel_dp;
    mx = ipar;
    tl = (hpar - rl * qpar - grav * parcel_ztop) / cp;
    ql = qpar;
    pl = IN2(pap, mx) * 0.01;
  } else {
    double hmax = 0.0;
    for (int k = lon; k >= max(pblt, msg + 1); --k) {
      double qk = IN2(qh, k), tk = IN2(t, k), zk = IN2(zm, k) + zs;
      double hmn = hmn_launch(tk, qk, zk);
      if (hmn > hmax) { hmax = hmn; mx = k; }
    }
    tl = IN2(t, mx);
    ql = IN2(qh, mx);
    pl = IN2(pap, mx) * 0.01;
  }
  const double lwmax = 1.e-3, tscool = 0.0;

  if (roleA) {
    // ================= first parcel loop (zm_conv.F90:5002-5144) =================
    const double dmpdz = w.dmpdz[col];
    const double landfrac = ORG ? in.landfrac[(size_t)c * pcols + i] : 0.0;
    int lcl = mx;
    double t_p = IN2(t, mx), q_p = IN2(qh, mx), p_p = IN2(pap, mx) * 0.01, z_p = IN2(zm, mx) + zs;
    double tmix1_p = t_p, qtmix_p, qsmix1_p, smix_p;
    double sp = 0.0, qtp = 0.0, mp = 0.0, sp0, qtp0;
    const double mp0 = 1.0;
    double dum;
    if (P.lparcel_pbl) {
      qtp0 = ql; sp0 = enthalpy_q(tl, pl, qtp0, zl, dum);
      (void)enthalpy_q(tmix1_p, p_p, qtp0, z_p, qsmix1_p);     // qsmix = qsat_hPa(tmix, p)
    } else {
      qtp0 = q_p; sp0 = enthalpy_q(t_p, p_p, qtp0, z_p, qsmix1_p);
    }
    smix_p = sp0; qtmix_p = qtp0;
    ab_qs[(size_t)(mx - 1) * ncolpad] = qsmix1_p;              // the second loop starts from qsmix(mx)
    __threadfence_block();
    prog[lane] = mx;
    for (int k = mx - 1; k >= msg + 1; --k) {
      const double t_k = IN2(t, k), q_k = IN2(qh, k), p_k = IN2(pap, k) * 0.01, z_k = IN2(zm, k) + zs;
      const double org_k = ORG ? IN2(org, k) : 0.0;
      double dp = (p_k - p_p);
      double qtenv = 0.5 * (q_k + q_p);
      double tenv = 0.5 * (t_k + t_p);
      double penv = 0.5 * (p_k + p_p);
      double zenv = 0.5 * (z_k + z_p);
      double senv = enthalpy_q(tenv, penv, qtenv, zenv, dum);
      double dpdz = -(penv * grav) / (P.rgas * tenv);
      double dzdp = 1.0 / dpdz;
      double dmpdp;
      if (ORG) {                                   // tht_tweaks: dmpdz_lnd = dmpdz_mask (zm_conv.F90:5072)
        double dmpdz_mask = dmpdz;
        const double dmpdz_lnd = dmpdz_mask;
        dmpdz_mask = landfrac * dmpdz_lnd + (1.0 - landfrac) * dmpdz_mask;
        dmpdp = (dmpdz_mask / (1.0 + org_k * org2rkm)) * dzdp;
      } else {
        dmpdp = dmpdz * dzdp;
      }
      sp = sp - dmpdp * dp * senv;
      qtp = qtp - dmpdp * dp * qtenv;
      mp = mp - dmpdp * dp;
      double smix_k = (sp0 + sp) / (mp0 + mp);
      double qtmix_k = (qtp0 + qtp) / (mp0 + mp);
      double tmix_k, qsmix_k;
      if (!invert<1>(smix_k, p_k, z_k, qtmix_k, tmix1_p, tmix_k, qsmix_k))
        report_fail(w, 2, col, p_k, tmix1_p, qtmix_k, smix_k);
      // hand level k to the second loop before the (rare) LCL inversion
      ab_t[(size_t)(k - 1) * ncolpad] = tmix_k;
      ab_qs[(size_t)(k - 1) * ncolpad] = qsmix_k;
      ab_qt[(size_t)(k - 1) * ncolpad] = qtmix_k;
      __threadfence_block();
      prog[lane] = k;
      if (qsmix_k <= qtmix_k && qsmix1_p > qtmix_p) {
        lcl = k;
        double qxsk = qtmix_k - qsmix_k;
        double qxskp1 = qtmix_p - qsmix1_p;
        double dqxsdp = (qxsk - qxskp1) / dp;
        pl = p_p - qxskp1 / dqxsdp;
        zl = z_p - qxskp1 / dqxsdp * dzdp;
        double dsdp = (smix_k - smix_p) / dp;
        double dqtdp = (qtmix_k - qtmix_p) / dp;
        double slcl = smix_p + dsdp * (pl - p_p);
        double qtlcl = qtmix_p + dqtdp * (pl - p_p);
        double qslcl;
        if (!invert<1>(slcl, pl, zl, qtlcl, tmix_k, tl, qslcl))
          report_fail(w, 3, col, pl, tmix_k, qtlcl, slcl);
      }
      t_p = t_k; q_p = q_k; p_p = p_k; z_p = z_k;
      tmix1_p = tmix_k; qtmix_p = qtmix_k; qsmix1_p = qsmix_k; smix_p = smix_k;
    }
    // lcl, pl, tl are final: the second loop's CAPE sums wait for them
    w.tl[col] = tl;
    w.cin[col] = pl;                                // pl travels through the cin slot until warp 1 overwrites it
    sh_i[lane] = lcl;
    __threadfence_block();
    prog[lane] = 0;
    return;
  }

  // ================= second parcel loop (zm_conv.F90:5180-5269), CAPE / CIN =================
  double* tp_o = w.tp + col;        // stride ncolpad per level
  double* qstp_o = w.qstp + col;
  // levels outside [msg+1, mx] keep environment values (zm_conv.F90:4597-4598, 4760-4761)
  for (int k = 1; k <= pver; ++k)
    if (k <= msg || k > mx) {
      tp_o[(size_t)(k - 1) * ncolpad] = IN2(t, k);
      qstp_o[(size_t)(k - 1) * ncolpad] = IN2(qh, k);
    }
  double xsh2o_p = 0.0, ds_xsh2o_p = 0.0, ds_freeze_p = 0.0;
  {
    const int k = mx;                        // launch level (zm_conv.F90:5180-5200)
    const double t_p = IN2(t, k), q_p = IN2(qh, k);
    double tpk = t_p, qstpk = q_p;
    double tpv;
    if (ORG) tpv = (tpk + (org2Tpert * IN2(org, k) + tpert)) * (1.0 + qstpk / eps1) / (1.0 + qstpk);
    else     tpv = (tpk + tpert) * (1.0 + qstpk / eps1) / (1.0 + qstpk);
    double tv = t_p * (1.0 + q_p / eps1) / (1.0 + q_p);
    BUOY(k) = tpv - tv + P.tiedke_add;
    tp_o[(size_t)(k - 1) * ncolpad] = tpk;
    qstp_o[(size_t)(k - 1) * ncolpad] = qstpk;
  }
  while (prog[lane] > mx) { }
  __threadfence_block();
  double qsmix2_p = *((volatile double*)&ab_qs[(size_t)(mx - 1) * ncolpad]);
  for (int k = mx - 1; k >= msg + 1; --k) {
    const double t_k = IN2(t, k), q_k = IN2(qh, k), p_k = IN2(pap, k) * 0.01;
    const double org_k = ORG ? IN2(org, k) : 0.0;
    while (prog[lane] > k) { }
    __threadfence_block();
    const double tmix_k = *((volatile double*)&ab_t[(size_t)(k - 1) * ncolpad]);
    const double qsmix_k = *((volatile double*)&ab_qs[(size_t)(k - 1) * ncolpad]);
    const double qtmix_k = *((volatile double*)&ab_qt[(size_t)(k - 1) * ncolpad]);
    double dum;
    double tmix2 = tmix_k, qsmix2 = qsmix_k;
    double smix2 = entropy_q(tmix2, p_k, qtmix_k, dum);
    double xsh2o_k = 0.0, ds_xsh2o_k = 0.0, ds_freeze_k = 0.0, new_s = 0.0, new_q = 0.0;
#pragma unroll 1
    for (int ii = 0; ii < 2; ++ii) {
      xsh2o_k = fmax2(0.0, qtmix_k - qsmix2 - lwmax);
      ds_xsh2o_k = ds_xsh2o_p - P.cpliq * zmm::log_(tmix2 / P.tfreez) * fmax2(0.0, (xsh2o_k - xsh2o_p));
      if (tmix2 <= P.tfreez + tscool && ds_freeze_p == 0.0)
        ds_freeze_k = (P.latice / tmix2) * fmax2(0.0, qtmix_k - qsmix2 - xsh2o_k);
      if (tmix2 <= P.tfreez + tscool && ds_freeze_p != 0.0)
        ds_freeze_k = ds_freeze_p + (P.latice / tmix2) * fmax2(0.0, (qsmix2_p - qsmix2));
      new_s = smix2 + ds_xsh2o_k + ds_freeze_k;
      new_q = qtmix_k - xsh2o_k;
      double tfg = tmix2;
      if (!invert<0>(new_s, p_k, 0.0, new_q, tfg, tmix2, qsmix2))
        report_fail(w, 4, col, p_k, tfg, new_q, new_s);
    }
    double tpk = tmix2;
    double qstpk = (new_q > qsmix2) ? qsmix2 : new_q;
    double tpv;
    if (ORG) tpv = (tpk + (org2Tpert * org_k + tpert)) * (1.0 + qstpk / eps1) / (1.0 + new_q);
    else     tpv = (tpk + tpert) * (1.0 + qstpk / eps1) / (1.0 + new_q);
    double tv = t_k * (1.0 + q_k / eps1) / (1.0 + q_k);
    BUOY(k) = tpv - tv + P.tiedke_add;
    tp_o[(size_t)(k - 1) * ncolpad] = tpk;
    qstp_o[(size_t)(k - 1) * ncolpad] = qstpk;
    qsmix2_p = qsmix2; xsh2o_p = xsh2o_k; ds_xsh2o_p = ds_xsh2o_k; ds_freeze_p = ds_freeze_k;
  }
  while (prog[lane] > 0) { }
  __threadfence_block();
  const int lcl = sh_i[lane];
  pl = *((volatile double*)&w.cin[col]);

  // ---- CAPE / CIN (zm_conv.F90:4742-4816) ----------------------------------------------------
  const bool plge600 = pl >= P.plclmin;
  double cape = 0.0, cin = 0.0;
  int lel = pver;
  if (!plge600) {
    for (int k = msg + 1; k <= mx; ++k) {
      tp_o[(size_t)(k - 1) * ncolpad] = IN2(t, k);
      qstp_o[(size_t)(k - 1) * ncolpad] = IN2(qh, k);
    }
  } else {
    int lelten[ZM_MAXCIN];
    double capeten[ZM_MAXCIN], cinten[ZM_MAXCIN];
#pragma unroll
    for (int n = 0; n < ZM_MAXCIN; ++n) { lelten[n] = pver; capeten[n] = 0.0; cinten[n] = 0.0; }
    int knt = 0;
    for (int k = msg + 2; k <= pver; ++k) {
      if (k < lcl) {
        if (BUOY(k + 1) > 0.0 && BUOY(k) <= 0.0) {
          knt = min(P.num_cin, knt + 1);
#pragma unroll
          for (int n = 0; n < ZM_MAXCIN; ++n) if (n == knt - 1) lelten[n] = k;
        }
      }
    }
    double pf_k = IN2P(paph, msg + 1) * 0.01, pf_n = IN2P(paph, msg + 2) * 0.01;
    for (int k = msg + 1; k <= mx; ++k) {
      const double pf_k1 = pf_n;
      if (k < mx) pf_n = IN2P(paph, k + 2) * 0.01;
      double lg = zmm::log_hot(div_hot(pf_k1, pf_k));        // log(pf(k+1)/pf(k)), zm_conv.F90:4789
      pf_k = pf_k1;
      double b = BUOY(k);
#pragma unroll
      for (int n = 0; n < ZM_MAXCIN; ++n) {
        if (n < P.num_cin && k > lelten[n]) {
          capeten[n] = capeten[n] + P.rgas * b * lg;
          cinten[n] = cinten[n] - P.rgas * fmin2(b, 0.0) * lg;
        }
      }
    }
#pragma unroll
    for (int n = 0; n < ZM_MAXCIN; ++n) {
      if (n < P.num_cin && capeten[n] > cape) { cape = capeten[n]; cin = cinten[n]; lel = lelten[n]; }
    }
    cape = fmax2(cape, 0.0);
  }
  w.cape[col] = cape; w.cin[col] = cin;
  w.lcl[col] = lcl; w.lel[col] = lel; w.mx[col] = mx;
#undef BUOY
#undef IN2
#undef IN2P
}

// ---- buoyan: undilute CAPE (cam3 physics only), one thread per column ---------------------------------
// zm_conv.F90:2719-3022, reached when cam_physpkg_is('cam3') (zm_conv.F90:871-880) as the FIRST trigger
// pass; the second pass is buoyan_dilute like everywhere else (zm_conv.F90:1080).  The reference then
// tests an undefined `cin` at zm_conv.F90:909 (buoyan does not set it): this build defines cin = 0 for
// that first test.  lelten/capeten are 5 wide as the reference's `do n = 1,5` loops assume.
__global__ void __launch_bounds__(128)
k_buoyan_undilute(ConvrIn in, ConvrWork w) {
  extern __shared__ double sm_buoy[];
  const int pcols = P.pcols, pver = P.pver, msg = P.msg;
  const int ncolpad = in.nchunks * pcols;
  const int nthr = blockDim.x;
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= ncolpad) return;
  const int c = col / pcols, i = col - c * pcols;
  if (i >= in.ncol[c]) return;
#define BUOY(k) sm_buoy[(k) * nthr + threadIdx.x]
#define IN2(a, k) in.a[cidx(c, (k) - 1, i, pver)]
#define IN2P(a, k) in.a[cidx(c, (k) - 1, i, pver + 1)]
  const double eps1 = P.eps1, grav = P.grav, cp = P.cpres, rl = P.rl, rd = P.rgas;
  const double zs = in.geos[(size_t)c * pcols + i] * P.rgrav;
  const double pblh = in.pblh[(size_t)c * pcols + i];
  const double tpert = in.tpert[(size_t)c * pcols + i];
  int pblt = pver;
  for (int k = pver - 1; k >= msg + 1; --k) {
    double zk = IN2(zm, k) + zs;
    double zfk = IN2P(zi, k) + zs, zfk1 = IN2P(zi, k + 1) + zs;
    if (fabs(zk - zs - pblh) < (zfk - zfk1) * 0.5) pblt = k;
  }
  const int lon = pver;
  int mx = lon;
  double hmax = 0.0;
  for (int k = pver; k >= msg + 1; --k) {
    const double hmn = cp * IN2(t, k) + grav * (IN2(zm, k) + zs) + rl * IN2(qh, k);
    if (k >= pblt && k <= lon && hmn > hmax) { hmax = hmn; mx = k; }
  }
  const double t_mx = IN2(t, mx), q_mx = IN2(qh, mx), p_mx = IN2(pap, mx) * 0.01;
  int lcl = mx;
  const double e = p_mx * q_mx / (eps1 + q_mx);
  double tl = 2840.0 / (3.5 * zmm::log_(t_mx) - zmm::log_(e) - 4.805) + 55.0;
  double pl;
  if (tl < t_mx) {
    const double plexp = (1.0 / (0.2854 * (1.0 - 0.28 * q_mx)));
    pl = p_mx * zmm::pow_(tl / t_mx, plexp);
  } else {
    tl = t_mx;
    pl = p_mx;
  }
  for (int k = pver; k >= msg + 2; --k)
    if (k <= mx && (IN2(pap, k) * 0.01 > pl && IN2(pap, k - 1) * 0.01 <= pl)) lcl = k - 1;
  const bool plge600 = pl >= P.plclmin;

  double* tp_o = w.tp + col;
  double* qstp_o = w.qstp + col;
  double tp_p = 0.0, qstp_p = 0.0, p_p = 0.0;        // parcel at level k+1
  for (int k = pver; k >= 1; --k) {
    const double tk = IN2(t, k), qk = IN2(qh, k), pk = IN2(pap, k) * 0.01;
    double tpk = tk, qstpk = qk;                      // defaults (zm_conv.F90:2822-2823)
    if (k >= msg + 1 && plge600) {
      const double tv = tk * (1.0 + 1.608 * qk) / (1.0 + qk);
      bool parcel = false;
      double tpv = 0.0;
      if (k > lcl && k <= mx) {                        // sub-cloud layer, zm_conv.F90:2896-2911
        qstpk = q_mx;
        tpk = t_mx * zmm::pow_(pk / p_mx, 0.2854 * (1.0 - 0.28 * q_mx));
        tpv = (tpk + tpert) * (1.0 + 1.608 * q_mx) / (1.0 + q_mx);
        parcel = true;
      } else if (k == lcl || (k < lcl && k <= pver - 1)) {
        double ybase;
        if (k == lcl) {                                // zm_conv.F90:2916-2948
          qstpk = q_mx;
          tpk = tl * zmm::pow_(pk / pl, 0.2854 * (1.0 - 0.28 * qstpk));
          ybase = q_mx;
        } else {                                       // zm_conv.F90:2952-2976
          qstpk = qstp_p;
          tpk = tp_p * zmm::pow_(pk / p_p, 0.2854 * (1.0 - 0.28 * qstpk));
          ybase = qstp_p;
        }
        double est;
        qsat_hPa(tpk, pk, est, qstpk);
        double a1 = cp / rl + qstpk * (1.0 + qstpk / eps1) * rl * eps1 / (rd * (tpk * tpk));
        double a2 = .5 * (qstpk * (1.0 + 2.0 / eps1 * qstpk) * (1.0 + qstpk / eps1) * (eps1 * eps1) * rl * rl /
                              ((rd * rd) * ((tpk * tpk) * (tpk * tpk))) -
                          qstpk * (1.0 + qstpk / eps1) * 2.0 * eps1 * rl / (rd * ((tpk * tpk) * tpk)));
        a1 = 1.0 / a1;
        a2 = -a2 * ((a1 * a1) * a1);
        const double y = ybase - qstpk;
        tpk = tpk + a1 * y + a2 * (y * y);
        qsat_hPa(tpk, pk, est, qstpk);
        tpv = (tpk + tpert) * (1.0 + 1.608 * qstpk) / (1.0 + q_mx);
        parcel = true;
      }
      BUOY(k) = parcel ? (tpv - tv + P.tiedke_add) : 0.0;
    } else {
      BUOY(k) = 0.0;
    }
    tp_o[(size_t)(k - 1) * ncolpad] = tpk;
    qstp_o[(size_t)(k - 1) * ncolpad] = qstpk;
    tp_p = tpk; qstp_p = qstpk; p_p = pk;
  }
  double cape = 0.0;
  int lel = pver;
  if (plge600) {
    int lelten[5];
    double capeten[5];
#pragma unroll
    for (int n = 0; n < 5; ++n) { lelten[n] = pver; capeten[n] = 0.0; }
    int knt = 0;
    for (int k = msg + 2; k <= pver; ++k)
      if (k < lcl)
        if (BUOY(k + 1) > 0.0 && BUOY(k) <= 0.0) {
          knt = min(5, knt + 1);
#pragma unroll
          for (int n = 0; n < 5; ++n) if (n == knt - 1) lelten[n] = k;
        }
    for (int k = msg + 1; k <= mx; ++k) {
      const double lg = zmm::log_((IN2P(paph, k + 1) * 0.01) / (IN2P(paph, k) * 0.01));
      const double b = BUOY(k);
#pragma unroll
      for (int n = 0; n < 5; ++n)
        if (k > lelten[n]) capeten[n] = capeten[n] + rd * b * lg;
    }
#pragma unroll
    for (int n = 0; n < 5; ++n)
      if (capeten[n] > cape) { cape = capeten[n]; lel = lelten[n]; }
    cape = fmax2(cape, 0.0);
  }
  w.cape[col] = cape; w.cin[col] = 0.0; w.tl[col] = tl;
  w.lcl[col] = lcl; w.lel[col] = lel; w.mx[col] = mx;
#undef BUOY
#undef IN2
#undef IN2P
}

// ---- trigger + order-preserving compaction, one warp per chunk -------------------------------
// zm_conv.F90:905-915 (FINAL=0: pass-1 worklist) and 1095-1111 (FINAL=1: ideep/lengath outputs).
template <int FINAL>
__global__ void k_trigger(ConvrIn in, ConvrOut o, ConvrWork w) {
  const int pcols = P.pcols;
  const int lane = threadIdx.x & 31;
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (c >= in.nchunks) return;
  const int ncol = in.ncol[c];
  int base = 0;
  int wlbase = 0;
  // first sweep: count; second sweep: write (keeps the worklist range of a chunk contiguous)
  int total = 0;
  for (int i0 = 0; i0 < ncol; i0 += 32) {
    int i = i0 + lane;
    bool trig = false;
    if (i < ncol) {
      int col = c * pcols + i;
      double cape = w.cape[col];
      trig = (cape > P.capelmt) && (w.cin[col] < cape * P.cin_threshd);
    }
    total += __popc(__ballot_sync(0xffffffffu, trig));
  }
  if (lane == 0) wlbase = total ? atomicAdd(&w.count[FINAL], total) : 0;
  wlbase = __shfl_sync(0xffffffffu, wlbase, 0);
  for (int i0 = 0; i0 < ncol; i0 += 32) {
    int i = i0 + lane;
    bool trig = false;
    int col = c * pcols + i;
    if (i < ncol) {
      double cape = w.cape[col];
      trig = (cape > P.capelmt) && (w.cin[col] < cape * P.cin_threshd);
    }
    unsigned m = __ballot_sync(0xffffffffu, trig);
    int pos = base + __popc(m & ((1u << lane) - 1u));
    if (trig) {
      if (FINAL) {
        o.ideep[(size_t)c * pcols + pos] = i + 1;
        w.wl2[2 * (wlbase + pos)] = col;
        w.wl2[2 * (wlbase + pos) + 1] = c * pcols + pos;
      } else {
        w.wl1[wlbase + pos] = col;
      }
    }
    base += __popc(m);
  }
  if (!FINAL && lane == 0) w.n1chunk[c] = total;
  if (FINAL) {
    if (lane == 0) o.lengath[c] = total;
    for (int i = lane; i < ncol; i += 32) o.cape[(size_t)c * pcols + i] = w.cape[c * pcols + i];
  }
}
