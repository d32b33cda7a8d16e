// zm_transport.cuh -- zm_conv_evap, momtran, convtran kernels and the two neighbours of the path (geopotential_t,
// convect_diagnostics_calc).
//   zm_conv_evap  zm_conv.F90:1712-1972   thread per column, top-down scan, no per-level storage; inside the fused
//                                         step it also applies physics_update and stores the summed tendencies
//   momtran       zm_conv.F90:2315-2715   warp per gathered column, lane = level, the four wind recurrences in one
//                                         instruction stream
//   convtran      zm_conv.F90:1976-2311   block per chunk (k_convtran_c); thread per (gathered column, constituent)
//                                         as the fallback (k_convtran_t); both also as <true> instantiations that
//                                         read and write the convective columns' records (zm_conv_tend_2 gathered)
// The chunk-wide loop bounds ktm/kbm (zm_conv.F90:2076-2081, 2449-2454) are reproduced exactly
// by a tiny per-chunk reduction kernel so the level ranges match the reference bit for bit.
#pragma once
#include "zm_kernels.cuh"

// ---- zm_conv_evap ------------------------------------------------------------------------------
struct EvapArgs {
  int nchunks;
  const int* ncol;
  const double *t, *pmid, *pdel, *q, *landfrac, *prdprec, *cldfrc;
  double *tend_s, *tend_s_snwprd, *tend_s_snwevmlt, *tend_q, *prec, *snow, *ntprprd, *ntsnprd,
      *flxprec, *flxsnow;
  double deltat;
  // Fused zm_conv_tend step (k_conv_evap<true>): t, q above are the state BEFORE zm_convr's tendencies and the kernel
  // applies physics_update itself (t + heat*dt/cpair, q + qtnd*dt clipped at 1e-12: physics_types.F90:322-329, 427,
  // the statements of k_state_update), then stores the sums of the two ptend_loc instead of its own tend_s:
  // ps = heat + tend_s, pq = qtnd + tend_q (zm_conv_intr.F90:736, 803); tend_q still goes to a.tend_q (= evapcdp).
  const double *heat = nullptr, *qtnd = nullptr;
  double *ps = nullptr, *pq = nullptr;
};

// HIST (fused step with history fields attached, zm_conv_tend_hist_fields): the fused kernel also stores its own
// tend_s and the four diagnostics above, all five non-NULL (the caller substitutes scratch for unattached ones)
template <bool FUSED, bool HIST = false>
__global__ void __launch_bounds__(128)
k_conv_evap(EvapArgs a) {
  const int pcols = P.pcols, pver = P.pver, pverp = P.pverp;
  int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= a.nchunks * pcols) return;
  const int c = col / pcols, i = col - c * pcols;
  if (i >= a.ncol[c]) {
    // padding lanes: the reference leaves its intent(out) arrays untouched there; define them (zero) so that
    // what goes back to the host never depends on stale device memory
    for (int k = 0; k < pver; ++k) {
      const size_t e = cidx(c, k, i, pver);
      if (FUSED) { a.ps[e] = 0.0; a.pq[e] = 0.0; } else a.tend_s[e] = 0.0;
      if (HIST) a.tend_s[e] = 0.0;
      a.tend_q[e] = 0.0;
      // tend_s_snwprd, tend_s_snwevmlt, ntprprd, ntsnprd are history diagnostics (zm_conv_intr.F90:779-794): all four
      // NULL inside the fused zm_conv_tend step unless zm_conv_tend_hist_fields attached them
      if (a.ntprprd) { a.tend_s_snwprd[e] = 0.0; a.tend_s_snwevmlt[e] = 0.0; a.ntprprd[e] = 0.0; a.ntsnprd[e] = 0.0; }
    }
    for (int k = 0; k < pverp; ++k) { a.flxprec[cidx(c, k, i, pverp)] = 0.0; a.flxsnow[cidx(c, k, i, pverp)] = 0.0; }
    a.snow[col] = 0.0;
    return;
  }
  const double tmelt = P.tmelt, gravit = P.gravit, latice = P.latice, latvap = P.latvap;
  double prec = a.prec[col] * 1000.0;
  double flxprec = 0.0, flxsnow = 0.0, evpvint = 0.0;
  a.flxprec[cidx(c, 0, i, pverp)] = 0.0;
  a.flxsnow[cidx(c, 0, i, pverp)] = 0.0;
  for (int k = 1; k <= pver; ++k) {
    const size_t e = cidx(c, k - 1, i, pver);
    const double pmid = a.pmid[e], pdel = a.pdel[e], prdprec = a.prdprec[e], cldfrc = a.cldfrc[e];
    double t = a.t[e], q = a.q[e], heat_k = 0.0, qtnd_k = 0.0;
    if (FUSED) {
      heat_k = a.heat[e]; qtnd_k = a.qtnd[e];
      t = t + div_z(heat_k * a.deltat, P.cpair);
      const double qn = q + qtnd_k * a.deltat;
      q = (qn < 1.e-12) ? 1.e-12 : qn;
    }
    double es, qs, fice, fsnow_conv;
    qsat_table(t, pmid, es, qs);
    cldfrc_fice(t, fice, fsnow_conv);
    double flxsntm, snowmlt;
    if (t > tmelt) { flxsntm = 0.0; snowmlt = div_z(flxsnow * gravit, pdel); }
    else           { flxsntm = flxsnow; snowmlt = 0.0; }
    double evplimit = fmax2(1.0 - q / (1.0 + q) / qs, 0.0);
    // zm_conv.F90:1860-1864
    const double kemask = P.zm_org ? P.ke * (1.0 - a.landfrac[col]) + P.ke_lnd * a.landfrac[col] : P.ke;
    double evpprec = kemask * (1.0 - cldfrc) * evplimit * sqrt_z(flxprec);
    evplimit = fmin2(evplimit, div_z(flxprec * gravit, pdel));
    evplimit = fmin2(evplimit, div_z((prec - evpvint) * gravit, pdel));
    evpprec = fmin2(evplimit, evpprec);
    double evpsnow, work1, work2;
    if (flxprec > 0.0) {
      work1 = fmin2(fmax2(0.0, div_z(flxsntm, flxprec)), 1.0);
      evpsnow = evpprec * work1;
    } else {
      evpsnow = 0.0;
    }
    evpvint = evpvint + div_z(evpprec * pdel, gravit);
    const double ntprprd = prdprec - evpprec;
    if (flxprec > 0.0) work1 = fmin2(fmax2(0.0, div_z(flxsnow, flxprec)), 1.0);
    else work1 = 0.0;
    work2 = fmax2(fsnow_conv, work1);
    if (snowmlt > 0.0) work2 = 0.0;
    const double ntsnprd = prdprec * work2 - evpsnow - snowmlt;
    if (a.ntprprd) {
      a.tend_s_snwprd[e] = prdprec * work2 * latice;
      a.tend_s_snwevmlt[e] = -(evpsnow + snowmlt) * latice;
      a.ntprprd[e] = ntprprd;
      a.ntsnprd[e] = ntsnprd;
    }
    flxprec = flxprec + div_z(ntprprd * pdel, gravit);
    flxsnow = flxsnow + div_z(ntsnprd * pdel, gravit);
    flxprec = fmax2(flxprec, 0.0);
    flxsnow = fmax2(flxsnow, 0.0);
    a.flxprec[cidx(c, k, i, pverp)] = flxprec;
    a.flxsnow[cidx(c, k, i, pverp)] = flxsnow;
    const double tend_s = -evpprec * latvap + ntsnprd * latice;
    if (FUSED) { a.ps[e] = heat_k + tend_s; a.pq[e] = qtnd_k + evpprec; } else a.tend_s[e] = tend_s;
    if (HIST) a.tend_s[e] = tend_s;
    a.tend_q[e] = evpprec;
  }
  a.prec[col] = div_z(flxprec, 1000.0);
  a.snow[col] = div_z(flxsnow, 1000.0);
}

// ---- zm_org (organisation tracer, SURVEY N3) -------------------------------------------------------------
// org2d(i,:) = sum(dpp*org)/sum(dpp) over the levels with org > 0 (zm_conv.F90:793-819), orgt = 0 (:555-556).
// Thread per column, levels summed in the reference's order.  Padding lanes (i >= ncol) get 0.
__global__ void k_org2d(int nchunks, const int* ncol, const double* org, const double* dpp, double* orgt,
                        double* org2d) {
  const int pcols = P.pcols, pver = P.pver;
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= nchunks * pcols) return;
  const int c = col / pcols, i = col - c * pcols;
  double orgavg = 0.0, dptot = 0.0;
  if (i < ncol[c]) {
    for (int k = 0; k < pver; ++k) {
      const size_t e = cidx(c, k, i, pver);
      const double o = org[e];
      if (o > 0) { orgavg = orgavg + dpp[e] * o; dptot = dptot + dpp[e]; }
    }
    if (dptot > 0) orgavg = orgavg / dptot;
  }
  for (int k = 0; k < pver; ++k) { const size_t e = cidx(c, k, i, pver); org2d[e] = orgavg; orgt[e] = 0.0; }
}
// org tendency after zm_conv_evap (zm_conv_intr.F90:773-777), added to the zero tendency zm_convr returned
__global__ void k_org_tend(int nchunks, const int* ncol, const double* org, const double* evapcdp, double ztodt,
                           double* orgt) {
  const int pcols = P.pcols, pver = P.pver;
  const size_t n2 = (size_t)nchunks * pcols * pver;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n2; e += (size_t)gridDim.x * blockDim.x) {
    const int i = (int)(e % pcols), c = (int)(e / ((size_t)pcols * pver));
    if (i >= ncol[c]) continue;
    double x = fmin2(1.0, fmax2(0.0, (50.0 * 1000.0 * 1000.0 * fabs(evapcdp[e])) - (org[e] / 10800.0)));
    x = (x - org[e]) / ztodt;
    orgt[e] = orgt[e] + x;
  }
}

// ---- chunk-wide ktm / kbm (zm_conv.F90:2076-2081) + compact list of convective slots: warp per chunk --
// slots[0..count) lists the gathered slots (chunk*pcols + gathered position) that hold a convective
// column, so the transport kernels run dense warps; the order of the list does not matter.
__global__ void k_chunk_bounds(int nchunks, const int* jt, const int* mx, const int* lengath, int* ktm,
                               int* kbm, int* slots, int* count) {
  const int lane = threadIdx.x & 31;
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (c >= nchunks) return;
  const int pcols = P.pcols, n = lengath[c];
  int a = P.pver, b = P.pver;
  for (int i = lane; i < n; i += 32) {
    a = min(a, jt[(size_t)c * pcols + i]);
    b = min(b, mx[(size_t)c * pcols + i]);
  }
  for (int off = 16; off; off >>= 1) {
    a = min(a, __shfl_xor_sync(0xffffffffu, a, off));
    b = min(b, __shfl_xor_sync(0xffffffffu, b, off));
  }
  int base = 0;
  if (lane == 0) { ktm[c] = a; kbm[c] = b; base = n ? atomicAdd(count, n) : 0; }
  base = __shfl_sync(0xffffffffu, base, 0);
  for (int i = lane; i < n; i += 32) slots[base + i] = c * pcols + i;
}

// ---- momtran -------------------------------------------------------------------------------------
struct MomArgs {
  int nchunks, ncnst;
  const int *ncol, *jt, *mx, *ideep, *lengath, *ktm, *kbm, *slots, *count;
  int domom[2];
  const double *q, *mu, *md, *du, *eu, *ed, *dp;
  double *dqdt, *pguall, *pgdall, *icwu, *icwd, *seten;
  double dt;
  // Fused zm_conv_tend step: the two wind components come from / go to separate (pcols,pver) arrays (state%u, state%v
  // -> ptend%u, ptend%v) instead of the packed winds(pcols,pver,2) / wind_tends(pcols,pver,2) of zm_conv_intr.F90:814-826,
  // so the step neither packs the winds nor unpacks the tendencies.  NULL: the packed q / dqdt above.
  const double *q_u = nullptr, *q_v = nullptr;
  double *dq_u = nullptr, *dq_v = nullptr;   // (zero-filled, like seten, by the caller: momtran writes convective columns only)
};

// initialisation of the outgoing fields (zm_conv.F90:2429-2443, 2630)
__global__ void k_momtran_init(MomArgs a) {
  const int pcols = P.pcols, pver = P.pver;
  const size_t n2 = (size_t)a.nchunks * pcols * pver;
  size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
  for (size_t e = tid; e < n2 * a.ncnst; e += nth) {
    // e -> (c, m, k, i)
    size_t i = e % pcols, r = e / pcols;
    size_t m = (r / pver) % a.ncnst, c = r / ((size_t)pver * a.ncnst);
    // pguall / pgdall / icwu / icwd are history diagnostics (ZMUPGU ... ZMICVD, zm_conv_intr.F90:846-857): all four
    // NULL inside the fused zm_conv_tend step, which does not return them
    if (a.pguall) {
      a.pguall[e] = 0.0; a.pgdall[e] = 0.0;
      if ((int)i < a.ncol[c]) { a.icwu[e] = a.q[e]; a.icwd[e] = a.q[e]; }
    }
    if (m < 2 && a.domom[m]) a.dqdt[e] = 0.0;
  }
  for (size_t e = tid; e < n2; e += nth) a.seten[e] = 0.0;
}

// momtran's in-cloud winds icwu / icwd of the fused step with split winds, when zm_conv_tend_hist_fields attached
// them: the environment wind for i <= ncol (zm_conv.F90:2429-2443; state%u / state%v, component 1 = u), 0 in the
// padding columns.  k_momtran_t then overwrites the convective columns.  (pguall / pgdall start as zero: k_zero_fill.)
__global__ void k_icw_init(int nchunks, const int* ncol, const double* u, const double* v, double* icwu, double* icwd) {
  const int pcols = P.pcols, pver = P.pver;
  const size_t n2 = (size_t)nchunks * pcols * pver;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < 2 * n2; e += (size_t)gridDim.x * blockDim.x) {
    // e -> (c, m, k, i) of the (pcols,pver,2) arrays
    const size_t i = e % pcols, r = e / pcols;
    const size_t m = (r / pver) & 1, c = r / ((size_t)pver * 2), src = (c * pver + r % pver) * pcols + i;
    const double w = ((int)i < ncol[c]) ? (m ? v[src] : u[src]) : 0.0;
    icwu[e] = w; icwd[e] = w;
  }
}

// Warp per gathered (convective) column, lane = level.  Everything that is independent from level to level
// (pressure-gradient terms 2497-2530, the mass-flux weighted differences, tendencies 2596-2627, momentum
// flux and end-of-step wind 2646-2666, KE-dissipation heating 2675-2712) runs with one level per lane out of
// shared memory; only the two first-order recurrences -- in-cloud updraft wind bottom-up (zm_conv.F90:2536-2575)
// and downdraft wind top-down (2579-2589) -- are sequential, and those run for both wind components and both
// directions in ONE loop (four independent dependency chains) with their level-local terms precomputed.
// Expression order is the reference's everywhere, so results are bit-identical to the serial code.
// (Earlier versions ran one thread per column: 0.26 ms of dependent divisions for 19k columns.)
#define MOM_WARPS 4
// shared-memory arrays of one column.  Recurrence coefficients are stored per chain (0: updraft u, 1: updraft v,
// 2: downdraft u, 3: downdraft v) or per direction (0: up, 1: down) so that one lane can run one chain with
// the same instructions as its neighbours:  val = use ? ((A*prev + B1) + B2) / D : default
enum MomArr { M_MU = 0, M_MD, M_ED, M_DP, M_C, M_CHAT = M_C + 2, M_PGU = M_CHAT + 2, M_PGD = M_PGU + 2,
              M_CONU = M_PGD + 2, M_COND = M_CONU + 2,      // = "chain value" arrays M_CONU + chain
              M_B1 = M_COND + 2, M_B2 = M_B1 + 4,           // per chain
              // momentum flux and end-of-step wind are formed after the recurrences, when their numerator terms B1 are
              // dead: same storage (level pver+1 of MF is set ahead of the recurrences; B1 ends at level pver).
              // 32 instead of 36 arrays: six instead of five 4-warp blocks per SM at L32
              M_MF = M_B1, M_WF = M_B1 + 2,
              M_A = M_B2 + 4, M_D = M_A + 2, M_R = M_D + 2, M_USE = M_R + 2,   // per direction
              M_NARR = M_USE + 2 };
__host__ __device__ inline size_t momtran_smem_bytes(int pver) {
  return (size_t)MOM_WARPS * M_NARR * (pver + 2) * sizeof(double);
}
__global__ void __launch_bounds__(32 * MOM_WARPS)
k_momtran_t(MomArgs a) {
  extern __shared__ double sm_mom[];
  const int pcols = P.pcols, pver = P.pver;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int wid = blockIdx.x * MOM_WARPS + wib;
  if (wid >= *a.count) return;
  const int slot = a.slots[wid];
  const int c = slot / pcols, gi = slot - c * pcols;
  const int ii = a.ideep[slot] - 1;
  const int mx = a.mx[slot];
  const int ktm = a.ktm[c], kbm = a.kbm[c];
  const double mbsth = 1.e-15, dt = a.dt;
  const int ld = pver + 2;                                    // levels 1..pver+1 addressed directly
  double* S = sm_mom + (size_t)wib * M_NARR * ld;
#define SA(arr, k) S[(arr) * ld + (k)]
#define QI(m, k) ((((size_t)c * 2 + (m)) * pver + (k) - 1) * pcols + ii)
#define PAR _Pragma("unroll 1") for (int k = lane + 1; k <= pver; k += 32)
  // wind component m of level k: packed (pcols,pver,2) arrays or the split ones of the fused step
  const bool split = a.q_u != nullptr;
  const double* qsrc[2] = {split ? a.q_u : a.q, split ? a.q_v : a.q + (size_t)pver * pcols};
  double* qdst[2] = {split ? a.dq_u : a.dqdt, split ? a.dq_v : a.dqdt + (size_t)pver * pcols};
  const size_t wbase = (size_t)c * (split ? 1 : 2) * pver * pcols + ii;
#define WI(k) (wbase + (size_t)((k) - 1) * pcols)
  // ---- stage the column ----
  PAR {
    const size_t g = cidx(c, k - 1, gi, pver);
    SA(M_MU, k) = a.mu[g]; SA(M_MD, k) = a.md[g]; SA(M_ED, k) = a.ed[g]; SA(M_DP, k) = a.dp[g];
#pragma unroll
    for (int m = 0; m < 2; ++m) SA(M_C + m, k) = a.domom[m] ? qsrc[m][WI(k)] : 0.0;
  }
  if (lane == 0) { SA(M_MF, pver + 1) = 0.0; SA(M_MF + 1, pver + 1) = 0.0; }
  __syncwarp();
  // ---- level-local terms ----
  PAR {
    const int km1 = max(1, k - 1), kp1 = min(pver, k + 1);
    const double mu_k = SA(M_MU, k), md_k = SA(M_MD, k), dp_k = SA(M_DP, k), dp_km1 = SA(M_DP, km1);
    const double mu_kp1 = SA(M_MU, kp1), md_kp1 = SA(M_MD, kp1);
    const size_t g = cidx(c, k - 1, gi, pver);
    const double eu_k = a.eu[g];
    const double mup_k = mu_k + a.du[g] * dp_k;
    // Divisors of the two recurrences with their refined reciprocals: q = x*r; q += r*(x - b*q) in the sequential
    // loop is the IEEE quotient x/b (the compiler's own fast-path division with the reciprocal hoisted out of
    // the dependent chain); only used where the reference divides (|b| > mbsth).
    SA(M_D, k) = mup_k;      SA(M_R, k) = rcp_hot(mup_k);     SA(M_USE, k) = (mup_k > mbsth) ? 1.0 : 0.0;
    SA(M_D + 1, k) = md_k;   SA(M_R + 1, k) = rcp_hot(md_k);  SA(M_USE + 1, k) = (md_k < -mbsth) ? 1.0 : 0.0;
    SA(M_A, k) = mu_kp1;                                       // mu(kk+1) of the updraft step at level kk = k
    SA(M_A + 1, k) = SA(M_MD, km1);                            // md(k-1) of the downdraft step at level k
#pragma unroll
    for (int m = 0; m < 2; ++m) {
      const double c_k = SA(M_C + m, k), c_km1 = SA(M_C + m, km1), c_kp1 = SA(M_C + m, kp1);
      double pgu, pgd;
      if (k == 1) {
        pgu = 0.0; pgd = 0.0;
      } else if (k == pver) {
        pgu = -P.momcu * div_z(mu_k * (c_k - c_km1), dp_km1);
        pgd = -P.momcd * div_z(md_k * (c_k - c_km1), dp_km1);
      } else {
        pgu = -P.momcu * 0.5 * (div_z(mu_k * (c_k - c_km1), dp_km1) + div_z(mu_kp1 * (c_kp1 - c_k), dp_k));
        pgd = -P.momcd * 0.5 * (div_z(md_k * (c_k - c_km1), dp_km1) + div_z(md_kp1 * (c_kp1 - c_k), dp_k));
      }
      const double chat = 0.5 * (c_k + c_km1);
      SA(M_CHAT + m, k) = chat; SA(M_CONU + m, k) = chat; SA(M_COND + m, k) = chat;
      SA(M_PGU + m, k) = pgu; SA(M_PGD + m, k) = pgd;
      SA(M_B1 + m, k) = eu_k * c_k * dp_k;                    // updraft: eu*cnst*dp ...
      SA(M_B2 + m, k) = pgu * dp_k;                           // ... + pgu*dp (zm_conv.F90:2538, 2563)
    }
  }
  __syncwarp();
  PAR {          // terms of the downdraft recurrence at level k use level k-1 (needs pgd of all levels)
    const int km1 = max(1, k - 1);
#pragma unroll
    for (int m = 0; m < 2; ++m) {
      // downdraft: - ed(k-1)*cnst(k-1)*dp(k-1) - pgd(k-1)*dp(k-1), stored negated (x - y == x + (-y))
      SA(M_B1 + 2 + m, k) = -(SA(M_ED, km1) * SA(M_C + m, km1) * SA(M_DP, km1));
      SA(M_B2 + 2 + m, k) = -(SA(M_PGD + m, km1) * SA(M_DP, km1));
    }
  }
  __syncwarp();
  // ---- the recurrences: lane & 3 picks the chain (updraft u, updraft v, downdraft u, downdraft v), every chain
  // runs the same instruction stream (other lanes repeat one of the four).  Updraft (zm_conv.F90:2536-2575):
  // level kk = pver - n, conu = (mu(kk+1)*conu(kk+1) + eu*c*dp + pgu*dp)/mupdudp, without the first product at
  // kk = pver.  Downdraft (2579-2589): level k = n + 2, cond = (md(k-1)*cond(k-1) - ed*c*dp - pgd*dp)/md(k); at
  // k = 2 the reference's operator precedence (2554) makes it (-ed*c*dp) - (pgd*dp)/md(2).
  {
    const int chain = lane & 3, dir = chain >> 1, m = chain & 1;
    const bool on = a.domom[m] != 0;
    double prev = dir ? SA(M_COND + m, 1) : 0.0;
    for (int n = 0; n < pver; ++n) {
      const int lev = dir ? n + 2 : pver - n;
      if (lev <= pver && on) {
        const double b1 = SA(M_B1 + chain, lev), b2 = SA(M_B2 + chain, lev);
        const double dd = SA(M_D + dir, lev), rr = SA(M_R + dir, lev);
        const bool first = (n == 0);                   // updraft at pver: no flux from below; downdraft at 2: :2554
        const double num = first ? (dir ? b2 : b1 + b2) : (SA(M_A + dir, lev) * prev + b1) + b2;
        const double q = zmm::div_rcp(num, dd, rr);
        double val = (first && dir) ? b1 + q : q;
        if (SA(M_USE + dir, lev) == 0.0) val = SA(M_CONU + chain, lev);     // keeps chat
        prev = val;
        if (lane < 4) SA(M_CONU + chain, lev) = val;
      }
    }
  }
  __syncwarp();
  // ---- fluxes, tendencies, end-of-step wind (level-local) ----
  PAR {
    const int kp1 = min(pver, k + 1);
    const double dp_k = SA(M_DP, k);
#pragma unroll
    for (int m = 0; m < 2; ++m) {
      if (!a.domom[m]) { SA(M_MF + m, k) = 0.0; SA(M_WF + m, k) = 0.0; continue; }
      const double X_k = SA(M_MU, k) * (SA(M_CONU + m, k) - SA(M_CHAT + m, k));
      const double Y_k = SA(M_MD, k) * (SA(M_COND + m, k) - SA(M_CHAT + m, k));
      const double X_p = SA(M_MU, kp1) * (SA(M_CONU + m, kp1) - SA(M_CHAT + m, kp1));
      const double Y_p = SA(M_MD, kp1) * (SA(M_COND + m, kp1) - SA(M_CHAT + m, kp1));
      double dc = 0.0;
      if (k >= ktm) dc = +div_z(X_p - X_k + Y_p - Y_k, dp_k);
      if (k >= kbm && k == mx) dc = (1.0 / dp_k) * (-X_k - Y_k);
      qdst[m][WI(k)] = dc;
      if (a.pguall) {
        a.pguall[QI(m, k)] = -SA(M_PGU + m, k);
        a.pgdall[QI(m, k)] = -SA(M_PGD + m, k);
        a.icwu[QI(m, k)] = SA(M_CONU + m, k);
        a.icwd[QI(m, k)] = SA(M_COND + m, k);
      }
      SA(M_MF + m, k) = (k >= ktm) ? (-X_k - Y_k) : 0.0;
    }
  }
  __syncwarp();
  PAR {
#pragma unroll
    for (int m = 0; m < 2; ++m)
      if (a.domom[m])
        SA(M_WF + m, k) = (k >= ktm) ? SA(M_C + m, k) - div_z((SA(M_MF + m, k + 1) - SA(M_MF + m, k)) * dt, SA(M_DP, k)) : 0.0;
  }
  __syncwarp();
  // ---- KE dissipation heating (zm_conv.F90:2675-2712) ----
  PAR {
    double gset2 = 0.0;
    if (k >= ktm) {
      const int km1 = max(1, k - 1), kp1 = min(pver, k + 1);
      const double u0 = SA(M_C, k), v0 = SA(M_C + 1, k);
      const double utop = (u0 + SA(M_C, km1)) / 2.0;
      const double vtop = (v0 + SA(M_C + 1, km1)) / 2.0;
      const double ubot = (SA(M_C, kp1) + u0) / 2.0;
      const double vbot = (SA(M_C + 1, kp1) + v0) / 2.0;
      const double fket = utop * SA(M_MF, k) + vtop * SA(M_MF + 1, k);
      const double fkeb = ubot * SA(M_MF, k + 1) + vbot * SA(M_MF + 1, k + 1);
      const double ketend_cons = div_z(fket - fkeb, SA(M_DP, k));
      const double uf = SA(M_WF, k), vf = SA(M_WF + 1, k);
      const double ketend = div_z(((uf * uf + vf * vf) - (u0 * u0 + v0 * v0)) * 0.5, dt);
      gset2 = ketend_cons - ketend;
    }
    a.seten[cidx(c, k - 1, ii, pver)] = gset2;
  }
#undef SA
#undef QI
#undef WI
#undef PAR
}

// ---- convtran --------------------------------------------------------------------------------------
struct TranArgs {
  int nchunks, ncnst, nactive;
  const int *jt, *mx, *ideep, *lengath, *ktm, *kbm, *slots, *count;
  const int* active;        // [nactive] 0-based constituent indices with doconvtran (m >= 2)
  const int* is_dry;        // [ncnst]
  const double *q, *fracis, *mu, *md, *du, *eu, *ed, *dp, *dpdry;
  double* dqdt;
};
// Gathered instantiations of k_convtran_t / k_convtran_c (zm_conv_tend_2_batch_gathered): q, fracis and dqdt are the
// convective columns' records instead of (pcols,pver,ncnst) chunk arrays.  Chunk c's block starts at
// nactive*pver*rbase[c] (rbase, an extra kernel argument: exclusive prefix of lengath, k_lengath_scan); inside it the
// Fortran array g(lengath(c), pver, nactive), i.e. element (gathered slot gi, level k0, active constituent j) at
// (j*pver + k0)*lengath(c) + gi.  The default instantiations ignore rbase.

// dqdt(:,:,m) = 0 for every active constituent (zm_conv.F90:2298): one block per (chunk, active m) slice
__global__ void __launch_bounds__(128)
k_convtran_zero(TranArgs a) {
  const int per = P.pcols * P.pver;
  const int c = blockIdx.x / a.nactive, j = blockIdx.x - c * a.nactive;
  double* d = a.dqdt + ((size_t)c * a.ncnst + a.active[j]) * per;
  for (int e = threadIdx.x; e < per; e += blockDim.x) d[e] = 0.0;
}

// Interface value of the tracer between levels k-1 and k (zm_conv.F90:2119-2139).
// Divisions and the log use the straight-line variants (div_hot, log_hot: the IEEE / general results for normal
// operands): tracer mixing ratios are either 0 or far above 1e-280, where that holds.
__device__ __forceinline__ double convtran_chat(double cm, double ck) {
  const double small = 1.e-36;
  const double minc = fmin2(cm, ck), maxc = fmax2(cm, ck);
  double cdifr;
  if (minc < 0.0) cdifr = 0.0;
  else cdifr = div_hot(fabs(ck - cm), fmax2(maxc, small));
  if (cdifr > 1.E-6) {
    const double cabv = fmax2(cm, maxc * 1.e-12);
    const double cbel = fmax2(ck, maxc * 1.e-12);
    return div_hot(zmm::log_hot(div_hot(cabv, cbel)), cabv - cbel) * cabv * cbel;
  }
  return 0.5 * (ck + cm);
}

// Thread per (gathered column, active constituent), registers only.  Sweep 1 (bottom-up) computes the updraft
// mixing ratio conu(k) (zm_conv.F90:2152-2175) and parks it in the dqdt output slice; sweep 2 (top-down) computes
// the downdraft mixing ratio cond(k) (2178-2186) and, one level late, the limited fluxes and the tendency
// (2189-2254).  blockDim = (32 column slots, 4 constituents); grid x = constituent group (fastest), y = group of 32
// column slots, so the blocks that share a column's seven mass-flux arrays run back to back and those arrays
// come from L2 instead of HBM once per constituent group (ncu: 4.9 -> 3.9 GB of DRAM traffic per launch, of
// which 0.6 GB is useful -- with one convective column in three every pass over a [level][16 columns] row drags
// the whole row in; staging the tracer column in shared memory cut the traffic further but cost more in
// occupancy than it saved: 1.16 vs 0.98 ms).
// constituents per block: 4 up to 64 levels, 2 above
__host__ __device__ inline int convtran_cnst_per_block(int pver) { return pver <= 64 ? 4 : 2; }
// GATH: q / fracis / dqdt are records (see TranArgs); level k of the pair is element rb + (k-1)*len, the
// updraft value is parked in dqdt_rec the same way, and every record element is written (no k_convtran_zero)
template <bool GATH = false>
__global__ void __launch_bounds__(128)
k_convtran_t(TranArgs a, const int* rbase) {
  zmm::hot_tables_load();                              // before any return (block-wide barrier inside)
  const int pcols = P.pcols, pver = P.pver;
  const int tid = blockIdx.y * blockDim.x + threadIdx.x;
  const int j = blockIdx.x * blockDim.y + threadIdx.y;
  if (tid >= *a.count || j >= a.nactive) return;
  const int slot = a.slots[tid];
  const int c = slot / pcols, gi = slot - c * pcols;
  const int m = a.active[j];
  const int ii = GATH ? 0 : a.ideep[slot] - 1;
  const int mx = a.mx[slot];
  const int ktm = a.ktm[c], kbm = a.kbm[c];
  const double mbsth = 1.e-15;
  const bool dry = a.is_dry[m] != 0;
  const size_t mb = ((size_t)c * a.ncnst + m) * pver;
  size_t rb = 0;
  int rlen = 0;
  if (GATH) { rlen = a.lengath[c]; rb = ((size_t)rbase[c] * a.nactive + (size_t)j * rlen) * pver + gi; }
#define GA(arr, k) a.arr[cidx(c, (k) - 1, gi, pver)]
#define QI(k) (GATH ? rb + (size_t)((k) - 1) * rlen : (mb + (k) - 1) * pcols + ii)
#define QS(k) a.q[QI(k)]
#define CU(k) a.dqdt[QI(k)]
  // per-level mass-flux terms with the dry/moist switch of zm_conv.F90:2087-2105
  auto dptmp_of = [&](int k) { return dry ? GA(dpdry, k) : GA(dp, k); };
  auto scaled = [&](double x, int k) { return dry ? div_hot(x * GA(dp, k), GA(dpdry, k)) : x; };

  // ---------------- sweep 1: conu, k = pver .. 1 ----------------
  {
    double conu_kp1 = 0.0, mu_kp1 = 0.0;
    double c_k = QS(pver);
    for (int k = pver; k >= 1; --k) {
      const double c_km1 = QS(max(1, k - 1));
      const double mu_k = GA(mu, k), dpt = dptmp_of(k);
      const double dut = scaled(GA(du, k), k);
      const double mupdudp = mu_k + dut * dpt;
      double conu;
      if (mupdudp > mbsth) {
        const double eut = scaled(GA(eu, k), k), fis = a.fracis[QI(k)];
        if (k == pver) conu = div_hot(+eut * fis * c_k * dpt, mupdudp);
        else           conu = div_hot(mu_kp1 * conu_kp1 + eut * fis * c_k * dpt, mupdudp);
      } else {
        conu = convtran_chat(c_km1, c_k);
      }
      CU(k) = conu;
      conu_kp1 = conu; mu_kp1 = mu_k; c_k = c_km1;
    }
  }
  // ---------------- sweep 2: cond + fluxes, k = 1 .. pver, finishing level k-1 one step late ----------------
  {
    double c_km1 = QS(1), c_k = c_km1;
    double c_jm1 = c_km1;                       // const(max(1, j-1)) of the level being finished
    double cond_km1 = 0.0, md_km1 = 0.0, t_km1 = 0.0;   // t = edtmp*fisg*const*dptmp of level k-1
    double chat_j = 0.0, conu_j = 0.0, cond_j = 0.0, mu_j = 0.0, md_j = 0.0, dpt_j = 1.0;
    for (int k = 1; k <= pver + 1; ++k) {
      double chat_k = 0.0, conu_k = 0.0, cond_k = 0.0, mu_k = 0.0, md_k = 0.0, dpt_k = 1.0, c_kp1 = c_k, t_k = 0.0;
      if (k <= pver) {
        chat_k = convtran_chat(c_km1, c_k);
        conu_k = CU(k);
        mu_k = GA(mu, k); md_k = GA(md, k); dpt_k = dptmp_of(k);
        if (k < pver) c_kp1 = QS(k + 1);
        cond_k = chat_k;
        if (k == 2) {
          if (md_k < -mbsth) cond_k = div_hot(-t_km1, md_k);
        } else if (k >= 3) {
          if (md_k < -mbsth) cond_k = div_hot(md_km1 * cond_km1 - t_km1, md_k);
        }
        t_k = scaled(GA(ed, k), k) * a.fracis[QI(k)] * c_k * dpt_k;
      }
      if (k >= 2) {
        const int jl = k - 1;                   // level being finished; kp1 = min(pver, jl+1)
        const bool last = (jl == pver);
        const double mu_p = last ? mu_j : mu_k, md_p = last ? md_j : md_k;
        const double conu_p = last ? conu_j : conu_k, cond_p = last ? cond_j : cond_k;
        const double chat_p = last ? chat_j : chat_k;
        const double c_p = last ? c_km1 : c_k;  // const(kp1): c_km1 currently holds level jl
        const double cj = c_km1;                // const(jl)
        double dc = 0.0;
        if (jl >= ktm) {
          const double fluxin = mu_p * conu_p + mu_j * fmin2(chat_j, c_jm1) - (md_j * cond_j + md_p * fmin2(chat_p, c_p));
          const double fluxout = mu_j * conu_j + mu_p * fmin2(chat_p, cj) - (md_p * cond_p + md_j * fmin2(chat_j, cj));
          double netflux = fluxin - fluxout;
          if (fabs(netflux) < fmax2(fluxin, fluxout) * 1.e-12) netflux = 0.0;
          dc = div_hot(netflux, dpt_j);
        }
        if (jl >= kbm) {
          if (jl == mx) {
            const double fluxin = mu_j * fmin2(chat_j, c_jm1) - md_j * cond_j;
            const double fluxout = mu_j * conu_j - md_j * fmin2(chat_j, cj);
            double netflux = fluxin - fluxout;
            if (fabs(netflux) < fmax2(fluxin, fluxout) * 1.e-12) netflux = 0.0;
            dc = div_hot(netflux, dpt_j);
          } else if (jl > mx) {
            dc = 0.0;
          }
        }
        a.dqdt[QI(jl)] = dc;
      }
      // shift
      c_jm1 = (k == 1) ? c_k : c_km1;           // for the next finished level j' = k: const(max(1, k-1))
      chat_j = chat_k; conu_j = conu_k; cond_j = cond_k; mu_j = mu_k; md_j = md_k; dpt_j = dpt_k;
      cond_km1 = cond_k; md_km1 = md_k; t_km1 = t_k;
      c_km1 = c_k; c_k = c_kp1;
    }
  }
#undef GA
#undef QI
#undef QS
#undef CU
}

// ---- convtran, block per chunk slice -------------------------------------------------------------------
// The same statements (zm_conv.F90:2108-2302) organised around the memory system instead of around one column:
//   * a block owns one chunk and walks over groups of G = floor(32 / lengath) active constituents, i.e.
//     T = G*lengath <= 32 (column, constituent) pairs at a time: lane = pair, warp = level (levels w, w+NW, ...),
//     so every warp is 27-32 lanes wide whatever the chunk's number of convective columns (CTC_BPC blocks share
//     the groups of a chunk);
//   * every row of q and fracis is fetched once (phase A: gather, interface values chat, the level-local products
//     of the two recurrences -- all level-parallel); the only serial part are the two first-order recurrences
//     conu (bottom-up, warp 0) and cond (top-down, warp 1), which run side by side out of shared memory (phase B);
//   * fluxes and the limited tendency are level-parallel again (phase C), and the dqdt slices leave the block as
//     whole 128-byte rows with the zero-fill of zm_conv.F90:2298 in the same pass (phase D): no k_convtran_zero,
//     no updraft values parked in HBM, no second sweep over q / fracis.
// DRAM traffic per launch = q + fracis (touched sectors) + dqdt (once) + the mass-flux arrays once (the blocks of
// one chunk are neighbours in the grid: L2) -- 1.7 GB for 38 constituents on the f09 shard against 4.4 GB for
// k_convtran_zero + k_convtran_t.
// Shared memory, one row per level: [const | chat | eu*fis*c*dp -> conu | ed*fis*c*dp -> cond | mupdudp -> dcondt]
// x 32 lanes, then mu[pcols], md[pcols]; every access is lane pointer + level*row + compile-time offset.
// Used when pcols is a power of two from 2 to 32, the rows fit and dqdt is 16-byte aligned; k_convtran_t otherwise.
// The gathered instantiation (records in, records out) needs no alignment: it stores 8-byte elements.
#define CTC_T 32
#define CTC_NW 8
#define CTC_BPC 3
#define CTC_GZERO 8
#define CTC_CONST 0
#define CTC_CHAT 32
#define CTC_CONU 64
#define CTC_COND 96
#define CTC_DC 128
#define CTC_MU 160
__host__ __device__ inline int convtran_c_row(int pcols) { return CTC_MU + 2 * pcols; }
__host__ __device__ inline size_t convtran_c_smem_bytes(int pver, int pcols) {
  return (size_t)pver * convtran_c_row(pcols) * sizeof(double);
}
__host__ inline bool convtran_c_fits(int pver, int pcols) {
  return pcols >= 2 && pcols <= CTC_T && (pcols & (pcols - 1)) == 0 && convtran_c_smem_bytes(pver, pcols) <= 200 * 1024;
}
// blocks per chunk: no more than the constituent groups a chunk can have (smallest G: floor(32 / pcols))
__host__ inline int convtran_c_blocks_per_chunk(int nactive, int pcols) {
  const int gmin = CTC_T / pcols > 0 ? CTC_T / pcols : 1;
  const int groups = (nactive + gmin - 1) / gmin;
  return groups < CTC_BPC ? groups : CTC_BPC;
}

// GATH (zm_conv_tend_2_batch_gathered): q / fracis / dqdt are records (see TranArgs).  Phase A1 reads a pair's
// levels len apart from its record plane (no column map), phase D stores each constituent's pver x len plane
// contiguously, and a chunk without convective columns has nothing to write.
template <bool GATH = false>
__global__ void __launch_bounds__(32 * CTC_NW, 4)
k_convtran_c(TranArgs a, int bpc, const int* rbase) {
  extern __shared__ double sm_ctc[];
  __shared__ int s_inv[CTC_T];
  const int pcols = P.pcols, pver = P.pver;
  const int c = blockIdx.x / bpc, g0 = blockIdx.x - c * bpc;
  const int len = a.lengath[c];
  const int G = len > 0 ? CTC_T / len : CTC_GZERO;
  if (g0 * G >= a.nactive) return;                     // uniform over the block: more blocks than groups
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slice = pver * pcols;
  const size_t cbase = (size_t)c * a.ncnst * slice;    // this chunk's q / fracis / dqdt slices
  // gathered: this chunk's record block, a constituent's plane is pver*len doubles, a level len doubles
  const size_t rblk = GATH ? (size_t)rbase[c] * a.nactive * pver : 0;
  const int qs = GATH ? len : pcols;                   // stride between levels of q / fracis
  if (GATH && len == 0) return;
  if (len == 0) {                                      // nothing convective in this chunk: dqdt(:,:,m) = 0
    for (int g = g0; g * G < a.nactive; g += bpc)
      for (int j = g * G; j < min(g * G + G, a.nactive); ++j) {
        double* d = a.dqdt + cbase + (size_t)a.active[j] * slice;
        for (int e = threadIdx.x; e < slice; e += blockDim.x) d[e] = 0.0;
      }
    return;
  }
  const int row = convtran_c_row(pcols);
  const double mbsth = 1.e-15;
  // once per block: column -> gathered position, mu / md of the chunk's convective columns
  if (!GATH) {
    if (threadIdx.x < pcols) s_inv[threadIdx.x] = -1;
    __syncthreads();
    if (threadIdx.x < len) s_inv[a.ideep[(size_t)c * pcols + threadIdx.x] - 1] = threadIdx.x;
  }
  if (lane < len) {
    const double* mup = a.mu + (size_t)c * slice + lane;
    const double* mdp = a.md + (size_t)c * slice + lane;
    double* rg = sm_ctc + CTC_MU + lane;
#pragma unroll 4
    for (int k0 = warp; k0 < pver; k0 += CTC_NW) {
      rg[k0 * row] = mup[k0 * pcols];
      rg[k0 * row + pcols] = mdp[k0 * pcols];
    }
  }
  zmm::hot_tables_load();                              // ends with a block-wide barrier
  const int ktm = a.ktm[c], kbm = a.kbm[c];
  // phase D: a warp stores one constituent's slice, a lane two neighbouring columns of a row (16 bytes)
  const int hp = pcols >> 1;
  const int di = (lane % hp) * 2, dk = lane / hp, dstep = 32 / hp;
  const int ds0 = GATH ? 0 : s_inv[di], ds1 = GATH ? 0 : s_inv[di + 1];
  // this lane's (column, constituent) pair inside a group
  const int jl = lane / len, gi = lane - jl * len;
  const int ii = GATH ? gi : a.ideep[(size_t)c * pcols + gi] - 1;         // gathered: slot of the record plane
  const int mx = a.mx[(size_t)c * pcols + gi];
  const size_t go = (size_t)c * slice + gi;                                // gathered arrays, + k0*pcols
  double* rl = sm_ctc + lane;                                              // + k0*row + CTC_*
  const double* rg = sm_ctc + CTC_MU + gi;                                 // mu; md at + pcols

  for (int g = g0; g * G < a.nactive; g += bpc) {
    const int j0 = g * G, ng = min(G, a.nactive - j0);
    const bool on = jl < ng;
    const int m = a.active[j0 + (on ? jl : 0)];
    const bool dry = a.is_dry[m] != 0;
    const size_t qo = GATH ? rblk + (size_t)(j0 + (on ? jl : 0)) * pver * len + ii : cbase + (size_t)m * slice + ii;
    const double* qp = a.q + qo;                                           // + k0*qs
    const double* fp = a.fracis + qo;

    // ---- phase A1: gather const and fisg (every DRAM-latency load of the group is in flight here) ----
    if (on) {
#pragma unroll 4
      for (int k0 = warp; k0 < pver; k0 += CTC_NW) {
        rl[k0 * row + CTC_CONST] = qp[k0 * qs];
        rl[k0 * row + CTC_CONU] = fp[k0 * qs];         // fisg, replaced by the updraft term in phase A2
      }
    }
    __syncthreads();
    // ---- phase A2: chat (zm_conv.F90:2119-2147), the level-local terms of the two recurrences ----
    if (on) {
#pragma unroll 2
      for (int k0 = warp; k0 < pver; k0 += CTC_NW) {
        double* r = rl + k0 * row;
        const double ck = r[CTC_CONST], ckm1 = (k0 > 0) ? r[CTC_CONST - row] : ck;
        const double fis = r[CTC_CONU];
        const size_t gx = go + (size_t)(k0 * pcols);
        double dpt = a.dp[gx], eut = a.eu[gx], edt = a.ed[gx], dut = a.du[gx];
        if (dry) {                                     // zm_conv.F90:2087-2095: x*dp/dpdry, one reciprocal for the three
          const double dpd = a.dpdry[gx], rdpd = rcp_hot(dpd);
          dut = zmm::div_rcp(dut * dpt, dpd, rdpd); eut = zmm::div_rcp(eut * dpt, dpd, rdpd);
          edt = zmm::div_rcp(edt * dpt, dpd, rdpd);
          dpt = dpd;
        }
        r[CTC_CHAT] = convtran_chat(ckm1, ck);
        r[CTC_CONU] = eut * fis * ck * dpt;
        r[CTC_COND] = edt * fis * ck * dpt;
        r[CTC_DC] = rg[k0 * row] + dut * dpt;
      }
    }
    __syncthreads();
    // ---- phase B: conu bottom-up on warp 0 (2152-2175), cond top-down on warp 1 (2153-2186).  The operands of the
    // next level are loaded, and the reciprocal of its divisor refined, before this level's result is stored, so
    // that only  multiply-add, quotient, select  remain on the chain; the quotient is formed unconditionally and
    // selected (a discarded one may be inf / nan) ----
    if (on && warp == 0) {
      double conu_kp1 = 0.0, mu_kp1 = 0.0;
      double* r = rl + (pver - 1) * row;
      const double* q = rg + (pver - 1) * row;
      double b_n = r[CTC_DC], u_n = r[CTC_CONU], ch_n = r[CTC_CHAT], mu_n = q[0], rb_n = rcp_hot(b_n);
      for (int k0 = pver - 1; k0 >= 0; --k0, r -= row, q -= row) {
        const double mupdudp = b_n, u = u_n, ch = ch_n, rb = rb_n, mu_k = mu_n;
        const int nx = (k0 > 0) ? -row : 0;            // no branch: the last level reloads itself
        b_n = r[CTC_DC + nx]; u_n = r[CTC_CONU + nx]; ch_n = r[CTC_CHAT + nx]; mu_n = q[nx];
        rb_n = rcp_hot(b_n);
        const double num = (k0 == pver - 1) ? u : mu_kp1 * conu_kp1 + u;
        const double quo = zmm::div_rcp(num, mupdudp, rb);
        const double conu = (mupdudp > mbsth) ? quo : ch;
        r[CTC_CONU] = conu;
        conu_kp1 = conu; mu_kp1 = mu_k;
      }
    } else if (on && warp == 1) {
      double cond_km1 = 0.0, md_km1 = 0.0, t_km1 = 0.0;
      double* r = rl;
      const double* q = rg + pcols;
      double b_n = q[0], t_n = r[CTC_COND], ch_n = r[CTC_CHAT], rb_n = rcp_hot(b_n);
      for (int k0 = 0; k0 < pver; ++k0, r += row, q += row) {
        const double md_k = b_n, t_k = t_n, ch = ch_n, rb = rb_n;
        const int nx = (k0 < pver - 1) ? row : 0;
        b_n = q[nx]; t_n = r[CTC_COND + nx]; ch_n = r[CTC_CHAT + nx];
        rb_n = rcp_hot(b_n);
        const double num = (k0 == 1) ? -t_km1 : md_km1 * cond_km1 - t_km1;
        const double quo = zmm::div_rcp(num, md_k, rb);
        const double cond = (k0 >= 1 && md_k < -mbsth) ? quo : ch;
        r[CTC_COND] = cond;
        cond_km1 = cond; md_km1 = md_k; t_km1 = t_k;
      }
    }
    else if (warp >= 2 && (g + bpc) * G < a.nactive) {
      // the other warps pull the next group's q / fracis rows into L2 meanwhile
      const int j0n = (g + bpc) * G;
      if (jl < min(G, a.nactive - j0n)) {
        const size_t mo = GATH ? rblk + (size_t)(j0n + jl) * pver * len + ii : cbase + (size_t)a.active[j0n + jl] * slice + ii;
        for (int k0 = warp - 2; k0 < pver; k0 += CTC_NW - 2) {
          asm volatile("prefetch.global.L2 [%0];" ::"l"(a.q + mo + k0 * qs));
          asm volatile("prefetch.global.L2 [%0];" ::"l"(a.fracis + mo + k0 * qs));
        }
      }
    }
    __syncthreads();
    // ---- phase C: limited fluxes and the tendency (2189-2254) ----
    if (on) {
      const double* dpp = (dry ? a.dpdry : a.dp) + go;
#pragma unroll 2
      for (int k0 = warp; k0 < pver; k0 += CTC_NW) {
        const int k = k0 + 1;
        double* r = rl + k0 * row;
        const double* rm = (k0 > 0) ? r - row : r;
        const double* rp = (k0 < pver - 1) ? r + row : r;
        const double* q = rg + k0 * row;
        const double* qn = (k0 < pver - 1) ? q + row : q;
        const double dpt_j = dpp[k0 * pcols];
        const double mu_j = q[0], mu_p = qn[0], md_j = q[pcols], md_p = qn[pcols];
        const double conu_j = r[CTC_CONU], conu_p = rp[CTC_CONU];
        const double cond_j = r[CTC_COND], cond_p = rp[CTC_COND];
        const double chat_j = r[CTC_CHAT], chat_p = rp[CTC_CHAT];
        const double c_jm1 = rm[CTC_CONST], cj = r[CTC_CONST], c_p = rp[CTC_CONST];
        double dc = 0.0;
        if (k >= ktm) {
          const double fluxin = mu_p * conu_p + mu_j * fmin2(chat_j, c_jm1) - (md_j * cond_j + md_p * fmin2(chat_p, c_p));
          const double fluxout = mu_j * conu_j + mu_p * fmin2(chat_p, cj) - (md_p * cond_p + md_j * fmin2(chat_j, cj));
          double netflux = fluxin - fluxout;
          if (fabs(netflux) < fmax2(fluxin, fluxout) * 1.e-12) netflux = 0.0;
          dc = div_hot(netflux, dpt_j);
        }
        if (k >= kbm) {
          if (k == mx) {
            const double fluxin = mu_j * fmin2(chat_j, c_jm1) - md_j * cond_j;
            const double fluxout = mu_j * conu_j - md_j * fmin2(chat_j, cj);
            double netflux = fluxin - fluxout;
            if (fabs(netflux) < fmax2(fluxin, fluxout) * 1.e-12) netflux = 0.0;
            dc = div_hot(netflux, dpt_j);
          } else if (k > mx) {
            dc = 0.0;
          }
        }
        r[CTC_DC] = dc;
      }
    }
    __syncthreads();
    // ---- phase D: dqdt(:,:,m) = 0, dqdt(ideep(i),k,m) = dcondt(i,k) (2298-2304) as whole rows ----
    if (GATH) {                  // the records: a warp stores one constituent's pver x len plane contiguously
      for (int j = warp; j < ng; j += CTC_NW) {
        double* d = a.dqdt + rblk + (size_t)(j0 + j) * pver * len;
        const double* s = sm_ctc + CTC_DC + j * len;
        for (int e = lane; e < pver * len; e += 32) {
          const int k0 = e / len;
          d[e] = s[k0 * row + (e - k0 * len)];
        }
      }
    } else
    for (int j = warp; j < ng; j += CTC_NW) {
      double* d = a.dqdt + cbase + (size_t)a.active[j0 + j] * slice + (dk * pcols + di);
      const double* s = sm_ctc + CTC_DC + j * len + dk * row;
#pragma unroll 4
      for (int k0 = dk; k0 < pver; k0 += dstep, d += dstep * pcols, s += dstep * row) {
        double2 v;
        v.x = (ds0 >= 0) ? s[ds0] : 0.0;
        v.y = (ds1 >= 0) ? s[ds1] : 0.0;
        *reinterpret_cast<double2*>(d) = v;
      }
    }
    // the next group's phase A1 only writes const, which nobody reads any more; its barrier orders phase D above
    // against the writes of phase A2
  }
}

// ---- N4 neighbours of the path (SURVEY.md section 8f) ------------------------------------------------
// geopotential_t (physics/geopotential.F90:153-247): thread per column, bottom-up scan, registers only.
struct GeoArgs {
  int nchunks, dycore_lr;
  const int* ncol;
  const double *piln, *pint, *pmid, *pdel, *rpdel, *t, *q, *rair, *zvir;
  double gravit;
  double *zi, *zm;
};
__global__ void __launch_bounds__(128)
k_geopotential_t(GeoArgs a) {
  const int pcols = P.pcols, pver = P.pver, pverp = P.pverp;
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= a.nchunks * pcols) return;
  const int c = col / pcols, i = col - c * pcols;
  if (i >= a.ncol[c]) return;
  double zi_p = 0.0;
  a.zi[cidx(c, pverp - 1, i, pverp)] = 0.0;
  for (int k = pver; k >= 1; --k) {
    const size_t e = cidx(c, k - 1, i, pver);
    double hkl, hkk;
    if (a.dycore_lr) {
      hkl = a.piln[cidx(c, k, i, pverp)] - a.piln[cidx(c, k - 1, i, pverp)];
      hkk = 1.0 - a.pint[cidx(c, k - 1, i, pverp)] * hkl * a.rpdel[e];
    } else {
      hkl = a.pdel[e] / a.pmid[e];
      hkk = 0.5 * hkl;
    }
    const double rog = a.rair[e] / a.gravit;
    const double tvfac = 1.0 + a.zvir[e] * a.q[e];
    const double tv = a.t[e] * tvfac;
    a.zm[e] = zi_p + rog * tv * hkk;
    zi_p = zi_p + rog * tv * hkl;
    a.zi[cidx(c, k - 1, i, pverp)] = zi_p;
  }
}

// geopotential_t, generalized-virtual-temperature branch (physics/geopotential.F90:248-310; dycore MPAS / SE):
// thread per column; q3 is the chunk's q(pcols,pver,ncnst), species[] the 1-based indices of the thermodynamically
// active species.  The two species loops of the reference (wet-to-dry factor, sum of dry mixing ratios) run per
// level in the reference's order; the level's species values are read twice (L1-resident: the sweep is HBM-bound).
struct GeoGenArgs {
  int nchunks, dycore_lr, ncnst, nspecies;
  const int *ncol, *species;
  const double *piln, *pint, *pmid, *pdel, *rpdel, *t, *q3, *rair, *zvir;
  double gravit;
  double *zi, *zm;
};
__global__ void __launch_bounds__(128)
k_geopotential_t_gen(GeoGenArgs a) {
  const int pcols = P.pcols, pver = P.pver, pverp = P.pverp;
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= a.nchunks * pcols) return;
  const int c = col / pcols, i = col - c * pcols;
  if (i >= a.ncol[c]) return;
  const double* qc = a.q3 + (size_t)c * a.ncnst * pver * pcols + i;      // + (m*pver + k)*pcols
  double zi_p = 0.0;
  a.zi[cidx(c, pverp - 1, i, pverp)] = 0.0;
  for (int k = pver; k >= 1; --k) {
    const size_t e = cidx(c, k - 1, i, pver);
    double qfac = 1.0;
    for (int s = 0; s < a.nspecies; ++s) qfac = qfac - qc[((size_t)(a.species[s] - 1) * pver + (k - 1)) * pcols];
    qfac = 1.0 / qfac;
    double sdm = 1.0;
    for (int s = 0; s < a.nspecies; ++s) sdm = sdm + qc[((size_t)(a.species[s] - 1) * pver + (k - 1)) * pcols] * qfac;
    sdm = 1.0 / sdm;
    double hkl, hkk;
    if (a.dycore_lr) {
      hkl = a.piln[cidx(c, k, i, pverp)] - a.piln[cidx(c, k - 1, i, pverp)];
      hkk = 1.0 - a.pint[cidx(c, k - 1, i, pverp)] * hkl * a.rpdel[e];
    } else {
      hkl = a.pdel[e] / a.pmid[e];
      hkk = 0.5 * hkl;
    }
    const double rog = a.rair[e] / a.gravit;
    const double tvfac = (1.0 + (a.zvir[e] + 1.0) * qc[(size_t)(k - 1) * pcols] * qfac) * sdm;
    const double tv = a.t[e] * tvfac;
    a.zm[e] = zi_p + rog * tv * hkk;
    zi_p = zi_p + rog * tv * hkl;
    a.zi[cidx(c, k - 1, i, pverp)] = zi_p;
  }
}

// convect_diagnostics_calc for shallow_scheme == 'CLUBB_SGS' (physics/convect_diagnostics.F90:115-249)
struct CdiagArgs {
  int nchunks;
  const int* ncol;
  double *cmfmc, *qc, *qc2, *rliq, *rliq2, *cnt, *cnb, *cmfmc2, *rprdsh, *rprdtot, *pcnt, *pcnb;
  const double *pmid, *rprddp;
};
// Level-wise statements run one element per thread (grid-stride over the (chunk, level, column) elements, coalesced);
// the per-column statements (cloud top / base merge and their pressures) follow in a second grid-stride loop.
__global__ void __launch_bounds__(256)
k_convect_diagnostics(CdiagArgs a) {
  const int pcols = P.pcols, pver = P.pver, pverp = P.pverp;
  const size_t nth = (size_t)gridDim.x * blockDim.x, tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t n2p = (size_t)a.nchunks * pverp * pcols, n2 = (size_t)a.nchunks * pver * pcols;
  for (size_t e = tid; e < n2p; e += nth) {
    const int i = (int)(e % pcols), c = (int)(e / ((size_t)pverp * pcols));
    a.cmfmc2[e] = 0.0;                                   // zeroed for all pcols (whole-array assignment)
    if (i < a.ncol[c]) a.cmfmc[e] = a.cmfmc[e] + 0.0;
  }
  for (size_t e = tid; e < n2; e += nth) {
    const int i = (int)(e % pcols), c = (int)(e / ((size_t)pver * pcols));
    a.rprdsh[e] = 0.0; a.qc2[e] = 0.0;
    if (i < a.ncol[c]) { a.rprdtot[e] = 0.0 + a.rprddp[e]; a.qc[e] = a.qc[e] + 0.0; }
  }
  for (size_t col = tid; col < (size_t)a.nchunks * pcols; col += nth) {
    const int c = (int)(col / pcols), i = (int)(col - (size_t)c * pcols);
    a.rliq2[col] = 0.0;
    if (i < a.ncol[c]) {
      const double cnt2 = (double)pver, cnb2 = 1.0;
      double cnt = a.cnt[col], cnb = a.cnb[col];
      if (cnt2 < cnt) cnt = cnt2;
      if (cnb2 > cnb) cnb = cnb2;
      if (cnb == 1.0) cnb = cnt;
      a.cnt[col] = cnt; a.cnb[col] = cnb;
      a.pcnt[col] = a.pmid[cidx(c, (int)cnt - 1, i, pver)];
      a.pcnb[col] = a.pmid[cidx(c, (int)cnb - 1, i, pver)];
      a.rliq[col] = a.rliq[col] + 0.0;
    }
  }
}
