// zm_plume_warp.cuh -- per-column cloud model, ONE WARP PER CONVECTIVE COLUMN.
//
// cldprp + closure + q1q2_pjr + scatter + precipitation (reference zm_conv.F90:3024-4026, 4028-4260,
// 4262-4421 and the zm_convr glue 926-1027, 1047-1078, 1233-1331, 1495-1511, 1616-1649).
// The ~55 per-level work arrays of one column live in shared memory; loops whose iterations are
// independent across levels (saturation, exp/log/pow evaluations, gathers, scatters) run with
// lane == level, while the order-dependent recurrences (k1..i4, hu, su/qu, ql, hd, sd, pflx and the
// running sums) are executed redundantly by every lane in the reference's own order, so every sum
// is accumulated exactly as the serial Fortran does (bit-exact vs the CPU oracle).
// A convective column therefore costs one saturation-pressure evaluation of latency plus a few short
// scans instead of a 32-level serial chain per thread.
// The reference's chunk-wide loop bounds (khighest/klowest 3573-3578, kmin/kmax 4245-4246,
// ktm/kbm 4350-4355) only trim loops whose bodies are re-guarded per column, so a per-column
// formulation is numerically identical (SURVEY.md section 8a notes a6-a8).
#pragma once
#include "zm_kernels.cuh"

enum PlumeArr {
  A_Q, A_T, A_P, A_Z, A_S, A_ZF, A_DZ, A_DP, A_SHAT, A_QHAT,
  A_MU, A_EU, A_DU, A_QU, A_SU, A_QST, A_HMN, A_HSAT,
  A_GAMMA, A_HU, A_EPS, A_F, A_K1, A_I2, A_I3, A_I4, A_QSTHAT, A_HSTHAT, A_GAMHAT,
  A_W1,
  A_FRONT_COUNT,   // 30 arrays are all the first cldprp call touches (cldprp_warp<false>, up to the cloud-top reset):
                   // k_cldprp_pass1_w allocates only these -- 24-26 warps per SM at L32 instead of 20
  A_MD = A_FRONT_COUNT, A_ED, A_SD, A_QD, A_MC, A_QL, A_CMEG, A_PFLX, A_EVP, A_CU, A_RPRD,
  A_COUNT,     // 41 arrays: 4 warps x 41 x 34 doubles = 44.6 KB per block, FIVE blocks (20 warps) per SM at L32
  // Arrays with disjoint lifetimes share storage (occupancy of these kernels is bounded by shared memory).
  // Host array -> last use; guest -> first use, in the (straight-line) order of cldprp_warp / k_plume_w:
  A_W4 = A_K1,       // k1: entrainment Taylor series (ends with the f(z) evaluation); W4 from the hu recurrence on
  A_QCDE = A_I2,     // i2: as k1; qcde zero-filled with the tu initialisation, written by the rain-out section
  A_TU = A_I3,       // i3: as k1; tu from the updraft temperature section on
  A_W2 = A_I4,       // i4: as k1; W2 from the hu recurrence on
  A_W3 = A_GAMMA,    // gamma only feeds gamhat (interface values, right after the saturation section)
  A_W5 = A_QST,      // qst last read by the statement that first writes W5 (same level, same lane)
  A_HD = A_F,        // f: ends with eps; hd/td/qds are (re)initialised at the start of the downdraft section
  A_TD = A_EPS,      // eps: ends with the updraft mass flux
  A_QDS = A_HSAT     // hsat: last read by the hu recurrence coefficients
};

#define PL_WARPS 4      // most warps (columns) a block may hold; the launch picks 1..PL_WARPS, see plume_warps_per_block

// Per-warp shared-memory work arrays [array][level]; the leading dimension is a compile-time constant
// (32/64/128-level builds) so that S(A_X, k) is base + immediate + k instead of a multiply per access.
template <int LD>
struct PlumeShT {
  double* base;
  __device__ __forceinline__ double& operator()(int a, int k) const { return base[a * LD + k]; }
};

// lane == level loops: one trip up to L32 (two at most for the deeper grids), so unrolled copies and their trip-count
// dispatch are dead weight in a kernel whose 11k instructions already miss the instruction cache (k_plume_w
// 11,328 -> 9,736 instructions, 436 -> 425 us)
#define PAR(k, lo, hi) _Pragma("unroll 1") for (int k = (lo) + lane; k <= (hi); k += 32)
#define WSYNC() __syncwarp()

// Phase timers (built only with -DZM_PLUME_PHASE_CLOCKS, scripts/plume_phase_cycles.py): lane 0 of every warp adds the
// clock64() cycles since the previous mark to its kernel's row (0 = k_cldprp_pass1_w, 1 = k_plume_w); the last slot
// counts the columns.  cldprp_warp keeps a clock of its own (PH_BEGIN), the kernels restart theirs when it returns.
// Without the macro the marks expand to nothing and the kernels compile as without them.
enum PlumePhase {
  PH_GATHER, PH_INIT, PH_J0, PH_K1_PREP, PH_K1, PH_EXPDIF, PH_F, PH_FMAX, PH_MU, PH_HU, PH_JT, PH_CLDTOP,
  PH_EU_SCAN, PH_SUQU_PREP, PH_SUQU, PH_SAT_CU, PH_QL_PREP, PH_QL, PH_HD_PREP, PH_HD, PH_SD_PREP, PH_SD, PH_PFLX,
  PH_CLOSURE, PH_Q1Q2, PH_SCATTER,
  PH_COUNT
};
#ifdef ZM_PLUME_PHASE_CLOCKS
__device__ unsigned long long g_plume_phase[2][PH_COUNT + 1];
#define PH_BEGIN(kern)                                                                       \
  const int ph_kern_ = (kern);                                                               \
  long long ph_t_ = clock64()
#define PH_COLUMN() (lane == 0 ? (void)atomicAdd(&g_plume_phase[ph_kern_][PH_COUNT], 1ull) : (void)0)
#define PH_RESTART() (ph_t_ = clock64())
#define PH_MARK(ph)                                                                          \
  do {                                                                                       \
    const long long ph_now_ = clock64();                                                     \
    if (lane == 0) atomicAdd(&g_plume_phase[ph_kern_][ph], (unsigned long long)(ph_now_ - ph_t_)); \
    ph_t_ = ph_now_;                                                                         \
  } while (0)
#else
#define PH_BEGIN(kern) ((void)0)
#define PH_COLUMN() ((void)0)
#define PH_RESTART() ((void)0)
#define PH_MARK(ph) ((void)0)
#endif

// Warp collectives over lane == level values.  For the searches below they reproduce the serial scans exactly: each
// predicate or value is evaluated per level as the scan would, and only the position of a hit is reduced.
__device__ __forceinline__ double warp_min(double v) {
  for (int off = 16; off; off >>= 1) v = fmin2(v, __shfl_xor_sync(0xffffffffu, v, off));
  return v;
}
__device__ __forceinline__ int warp_max(int v) { return __reduce_max_sync(0xffffffffu, v); }

// Level where `for (k...) if (valid(k) && v(k) <= vmin) { vmin = v(k); kbest = k; }` (vmin starting at 1.E6) ends up:
// the highest valid level whose value equals the minimum over the valid levels with v <= 1.E6 (a value the running
// minimum accepts; NaN never is).  -0 == +0, so the level does not depend on which zero the reduction returns.
// Returns 0 when no level is accepted.  The caller reads the value back at that level, so it keeps its sign.
template <class PlumeSh>
__device__ __forceinline__ int warp_last_argmin(const PlumeSh& S, int arr, int lo, int hi, int lane) {
  double m = 1.E6;
  bool any = false;
  PAR(k, lo, hi) {
    const double v = S(arr, k);
    if (v <= 1.E6) { m = fmin2(m, v); any = true; }
  }
  m = warp_min(m);
  if (!__any_sync(0xffffffffu, any)) return 0;
  int kbest = 0;
  PAR(k, lo, hi) if (S(arr, k) == m) kbest = k;        // == never holds for a NaN or for a value above 1.E6 (m <= 1.E6)
  return warp_max(kbest);
}

// gather one column into shared arrays (zm_conv.F90:926-940, 980-1027 / 1114-1195); returns dsubcld
template <class PlumeSh>
__device__ __forceinline__ double gather_column_w(const PlumeSh& S, const ConvrIn& in, int c, int i, int maxg,
                                                  int lane) {
  const int pver = P.pver, pcols = P.pcols, msg = P.msg;
  const double zs = in.geos[(size_t)c * pcols + i] * P.rgrav;
  PAR(k, 1, pver) {
    size_t e = cidx(c, k - 1, i, pver);
    double qk = in.qh[e], tk = in.t[e];
    const double dppk = in.dpp[e];
    S(A_DP, k) = 0.01 * dppk;
    S(A_Q, k) = qk;
    S(A_T, k) = tk;
    S(A_P, k) = in.pap[e] * 0.01;
    double zk = in.zm[e] + zs;
    S(A_Z, k) = zk;
    S(A_S, k) = tk + (P.grav / ((1.0 + P.zvir * qk) * P.cpres)) * zk;
    S(A_ZF, k) = in.zi[cidx(c, k - 1, i, pver + 1)] + zs;
  }
  if (lane == 0) S(A_ZF, pver + 1) = in.zi[cidx(c, pver, i, pver + 1)] + zs;
  WSYNC();
  double dsubcld = 0.0;
  for (int k = msg + 1; k <= pver; ++k)
    if (k >= maxg) dsubcld = dsubcld + S(A_DP, k);
  PAR(k, 1, pver) {
    if (k <= msg + 1) {
      S(A_SHAT, k) = S(A_S, k); S(A_QHAT, k) = S(A_Q, k);
    } else {
      double sk = S(A_S, k), sm = S(A_S, k - 1), qk = S(A_Q, k), qm = S(A_Q, k - 1);
      double sdifr = 0.0, qdifr = 0.0;
      if (sk > 0.0 || sm > 0.0) sdifr = fabs((sk - sm) / fmax2(sm, sk));
      if (qk > 0.0 || qm > 0.0) qdifr = fabs((qk - qm) / fmax2(qm, qk));
      S(A_SHAT, k) = (sdifr > 1.E-6) ? zmm::log_(sm / sk) * sm * sk / (sm - sk) : 0.5 * (sk + sm);
      S(A_QHAT, k) = (qdifr > 1.E-6) ? zmm::log_(qm / qk) * qm * qk / (qm - qk) : 0.5 * (qk + qm);
    }
    S(A_DZ, k) = S(A_ZF, k) - S(A_ZF, k + 1);
  }
  WSYNC();
  return dsubcld;
}

struct PlumeIdx { int jt, jlcl, j0, jd; };

// cldprp for one column.  FULL=false stops after the cloud-top reset (zm_conv.F90:3646).
template <bool FULL, class PlumeSh>
__device__ __forceinline__ PlumeIdx cldprp_warp(const PlumeSh& S, int jb, int lel, double landfrac, int lane) {
  const int pver = P.pver, pverp = P.pverp, msg = P.msg, limcnv = P.limcnv;
  const double eps1 = P.eps1, zvir = P.zvir, cpvir = P.cpvir, dcol = P.dcol, tmelt = P.tmelt;
  const double rl = P.rl, rd = P.rgas, grav = P.grav, cp = P.cpres;
  const int mx = jb;
  const double c0mask = P.c0_ocn * (1.0 - landfrac) + P.c0_lnd * landfrac;
  const double tiedke_msk = P.tiedke_add * (1.0 - landfrac) + P.tiedke_lnd * landfrac;
  PH_BEGIN(FULL ? 1 : 0);

  // ---- level-parallel initialisation (zm_conv.F90:3256-3314) ----
  PAR(k, 1, pver + 1) {
    S(A_K1, k) = 0.0; S(A_I2, k) = 0.0; S(A_I3, k) = 0.0; S(A_I4, k) = 0.0;
    S(A_MU, k) = 0.0; S(A_F, k) = 0.0; S(A_EPS, k) = 0.0;
    if (FULL) S(A_QL, k) = 0.0;          // the arrays from A_MD on exist in the full kernel only
    if (k <= pver) {
      const double qk = S(A_Q, k), tk = S(A_T, k), pk = S(A_P, k), zk = S(A_Z, k), sk = S(A_S, k);
      S(A_EU, k) = 0.0; S(A_DU, k) = 0.0;
      if (FULL) {
        S(A_CU, k) = 0.0; S(A_EVP, k) = 0.0; S(A_CMEG, k) = 0.0;
        S(A_MD, k) = 0.0; S(A_ED, k) = 0.0; S(A_SD, k) = sk; S(A_QD, k) = qk;
        S(A_MC, k) = 0.0; S(A_RPRD, k) = 0.0;
      }
      S(A_QU, k) = qk; S(A_SU, k) = sk;
      double est, qs;
      qsat_hPa(tk, pk, est, qs);
      if (pk - est <= 0.0) qs = 1.0;
      S(A_QST, k) = qs;
      const double mrd = (1.0 + zvir * qk) * rd;
      const double mcp = (1.0 + cpvir * qk) * cp;
      const double mrl = (1.0 - dcol * (tk - tmelt)) * rl;
      S(A_GAMMA, k) = qs * (1.0 + qs / eps1) * eps1 * mrl / (mrd * (tk * tk)) * mrl / mcp;
      const double hmn = mcp * tk + grav * zk + mrl * qk;
      S(A_HMN, k) = hmn;
      S(A_HSAT, k) = mcp * tk + grav * zk + mrl * qs;
      S(A_HU, k) = hmn;
    }
  }
  if (FULL && lane == 0) S(A_PFLX, 1) = 0.0;
  WSYNC();
  PAR(k, 1, pver) {
    if (k <= msg + 1) {
      S(A_HSTHAT, k) = S(A_HSAT, k); S(A_QSTHAT, k) = S(A_QST, k); S(A_GAMHAT, k) = S(A_GAMMA, k);
    } else {
      const double q1 = S(A_QST, k - 1), q0 = S(A_QST, k), g1 = S(A_GAMMA, k - 1), g0 = S(A_GAMMA, k);
      const double qsthat = (fabs(q1 - q0) > 1.E-6) ? zmm::log_(q1 / q0) * q1 * q0 / (q1 - q0) : q0;
      S(A_QSTHAT, k) = qsthat;
      // mcp, mrl of level k recomputed (same expressions as above) instead of kept in two more arrays
      const double mcp = (1.0 + cpvir * S(A_Q, k)) * cp;
      const double mrl = (1.0 - dcol * (S(A_T, k) - tmelt)) * rl;
      S(A_HSTHAT, k) = mcp * S(A_SHAT, k) + mrl * qsthat;
      S(A_GAMHAT, k) = (fabs(g1 - g0) > 1.E-6) ? zmm::log_(g1 / g0) * g1 * g0 / (g1 - g0) : g0;
    }
  }
  WSYNC();
  PH_MARK(PH_INIT);

  // ---- scalars (redundant on every lane) ----
  int jt = max(lel, limcnv + 1);
  jt = min(jt, pver);
  int jd = pver, jlcl = lel;
  // zm_conv.F90:3422-3428: last level of least hsat in [jt, jb]
  int j0 = warp_last_argmin(S, A_HSAT, max(msg + 1, jt), min(pver, jb), lane);
  PH_MARK(PH_J0);
  j0 = min(j0, jb - 2);
  j0 = max(j0, jt + 2);
  j0 = min(j0, pver);
  const double hmn_mx = S(A_HMN, mx), s_mx = S(A_S, mx);
  PAR(k, msg + 1, pver) {
    if (k >= jt && k <= jb) {
      S(A_HU, k) = hmn_mx + cp * tiedke_msk;
      S(A_SU, k) = s_mx + tiedke_msk / (1.0 + cpvir * S(A_QU, k));
    }
  }
  WSYNC();
  // k1, i2, i3, i4 recurrences (zm_conv.F90:3430-3442) -- serial, redundant on every lane
  PAR(k, msg + 1, pver) S(A_W1, k) = (hmn_mx - S(A_HMN, k)) * S(A_DZ, k);
  WSYNC();
  PH_MARK(PH_K1_PREP);
  {
    // The reference walks k = pver-1 .. msg+1 and, outside [jt, jb), only carries k1..i4 of level k (the zeros of the
    // initialisation: nothing else has written these arrays yet) to the next level; below jb that leaves zeros, above
    // jt nothing reads them.  So the walk starts at jb-1 from zeros and stops at jt.  The next level's operands are
    // loaded before this level's stores (nvcc does not move a shared load above a shared store).
    double k1p = 0.0, i2p = 0.0, i3p = 0.0, i4p = 0.0;        // values at k+1
    const int klo = max(jt, msg + 1);
    double dz = S(A_DZ, jb - 1), w1 = S(A_W1, jb - 1);
    for (int k = jb - 1; k >= klo; --k) {
      const double dzn = S(A_DZ, k - 1), w1n = S(A_W1, k - 1);
      const double k1 = k1p + w1;
      const double ihat = 0.5 * (k1p + k1);
      const double i2 = i2p + ihat * dz;
      const double idag = 0.5 * (i2p + i2);
      const double i3 = i3p + idag * dz;
      const double iprm = 0.5 * (i3p + i3);
      const double i4 = i4p + iprm * dz;
      S(A_K1, k) = k1; S(A_I2, k) = i2; S(A_I3, k) = i3; S(A_I4, k) = i4;
      k1p = k1; i2p = i2; i3p = i3; i4p = i4;
      dz = dzn; w1 = w1n;
    }
  }
  PH_MARK(PH_K1);
  // zm_conv.F90:3444-3450: expdif from the last level of least hmn in [j0, jb]
  const int khmin = warp_last_argmin(S, A_HMN, max(msg + 1, j0), min(pver, jb), lane);
  const double expdif = khmin > 0 ? hmn_mx - S(A_HMN, khmin) : 0.0;
  WSYNC();
  PH_MARK(PH_EXPDIF);
  PAR(k, msg + 2, pver) {
    double expnum = 0.0;
    double k1 = S(A_K1, k);
    if (k < jt || k >= jb) {
      k1 = 0.0; S(A_K1, k) = 0.0;
    } else {
      expnum = hmn_mx - (S(A_HSAT, k - 1) * (S(A_ZF, k) - S(A_Z, k)) + S(A_HSAT, k) * (S(A_Z, k - 1) - S(A_ZF, k))) /
                            (S(A_Z, k - 1) - S(A_Z, k));
    }
    if ((expdif > 100.0 && expnum > 0.0) && k1 > expnum * S(A_DZ, k)) {
      const double ft = expnum / k1, K1 = k1, I2 = S(A_I2, k), I3 = S(A_I3, k), I4 = S(A_I4, k);
      double fk = ft + I2 / K1 * (ft * ft) + (2.0 * (I2 * I2) - K1 * I3) / (K1 * K1) * ((ft * ft) * ft) +
                  (-5.0 * K1 * I2 * I3 + 5.0 * ((I2 * I2) * I2) + (K1 * K1) * I4) / ((K1 * K1) * K1) *
                      ((ft * ft) * (ft * ft));
      fk = fmax2(fk, 0.0);
      fk = fmin2(fk, P.entrmn);
      S(A_F, k) = fk;
    }
  }
  WSYNC();
  PH_MARK(PH_F);
  if (j0 < jb)
    if (S(A_F, j0) < 1.E-6 && S(A_F, j0 + 1) > S(A_F, j0)) j0 = j0 + 1;
  {
    // running max of f over [max(jt, msg+2), j0], seeded with f one level above; the carried value is the one the
    // previous level stored, so fmax2 sees the same operands in the same order
    const int klo = max(jt, msg + 2);
    double fp = S(A_F, klo - 1), f = S(A_F, klo);
    for (int k = klo; k <= j0; ++k) {
      const double fn = S(A_F, k + 1);
      fp = fmax2(f, fp);
      S(A_F, k) = fp;
      f = fn;
    }
  }
  const double eps0 = S(A_F, j0);
  WSYNC();
  PAR(k, msg + 1, pver) {           // zm_conv.F90:3500-3518, same assignment order
    double v = S(A_EPS, k);
    if (k == jb) v = eps0;
    if (k >= j0 && k <= jb) v = eps0;
    if (k < j0 && k >= jt) v = S(A_F, k);
    S(A_EPS, k) = v;
  }
  WSYNC();
  PH_MARK(PH_FMAX);
  // updraft mass flux (zm_conv.F90:3550-3571): level parallel (mu(k) does not depend on mu(k+1))
  const double zf_jb = S(A_ZF, jb);
  if (eps0 > 0.0) {
    PAR(k, msg + 1, pver) {
      if (k == jb) {
        S(A_MU, k) = 1.0;
      } else if (k >= jt && k < jb) {
        const double zuef = S(A_ZF, k) - zf_jb;
        S(A_MU, k) = (1.0 / eps0) * (zmm::exp_(S(A_EPS, k) * zuef) - 1.0) / zuef;
        S(A_W1, k) = (1.0 / eps0) * (zmm::exp_(S(A_EPS, k + 1) * zuef) - 1.0) / zuef;     // rmue
      }
    }
    WSYNC();
    PAR(k, msg + 1, pver) {
      if (k == jb) {
        S(A_EU, k) = S(A_MU, k) / S(A_DZ, k);
      } else if (k >= jt && k < jb) {
        const double rmue = S(A_W1, k);
        S(A_EU, k) = (rmue - S(A_MU, k + 1)) / S(A_DZ, k);
        S(A_DU, k) = div_z(rmue - S(A_MU, k), S(A_DZ, k));
      }
    }
    WSYNC();
    // hu recurrence (zm_conv.F90:3579-3598): hu(k) = A(k)*hu(k+1) + B(k) -- the coefficients are
    // level parallel (mu(k+1) taken as the serial loop leaves it: zeroed if it was < 0.02), the
    // chain itself is one multiply-add per level
    PAR(k, msg + 1, pver) {
      if (k >= lel && k <= jb - 1) {
        const double muk = S(A_MU, k);
        double mup = S(A_MU, k + 1);
        if (k + 1 <= jb - 1 && mup < 0.02) mup = 0.0;
        if (muk < 0.02) {
          S(A_W3, k) = 1.0;
          S(A_W4, k) = mup / S(A_DZ, k);                       // new du(k)
        } else {
          S(A_W3, k) = 0.0;
          S(A_W1, k) = mup / muk;
          S(A_W2, k) = S(A_DZ, k) / muk * (S(A_EU, k) * S(A_HMN, k) - S(A_DU, k) * S(A_HSAT, k));
        }
      }
    }
    WSYNC();
    PAR(k, msg + 1, pver) {
      if (k >= lel && k <= jb - 1 && S(A_W3, k) != 0.0) { S(A_MU, k) = 0.0; S(A_EU, k) = 0.0; S(A_DU, k) = S(A_W4, k); }
    }
    PH_MARK(PH_MU);
    {
      // the next level's coefficients are loaded before this level's store
      double hup = S(A_HU, jb);
      double w3 = S(A_W3, jb - 1), hmn = S(A_HMN, jb - 1), a = S(A_W1, jb - 1), b = S(A_W2, jb - 1);
      for (int k = jb - 1; k >= lel; --k) {
        const double w3n = S(A_W3, k - 1), hmnn = S(A_HMN, k - 1), an = S(A_W1, k - 1), bn = S(A_W2, k - 1);
        hup = (w3 != 0.0) ? hmn : a * hup + b;
        S(A_HU, k) = hup;
        w3 = w3n; hmn = hmnn; a = an; b = bn;
      }
    }
    WSYNC();
    PH_MARK(PH_HU);
  }
  {
    // zm_conv.F90:3600-3618: the first level going up from jb-2 (down to lel-1) where the updraft stops; each level's
    // test reads only hu, hsthat and mu, so it is evaluated lane == level and the hit nearest jb is kept
    const double hu_jb = S(A_HU, jb);
    int khit = -1;
    PAR(k, lel - 1, jb - 2) {
      const double hu = S(A_HU, k), hst = S(A_HSTHAT, k), muk = S(A_MU, k);
      const bool stop = (hu <= hst && S(A_HU, k + 1) > S(A_HSTHAT, k + 1) && muk >= 0.02) || hu > hu_jb || muk < 0.02;
      if (stop) khit = k;
    }
    khit = warp_max(khit);
    if (khit >= 0) {
      const int k = khit;
      const double hu = S(A_HU, k), hst = S(A_HSTHAT, k), muk = S(A_MU, k);
      if (hu <= hst && S(A_HU, k + 1) > S(A_HSTHAT, k + 1) && muk >= 0.02) jt = (hu - hst < -2000.0) ? k + 1 : k;
      else jt = k + 1;
    }
  }
  PH_MARK(PH_JT);
  if (eps0 > 0.0) {
    // cloud-top reset (zm_conv.F90:3620-3634), level parallel: level jt reads mu(jt+1), which no level changes
    PAR(k, msg + 1, pver) {
      if (k >= lel && k <= jt) {
        S(A_MU, k) = 0.0; S(A_EU, k) = 0.0; S(A_DU, k) = 0.0; S(A_HU, k) = S(A_HMN, k);
      }
      if (k == jt) {
        S(A_DU, k) = S(A_MU, k + 1) / S(A_DZ, k);
        S(A_EU, k) = 0.0;
        S(A_MU, k) = 0.0;
      }
    }
  }
  WSYNC();
  PH_MARK(PH_CLDTOP);
  PlumeIdx R{jt, jlcl, j0, jd};
  if (!FULL) return R;

  PAR(k, 1, pver) S(A_QCDE, k) = 0.0;        // zm_conv.F90:3309 (its storage held i2 until now)
  // tu initialisation (zm_conv.F90:3649-3654)
  PAR(k, msg + 2, pver) {
    const double qu = S(A_QU, k);
    S(A_TU, k) = (S(A_HU, k) - grav * S(A_ZF, k) - (1.0 + dcol * tmelt) * rl * qu) /
                 (cp * (1.0 + (cpvir - dcol * (rl / cp)) * qu));
  }
  WSYNC();
  if (eps0 > 0.0) {
    if (jb >= msg + 2) {
      const double qu = S(A_Q, mx);
      const double tu = (S(A_HU, jb) - grav * S(A_ZF, jb) - (1.0 + dcol * tmelt) * rl * qu) /
                        (cp * (1.0 + (cpvir - dcol * (rl / cp)) * qu));
      S(A_QU, jb) = qu;
      S(A_TU, jb) = tu;
      S(A_SU, jb) = (S(A_HU, jb) - (1.0 - dcol * (tu - tmelt)) * rl * qu) / ((1.0 + cpvir * qu) * cp);
    }
    // su/qu recurrence (zm_conv.F90:3672-3688) evaluated speculatively for every k in (jt, jb) into
    // W1/W2 (it never feeds the saturation test's outcome back), then the saturation test runs level
    // parallel and only the levels the reference actually updated (k >= jlcl) are committed.
    PAR(k, msg + 2, pver) {
      if (k > jt && k < jb) {
        const double muk = S(A_MU, k), dz = S(A_DZ, k), eu = S(A_EU, k), du = S(A_DU, k);
        S(A_W3, k) = S(A_MU, k + 1) / muk;
        S(A_W4, k) = dz / muk * (eu - du) * S(A_S, k);
        S(A_W5, k) = dz / muk * (eu * S(A_Q, k) - du * S(A_QST, k));
      }
    }
    WSYNC();
    PH_MARK(PH_SUQU_PREP);
    {
      // the next level's coefficients are loaded before this level's stores
      double sup = S(A_SU, jb), qup = S(A_QU, jb);
      const int klo = max(jt + 1, msg + 2);
      double a = S(A_W3, jb - 1), bs = S(A_W4, jb - 1), bq = S(A_W5, jb - 1);
      for (int k = jb - 1; k >= klo; --k) {
        const double an = S(A_W3, k - 1), bsn = S(A_W4, k - 1), bqn = S(A_W5, k - 1);
        sup = a * sup + bs;
        qup = a * qup + bq;
        S(A_W1, k) = sup; S(A_W2, k) = qup;
        a = an; bs = bsn; bq = bqn;
      }
    }
    WSYNC();
    PH_MARK(PH_SUQU);
    int kfirst = 0;      // highest k (first met going up from jb-1) with qu >= qstu
    PAR(k, msg + 2, pver) {
      bool sat = false;
      if (k > jt && k < jb) {
        const double su = S(A_W1, k), qu = S(A_W2, k);
        // default-real literal 0.85 in the reference (zm_conv.F90:3680) == (double)0.85f
        const double tu = su - grav / ((1.0 + 0.85000002384185791015625 * qu) * cp) * S(A_ZF, k);
        S(A_W3, k) = tu;
        const double qstu = qsat_hPa_q(tu, (S(A_P, k) + S(A_P, k - 1)) / 2.0);
        sat = qu >= qstu;
      }
      kfirst = max(kfirst, sat ? k : 0);
    }
    for (int off = 16; off; off >>= 1) kfirst = max(kfirst, __shfl_xor_sync(0xffffffffu, kfirst, off));
    if (kfirst > 0) jlcl = kfirst;
    const int kstop = (kfirst > 0) ? kfirst : (jt + 1);      // recurrence ran for k = jb-1 .. kstop
    WSYNC();
    PAR(k, msg + 2, pver) {
      if (k > jt && k < jb && k >= kstop) { S(A_SU, k) = S(A_W1, k); S(A_QU, k) = S(A_W2, k); S(A_TU, k) = S(A_W3, k); }
    }
    WSYNC();
    PAR(k, msg + 2, pver) {
      if (k > jt && k <= jlcl) {
        const double gh = S(A_GAMHAT, k), dh = S(A_HU, k) - S(A_HSTHAT, k);
        const double qu = S(A_QSTHAT, k) + gh * dh / ((1.0 - dcol * (S(A_TU, k) - tmelt)) * rl * (1.0 + gh));
        const double su = S(A_SHAT, k) + dh / ((1.0 + cpvir * qu) * cp * (1.0 + gh));
        S(A_QU, k) = qu; S(A_SU, k) = su;
        S(A_TU, k) = su - grav / ((1.0 + cpvir * qu) * cp) * S(A_ZF, k);
      }
    }
    WSYNC();
    PAR(k, msg + 2, pver) {
      if (k >= jt && k < jb) {
        double cuk = ((S(A_MU, k) * S(A_SU, k) - S(A_MU, k + 1) * S(A_SU, k + 1)) / S(A_DZ, k) -
                      (S(A_EU, k) - S(A_DU, k)) * S(A_S, k)) / (rl / cp) *
                     ((1.0 + cpvir * S(A_QU, k)) / (1.0 - dcol * (S(A_TU, k) - tmelt)));
        if (k == jt) cuk = 0.0;
        S(A_CU, k) = fmax2(0.0, cuk);
      }
    }
    WSYNC();
  }
  PH_MARK(PH_SAT_CU);
  // rain production (zm_conv.F90:3846-3870), serial
  double totpcp = 0.0, totevp = 0.0;
  PAR(k, msg + 2, pver) {
    S(A_RPRD, k) = 0.0;
    if (k >= jt && k < jb && eps0 > 0.0 && S(A_MU, k) >= 0.0) {
      const double muk = S(A_MU, k), dz = S(A_DZ, k);
      double mus = (muk > 0.0) ? muk : 1.0;       // no 1/0 on the idle path (it would leave the inline division)
      asm("" : "+d"(mus));
      S(A_W1, k) = (muk > 0.0) ? 1.0 / mus : 0.0;
      S(A_W2, k) = dz * S(A_DU, k);
      S(A_W3, k) = dz * S(A_CU, k);
      S(A_W4, k) = 1.0 + dz * c0mask;
      S(A_W5, k) = rcp_hot(1.0 + dz * c0mask);          // divisor's refined reciprocal: off the serial chain
    }
  }
  WSYNC();
  PH_MARK(PH_QL_PREP);
  if (eps0 > 0.0) {
    // The reference walks k = pver .. msg+2; a level outside [jt, jb) or with mu < 0 only carries ql(k), a zero of the
    // initialisation (this loop is the only writer of ql), to the next level.  So the walk starts at jb-1 from zero,
    // stops at jt and carries zero past a level with mu < 0.  mu and the coefficients of the next level are loaded
    // before this level's store.
    double qlp = 0.0;
    const int khi = min(pver, jb - 1), klo = max(jt, msg + 2);
    double mup = S(A_MU, khi + 1), mu = S(A_MU, khi);
    double w1 = S(A_W1, khi), w2 = S(A_W2, khi), w3 = S(A_W3, khi), w4 = S(A_W4, khi), w5 = S(A_W5, khi);
    for (int k = khi; k >= klo; --k) {
      const double mun = S(A_MU, k - 1);
      const double w1n = S(A_W1, k - 1), w2n = S(A_W2, k - 1), w3n = S(A_W3, k - 1), w4n = S(A_W4, k - 1),
                   w5n = S(A_W5, k - 1);
      const double dz = S(A_DZ, k), cu = S(A_CU, k), du = S(A_DU, k);
      if (mu >= 0.0) {
        double ql = 0.0;
        if (mu > 0.0) {
          const double ql1 = w1 * (mup * qlp - w2 * qlp + w3);
          ql = zmm::div_rcp(ql1, w4, w5);    // == ql1 / (1 + dz*c0mask)
        }
        S(A_QL, k) = ql;
        totpcp = totpcp + dz * (cu - du * qlp);
        qlp = ql;
      } else {
        qlp = 0.0;
      }
      mup = mu; mu = mun;
      w1 = w1n; w2 = w2n; w3 = w3n; w4 = w4n; w5 = w5n;
    }
  }
  WSYNC();
  PH_MARK(PH_QL);
  PAR(k, msg + 2, pver) {
    if (k >= jt && k < jb && eps0 > 0.0 && S(A_MU, k) >= 0.0) {
      const double ql = S(A_QL, k);
      S(A_RPRD, k) = c0mask * S(A_MU, k) * ql;
      S(A_QCDE, k) = ql;
    }
  }
  WSYNC();
  // downdraft (zm_conv.F90:3880-3975).  hd, qds, td start from their environment values (zm_conv.F90:3283-3312);
  // set here because their storage held f / hsat / eps until now.
  PAR(k, 1, pver) {
    const double qk = S(A_Q, k), hmn = S(A_HMN, k);
    S(A_HD, k) = hmn;
    S(A_QDS, k) = qk;
    S(A_TD, k) = (hmn - grav * S(A_ZF, k) - (1.0 + dcol * tmelt) * rl * qk) /
                 (cp * (1.0 + (cpvir - dcol * (rl / cp)) * qk));
  }
  WSYNC();
  const double alfa = P.alfadet;
  double epsm = 0.0;
  jt = min(jt, jb - 1);
  jd = max(j0, jt + 1);
  jd = min(jd, jb);
  S(A_HD, jd) = S(A_HMN, jd - 1);
  if (jd < jb && eps0 > 0.0) {
    epsm = eps0;
    S(A_MD, jd) = -alfa * epsm / eps0;
  }
  WSYNC();
  if (eps0 > 0.0) {
    const double zf_jd = S(A_ZF, jd);
    PAR(k, msg + 1, pver) {
      if (k > jd && k <= jb) {
        const double zdef = zf_jd - S(A_ZF, k);
        S(A_MD, k) = -alfa / (2.0 * eps0) * (zmm::exp_(2.0 * epsm * zdef) - 1.0) / zdef;
      }
    }
    WSYNC();
    if (jd < jb) {
      // ratmjb is recomputed every k in the reference from the already-rescaled md(jb) once k passes
      // jb?  No: k runs upward to jb, md(jb) is only modified at k = jb itself, so every k uses the
      // unscaled md(jb) (zm_conv.F90:3906-3913).
      const double ratmjb = fmin2(fabs(S(A_MU, jb) / S(A_MD, jb)), 1.0);
      PAR(k, msg + 1, pver) {
        if (k >= jt && k <= jb) S(A_MD, k) = S(A_MD, k) * ratmjb;
      }
      WSYNC();
    }
    const double small = 1.e-20;
    // ed level parallel, hd serial (zm_conv.F90:3916-3924)
    PAR(k, msg + 1, pver) {
      if (k >= jt) S(A_ED, k - 1) = div_z(S(A_MD, k - 1) - S(A_MD, k), S(A_DZ, k - 1));
    }
    WSYNC();
    PAR(k, msg + 1, pver) {
      if (k >= jt) {
        S(A_W1, k) = S(A_DZ, k - 1) * S(A_ED, k - 1) * S(A_HMN, k - 1);
        S(A_W2, k) = fmin2(S(A_MD, k), -small);
        S(A_W3, k) = rcp_hot(fmin2(S(A_MD, k), -small));
      }
    }
    WSYNC();
    PH_MARK(PH_HD_PREP);
    {
      // The reference runs hd down to pver, but below jb nothing reads it (qds, td and sd use hd of [jd, jb] only, and
      // hd's storage is not read again after the downdraft), so the walk stops at jb.  The next level's operands are
      // loaded before this level's store.
      const int k0 = max(jt, msg + 1), khi = min(jb, pver);
      double hdp = S(A_HD, k0 - 1);
      double md = S(A_MD, k0 - 1), w1 = S(A_W1, k0), w2 = S(A_W2, k0), w3 = S(A_W3, k0);
      for (int k = k0; k <= khi; ++k) {
        const double mdn = S(A_MD, k), w1n = S(A_W1, k + 1), w2n = S(A_W2, k + 1), w3n = S(A_W3, k + 1);
        hdp = zmm::div_rcp(md * hdp - w1, w2, w3);
        S(A_HD, k) = hdp;
        md = mdn; w1 = w1n; w2 = w2n; w3 = w3n;
      }
    }
    WSYNC();
    PH_MARK(PH_HD);
    if (jd < jb) {
      PAR(k, msg + 2, pver) {
        if (k >= jd && k <= jb) {
          const double gh = S(A_GAMHAT, k), dh = S(A_HD, k) - S(A_HSTHAT, k);
          double qds = S(A_QSTHAT, k) + gh * dh / (rl * (1.0 + gh));
          const double td = (S(A_HD, k) - grav * S(A_ZF, k) - (1.0 + dcol * tmelt) * rl * qds) /
                            (cp * (1.0 + (cpvir - dcol * (rl / cp)) * qds));
          qds = S(A_QSTHAT, k) + gh * dh / ((1.0 - dcol * (td - tmelt)) * rl * (1.0 + gh));
          S(A_TD, k) = td; S(A_QDS, k) = qds;
        }
      }
      WSYNC();
    }
  }
  {
    const int k = jd;
    const double qd = S(A_QDS, jd);
    S(A_QD, jd) = qd;
    const double sd = (S(A_HD, jd) - (1.0 - dcol * (S(A_TD, k) - tmelt)) * rl * qd) / ((1.0 + cpvir * qd) * cp);
    S(A_SD, jd) = sd;
    S(A_TD, k) = sd - grav / ((1.0 + cpvir * qd) * cp) * S(A_ZF, k);
  }
  if (eps0 > 0.0) {
    const double small = 1.e-20;
    const int k0 = max(jd, msg + 2);
    WSYNC();
    PAR(k, msg + 2, pver) {
      if (k >= k0 && k < jb) {
        const double qdn = S(A_QDS, k + 1);
        const double qd = S(A_QDS, k);                      // qd(k): qd(jd) = qds(jd), qd(k>jd) = qds(k)
        S(A_QD, k + 1) = qdn;
        const double dz = S(A_DZ, k), ed = S(A_ED, k), md = S(A_MD, k);
        double ev = -ed * S(A_Q, k) + (md * qd - S(A_MD, k + 1) * qdn) / dz;
        ev = fmax2(ev, 0.0);
        S(A_EVP, k) = ev;
        S(A_W1, k) = ((1.0 - dcol * (S(A_TD, k) - tmelt)) * rl / ((1.0 + cpvir * qd) * cp) * ev - ed * S(A_S, k)) * dz;
        S(A_W2, k) = fmin2(S(A_MD, k + 1), -small);
        S(A_W4, k) = rcp_hot(fmin2(S(A_MD, k + 1), -small));
        S(A_W3, k) = dz * ed * S(A_Q, k);
      }
    }
    WSYNC();
    PH_MARK(PH_SD_PREP);
    // the next level's operands are loaded before this level's store
    double sdp = S(A_SD, k0);
    double w1 = S(A_W1, k0), md = S(A_MD, k0), w2 = S(A_W2, k0), w4 = S(A_W4, k0);
    for (int k = k0; k < jb; ++k) {
      const double w1n = S(A_W1, k + 1), mdn = S(A_MD, k + 1), w2n = S(A_W2, k + 1), w4n = S(A_W4, k + 1);
      const double w3 = S(A_W3, k);
      sdp = zmm::div_rcp(w1 + md * sdp, w2, w4);
      S(A_SD, k + 1) = sdp;
      totevp = totevp - w3;
      w1 = w1n; md = mdn; w2 = w2n; w4 = w4n;
    }
    PH_MARK(PH_SD);
  }
  totevp = totevp + S(A_MD, jd) * S(A_QD, jd) - S(A_MD, jb) * S(A_QD, jb);
  totpcp = fmax2(totpcp, 0.0);
  totevp = fmax2(totevp, 0.0);
  WSYNC();
  {
    const bool both = totevp > 0.0 && totpcp > 0.0;
    const double fac = both ? fmin2(1.0, totpcp / (totevp + totpcp)) : 0.0;
    PAR(k, msg + 2, pver) {
      double ev;
      if (both) {
        S(A_MD, k) = S(A_MD, k) * fac; S(A_ED, k) = S(A_ED, k) * fac; ev = S(A_EVP, k) * fac;
      } else {
        S(A_MD, k) = 0.0; S(A_ED, k) = 0.0; ev = 0.0;
      }
      S(A_EVP, k) = ev;
      S(A_CMEG, k) = S(A_CU, k) - ev;
      S(A_RPRD, k) = S(A_RPRD, k) - ev;
    }
  }
  WSYNC();
  {
    PAR(k, 1, pver) S(A_W1, k) = S(A_RPRD, k) * S(A_DZ, k);
    WSYNC();
    double pf = 0.0;
    S(A_PFLX, 1) = 0.0;
    double w = S(A_W1, 1);
    for (int k = 2; k <= pverp; ++k) {
      const double wn = S(A_W1, k);           // loaded before this level's store
      pf = pf + w;
      S(A_PFLX, k) = pf;
      w = wn;
    }
  }
  PAR(k, msg + 1, pver) S(A_MC, k) = S(A_MU, k) + S(A_MD, k);
  WSYNC();
  PH_MARK(PH_PFLX);
  R.jt = jt; R.j0 = j0; R.jlcl = jlcl; R.jd = jd;
  return R;
}

// leading dimension of the per-warp arrays for a given level count (levels 0..pver+1 are addressed)
inline int plume_ld(int pver) { return pver <= 32 ? 34 : (pver <= 64 ? 66 : 130); }
// Warps per block: shared memory bounds the residency of these kernels, and what is left over after the last
// whole block is wasted -- pick the block size that leaves the most warps resident per SM (227 KB, 1 KB reserved
// per block).  L32: 4 warps x 5 blocks = 20 warps; L58/L64: 1 warp x 10 blocks (4-warp blocks would hold 8).
inline int plume_warps_per_block(int pver, int narr = A_COUNT) {
  const size_t per_warp = (size_t)narr * plume_ld(pver) * sizeof(double), sm = 227 * 1024;
  int best = 1; size_t best_res = 0;
  for (int w = PL_WARPS; w >= 1; --w) {
    const size_t blocks = sm / (w * per_warp + 1024);
    const size_t res = (blocks > 32 ? 32 : blocks) * w;
    if (res > best_res) { best_res = res; best = w; }
  }
  return best;
}
inline size_t plume_smem_bytes(int pver, int narr = A_COUNT) {
  return (size_t)plume_warps_per_block(pver, narr) * narr * plume_ld(pver) * sizeof(double);
}

// ---- pass-1 plume: diagnose the pass-2 test-parcel entrainment rate (zm_conv.F90:1047-1078) ---
template <int LD>
__global__ void __launch_bounds__(32 * PL_WARPS)
k_cldprp_pass1_w(ConvrIn in, ConvrWork w) {
  extern __shared__ double sm_pl[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int gw = blockIdx.x * (blockDim.x >> 5) + wib;
  if (gw >= w.count[0]) return;
  const int col = w.wl1[gw];
  const int pcols = P.pcols, pver = P.pver, msg = P.msg;
  const int c = col / pcols, i = col - c * pcols;
  const PlumeShT<LD> S{sm_pl + (size_t)wib * A_FRONT_COUNT * LD};     // the front arrays only
  const int maxg = w.mx[col];
  PH_BEGIN(0);
  PH_COLUMN();
  gather_column_w(S, in, c, i, maxg, lane);
  PH_MARK(PH_GATHER);
  cldprp_warp<false>(S, maxg, w.lel[col], in.landfrac[(size_t)c * pcols + i], lane);
  PH_RESTART();
  double hk = 0.0, dmmx = 0.0, dmsm = 0.0;
  const double orgc = 1.0;
  double dm = -1.0;
  for (int k = pver; k >= msg + 1; --k) {
    const double eu = S(A_EU, k);
    if (eu > 0.0) {
      dmmx = -fmax2(-dmmx, eu);
      dmsm = dmsm - eu;
      hk = hk + 1.0;
    }
  }
  if (hk > 0.0) {
    dmsm = dmsm / hk;
    dm = dmsm * orgc + dmmx * (1.0 - orgc);
  }
  if (lane == 0) w.dmpdz[col] = dm;
  PH_MARK(PH_EU_SCAN);
}

// ---- final plume: cldprp #2 + closure + limiter + q1q2 + scatter + prec -----------------------
template <int LD>
__global__ void __launch_bounds__(32 * PL_WARPS)
k_plume_w(ConvrIn in, ConvrOut o, ConvrWork w) {
  extern __shared__ double sm_pl[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int gw = blockIdx.x * (blockDim.x >> 5) + wib;
  if (gw >= w.count[1]) return;
  const int col = w.wl2[2 * gw], slot = w.wl2[2 * gw + 1];
  const int pcols = P.pcols, pver = P.pver, pverp = P.pverp, msg = P.msg;
  const int ncolpad = in.nchunks * pcols;
  const int c = col / pcols, i = col - c * pcols;      // ungathered position
  const int gi = slot - c * pcols;                     // gathered position (0-based)
  const double eps1 = P.eps1, rl = P.rl, rd = P.rgas, grav = P.grav, cp = P.cpres;
  const double delt = in.delt;
  const PlumeShT<LD> S{sm_pl + (size_t)wib * A_COUNT * LD};
  const int maxg = w.mx[col], lel = w.lel[col], lcl = w.lcl[col];
  const double capeg = w.cape[col], tlg = w.tl[col];
  const double landfrac = in.landfrac[(size_t)c * pcols + i];
  PH_BEGIN(1);
  PH_COLUMN();
  const double dsubcld = gather_column_w(S, in, c, i, maxg, lane);
  PH_MARK(PH_GATHER);
  const PlumeIdx R = cldprp_warp<true>(S, maxg, lel, landfrac, lane);
  PH_RESTART();
  const int jt = R.jt, mx = maxg;
  const double dmpdz = w.dmpdz[col];

  // 1/m -> 1/mb (zm_conv.F90:1252-1262)
  PAR(k, msg + 1, pver) {
    const double dzf = S(A_ZF, k) - S(A_ZF, k + 1), dp = S(A_DP, k);
    S(A_DU, k) = div_z(S(A_DU, k) * dzf, dp);
    S(A_EU, k) = div_z(S(A_EU, k) * dzf, dp);
    S(A_ED, k) = div_z(S(A_ED, k) * dzf, dp);
    S(A_CU, k) = div_z(S(A_CU, k) * dzf, dp);
    S(A_CMEG, k) = div_z(S(A_CMEG, k) * dzf, dp);
    S(A_RPRD, k) = div_z(S(A_RPRD, k) * dzf, dp);
    S(A_EVP, k) = div_z(S(A_EVP, k) * dzf, dp);
  }
  WSYNC();

  // ---- closure (zm_conv.F90:4028-4260) ----
  double mb = 0.0;
  {
    const double q_mx = S(A_Q, mx), t_mx = S(A_T, mx), p_mx = S(A_P, mx);
    const double eb = p_mx * q_mx / (eps1 + q_mx);
    const double dtbdt = (1.0 / dsubcld) * (S(A_MU, mx) * (S(A_SHAT, mx) - S(A_SU, mx)) + S(A_MD, mx) * (S(A_SHAT, mx) - S(A_SD, mx)));
    const double dqbdt = (1.0 / dsubcld) * (S(A_MU, mx) * (S(A_QHAT, mx) - S(A_QU, mx)) + S(A_MD, mx) * (S(A_QHAT, mx) - S(A_QD, mx)));
    const double epq = eps1 + q_mx;
    const double debdt = eps1 * p_mx / (epq * epq) * dqbdt;
    const double den = 3.5 * zmm::log_(t_mx) - zmm::log_(eb) - 4.805;
    const double dtldt = -2840.0 * (3.5 / t_mx * dtbdt - debdt / eb) / (den * den);
    const double beta = 0.0;
    // W1 = dboydt(k) * (zf(k)-zf(k+1)) term inputs: compute dtmdt/dqmdt and dboydt level parallel
    PAR(k, msg + 1, pver) {
      double dtmdt = 0.0, dqmdt = 0.0;
      if (k <= pver - 1) {
        if (k == jt) {
          dqmdt = (1.0 / S(A_DP, k)) * (S(A_MU, k + 1) * (S(A_QU, k + 1) - S(A_QHAT, k + 1) + S(A_QL, k + 1)) +
                                        S(A_MD, k + 1) * (S(A_QD, k + 1) - S(A_QHAT, k + 1)));
          dtmdt = (1.0 / S(A_DP, k)) * (S(A_MU, k + 1) * (S(A_SU, k + 1) - S(A_SHAT, k + 1) - rl / cp * S(A_QL, k + 1)) +
                                        S(A_MD, k + 1) * (S(A_SD, k + 1) - S(A_SHAT, k + 1)));
        }
        if (k > jt && k < mx) {
          const double sk = S(A_S, k);
          dtmdt = (S(A_MC, k) * (S(A_SHAT, k) - sk) - S(A_MC, k + 1) * (S(A_SHAT, k + 1) - sk)) / S(A_DP, k) -
                  rl / cp * S(A_DU, k) * (beta * S(A_QL, k) + (1 - beta) * S(A_QL, k + 1));
          dqmdt = (S(A_MU, k + 1) * (S(A_QU, k + 1) - S(A_QHAT, k + 1) + cp / rl * (S(A_SU, k + 1) - sk)) -
                   S(A_MU, k) * (S(A_QU, k) - S(A_QHAT, k) + cp / rl * (S(A_SU, k) - sk)) +
                   S(A_MD, k + 1) * (S(A_QD, k + 1) - S(A_QHAT, k + 1) + cp / rl * (S(A_SD, k + 1) - sk)) -
                   S(A_MD, k) * (S(A_QD, k) - S(A_QHAT, k) + cp / rl * (S(A_SD, k) - sk))) / S(A_DP, k) +
                  S(A_DU, k) * (beta * S(A_QL, k) + (1 - beta) * S(A_QL, k + 1));
        }
      }
      double dboydt = 0.0;
      // parcel temperature / humidity of the final CAPE pass, straight from the scratch arrays
      const double tpk = w.tp[(size_t)(k - 1) * ncolpad + col], qstpk = w.qstp[(size_t)(k - 1) * ncolpad + col];
      const double tk = S(A_T, k), qk = S(A_Q, k);
      if (k >= lel && k <= lcl) {
        const double pw = zmm::pow_(1000.0 / S(A_P, k), rd / cp);
        const double thetavp = tpk * pw * (1.0 + 1.608 * qstpk - q_mx);
        const double thetavm = tk * pw * (1.0 + 0.608 * qk);
        const double dqsdtp = qstpk * (1.0 + qstpk / eps1) * eps1 * rl / (rd * (tpk * tpk));
        const double dtpdt = tpk / (1.0 + rl / cp * (dqsdtp - qstpk / tpk)) *
                             (dtbdt / t_mx + rl / cp * (dqbdt / tlg - q_mx / (tlg * tlg) * dtldt));
        dboydt = ((dtpdt / tpk + 1.0 / (1.0 + 1.608 * qstpk - q_mx) * (1.608 * dqsdtp * dtpdt - dqbdt)) -
                  (dtmdt / tk + 0.608 / (1.0 + 0.608 * qk) * dqmdt)) * grav * thetavp / thetavm;
      }
      if (k > lcl && k < mx) {
        const double pw = zmm::pow_(1000.0 / S(A_P, k), rd / cp);
        const double thetavp = tpk * pw * (1.0 + 0.608 * q_mx);
        const double thetavm = tk * pw * (1.0 + 0.608 * qk);
        dboydt = (dtbdt / t_mx + 0.608 / (1.0 + 0.608 * q_mx) * dqbdt - dtmdt / tk -
                  0.608 / (1.0 + 0.608 * qk) * dqmdt) * grav * thetavp / thetavm;
      }
      S(A_W1, k) = dboydt * (S(A_ZF, k) - S(A_ZF, k + 1));
    }
    WSYNC();
    double dadt = 0.0;
    for (int k = msg + 1; k <= pver; ++k)
      if (k >= lel && k <= mx - 1) dadt = dadt + S(A_W1, k);
    const double dltaa = -1.0 * (capeg - P.capelmt);
    if (dadt != 0.0) mb = fmax2(dltaa / P.tau / dadt, 0.0);
  }
  // mass-flux limiter (zm_conv.F90:1285-1308)
  {
    double mumax = 0.0;                        // max is exact in any order: lane-parallel + shuffle
    PAR(k, msg + 2, pver) mumax = fmax2(mumax, div_z(S(A_MU, k), S(A_DP, k)));
    for (int off = 16; off; off >>= 1) mumax = fmax2(mumax, __shfl_xor_sync(0xffffffffu, mumax, off));
    if (mumax > 0.0) mb = fmin2(mb, 0.5 / (delt * mumax));
    else mb = 0.0;
    if (P.no_deep_pbl)
      if (in.zm[cidx(c, jt - 1, i, pver)] < in.pblh[(size_t)c * pcols + i]) mb = 0.0;
  }
  WSYNC();
  PAR(k, msg + 1, pver) {
    S(A_MU, k) = S(A_MU, k) * mb; S(A_MD, k) = S(A_MD, k) * mb; S(A_MC, k) = S(A_MC, k) * mb;
    S(A_DU, k) = S(A_DU, k) * mb; S(A_EU, k) = S(A_EU, k) * mb; S(A_ED, k) = S(A_ED, k) * mb;
    S(A_CMEG, k) = S(A_CMEG, k) * mb; S(A_RPRD, k) = S(A_RPRD, k) * mb; S(A_CU, k) = S(A_CU, k) * mb;
    S(A_EVP, k) = S(A_EVP, k) * mb;
    S(A_PFLX, k + 1) = div_z(S(A_PFLX, k + 1) * mb * 100.0, grav);
  }
  WSYNC();
  PH_MARK(PH_CLOSURE);

  // ---- q1q2_pjr (zm_conv.F90:4262-4421): dsdt -> W1, dqdt -> W2, dl -> W3 ----
  PAR(k, msg + 1, pver) {
    double dsdt = 0.0, dqdt = 0.0, dl = 0.0;
    if (k <= pver - 1) {
      const double emc = -S(A_CU, k) + S(A_EVP, k);
      dsdt = -rl / cp * emc + div_z(S(A_MU, k + 1) * (S(A_SU, k + 1) - S(A_SHAT, k + 1)) - S(A_MU, k) * (S(A_SU, k) - S(A_SHAT, k)) +
                                    S(A_MD, k + 1) * (S(A_SD, k + 1) - S(A_SHAT, k + 1)) - S(A_MD, k) * (S(A_SD, k) - S(A_SHAT, k)), S(A_DP, k));
      dqdt = emc + div_z(S(A_MU, k + 1) * (S(A_QU, k + 1) - S(A_QHAT, k + 1)) - S(A_MU, k) * (S(A_QU, k) - S(A_QHAT, k)) +
                         S(A_MD, k + 1) * (S(A_QD, k + 1) - S(A_QHAT, k + 1)) - S(A_MD, k) * (S(A_QD, k) - S(A_QHAT, k)), S(A_DP, k));
      dl = S(A_DU, k) * S(A_QCDE, k + 1);
    }
    S(A_W1, k) = dsdt; S(A_W2, k) = dqdt; S(A_W3, k) = dl;
  }
  WSYNC();
  {
    const double dsb = (1.0 / dsubcld) * (-S(A_MU, mx) * (S(A_SU, mx) - S(A_SHAT, mx)) - S(A_MD, mx) * (S(A_SD, mx) - S(A_SHAT, mx)));
    const double dqb = (1.0 / dsubcld) * (-S(A_MU, mx) * (S(A_QU, mx) - S(A_QHAT, mx)) - S(A_MD, mx) * (S(A_QD, mx) - S(A_QHAT, mx)));
    WSYNC();
    PAR(k, msg + 1, pver) {
      if (k >= mx) { S(A_W1, k) = dsb; S(A_W2, k) = dqb; }
    }
  }
  WSYNC();
  PH_MARK(PH_Q1Q2);
  // scatter to the ungathered column i of chunk c (zm_conv.F90:1495-1511, 1616-1620)
  PAR(k, msg + 1, pver) {
    const size_t e = cidx(c, k - 1, i, pver);
    o.qtnd[e] = S(A_W2, k);
    o.cme[e] = S(A_CMEG, k);
    o.rprd[e] = S(A_RPRD, k);
    o.zdu[e] = S(A_DU, k);
    o.heat[e] = S(A_W1, k) * P.cpres;
    o.dlf[e] = S(A_W3, k);
    o.ql[e] = S(A_QL, k);
    if (o.eurt) o.eurt[e] = -dmpdz;
    const size_t ep = cidx(c, k - 1, i, pverp);
    o.mcon[ep] = o.mcon_kgm2s ? div_z(S(A_MC, k) * 100.0, P.gravit) : S(A_MC, k);
    o.pflx[ep] = S(A_PFLX, k);
  }
  // gathered outputs at gathered position gi of chunk c
  PAR(k, 1, pver) {
    const size_t e = cidx(c, k - 1, gi, pver);
    o.mu[e] = S(A_MU, k); o.md[e] = S(A_MD, k); o.du[e] = S(A_DU, k); o.eu[e] = S(A_EU, k); o.ed[e] = S(A_ED, k);
    o.dp[e] = S(A_DP, k);
  }
  // precipitation and reserved liquid (zm_conv.F90:1629-1649), serial sums in the reference's order
  double prec = 0.0, rliq = 0.0;
  WSYNC();
  PAR(k, 1, pver) {
    const double dppk = in.dpp[cidx(c, k - 1, i, pver)], qhk = S(A_Q, k);
    const double dlfk = (k >= msg + 1) ? S(A_W3, k) : 0.0;
    const double qnew = qhk + 2.0 * delt * ((k >= msg + 1) ? S(A_W2, k) : 0.0);
    S(A_W4, k) = dppk * (qnew - qhk);
    S(A_W5, k) = dppk * (dlfk + 0.0) * 2.0 * delt;
    S(A_W1, k) = div_z((dlfk + 0.0) * dppk, P.gravit);
  }
  WSYNC();
  for (int k = pver; k >= msg + 1; --k) prec = prec - S(A_W4, k) - S(A_W5, k);
  prec = P.rgrav * fmax2(prec, 0.0) / (2.0 * delt) / 1000.0;
  for (int k = 1; k <= pver; ++k) rliq = rliq + S(A_W1, k);
  rliq = rliq / 1000.0;
  if (lane == 0) {
    o.pflx[cidx(c, pverp - 1, i, pverp)] = S(A_PFLX, pverp);
    o.prec[(size_t)c * pcols + i] = prec;
    o.rliq[(size_t)c * pcols + i] = rliq;
    o.jctop[(size_t)c * pcols + i] = (double)jt;
    o.jcbot[(size_t)c * pcols + i] = (double)maxg;
    o.dsubcld[(size_t)c * pcols + gi] = dsubcld;
    o.jt[(size_t)c * pcols + gi] = jt;
    o.maxg[(size_t)c * pcols + gi] = maxg;
  }
  PH_MARK(PH_SCATTER);
}
#undef PAR
#undef WSYNC
