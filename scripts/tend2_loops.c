/* The host loops around zm_conv_tend_2 in the batched binding (fortran/zm_conv_intr_batched.F90), in the two forms:
 * loop 1 (zm_batch_gather_2) before the call and loop 2 (zm_batch_scatter_2) after it.  Built at run time by
 * scripts/tend2_gathered_cost.py (gcc -O2 -fopenmp -shared) and loaded through ctypes.
 *
 * Chunk arrays are [chunk][m][k][i] in C terms, as state%q / fracis / ptend%q are (pcols,pver,pcnst) per chunk;
 * pdeldry is [chunk][k][i].  iact[nact] are the 0-based flagged constituents, ascending.  Records: chunk c's block of
 * q_rec / fracis_rec / dqdt_rec at nact*pver*base(c) is g(n, pver, nact) in Fortran order, pdeldry_rec's at
 * pver*base(c), base(c) = sum(lengath(1:c-1)).
 * Loop 2 starts, in both forms, with physics_ptend_init's zero-fill of the chunk's ptend%q.  dst_stride = 0: every
 * thread reuses one chunk ptend buffer of its own (dst + thread * chunk size), which stays in cache as the model's
 * chunk-local ptend does; dst_stride > 0: chunk c goes to dst + c * dst_stride (to check the result). */
#include <omp.h>
#include <string.h>

/* dense loop 1: the chunk's q, fracis, pdeldry whole into the rank-level arrays, and the chunk's slice of the
 * rank-level ptend_q zeroed (ptend_q3_b = 0 before the call) */
void loop1_dense(int nthreads, int nchunks, int pcols, int pver, int pcnst, const double* q, const double* fracis,
                 const double* pdeldry, double* q_b, double* fracis_b, double* pdeldry_b, double* ptend_q_b) {
  const long long n3 = (long long)pcols * pver * pcnst, n2 = (long long)pcols * pver;
#pragma omp parallel for num_threads(nthreads) schedule(static)
  for (int c = 0; c < nchunks; ++c) {
    memcpy(q_b + c * n3, q + c * n3, (size_t)n3 * sizeof(double));
    memcpy(fracis_b + c * n3, fracis + c * n3, (size_t)n3 * sizeof(double));
    memcpy(pdeldry_b + c * n2, pdeldry + c * n2, (size_t)n2 * sizeof(double));
    memset(ptend_q_b + c * n3, 0, (size_t)n3 * sizeof(double));
  }
}

/* gathered loop 1: pack the chunk's convective columns ideep(1:n) of the flagged constituents; pdeldry_rec NULL: no
 * flagged constituent is dry and pdeldry does not travel */
void loop1_gathered(int nthreads, int nchunks, int pcols, int pver, int pcnst, int nact, const int* iact,
                    const int* lengath, const int* ideep, const double* q, const double* fracis, const double* pdeldry,
                    double* q_rec, double* fracis_rec, double* pdeldry_rec) {
  const long long n3 = (long long)pcols * pver * pcnst, n2 = (long long)pcols * pver;
#pragma omp parallel num_threads(nthreads)
  {
    long long base = 0;              /* chunk c's first record column, as the binding keeps it in rec_base_b */
    int next = 0;
#pragma omp for schedule(static)
    for (int c = 0; c < nchunks; ++c) {
      for (; next < c; ++next) base += lengath[next];
      const int n = lengath[c];
      const int* id = ideep + (long long)c * pcols;
      double* qd = q_rec + (long long)nact * pver * base;
      double* fd = fracis_rec + (long long)nact * pver * base;
      for (int a = 0; a < nact; ++a)
        for (int k = 0; k < pver; ++k) {
          const long long s = c * n3 + ((long long)iact[a] * pver + k) * pcols;
          for (int i = 0; i < n; ++i) { qd[i] = q[s + id[i] - 1]; fd[i] = fracis[s + id[i] - 1]; }
          qd += n; fd += n;
        }
      if (pdeldry_rec) {
        double* pd = pdeldry_rec + (long long)pver * base;
        for (int k = 0; k < pver; ++k, pd += n)
          for (int i = 0; i < n; ++i) pd[i] = pdeldry[c * n2 + (long long)k * pcols + id[i] - 1];
      }
    }
  }
}

/* dense loop 2: zero the chunk's ptend%q, copy the flagged slices of the rank-level ptend_q */
void loop2_dense(int nthreads, int nchunks, int pcols, int pver, int pcnst, int nact, const int* iact,
                 const double* ptend_q_b, double* dst, long long dst_stride) {
  const long long n3 = (long long)pcols * pver * pcnst, n2 = (long long)pcols * pver;
#pragma omp parallel for num_threads(nthreads) schedule(static)
  for (int c = 0; c < nchunks; ++c) {
    double* b = dst + (dst_stride ? (long long)c * dst_stride : (long long)omp_get_thread_num() * n3);
    memset(b, 0, (size_t)n3 * sizeof(double));
    for (int a = 0; a < nact; ++a)
      memcpy(b + iact[a] * n2, ptend_q_b + c * n3 + iact[a] * n2, (size_t)n2 * sizeof(double));
  }
}

/* gathered loop 2: zero the chunk's ptend%q, scatter the chunk's records into columns ideep(1:n) */
void loop2_gathered(int nthreads, int nchunks, int pcols, int pver, int pcnst, int nact, const int* iact,
                    const int* lengath, const int* ideep, const double* dqdt_rec, double* dst, long long dst_stride) {
  const long long n3 = (long long)pcols * pver * pcnst;
#pragma omp parallel num_threads(nthreads)
  {
    long long base = 0;
    int next = 0;
#pragma omp for schedule(static)
    for (int c = 0; c < nchunks; ++c) {
      for (; next < c; ++next) base += lengath[next];
      double* b = dst + (dst_stride ? (long long)c * dst_stride : (long long)omp_get_thread_num() * n3);
      memset(b, 0, (size_t)n3 * sizeof(double));
      const int n = lengath[c];
      const int* id = ideep + (long long)c * pcols;
      const double* r = dqdt_rec + (long long)nact * pver * base;
      for (int a = 0; a < nact; ++a)
        for (int k = 0; k < pver; ++k, r += n) {
          double* row = b + ((long long)iact[a] * pver + k) * pcols;
          for (int i = 0; i < n; ++i) row[id[i] - 1] = r[i];
        }
    }
  }
}
