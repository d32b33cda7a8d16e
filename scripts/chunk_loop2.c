/* Loop 2 of the batched binding's split chunk loop (fortran/zm_conv_intr_batched.F90, zm_batch_scatter), reduced to
 * the twenty (pcols,pver[p]) outputs of zm_conv_tend: what the host does with them after the step, in the two return
 * forms.  Built at run time by scripts/tend_gathered_cost.py (gcc -O2 -fopenmp -shared) and loaded through ctypes.
 *
 * A chunk's outputs go to a chunk buffer of the twenty fields back to back, each (pcols,nlev) column-major as
 * ptend_all and the dummy outputs are ([k][i] in C terms), in the record order of zm_conv_tend_batch_gathered:
 * ptend_s ptend_q ptend_u ptend_v cme zdu ql rprd evapcdp dlf (pver), mcon pflx flxprec flxsnow (pver+1),
 * mu md du eu ed dp (pver; rows = gathered slots).  dst_stride = 0: every thread reuses one chunk buffer of its own
 * (dst + thread * chunk size), which stays in cache as the model's chunk-local ptend does; dst_stride > 0: chunk c
 * goes to dst + c * dst_stride (to check the result). */
#include <omp.h>
#include <string.h>

#define NF 20
#define NCOL_FIELDS 14

static int nlev_of(int f, int pver) { return (f >= 10 && f < 14) ? pver + 1 : pver; }
static long long chunk_doubles(int pcols, int pver) { return (long long)pcols * (20 * pver + 4); }

/* dense: copy the chunk's slices of the twenty rank-level arrays (fields[f] is [nchunks][nlev][pcols]) */
void loop2_dense(int nthreads, int nchunks, int pcols, int pver, const double* const* fields, double* dst,
                 long long dst_stride) {
  const long long cd = chunk_doubles(pcols, pver);
#pragma omp parallel for num_threads(nthreads) schedule(static)
  for (int c = 0; c < nchunks; ++c) {
    double* b = dst + (dst_stride ? (long long)c * dst_stride : (long long)omp_get_thread_num() * cd);
    for (int f = 0; f < NF; ++f) {
      const long long n = (long long)pcols * nlev_of(f, pver);
      memcpy(b, fields[f] + (long long)c * n, (size_t)n * sizeof(double));
      b += n;
    }
  }
}

/* gathered: zero the chunk buffer, then scatter the chunk's records (rec_len = 20 pver + 4 with the pbuf fields,
 * 14 pver + 4 without; then the pbuf fields of the chunk buffer stay 0) */
void loop2_gathered(int nthreads, int nchunks, int pcols, int pver, int with_pbuf, const int* lengath,
                    const int* ideep, const double* rec, double* dst, long long dst_stride) {
  const long long cd = chunk_doubles(pcols, pver);
  const int rec_len = (with_pbuf ? 20 : 14) * pver + 4, nf = with_pbuf ? NF : NCOL_FIELDS;
#pragma omp parallel num_threads(nthreads)
  {
    /* chunk c's first record: the exclusive prefix of lengath, as the binding keeps it in rec_base_b */
    long long base = 0;
    int next = 0;
#pragma omp for schedule(static)
    for (int c = 0; c < nchunks; ++c) {
      for (; next < c; ++next) base += lengath[next];
      double* b = dst + (dst_stride ? (long long)c * dst_stride : (long long)omp_get_thread_num() * cd);
      memset(b, 0, (size_t)cd * sizeof(double));
      for (int j = 0; j < lengath[c]; ++j) {
        const double* r = rec + (base + j) * rec_len;
        const int i = ideep[(long long)c * pcols + j] - 1;
        double* fb = b;
        for (int f = 0; f < nf; ++f) {
          const int nl = nlev_of(f, pver), col = f < NCOL_FIELDS ? i : j;
          for (int k = 0; k < nl; ++k) fb[(long long)k * pcols + col] = r[k];
          r += nl;
          fb += (long long)pcols * nl;
        }
      }
    }
  }
}
