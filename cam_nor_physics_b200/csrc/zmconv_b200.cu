// zmconv_b200.cu -- C ABI (include/zmconv_b200.h) over the sm_100a kernels.
// Replaces module zm_conv's public procedures (reference physics/zm_conv.F90:33-37) as called from
// physics/zm_conv_intr.F90:376-379, 662-673, 764-769, 822-826, 875-879, 1020-1024.
// Host side: per-thread workspaces (device arena + stream), no global mutable state after
// zm_init => re-entrant from OpenMP threads like the reference (physpkg.F90:1147-1161).
#include "../../include/zmconv_b200.h"
#include "zm_plume_warp.cuh"
#include "zm_transport.cuh"
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <vector>
#include <algorithm>
#include <string>
#include <mutex>
#include <chrono>
#include <thread>
#include <condition_variable>
#include <functional>
#include <atomic>
#include <deque>

namespace {

zm_params_t g_params;
bool g_inited = false;
std::mutex g_mu;
thread_local std::string tls_err;
thread_local long long tls_launches = 0;
bool g_profile = false;

#define CK(call)                                                                          \
  do {                                                                                    \
    cudaError_t _e = (call);                                                              \
    if (_e != cudaSuccess) {                                                              \
      char _b[512];                                                                       \
      snprintf(_b, sizeof _b, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(_e),      \
               __FILE__, __LINE__, #call);                                                \
      tls_err = _b;                                                                       \
      return -100;                                                                        \
    }                                                                                     \
  } while (0)
#define NEED_INIT()                                                         \
  do {                                                                      \
    if (!g_inited) { tls_err = "zm_init has not been called"; return -1; }  \
  } while (0)

struct Workspace {
  cudaStream_t stream = nullptr;
  char* dbuf = nullptr; size_t dcap = 0, dtop = 0;
  std::vector<const char*> tnames;
  std::vector<cudaEvent_t> tev;
  int* last_count = nullptr;          // device: [0]=n pass-1, [1]=n final, [2]=brent failures
  double* last_err = nullptr;
  int chunk0 = 0;                     // first chunk of this arena's (sub-)batch, for error messages
  cudaStream_t side = nullptr;        // zm_conv_evap runs here, concurrently with momtran
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaStream_t side2 = nullptr;       // convtran1 runs here, concurrently with momtran and zm_conv_evap
  cudaEvent_t ev_fork2 = nullptr, ev_join2 = nullptr;
  int side_priority = 0; bool side_priority_set = false;
  int ensure_side() {
    if (!side) {
      if (side_priority_set) CK(cudaStreamCreateWithPriority(&side, cudaStreamNonBlocking, side_priority));
      else CK(cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking));
    }
    if (!ev_fork) CK(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
    if (!ev_join) CK(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
    return 0;
  }
  int ensure_side2() {
    if (side2) return 0;
    if (side_priority_set) CK(cudaStreamCreateWithPriority(&side2, cudaStreamNonBlocking, side_priority));
    else CK(cudaStreamCreateWithFlags(&side2, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ev_fork2, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ev_join2, cudaEventDisableTiming));
    return 0;
  }
  int ensure(size_t bytes) {
    if (!stream) CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    if (bytes > dcap) {
      if (dbuf) { CK(cudaDeviceSynchronize()); CK(cudaFree(dbuf)); dbuf = nullptr; dcap = 0; }
      size_t cap = bytes + (bytes >> 3) + (1u << 20);
      CK(cudaMalloc((void**)&dbuf, cap));
      dcap = cap;
    }
    dtop = 0;
    return 0;
  }
  void release() {                      // frees this arena's device memory, streams and events
    for (auto e : tev) cudaEventDestroy(e);
    tev.clear(); tnames.clear();
    if (dbuf) { cudaFree(dbuf); dbuf = nullptr; dcap = 0; dtop = 0; }
    if (ev_fork) { cudaEventDestroy(ev_fork); ev_fork = nullptr; }
    if (ev_join) { cudaEventDestroy(ev_join); ev_join = nullptr; }
    if (side) { cudaStreamDestroy(side); side = nullptr; }
    if (ev_fork2) { cudaEventDestroy(ev_fork2); ev_fork2 = nullptr; }
    if (ev_join2) { cudaEventDestroy(ev_join2); ev_join2 = nullptr; }
    if (side2) { cudaStreamDestroy(side2); side2 = nullptr; }
    if (stream) { cudaStreamDestroy(stream); stream = nullptr; }
    last_count = nullptr; last_err = nullptr;
  }
  template <class T> T* take(size_t n) {
    size_t b = (n * sizeof(T) + 255) & ~(size_t)255;
    T* p = (T*)(dbuf + dtop);
    dtop += b;
    return p;
  }
};
// Device-resident copy of the pbuf fields zm_conv_tend hands to zm_conv_tend_2 (ZM_MU..ZM_IDEEP,
// zm_conv_intr.F90:113-132, 994-1004): they live in an arena of their own (tls_mirror_ws, touched by nothing but
// zm_conv_tend_batch) until the calling thread's next zm_conv_tend_batch call, so convtran2 needs no second H2D
// of them and the calls the model makes in between (geopotential_t, convect_diagnostics_calc, physpkg.F90:2820-2885)
// cannot disturb them.  Set only when zm_conv_tend_batch succeeded; cleared on entry and on failure.
struct PbufMirror {
  int nchunks = 0;
  const double *mu = nullptr, *md = nullptr, *du = nullptr, *eu = nullptr, *ed = nullptr, *dp = nullptr, *dsubcld = nullptr;
  const int *jt = nullptr, *maxg = nullptr, *ideep = nullptr, *lengath = nullptr;
};
thread_local PbufMirror tls_mirror;
// zm_org = 1: the pointer dummies org / orgt / org2d of zm_convr (zm_conv.F90:421-423), attached per call
// with zm_org_fields (host pointers for the host-pointer entry points, device pointers for *_dev)
struct OrgFields { const double* org = nullptr; double* orgt = nullptr; double* org2d = nullptr; };
thread_local OrgFields tls_org;
// convtran1 of zm_conv_tend (zm_conv_intr.F90:865-880), attached per call with zm_convtran1_fields: state%q,
// fracis and ptend_loc%q, (pcols,pver,pcnst) per chunk (host or device pointers like zm_org_fields)
struct Tran1Fields { int pcnst = 0; const double* q = nullptr; const double* fracis = nullptr; double* ptend_q = nullptr; };
thread_local Tran1Fields tls_tran1;
struct Tran1Dev { int ncnst, nactive; const int* active; const int* is_dry; bool any_dry;
                  const double* q; const double* fracis; double* dqdt; };
// zm_conv_tend's history fields (zm_conv_intr.F90:676-857), attached per call with zm_conv_tend_hist_fields (host or
// device pointers like zm_org_fields): the outputs of zm_convr, zm_conv_evap and momtran inside the step.  NULL =
// not materialised.  pguall, pgdall, icwu, icwd are (pcols,pver,2) per chunk, everything else (pcols,pver).
enum { H_HEAT, H_QTND, H_EURT, H_DIF, H_DNLF, H_DNIF,                  // zm_convr
       H_TEND_S, H_SNWPRD, H_SNWEVMLT, H_NTPRPRD, H_NTSNPRD,          // zm_conv_evap
       H_SETEN, H_PGUALL, H_PGDALL, H_ICWU, H_ICWD,                   // momtran
       H_N };
struct HistFields {
  double* p[H_N] = {};                   // argument order of zm_conv_tend_hist_fields
  static bool is3d(int j) { return j >= H_PGUALL; }
  bool any() const { for (int j = 0; j < H_N; ++j) if (p[j]) return true; return false; }
  // the sub-batch that starts at chunk c0 (s2 = pcols*pver)
  HistFields slice(size_t c0, size_t s2) const {
    HistFields h = *this;
    for (int j = 0; j < H_N; ++j)
      if (h.p[j]) h.p[j] += c0 * s2 * (is3d(j) ? 2 : 1);
    return h;
  }
};
thread_local HistFields tls_hist;
thread_local Workspace tls_work;     // kernel work arrays
thread_local Workspace tls_stage;    // device staging of user arrays for the host-pointer API
thread_local Workspace tls_stage2;   // staging for zm_conv_tend_2_batch
// bytes the thread's last zm_conv_tend_2_batch[_gathered] moved over PCIe (zm_tend_2_transfer_bytes)
thread_local long long tls_t2_h2d = 0, tls_t2_d2h = 0;
thread_local Workspace tls_mirror_ws; // the device pbuf mirror (see PbufMirror)

// Host worker threads of the sparse return path (zero-fill of the caller's dense output arrays while the GPU works,
// then the scatter of the convective columns' records): ZM_HOST_THREADS, default min(8, hardware threads).
class HostPool {
 public:
  explicit HostPool(int n) {
    for (int i = 0; i < n; ++i) th_.emplace_back([this] { run(); });
  }
  ~HostPool() {
    { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }
    cv_.notify_all();
    for (auto& t : th_) t.join();
  }
  int size() const { return (int)th_.size(); }
  void submit(std::function<void()> f) {
    { std::lock_guard<std::mutex> lk(mu_); q_.push_back(std::move(f)); ++pending_; }
    cv_.notify_one();
  }
  void wait_all() {
    std::unique_lock<std::mutex> lk(mu_);
    done_.wait(lk, [this] { return pending_ == 0; });
  }
 private:
  void run() {
    for (;;) {
      std::function<void()> f;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [this] { return stop_ || !q_.empty(); });
        if (stop_ && q_.empty()) return;
        f = std::move(q_.front()); q_.pop_front();
      }
      f();
      { std::lock_guard<std::mutex> lk(mu_); if (--pending_ == 0) done_.notify_all(); }
    }
  }
  std::vector<std::thread> th_;
  std::deque<std::function<void()>> q_;
  std::mutex mu_;
  std::condition_variable cv_, done_;
  int pending_ = 0;
  bool stop_ = false;
};
HostPool& host_pool() {
  static HostPool* pool = [] {
    int n = 0;
    if (const char* e = getenv("ZM_HOST_THREADS")) n = atoi(e);
    if (n <= 0) { n = (int)std::thread::hardware_concurrency(); n = n > 8 ? 8 : (n < 1 ? 1 : n); }
    return new HostPool(n > 64 ? 64 : n);
  }();
  return *pool;
}

// Sparse return of zm_conv_tend_batch: the 2-D outputs are zero outside the convective columns (zm_conv.F90:559-563,
// 625-650; zm_conv_evap and momtran add nothing where zm_convr produced no rain and no mass flux), so only the
// convective columns' levels travel device -> host, as one record per column, and worker threads scatter them into
// the caller's arrays, which they zero-filled while the GPU was busy.  Field order of a record:
enum { SF_PS, SF_PQ, SF_PU, SF_PV, SF_CME, SF_ZDU, SF_QL, SF_RPRD, SF_EVAP, SF_DLF,     // (pcols,pver), by column
       SF_MCON, SF_PFLX, SF_FP, SF_FS,                                                   // (pcols,pverp), by column
       SF_MU, SF_MD, SF_DU, SF_EU, SF_ED, SF_DP,                                         // (pcols,pver), by gathered slot
       SF_N };
struct SparseFields {
  const double* d[SF_N];     // device arrays (sub-batch slice), NULL = not packed
  int off[SF_N];             // offset of the field inside a record (doubles), -1 = absent
  int rec_len;               // doubles per record
};
// zm_conv_tend_batch_gathered: the same records go straight to the caller, who scatters them in its own chunk loop
struct GatheredOut {
  double* rec;               // caller's record buffer (capacity checked by the entry point)
  bool pbuf;                 // the slot-indexed pbuf fields mu..dp are part of the records
};
// exclusive prefix of lengath over the chunks of a sub-batch (one block): base[c], total in base[nchunks]
__global__ void k_lengath_scan(int nchunks, const int* lengath, int* base) {
  __shared__ int part[1024];
  const int t = threadIdx.x, per = (nchunks + blockDim.x - 1) / blockDim.x;
  const int lo = min(t * per, nchunks), hi = min(lo + per, nchunks);
  int sum = 0;
  for (int c = lo; c < hi; ++c) sum += lengath[c];
  part[t] = sum;
  __syncthreads();
  if (t == 0) {
    int acc = 0;
    for (int i = 0; i < blockDim.x; ++i) { const int v = part[i]; part[i] = acc; acc += v; }
    base[nchunks] = acc;
  }
  __syncthreads();
  int acc = part[t];
  for (int c = lo; c < hi; ++c) { base[c] = acc; acc += lengath[c]; }
}
// one block per (chunk, gathered slot): the column's record
__global__ void __launch_bounds__(64) k_pack_records(int nchunks, const int* lengath, const int* ideep, const int* base,
                                                     SparseFields f, double* rec) {
  const int pcols = P.pcols, pver = P.pver;
  const int c = blockIdx.x / pcols, slot = blockIdx.x - c * pcols;
  if (c >= nchunks || slot >= lengath[c]) return;
  const int i = ideep[(size_t)c * pcols + slot] - 1;
  double* r = rec + (size_t)(base[c] + slot) * f.rec_len;
#pragma unroll
  for (int q = 0; q < SF_N; ++q) {
    if (f.off[q] < 0) continue;
    const int nlev = (q >= SF_MCON && q <= SF_FS) ? pver + 1 : pver;
    for (int k = threadIdx.x; k < nlev; k += blockDim.x)
      r[f.off[q] + k] = f.d[q][cidx(c, k, q >= SF_MU ? slot : i, nlev)];
  }
}

// Streams, events and per-sub-batch work arenas of the pipelined host-pointer zm_conv_tend_batch.
struct TendPipe {
  static const int MAXB = 8;
  Workspace work[MAXB];
  cudaStream_t h2d = nullptr, d2h_early = nullptr, d2h_final = nullptr;
  cudaEvent_t in_ready[MAXB] = {}, late_ready[MAXB] = {}, convr_done[MAXB] = {}, done[MAXB] = {};
  cudaEvent_t early_back[MAXB] = {}, final_back[MAXB] = {}, t0 = nullptr;   // timeline of the last call (zm_tend_trace)
  int ninit = 0, last_nb = 0, dev_nb = 0;
  // sparse return: pinned host staging of the records and of the per-sub-batch (lengath, ideep, count) triple
  cudaEvent_t small_back[MAXB] = {}, rec_back[MAXB] = {};
  double* h_rec = nullptr; size_t h_rec_cap = 0;       // doubles
  int* h_small = nullptr; size_t h_small_cap = 0;      // ints
  long long last_h2d = 0, last_d2h = 0;                // bytes moved by the last call (zm_tend_transfer_bytes)
  int ensure_pinned(size_t rec_doubles, size_t small_ints) {
    if (rec_doubles > h_rec_cap) {
      if (h_rec) { CK(cudaDeviceSynchronize()); CK(cudaFreeHost(h_rec)); h_rec = nullptr; }
      h_rec_cap = rec_doubles + (rec_doubles >> 2) + 1024;
      CK(cudaHostAlloc((void**)&h_rec, h_rec_cap * sizeof(double), cudaHostAllocDefault));
    }
    if (small_ints > h_small_cap) {
      if (h_small) { CK(cudaDeviceSynchronize()); CK(cudaFreeHost(h_small)); h_small = nullptr; }
      h_small_cap = small_ints + 1024;
      CK(cudaHostAlloc((void**)&h_small, h_small_cap * sizeof(int), cudaHostAllocDefault));
    }
    return 0;
  }
  // ZM_TEND_SUBBATCHES (1..8, default 8); a sub-batch is never smaller than 128 chunks
  int subbatches(int nchunks) const {
    int nb = 8;
    if (const char* e = getenv("ZM_TEND_SUBBATCHES")) nb = atoi(e);
    nb = nb < 1 ? 1 : (nb > MAXB ? MAXB : nb);
    while (nb > 1 && nchunks / nb < 128) --nb;
    return nb;
  }
  static int first(int b, int nchunks, int nb) { return (int)((long long)nchunks * b / nb); }
  // Host-pointer pipeline: sub-batch boundaries in sixteenths of the batch.  Default for large batches: four equal
  // sub-batches (with the round-2 kernels a sub-batch's chain of kernels is ~1.5 ms whatever its size, and the return
  // stream -- 289 MB at 47-56 GB/s -- is the long pole from the moment the first results exist; fewer, larger copies
  // serve it best: 7.84 ms against 8.11 ms for the earlier 1,1,2,4,4,4 ramp, scripts/e2e_schedule_sweep.py).
  // ZM_TEND_SCHEDULE=uniform keeps ZM_TEND_SUBBATCHES equal parts, ZM_TEND_SCHEDULE="1,1,2,4,4,4" sets explicit sizes.
  int sched_nb = 0, sched_first[MAXB + 1] = {};
  int plan(int nchunks) {
    const char* e = getenv("ZM_TEND_SCHEDULE");
    const bool ramp = !(e && !strcmp(e, "uniform")) && !getenv("ZM_TEND_SUBBATCHES") && nchunks >= 16 * 64;
    if (e && strchr(e, ',')) {                 // explicit sizes in sixteenths, e.g. "1,2,3,4,6"
      // every entry >= 1, at most MAXB entries, sum 16; anything else falls back to the default schedule
      int sizes[MAXB], n = 0, tot = 0;
      bool ok = true;
      for (const char* p = e; *p;) {
        const int v = atoi(p);
        if (v < 1 || n >= MAXB) { ok = false; break; }
        sizes[n++] = v; tot += v;
        p = strchr(p, ',');
        if (!p) break;
        ++p;
      }
      if (ok && tot == 16 && nchunks >= 16 * 64) {
        sched_nb = n;
        int acc = 0;
        for (int b = 0; b <= n; ++b) { sched_first[b] = (int)((long long)nchunks * acc / 16); if (b < n) acc += sizes[b]; }
        return sched_nb;
      }
    }
    if (ramp) {
      static const int sixteenths[5] = {0, 4, 8, 12, 16};
      sched_nb = 4;
      for (int b = 0; b <= 4; ++b) sched_first[b] = (int)((long long)nchunks * sixteenths[b] / 16);
    } else {
      sched_nb = subbatches(nchunks);
      for (int b = 0; b <= sched_nb; ++b) sched_first[b] = first(b, nchunks, sched_nb);
    }
    return sched_nb;
  }
  void release() {
    for (int b = 0; b < MAXB; ++b) work[b].release();
    for (int b = 0; b < ninit; ++b) {
      cudaEventDestroy(in_ready[b]); cudaEventDestroy(late_ready[b]); cudaEventDestroy(convr_done[b]);
      cudaEventDestroy(done[b]); cudaEventDestroy(early_back[b]); cudaEventDestroy(final_back[b]);
      cudaEventDestroy(small_back[b]); cudaEventDestroy(rec_back[b]);
    }
    if (h_rec) { cudaFreeHost(h_rec); h_rec = nullptr; h_rec_cap = 0; }
    if (h_small) { cudaFreeHost(h_small); h_small = nullptr; h_small_cap = 0; }
    ninit = 0; last_nb = 0; dev_nb = 0;
    if (t0) { cudaEventDestroy(t0); t0 = nullptr; }
    if (h2d) { cudaStreamDestroy(h2d); cudaStreamDestroy(d2h_early); cudaStreamDestroy(d2h_final); h2d = d2h_early = d2h_final = nullptr; }
  }
  int init(int nb) {
    if (!h2d) {
      CK(cudaStreamCreateWithFlags(&h2d, cudaStreamNonBlocking));
      CK(cudaStreamCreateWithFlags(&d2h_early, cudaStreamNonBlocking));
      CK(cudaStreamCreateWithFlags(&d2h_final, cudaStreamNonBlocking));
      CK(cudaEventCreate(&t0));
    }
    for (; ninit < nb; ++ninit) {
      CK(cudaEventCreate(&in_ready[ninit]));
      CK(cudaEventCreate(&late_ready[ninit]));
      CK(cudaEventCreate(&convr_done[ninit]));
      CK(cudaEventCreate(&done[ninit]));
      CK(cudaEventCreate(&early_back[ninit]));
      CK(cudaEventCreate(&final_back[ninit]));
      CK(cudaEventCreateWithFlags(&small_back[ninit], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&rec_back[ninit], cudaEventDisableTiming));
      // earlier sub-batches get higher stream priority: the first results reach the return stream sooner
      int lo = 0, hi = 0;
      CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));       // hi = greatest priority (numerically lowest)
      int pr = hi + ninit; if (pr > lo) pr = lo;
      if (!work[ninit].stream) CK(cudaStreamCreateWithPriority(&work[ninit].stream, cudaStreamNonBlocking, pr));
      work[ninit].side_priority = pr; work[ninit].side_priority_set = true;
      if (!work[ninit].side) {
        CK(cudaStreamCreateWithPriority(&work[ninit].side, cudaStreamNonBlocking, pr));
        CK(cudaEventCreateWithFlags(&work[ninit].ev_fork, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&work[ninit].ev_join, cudaEventDisableTiming));
      }
    }
    last_nb = nb;
    return 0;
  }
};
thread_local TendPipe tls_pipe;

// CUDA graph of one device-resident zm_conv_tend step (19 kernels, one memset, a fork/join with the side stream).
// A step is launch-gap sensitive (several kernels run 10-50 us), and a model calls it every time step with the same
// device arrays: the second call with an identical argument list is captured, later ones replay the graph.
struct TendGraph {
  std::vector<const void*> key;
  cudaGraphExec_t exec = nullptr;
  long long launches = 0;
  void clear() { if (exec) { cudaGraphExecDestroy(exec); exec = nullptr; } key.clear(); launches = 0; }
};
thread_local TendGraph tls_graph;
int g_epoch = 0;                       // bumped by zm_init: parameters are baked into captured kernels' constants

inline size_t al(size_t n, size_t sz) { return (n * sz + 255) & ~(size_t)255; }

void tick(Workspace& ws, cudaStream_t s, const char* name) {
  if (!g_profile) return;
  cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s);
  ws.tnames.push_back(name); ws.tev.push_back(e);
}

int lmax_for(int pver) { return pver <= 32 ? 32 : (pver <= 64 ? 64 : (pver <= 128 ? 128 : 0)); }

size_t convr_work_bytes(size_t ncolpad, int pver) {
  return 4 * al(ncolpad, 8) + 3 * al(ncolpad, 4) + 5 * al(ncolpad * pver, 8) + al(ncolpad, 4) +
         al(2 * ncolpad, 4) + 4 * al(ncolpad, 4) + al(4 + ZM_ORD_INTS, 4) + al(8, 8) + 4096;
}

// enqueue the whole zm_convr pipeline on stream s (no host synchronisation)
int convr_launch(Workspace& ws, cudaStream_t s, const ConvrIn& in, const ConvrOut& o,
                 bool own_arena = true, double* orgt = nullptr, double* org2d = nullptr,
                 const FillList* extra_fill = nullptr) {
  const int pcols = g_params.pcols, pver = g_params.pver;
  const bool org_on = g_params.zm_org != 0;
  if (org_on && !(in.org && orgt && org2d)) {
    tls_err = "zm_org = 1: call zm_org_fields(org, orgt, org2d) before zm_convr / zm_conv_tend";
    return -8;
  }
  const size_t ncolpad = (size_t)in.nchunks * pcols;
  if (own_arena && ws.ensure(convr_work_bytes(ncolpad, pver))) return -100;
  ConvrWork w;
  w.cape = ws.take<double>(ncolpad); w.cin = ws.take<double>(ncolpad); w.tl = ws.take<double>(ncolpad);
  w.dmpdz = ws.take<double>(ncolpad);
  w.lcl = ws.take<int>(ncolpad); w.lel = ws.take<int>(ncolpad); w.mx = ws.take<int>(ncolpad);
  w.tp = ws.take<double>(ncolpad * pver); w.qstp = ws.take<double>(ncolpad * pver);
  w.ab = ws.take<double>(3 * ncolpad * pver);
  w.wl1 = ws.take<int>(ncolpad); w.wl2 = ws.take<int>(2 * ncolpad);
  w.okey = ws.take<int>(ncolpad); w.ord1 = ws.take<int>(ncolpad); w.ord2 = ws.take<int>(ncolpad);
  w.count = ws.take<int>(4 + ZM_ORD_INTS); w.errinfo = ws.take<double>(8);
  w.n1chunk = ws.take<int>((size_t)in.nchunks); w.skip_idle_chunks = 0;
  // Two-warp CAPE kernel (first parcel loop on one warp, second on another): for launches that leave the schedulers
  // mostly idle.  Six 64-thread blocks (32 columns each) are resident per SM at <= 170 registers: one wave holds
  // 6 x 32 x SMs columns (28,416 on a B200); larger launches keep one thread per column.
  static const int ws_env = getenv("ZM_CAPE_TWO_WARPS") ? atoi(getenv("ZM_CAPE_TWO_WARPS")) : 1;
  static const int ws_sms = [] {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
  }();
  // resident blocks per SM: 6 by registers, fewer when the buoyancy rows of a deep grid fill the shared memory
  const size_t ws_block_smem = (size_t)(pver + 2) * 32 * sizeof(double) + 64 * sizeof(int) + ZMM_HOT_SMEM_BYTES + 1024;
  const int ws_bps = (int)std::min<size_t>(6, (227 * 1024) / ws_block_smem);
  w.ws_gate = ws_env ? ws_bps * 32 * ws_sms : -1;
  ws.last_count = w.count; ws.last_err = w.errinfo;
  for (auto e : ws.tev) cudaEventDestroy(e);
  ws.tev.clear(); ws.tnames.clear();

  const int TB = 128;
  const int nblk_cols = (int)((ncolpad + TB - 1) / TB);
  const size_t smem = (size_t)(pver + 2) * TB * sizeof(double);
  const int nwarpblk = (int)(((size_t)in.nchunks * 32 + 127) / 128);
  const int pl_warps = plume_warps_per_block(pver);
  const int nblk_pl = (int)((ncolpad + pl_warps - 1) / pl_warps);     // one warp per convective column
  const size_t smem_pl = plume_smem_bytes(pver);
  // plume kernels are built for 32/64/128-level leading dimensions (compile-time shared-memory strides)
  const int pl_ld = plume_ld(pver);
  auto k_cld1 = pl_ld == 34 ? k_cldprp_pass1_w<34> : (pl_ld == 66 ? k_cldprp_pass1_w<66> : k_cldprp_pass1_w<130>);
  auto k_plm = pl_ld == 34 ? k_plume_w<34> : (pl_ld == 66 ? k_plume_w<66> : k_plume_w<130>);
  // the first cldprp call needs 30 of the 41 work arrays: its own (smaller) blocks, more warps per SM
  const int pl1_warps = plume_warps_per_block(pver, A_FRONT_COUNT);
  const int nblk_pl1 = (int)((ncolpad + pl1_warps - 1) / pl1_warps);
  const size_t smem_pl1 = plume_smem_bytes(pver, A_FRONT_COUNT);
  CK(cudaFuncSetAttribute(k_cld1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pl1));
  CK(cudaFuncSetAttribute(k_plm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pl));
  {   // static tables (ZMM_HOT_SMEM_BYTES, 26 KB) + the buoyancy rows exceed the 48 KB default: opt in (dynamic part)
    CK(cudaFuncSetAttribute(k_buoyan_dilute<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaFuncSetAttribute((k_buoyan_dilute<1, false, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaFuncSetAttribute(k_buoyan_dilute<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaFuncSetAttribute(k_buoyan_undilute, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaFuncSetAttribute((k_buoyan_dilute<1, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaFuncSetAttribute((k_buoyan_dilute<2, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  const int nblk_ws = (int)((ncolpad + 31) / 32);
  const size_t smem_ws = (size_t)(pver + 2) * 32 * sizeof(double) + 64 * sizeof(int);
  if (smem_ws + ZMM_HOT_SMEM_BYTES > 48 * 1024) {
    CK(cudaFuncSetAttribute((k_buoyan_dilute_ws<1, false>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ws));
    CK(cudaFuncSetAttribute((k_buoyan_dilute_ws<1, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ws));
    CK(cudaFuncSetAttribute((k_buoyan_dilute_ws<2, false>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ws));
    CK(cudaFuncSetAttribute((k_buoyan_dilute_ws<2, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ws));
  }
  const bool ws1 = w.ws_gate > 0 && ncolpad <= (size_t)w.ws_gate;       // first pass: the host knows the column count
  tick(ws, s, "start");
  k_convr_init_cols<<<(unsigned)((ncolpad + 255) / 256), 256, 0, s>>>(in, o, w); ++tls_launches;
  // zero-fill of the per-level outputs and of what the caller adds (the fused step's wind tendencies and KE heating)
  FillList fl{};
  {
    const size_t n2 = ncolpad * pver, n2p = ncolpad * (pver + 1);
    bool full = false;
    auto add = [&](double* p, size_t n) {
      if (!p) return;
      if (fl.cnt == ZM_FILL_MAX) { full = true; return; }
      fl.p[fl.cnt] = p; fl.n[fl.cnt] = n; ++fl.cnt;
    };
    for (double* p : {o.qtnd, o.heat, o.cme, o.dlf, o.zdu, o.rprd, o.mu, o.md, o.du, o.eu, o.ed, o.dp, o.ql}) add(p, n2);
    // eurt, dif, dnlf, dnif: NULL inside the fused sequence unless zm_conv_tend_hist_fields attached them
    for (double* p : {o.eurt, o.dif, o.dnlf, o.dnif}) add(p, n2);
    add(o.mcon, n2p); add(o.pflx, n2p);
    if (extra_fill) for (int a = 0; a < extra_fill->cnt; ++a) add(extra_fill->p[a], extra_fill->n[a]);
    if (full) {      // an array left out would return stale arena contents
      tls_err = "internal: zero-fill list of zm_convr exceeds ZM_FILL_MAX";
      return -100;
    }
  }
  // the work ordering of the first CAPE pass (latency-bound, inputs only) runs on the side stream beside the fill
  // (bandwidth-bound); ZM_ORDER_SIDE=0 keeps both on this stream
  const bool order_side = !g_profile && !(getenv("ZM_ORDER_SIDE") && atoi(getenv("ZM_ORDER_SIDE")) == 0);
  const int nblk_ord = (int)((ncolpad + 255) / 256);
  if (order_side) {
    if (ws.ensure_side()) return -100;
    CK(cudaEventRecord(ws.ev_fork, s));                        // after k_convr_init_cols: the counters are zero
    CK(cudaStreamWaitEvent(ws.side, ws.ev_fork, 0));
    k_order_count<1><<<nblk_ord, 256, 0, ws.side>>>(in, w);
    k_order_scatter<1><<<nblk_ord, 256, 0, ws.side>>>(in, w);
    CK(cudaEventRecord(ws.ev_join, ws.side));
  }
  k_zero_fill<<<1184, 256, 0, s>>>(fl); ++tls_launches;
  if (org_on) {      // zm_conv.F90:555-556, 793-819
    k_org2d<<<nblk_cols, TB, 0, s>>>(in.nchunks, in.ncol, in.org, in.dpp, orgt, org2d); ++tls_launches;
  }
  if (order_side) {
    CK(cudaStreamWaitEvent(s, ws.ev_join, 0));
  } else {
    k_order_count<1><<<nblk_ord, 256, 0, s>>>(in, w);           // CAPE work order: most parcel levels first
    k_order_scatter<1><<<nblk_ord, 256, 0, s>>>(in, w);
  }
  tls_launches += 2;
  tick(ws, s, "convr_init");
  if (g_params.cam3) k_buoyan_undilute<<<nblk_cols, TB, smem, s>>>(in, w);     // zm_conv.F90:871-880
  else if (ws1 && org_on) k_buoyan_dilute_ws<1, true><<<nblk_ws, 64, smem_ws, s>>>(in, w);
  else if (ws1)           k_buoyan_dilute_ws<1, false><<<nblk_ws, 64, smem_ws, s>>>(in, w);
  else if (org_on)   k_buoyan_dilute<1, true><<<nblk_cols, TB, smem, s>>>(in, w);
  else if (ncolpad <= 24576)                 // few columns: the per-column chain is all that counts (latency mode)
    k_buoyan_dilute<1, false, true><<<nblk_cols, TB, smem, s>>>(in, w);
  else               k_buoyan_dilute<1><<<nblk_cols, TB, smem, s>>>(in, w);
  ++tls_launches;
  tick(ws, s, "buoyan_dilute_pass1");
  k_trigger<0><<<nwarpblk, 128, 0, s>>>(in, o, w); ++tls_launches;
  k_order_count<2><<<nblk_ord, 256, 0, s>>>(in, w); ++tls_launches;
  k_order_scatter<2><<<nblk_ord, 256, 0, s>>>(in, w); ++tls_launches;
  tick(ws, s, "trigger_pass1");
  k_cld1<<<nblk_pl1, 32 * pl1_warps, smem_pl1, s>>>(in, w);
  ++tls_launches;
  tick(ws, s, "cldprp_pass1");
  // The reference's second call covers every column of a chunk that has a convective column after the first gather
  // (zm_conv.F90:917, 1080-1091).  After a dilute first pass the columns that did not trigger keep their dmpdz row,
  // so their second-pass result is the first-pass result and only the worklist is recomputed; after cam3's undilute
  // first pass (zm_conv.F90:871) every column of those chunks needs the dilute pass.
  if (g_params.cam3) {
    ConvrWork w2 = w;
    w2.skip_idle_chunks = 1;
    if (org_on)                k_buoyan_dilute<1, true><<<nblk_cols, TB, smem, s>>>(in, w2);
    else if (ncolpad <= 24576) k_buoyan_dilute<1, false, true><<<nblk_cols, TB, smem, s>>>(in, w2);
    else                       k_buoyan_dilute<1><<<nblk_cols, TB, smem, s>>>(in, w2);
  } else {
    // latency mode: one warp per block, so that the blocks spread evenly over the schedulers of all SMs whatever the
    // size of the worklist (with 128-thread blocks the last few SMs get a second block: pass 2 0.816 -> 0.808 ms)
    const int tb2 = 32, nblk2 = (int)((ncolpad + tb2 - 1) / tb2);
    const size_t smem2 = (size_t)(pver + 2) * tb2 * sizeof(double);
    if (org_on) k_buoyan_dilute<2, true><<<nblk2, tb2, smem2, s>>>(in, w);
    else        k_buoyan_dilute<2><<<nblk2, tb2, smem2, s>>>(in, w);
    if (w.ws_gate > 0) {       // worklists up to ws_gate columns take the two-warp kernel instead (device-side gate)
      const int nb = (int)std::min<size_t>((size_t)nblk_ws, (size_t)(w.ws_gate + 31) / 32);
      if (org_on) k_buoyan_dilute_ws<2, true><<<nb, 64, smem_ws, s>>>(in, w);
      else        k_buoyan_dilute_ws<2, false><<<nb, 64, smem_ws, s>>>(in, w);
      ++tls_launches;
    }
  }
  ++tls_launches;
  tick(ws, s, "buoyan_dilute_pass2");
  k_trigger<1><<<nwarpblk, 128, 0, s>>>(in, o, w); ++tls_launches;
  tick(ws, s, "trigger_final");
  k_plm<<<nblk_pl, 32 * pl_warps, smem_pl, s>>>(in, o, w);
  ++tls_launches;
  tick(ws, s, "plume_closure_q1q2");
  CK(cudaGetLastError());
  return 0;
}

// after a sync: number of Brent failures of the last convr call on this thread
int read_failures(Workspace& ws, cudaStream_t s) {
  if (!ws.last_count) return 0;
  int cnt[4]; double info[8];
  CK(cudaMemcpyAsync(cnt, ws.last_count, sizeof cnt, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(info, ws.last_err, sizeof info, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (cnt[2] > 0) {
    char b[512];
    const int col = (int)info[1], pc = g_params.pcols;
    snprintf(b, sizeof b,
             "*** ZM_CONV: %s failed to converge (%d events); first: call#=%d lchnk=%d icol=%d "
             "P(mb)=%.2f Tfg(K)=%.2f qt(g/kg)=%.2f s(J/kg)=%.2f",
             (int)info[0] == 4 ? "IENTROPY" : "IENTHALPY", cnt[2], (int)info[0], ws.chunk0 + col / pc + 1,
             col % pc + 1, info[2], info[3], 1000.0 * info[4], info[5]);
    tls_err = b;
  }
  return cnt[2];
}

struct Stager {      // host-pointer API: bump-allocate device copies of user arrays
  Workspace& ws; cudaStream_t s; int rc = 0;
  struct Out { void* h; void* d; size_t bytes; };
  std::vector<Out> outs, early;
  Stager(Workspace& w) : ws(w), s(w.stream) {}
  template <class T> const T* in(const T* h, size_t n, cudaStream_t on = nullptr) {
    T* d = ws.take<T>(n);
    if (cudaMemcpyAsync(d, h, n * sizeof(T), cudaMemcpyHostToDevice, on ? on : s) != cudaSuccess) rc = -100;
    return d;
  }
  template <class T> T* out(T* h, size_t n, bool is_early = false) {
    T* d = ws.take<T>(n);
    if (h) (is_early ? early : outs).push_back({(void*)h, (void*)d, n * sizeof(T)});   // NULL: stays on device
    return d;
  }
  void flush_early(cudaStream_t on) {      // D2H of outputs that are final before the step ends
    for (auto& o : early)
      if (cudaMemcpyAsync(o.h, o.d, o.bytes, cudaMemcpyDeviceToHost, on) != cudaSuccess) rc = -100;
    early.clear();
  }
  template <class T> T* inout(T* h, size_t n) {
    T* d = ws.take<T>(n);
    if (cudaMemcpyAsync(d, h, n * sizeof(T), cudaMemcpyHostToDevice, s) != cudaSuccess) rc = -100;
    outs.push_back({(void*)h, (void*)d, n * sizeof(T)});
    return d;
  }
  int flush() {
    for (auto& o : outs)
      if (cudaMemcpyAsync(o.h, o.d, o.bytes, cudaMemcpyDeviceToHost, s) != cudaSuccess) rc = -100;
    if (cudaStreamSynchronize(s) != cudaSuccess) rc = -100;
    if (rc) tls_err = std::string("CUDA copy error: ") + cudaGetErrorString(cudaGetLastError());
    return rc;
  }
};

int evap_launch(cudaStream_t s, const EvapArgs& a) {
  const int ncolpad = a.nchunks * g_params.pcols;
  if (a.heat && a.tend_s) k_conv_evap<true, true><<<(ncolpad + 127) / 128, 128, 0, s>>>(a);
  else if (a.heat)        k_conv_evap<true><<<(ncolpad + 127) / 128, 128, 0, s>>>(a);
  else                    k_conv_evap<false><<<(ncolpad + 127) / 128, 128, 0, s>>>(a);
  ++tls_launches;
  CK(cudaGetLastError());
  return 0;
}

// ktm / kbm of momtran and convtran (zm_conv.F90:2076-2081, 2449-2454) + the compact list of convective slots
struct ChunkBounds { int *ktm = nullptr, *kbm = nullptr, *slots = nullptr, *count = nullptr; };
size_t chunk_bounds_bytes(int nchunks, int ncolpad) { return 2 * al(nchunks, 4) + al(ncolpad, 4) + 2048; }
int chunk_bounds_enqueue(Workspace& ws, cudaStream_t s, int nchunks, const int* jt, const int* mx, const int* lengath,
                         ChunkBounds& cb) {
  const int ncolpad = nchunks * g_params.pcols;
  cb.ktm = ws.take<int>(nchunks); cb.kbm = ws.take<int>(nchunks);
  cb.slots = ws.take<int>(ncolpad); cb.count = ws.take<int>(1);
  CK(cudaMemsetAsync(cb.count, 0, sizeof(int), s));
  k_chunk_bounds<<<(nchunks * 32 + 127) / 128, 128, 0, s>>>(nchunks, jt, mx, lengath, cb.ktm, cb.kbm, cb.slots, cb.count);
  ++tls_launches;
  CK(cudaGetLastError());
  return 0;
}

// own_arena: the bounds come from this call's own arena; otherwise `cb` holds them already
int momtran_launch(Workspace& ws, cudaStream_t s, MomArgs a, bool own_arena = true, const ChunkBounds* cb = nullptr) {
  const int pcols = g_params.pcols, pver = g_params.pver;
  const int ncolpad = a.nchunks * pcols;
  ChunkBounds own;
  if (!cb) {
    if (own_arena && ws.ensure(chunk_bounds_bytes(a.nchunks, ncolpad))) return -100;
    if (chunk_bounds_enqueue(ws, s, a.nchunks, a.jt, a.mx, a.lengath, own)) return -100;
    cb = &own;
  }
  a.ktm = cb->ktm; a.kbm = cb->kbm; a.slots = cb->slots; a.count = cb->count;
  // fused step with split wind arrays: dq_u, dq_v and seten were zero-filled with zm_convr's outputs at the start of
  // the step (k_zero_fill); the packed form initialises its outgoing fields here
  if (!a.q_u) { k_momtran_init<<<592, 256, 0, s>>>(a); ++tls_launches; }
  const size_t smem_mom = momtran_smem_bytes(pver);
  if (smem_mom > 48 * 1024)
    CK(cudaFuncSetAttribute(k_momtran_t, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_mom));
  k_momtran_t<<<(ncolpad + MOM_WARPS - 1) / MOM_WARPS, 32 * MOM_WARPS, smem_mom, s>>>(a);   // warp per convective column
  ++tls_launches;
  CK(cudaGetLastError());
  return 0;
}

// Constituent flags of a convtran call on the device: [0, nactive) the 0-based indices m >= 1 with doconvtran(m),
// then ncnst dry flags.  Kept per thread and re-uploaded (synchronously) only when the flags change, so that a
// step that repeats -- every model time step -- enqueues no host->device copy and can be captured in a CUDA graph.
struct TranMeta {
  int* d = nullptr; int cap = 0;
  std::vector<int> host;
  int ncnst = 0, nactive = 0, version = 0; bool any_dry = false;
  const int* active() const { return d; }
  const int* dry() const { return d + nactive; }
  int set(const int* doconvtran, const int* is_dry, int n) {
    std::vector<int> h;
    for (int m = 1; m < n; ++m)            // reference loops m = 2, ncnst (1-based)
      if (doconvtran[m]) h.push_back(m);
    const int na = (int)h.size();
    bool dry_any = false;
    for (int m = 0; m < n; ++m) { h.push_back(is_dry ? is_dry[m] : 0); }
    for (int j = 0; j < na; ++j) dry_any = dry_any || (is_dry && is_dry[h[j]]);
    return upload(h, n, na, dry_any);
  }
  // compact form: `na` constituents 0..na-1, all active, with their dry flags
  int set_compact(const std::vector<int>& dry_of_active) {
    const int na = (int)dry_of_active.size();
    std::vector<int> h;
    bool dry_any = false;
    for (int j = 0; j < na; ++j) h.push_back(j);
    for (int j = 0; j < na; ++j) { h.push_back(dry_of_active[j]); dry_any = dry_any || dry_of_active[j]; }
    return upload(h, na, na, dry_any);
  }
  int upload(const std::vector<int>& h, int n, int na, bool dry_any) {
    if (h == host && n == ncnst && d) return 0;
    if ((int)h.size() > cap) {
      if (d) { CK(cudaDeviceSynchronize()); CK(cudaFree(d)); d = nullptr; }
      cap = (int)h.size() + 64;
      CK(cudaMalloc((void**)&d, cap * sizeof(int)));
    }
    CK(cudaMemcpy(d, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice));
    host = h; ncnst = n; nactive = na; any_dry = dry_any; ++version;
    return 0;
  }
  void release() { if (d) { cudaFree(d); d = nullptr; } cap = 0; host.clear(); ncnst = nactive = 0; }
};
thread_local TranMeta tls_tmeta;      // zm_convtran_batch[_dev] / zm_conv_tend_2_batch
thread_local TranMeta tls_tmeta1;     // convtran1 attached to zm_conv_tend_batch_dev (caller's constituent layout)
thread_local TranMeta tls_tmeta1c;    // convtran1 of the host-pointer zm_conv_tend_batch (compact: active slices only)
thread_local std::vector<int> tls_tran1_flags;   // host copy of (doconvtran, cnst_is_dry) given to zm_convtran1_fields

// a.active / a.is_dry / a.nactive and the chunk bounds are set: zero the active slices, transport
int convtran_enqueue(cudaStream_t s, TranArgs a, const ChunkBounds& cb) {
  const int pcols = g_params.pcols, pver = g_params.pver;
  const int ncolpad = a.nchunks * pcols;
  if (a.nactive == 0) return 0;
  a.ktm = cb.ktm; a.kbm = cb.kbm; a.slots = cb.slots; a.count = cb.count;
  // block per (chunk, constituent group) with every row of q / fracis / dqdt moved once (ZM_CONVTRAN_KERNEL=t keeps
  // the thread-per-(column, constituent) kernel, which also serves shapes whose work arrays do not fit an SM)
  static const bool force_t = [] { const char* e = getenv("ZM_CONVTRAN_KERNEL"); return e && e[0] == 't'; }();
  if (!force_t && convtran_c_fits(pver, pcols) && (reinterpret_cast<uintptr_t>(a.dqdt) & 15) == 0) {
    const size_t smem = convtran_c_smem_bytes(pver, pcols);
    static size_t smem_set = 0;
    if (smem > smem_set) {
      CK(cudaFuncSetAttribute(k_convtran_c<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      smem_set = smem;
    }
    const int bpc = convtran_c_blocks_per_chunk(a.nactive, pcols);
    k_convtran_c<false><<<(unsigned)((size_t)a.nchunks * bpc), 32 * CTC_NW, smem, s>>>(a, bpc, nullptr); ++tls_launches;
    CK(cudaGetLastError());
    return 0;
  }
  k_convtran_zero<<<a.nchunks * a.nactive, 128, 0, s>>>(a); ++tls_launches;
  const int cpb = convtran_cnst_per_block(pver);
  dim3 blk(32, cpb);
  dim3 grd((a.nactive + cpb - 1) / cpb, (ncolpad + 31) / 32);       // x: constituent groups, y: column groups
  k_convtran_t<false><<<grd, blk, 0, s>>>(a, nullptr);
  ++tls_launches;
  CK(cudaGetLastError());
  return 0;
}

// The same transport on the convective columns' records (zm_conv_tend_2_batch_gathered): q / fracis / dqdt are record
// buffers and rbase[c] is chunk c's first record column (k_lengath_scan).  Every record element is written, so there
// is no zero-fill launch; the block kernel takes any dqdt alignment.  One launch.
int convtran_enqueue_gathered(cudaStream_t s, TranArgs a, const int* rbase, const ChunkBounds& cb) {
  const int pcols = g_params.pcols, pver = g_params.pver;
  const int ncolpad = a.nchunks * pcols;
  if (a.nactive == 0) return 0;
  a.ktm = cb.ktm; a.kbm = cb.kbm; a.slots = cb.slots; a.count = cb.count;
  static const bool force_t = [] { const char* e = getenv("ZM_CONVTRAN_KERNEL"); return e && e[0] == 't'; }();
  if (!force_t && convtran_c_fits(pver, pcols)) {
    const size_t smem = convtran_c_smem_bytes(pver, pcols);
    static size_t smem_set = 0;
    if (smem > smem_set) {
      CK(cudaFuncSetAttribute(k_convtran_c<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      smem_set = smem;
    }
    const int bpc = convtran_c_blocks_per_chunk(a.nactive, pcols);
    k_convtran_c<true><<<(unsigned)((size_t)a.nchunks * bpc), 32 * CTC_NW, smem, s>>>(a, bpc, rbase); ++tls_launches;
    CK(cudaGetLastError());
    return 0;
  }
  const int cpb = convtran_cnst_per_block(pver);
  dim3 blk(32, cpb);
  dim3 grd((a.nactive + cpb - 1) / cpb, (ncolpad + 31) / 32);
  k_convtran_t<true><<<grd, blk, 0, s>>>(a, rbase);
  ++tls_launches;
  CK(cudaGetLastError());
  return 0;
}

int convtran_launch(Workspace& ws, cudaStream_t s, TranArgs a, const int* doconvtran_h,
                    const int* is_dry_h) {
  const int ncolpad = a.nchunks * g_params.pcols;
  if (tls_tmeta.set(doconvtran_h, is_dry_h, a.ncnst)) return -100;
  a.nactive = tls_tmeta.nactive;
  if (a.nactive == 0) return 0;
  a.active = tls_tmeta.active(); a.is_dry = tls_tmeta.dry();
  if (ws.ensure(chunk_bounds_bytes(a.nchunks, ncolpad))) return -100;
  ChunkBounds cb;
  if (chunk_bounds_enqueue(ws, s, a.nchunks, a.jt, a.mx, a.lengath, cb)) return -100;
  return convtran_enqueue(s, a, cb);
}

// ---- zm_conv_tend glue (zm_conv_intr.F90:662-836) ------------------------------------------------
// state1 after physics_update(ptend_loc of zm_convr): physics_types.F90:322-329 (q + qneg3 clip at
// qmin(1)=1e-12) and :427 (t += s*dt/cpair); winds(:,:,1:2) = state1%u,v (zm_conv_intr.F90:815-816)
// PART 0: both; 1: t1, q1 only (what zm_conv_evap needs); 2: winds only (what momtran needs) -- the two halves run on
// the two branches of the evap / momtran fork
template <int PART>
__global__ void k_state_update(int n2, int nper, const double* t, const double* q, const double* heat,
                               const double* qtnd, const double* u, const double* v, double ztodt,
                               double* t1, double* q1, double* winds) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n2; e += gridDim.x * blockDim.x) {
    if (PART != 2) {
      t1[e] = t[e] + div_z(heat[e] * ztodt, P.cpair);
      double qn = q[e] + qtnd[e] * ztodt;
      q1[e] = (qn < 1.e-12) ? 1.e-12 : qn;
    }
    if (PART != 1) {
      int c = e / nper, r = e - c * nper;            // nper = pcols*pver
      winds[(size_t)c * 2 * nper + r] = u[e];
      winds[(size_t)c * 2 * nper + nper + r] = v[e];
    }
  }
}
// ptend_all = sum of the three ptend_loc (physics_ptend_sum, physics_types.F90:698-844) and, unless the plume kernel
// has done it (MCON = false), the mcon unit conversion mb/s -> kg/m2/s (zm_conv_intr.F90:693).
// MODE 0: cam3, no momentum transport (zm_conv_intr.F90:808); 1: wind tendencies unpacked from wind_tends(pcols,pver,2);
// 2: momtran has written ptend_u / ptend_v itself (split wind arrays).  evapcdp == ev_q when zm_conv_evap wrote its
// tend_q straight into the caller's evapcdp.
template <int MODE, bool MCON>
__global__ void k_tend_finalize(int n2, int n2p, int nper, const double* heat, const double* qtnd,
                                const double* ev_s, const double* ev_q, const double* seten,
                                const double* wtend, double* ps, double* pq, double* pu, double* pv,
                                double* evapcdp, double* mcon) {
  const int n = MCON ? n2p : n2;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    if (MCON) mcon[e] = div_z(mcon[e] * 100.0, P.gravit);
    if (e < n2) {
      const double evq = ev_q[e];
      pq[e] = qtnd[e] + evq;
      if (MODE) {
        ps[e] = (heat[e] + ev_s[e]) + seten[e];
        if (MODE == 1) {
          int c = e / nper, r = e - c * nper;
          pu[e] = wtend[(size_t)c * 2 * nper + r];
          pv[e] = wtend[(size_t)c * 2 * nper + nper + r];
        }
      } else {
        ps[e] = heat[e] + ev_s[e];
        pu[e] = 0.0; pv[e] = 0.0;
      }
      if (evapcdp != ev_q) evapcdp[e] = evq;
    }
  }
}

// the last term of ptend_s when zm_conv_evap has stored heat + tend_s itself: ptend_s = (heat + tend_s) + seten
// (zm_conv_intr.F90:833), every element like the reference (seten is +0 outside the columns momtran wrote)
__global__ void k_add_seten(size_t nhalf, double2* ps, const double2* seten) {
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < nhalf; e += (size_t)gridDim.x * blockDim.x) {
    double2 a = ps[e];
    const double2 b = seten[e];
    a.x = a.x + b.x; a.y = a.y + b.y;
    ps[e] = a;
  }
}

// ---- global water / energy budget terms (what check_energy_chng tests after ZM, physpkg.F90:2865) --
// Deterministic two-stage reduction (the result depends on nothing but the inputs and the fixed grid): a block walks
// over chunks blockIdx.x, blockIdx.x + gridDim.x, ...; its threads take the (level, column) elements of the chunk in
// storage order (coalesced) and the chunk's columns, each thread adding its terms in that order; a fixed tree adds
// the 256 threads of a block, then one warp per quantity adds the block partials -- each lane its own stride-32
// subsequence in order, then a fixed shuffle tree.  (The first version summed a column per thread: 52 us for 42 MB,
// 12 warps per SM waiting on strided loads; this one streams.)
#define ZM_CONS_BLOCKS 1184
__global__ void __launch_bounds__(256)
k_conservation_partial(int nchunks, const int* ncol, const double* pdel, const double* pq,
                       const double* ps, const double* prec, const double* snow,
                       const double* rliq, const int* lengath, double* partial) {
  __shared__ double sh[6][256];
  const int pcols = P.pcols, pver = P.pver, nper = pcols * pver;
  double a[6] = {0, 0, 0, 0, 0, 0};
  for (int c = blockIdx.x; c < nchunks; c += gridDim.x) {
    const int n = ncol[c];
    const size_t base = (size_t)c * nper;
    for (int r = threadIdx.x; r < nper; r += 256) {
      if (r % pcols < n) {
        const size_t e = base + r;
        const double m = div_hot(pdel[e], P.gravit);      // layer mass: pdel/g (the IEEE quotient for these operands)
        a[0] += m * pq[e];
        a[2] += m * ps[e];
      }
    }
    for (int i = threadIdx.x; i < n; i += 256) {
      const size_t col = (size_t)c * pcols + i;
      a[1] += 1000.0 * (prec[col] + rliq[col]);
      a[3] += 1000.0 * (P.latvap * (prec[col] + rliq[col]) + P.latice * snow[col]);
      a[5] += 1.0;
      if (i == 0) a[4] += (double)lengath[c];
    }
  }
  for (int j = 0; j < 6; ++j) sh[j][threadIdx.x] = a[j];
  __syncthreads();
  for (int off = 128; off; off >>= 1) {
    if (threadIdx.x < off)
      for (int j = 0; j < 6; ++j) sh[j][threadIdx.x] += sh[j][threadIdx.x + off];
    __syncthreads();
  }
  if (threadIdx.x < 6) partial[blockIdx.x * 6 + threadIdx.x] = sh[threadIdx.x][0];
}
__global__ void __launch_bounds__(192) k_conservation_final(int nblocks, const double* partial, double* out6) {
  const int j = threadIdx.x >> 5, lane = threadIdx.x & 31;       // one warp per quantity
  double s = 0.0;
  for (int b = lane; b < nblocks; b += 32) s += partial[b * 6 + j];
  for (int off = 16; off; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
  if (lane == 0) out6[j] = s;
}

// freqzm, mu_out / md_out, pcont / pconb of zm_conv_tend (zm_conv_intr.F90:685-688, 575-576 + 700-706, 721-729):
// one block per chunk.  The chunk's map column -> gathered slot is built in shared memory, then the (pcols,pver)
// rows are written in order (coalesced): the scaled mass flux where the column convects, zero elsewhere.
// pcont / pconb are assigned for i <= ncol only (:721-722); the rest of the row is zero-filled.
__global__ void __launch_bounds__(128)
k_tend_diag(int nchunks, const int* ncol, const double* ps, const double* pmid, const double* mu,
            const double* md, const int* jt, const int* maxg, const int* ideep, const int* lengath,
            double* freqzm, double* mu_out, double* md_out, double* pcont, double* pconb) {
  extern __shared__ int sh_inv[];                  // [pcols] gathered slot of a column, -1 if it does not convect
  const int pcols = P.pcols, pver = P.pver;
  const int c = blockIdx.x;
  if (c >= nchunks) return;
  const int n = ncol[c], len = lengath[c];
  const size_t c1 = (size_t)c * pcols;
  for (int i = threadIdx.x; i < pcols; i += blockDim.x) sh_inv[i] = -1;
  __syncthreads();
  for (int g = threadIdx.x; g < len; g += blockDim.x) sh_inv[ideep[c1 + g] - 1] = g;
  __syncthreads();
  for (int i = threadIdx.x; i < pcols; i += blockDim.x) {
    const int g = sh_inv[i];
    freqzm[c1 + i] = (g >= 0) ? 1.0 : 0.0;
    double pt = (i < n) ? ps[c1 + i] : 0.0, pb = pt;
    if (g >= 0) {
      const int j = jt[c1 + g], mx = maxg[c1 + g];
      if (mx > j) { pt = pmid[cidx(c, j - 1, i, pver)]; pb = pmid[cidx(c, mx - 1, i, pver)]; }
    }
    pcont[c1 + i] = pt; pconb[c1 + i] = pb;
  }
  for (int e = threadIdx.x; e < pcols * pver; e += blockDim.x) {
    const int k = e / pcols, i = e - k * pcols;
    const int g = sh_inv[i];
    double vu = 0.0, vd = 0.0;
    if (g >= 0) { vu = div_z(mu[cidx(c, k, g, pver)] * 100.0, P.gravit); vd = div_z(md[cidx(c, k, g, pver)] * 100.0, P.gravit); }
    mu_out[(size_t)c * pcols * pver + e] = vu;
    md_out[(size_t)c * pcols * pver + e] = vd;
  }
}

__global__ void k_dpdry_gather(int nchunks, const int* ideep, const int* lengath, const double* pdeldry,
                               double* dpdry) {
  const int pcols = P.pcols, pver = P.pver, nper = pcols * pver;
  for (int c = blockIdx.x; c < nchunks; c += gridDim.x) {        // a block per chunk: 32-bit index arithmetic only
    const int len = lengath[c];
    for (int r = threadIdx.x; r < nper; r += blockDim.x) {
      const int k = r / pcols, i = r - k * pcols;
      double v = 0.0;
      if (i < len) v = pdeldry[cidx(c, k, ideep[(size_t)c * pcols + i] - 1, pver)] / 100.0;
      dpdry[(size_t)c * nper + r] = v;
    }
  }
}
// the same from the records of zm_conv_tend_2_batch_gathered: chunk c's pdeldry(ideep(1:n),:) is the Fortran array
// (n, pver) at pver*base(c)
__global__ void k_dpdry_gather_rec(int nchunks, const int* lengath, const int* base, const double* pdeldry_rec,
                                   double* dpdry) {
  const int pcols = P.pcols, pver = P.pver, nper = pcols * pver;
  for (int c = blockIdx.x; c < nchunks; c += gridDim.x) {
    const int len = lengath[c];
    const double* src = pdeldry_rec + (size_t)base[c] * pver;
    for (int r = threadIdx.x; r < nper; r += blockDim.x) {
      const int k = r / pcols, i = r - k * pcols;
      double v = 0.0;
      if (i < len) v = src[k * len + i] / 100.0;
      dpdry[(size_t)c * nper + r] = v;
    }
  }
}

// ---- diagnostics kernels ----------------------------------------------------------------------
__global__ void k_math_eval(int id, int n, const double* x, const double* y, double* o) {
  zmm::hot_tables_load();
  zmm::hot_svp_load();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  switch (id) {
    case 0: o[i] = zmm::log_(x[i]); break;
    case 1: o[i] = zmm::log10_(x[i]); break;
    case 2: o[i] = zmm::exp_(x[i]); break;
    case 3: o[i] = zmm::pow10_(x[i]); break;
    case 5: o[i] = zmm::log_hot(x[i]); break;
    case 6: o[i] = zmm::log10_hot(x[i]); break;
    case 7: o[i] = zmm::pow10_hot(x[i]); break;
    case 8: o[i] = zmm::div_rcp(x[i], y[i], 1.0 / y[i]); break;
    case 9: o[i] = div_hot(x[i], y[i]); break;
    case 10: o[i] = zmm::svp_water<false>(x[i]); break;
    case 11: o[i] = zmm::svp_water_formula(x[i]); break;
    case 12: o[i] = zmm::svp_water<true>(x[i]); break;
    default: o[i] = zmm::pow_(x[i], y[i]); break;
  }
}
__global__ void k_thermo_eval(int id, int n, const double* a, const double* b, const double* c,
                              const double* d, const double* e, double* o0, double* o1) {
  zmm::hot_tables_load();
  zmm::hot_svp_load();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double r0 = 0.0, r1 = 0.0;
  switch (id) {
    case 0: r0 = entropy_q(a[i], b[i], c[i], r1); break;
    case 1: r0 = enthalpy_q(a[i], b[i], c[i], d[i], r1); break;
    case 2: invert<0>(a[i], b[i], 0.0, c[i], d[i], r0, r1); break;
    case 3: invert<1>(a[i], b[i], c[i], d[i], e[i], r0, r1); break;
    case 4: qsat_hPa(a[i], b[i], r0, r1); break;
    default: qsat_table(a[i], b[i], r0, r1); break;
  }
  o0[i] = r0; o1[i] = r1;
}
// single-warp latency microbenchmark (cycles per dependent call), see zm_microbench
__global__ void k_microbench(double* out, long long* cyc, int n) {
  zmm::hot_tables_load();
  zmm::hot_svp_load();
  double x = 290.0 + threadIdx.x * 0.01, acc = 0.0, q;
  long long t0, t1;
  int j = 0;
#define MB(expr)                                      \
  t0 = clock64();                                     \
  for (int i = 0; i < n; ++i) { expr; }               \
  t1 = clock64();                                     \
  if (threadIdx.x == 0) cyc[j] = (t1 - t0) / n;       \
  ++j;
  MB(x = 300.0 + 1e-3 * (373.16 / x));                                   // 0 division
  MB(x = 300.0 + 1e-3 * zmm::log_(x));                                   // 1 log
  MB(x = 300.0 + 1e-3 * zmm::log10_(x));                                 // 2 log10
  MB(x = 300.0 + 1e-3 * zmm::pow10_(x * 1e-2));                          // 3 pow10
  MB(x = 300.0 + 1e-3 * zmm::exp_(x * 1e-2));                            // 4 exp
  MB(x = 300.0 + 1e-6 * gg_svp_water(x));                                // 5 goff-gratch
  MB(x = 300.0 + 1e-9 * enthalpy_q(x, 900.0, 0.015, 500.0, q));          // 6 enthalpy
  MB(x = 300.0 + 1e-6 * entropy_q(x, 900.0, 0.015, q));                  // 7 entropy
  MB(invert_k<1>(3.5e5 + x, 900.0, 500.0, 0.015, 295.0, acc, q); x = 290.0 + 1e-3 * acc);  // 8 ienthalpy
  MB(invert_k<0>(250.0 + 1e-3 * x, 900.0, 0.0, 0.015, 295.0, acc, q); x = 290.0 + 1e-3 * acc);  // 9 ientropy
  MB(x = 300.0 + 1e-3 * zmm::pow_(x, 0.2857));                           // 10 pow
  MB(x = 300.0 + 1e-6 * zmm::svp_water_formula(x));                      // 11 goff-gratch formula
  MB(x = fma(x, 0.999999, 1e-4));                                        // 12 dependent DFMA
  MB(x = x + 1e-9);                                                      // 13 dependent DADD
  MB(x = x * 1.0000001);                                                 // 14 dependent DMUL
  MB(x = 300.0 + 1e-3 * div_hot(373.16, x));                             // 15 div_hot
  MB(x = 300.0 + 1e-3 * zmm::log_hot(x));                                // 16 log_hot
  MB(x = 300.0 + 1e-6 * zmm::svp_water<true>(x));                        // 17 svp table (shared memory)
  MB(x = (x > 300.5) ? x - 0.75 : x + 0.5);                              // 18 DSETP + select
  MB(x = (double)((int)x) + 0.25);                                       // 19 F2I + I2F
  out[threadIdx.x] = x + acc;
}
__global__ void k_fp64_peak(double* out, int iters) {
  double a0 = 1.0 + threadIdx.x * 1e-9, a1 = 1.1, a2 = 1.2, a3 = 1.3, a4 = 1.4, a5 = 1.5, a6 = 1.6, a7 = 1.7;
  const double m = 0.999999, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

}  // namespace

extern "C" {

void zm_params_default(zm_params_t* p, int pcols, int pver, int limcnv) {
  std::memset(p, 0, sizeof(*p));
  p->pcols = pcols; p->pver = pver; p->limcnv = limcnv;
  p->num_cin = 1; p->masterproc = 1;
  p->c0_lnd = 0.0075; p->c0_ocn = 0.03; p->ke = 5.0e-6; p->ke_lnd = 1.0e-5;
  p->momcu = 0.7; p->momcd = 0.7; p->tiedke_add = 0.5; p->capelmt = 70.0; p->dmpdz = -1.0e-3;
  p->tau = 3600.0;
  const double boltz = 1.38065e-23, avogad = 6.02214e26, rgas = avogad * boltz;
  const double mwdair = 28.966, mwwv = 18.016;
  p->cpair = 1.00464e3; p->epsilo = mwwv / mwdair; p->gravit = 9.80616; p->latice = 3.337e5;
  p->latvap = 2.501e6; p->tmelt = 273.15; p->rair = rgas / mwdair; p->cpwv = 1.810e3;
  p->cpliq = 4.188e3; p->rh2o = rgas / mwwv; p->cpvir = p->cpwv / p->cpair - 1.0;
  p->zvir = p->rh2o / p->rair - 1.0;
}

// zm_convi (zm_conv.F90:115-227)
int zm_init(const zm_params_t* p) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (p->microp) { tls_err = "zmconv_microp is out of scope (zm_microphysics is not part of the reference tree)"; return -2; }
  if (p->masterproc && p->num_cin > 5) { tls_err = "**** ZM_CONVI : NUM_CIN must not exceeed 5 ****"; return -3; }
  if (p->num_cin < 1 || p->num_cin > ZM_MAXCIN) { tls_err = "num_cin out of range 1..5"; return -3; }
  if (p->cam3 && p->num_cin != 5) {
    // buoyan declares capeten(pcols,num_cin) but loops n = 1,5 (zm_conv.F90:2770 vs 2992,3006)
    tls_err = "cam3 (undilute buoyan) is only well defined for num_cin = 5"; return -4;
  }
  if (lmax_for(p->pver) == 0 || p->pcols < 1 || p->limcnv < 2 || p->limcnv > p->pver) {
    tls_err = "unsupported grid (need 1 <= pver <= 128, 2 <= limcnv <= pver)"; return -5;
  }
  g_params = *p;
  ++g_epoch;
  ZmDevParams d;
  d.pcols = p->pcols; d.pver = p->pver; d.pverp = p->pver + 1; d.limcnv = p->limcnv; d.msg = p->limcnv - 1;
  d.num_cin = p->num_cin; d.no_deep_pbl = p->no_deep_pbl; d.lparcel_pbl = p->lparcel_pbl; d.cam3 = p->cam3; d.zm_org = p->zm_org != 0;
  d.rl = p->latvap; d.cpres = p->cpair; d.ke = p->ke; d.ke_lnd = p->ke_lnd; d.c0_lnd = p->c0_lnd;
  d.c0_ocn = p->c0_ocn; d.tau = p->tau; d.tfreez = p->tmelt; d.eps1 = p->epsilo; d.momcu = p->momcu;
  d.momcd = p->momcd; d.rgrav = 1.0 / p->gravit; d.rgas = p->rair; d.grav = p->gravit; d.cp = p->cpair;
  d.dcol = (p->cpliq - p->cpwv) / p->latvap;
  d.capelmt = p->capelmt; d.tiedke_add = p->tiedke_add; d.tiedke_lnd = 1.0; d.entrmn = 2e-4;
  d.alfadet = 0.1; d.plclmin = 6.e2; d.cin_threshd = 0.33; d.parcel_hscale = 0.5;
  d.rtfreez = 1.0 / p->tmelt;
  d.tentrm = p->masterproc ? -p->dmpdz : 1e-3;          // zm_conv.F90:90,213
  d.cpair = p->cpair; d.epsilo = p->epsilo; d.gravit = p->gravit; d.latice = p->latice;
  d.latvap = p->latvap; d.tmelt = p->tmelt; d.rair = p->rair; d.cpwv = p->cpwv; d.cpliq = p->cpliq;
  d.rh2o = p->rh2o; d.cpvir = p->cpvir; d.zvir = p->zvir; d.omeps = 1.0 - p->epsilo;
  CK(cudaMemcpyToSymbol(P, &d, sizeof d));
  // CAM's estbl table (wv_saturation): svp_trans at 1-K steps from 127.16 K, ttrice = 20 K
  double tbl[ZM_ESTBL_LEN];
  auto svp_w = [](double t) { return zmm::svp_water<false>(t); };
  auto svp_i = [](double t) {
    const double t3 = 273.16;
    return zmm::pow10_(-9.09718 * (t3 / t - 1.0) - 3.56654 * zmm::log10_(t3 / t) + 0.876793 * (1.0 - t / t3) +
                       0.7858350313586662) * 100.0;
  };
  const double tmelt = p->tmelt, ttrice = 20.0;
  for (int i = 0; i < ZM_ESTBL_LEN - 1; ++i) {
    double t = 127.16 + (double)i, es;
    if (t >= (tmelt - ttrice)) es = svp_w(t); else es = 0.0;
    if (t < tmelt) {
      double esice = svp_i(t), weight;
      if ((tmelt - t) > ttrice) weight = 1.0; else weight = (tmelt - t) / ttrice;
      es = weight * esice + (1.0 - weight) * es;
    }
    tbl[i] = es;
  }
  tbl[ZM_ESTBL_LEN - 1] = tbl[ZM_ESTBL_LEN - 2];
  CK(cudaMemcpyToSymbol(g_estbl, tbl, sizeof tbl));
  CK(cudaDeviceSynchronize());
  g_inited = true;
  return 0;
}

// Marks the library uninitialised and releases the CALLING thread's device arenas, streams and events
// (other threads' per-thread resources live until those threads call zm_finalize themselves or the
// process ends).
int zm_finalize(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  g_inited = false;
  cudaDeviceSynchronize();
  tls_graph.clear();
  tls_work.release(); tls_stage.release(); tls_stage2.release(); tls_mirror_ws.release(); tls_pipe.release();
  tls_tmeta.release(); tls_tmeta1.release(); tls_tmeta1c.release(); tls_tran1 = Tran1Fields{};
  tls_mirror = PbufMirror{};
  return 0;
}

int zm_last_error(char* buf, int buflen) {
  if (buf && buflen > 0) { std::strncpy(buf, tls_err.c_str(), buflen - 1); buf[buflen - 1] = 0; }
  return (int)tls_err.size();
}

#ifndef ZM_SOURCE_HASH
#define ZM_SOURCE_HASH "unknown"
#endif
// hash of the sources and flags this binary was built from (cam_nor_physics_b200/build.py compares it with the tree)
const char* zm_build_info(void) { return "ZMSRCHASH:" ZM_SOURCE_HASH " sm_100a"; }

int zm_set_profiling(int on) { g_profile = on != 0; return 0; }
long long zm_launch_count(int reset) { long long v = tls_launches; if (reset) tls_launches = 0; return v; }

int zm_get_kernel_times(int* n, const char** names, float* ms) {
  Workspace& ws = tls_work;
  int cnt = 0;
  if (ws.tev.size() >= 2) {
    cudaEventSynchronize(ws.tev.back());
    for (size_t i = 1; i < ws.tev.size() && cnt < *n; ++i, ++cnt) {
      cudaEventElapsedTime(&ms[cnt], ws.tev[i - 1], ws.tev[i]);
      names[cnt] = ws.tnames[i];
    }
  }
  *n = cnt;
  return 0;
}

// The same per-kernel times folded into the reference's GPTL timer names (t_startf / t_stopf in
// zm_conv_intr.F90:654-711 'zm_convr', :763-798 'zm_conv_evap', :821-827 'momtran', :874-880 'convtran1',
// :1019-1025 'convtran2'); the glue kernels of physics_update / physics_ptend_sum are reported beside them.
int zm_get_timers(int* n, const char** names, float* ms) {
  static const char* const gptl[] = {"zm_convr", "zm_conv_evap", "momtran", "convtran1", "convtran2", "physics_update"};
  float acc[6] = {0, 0, 0, 0, 0, 0};
  auto bucket = [](const char* k) {
    if (!strcmp(k, "zm_conv_evap")) return 1;
    if (!strcmp(k, "momtran")) return 2;
    if (!strcmp(k, "convtran1")) return 3;
    if (!strcmp(k, "convtran2")) return 4;
    if (!strcmp(k, "state_update") || !strcmp(k, "tend_finalize")) return 5;
    return 0;                                        // every kernel of zm_convr
  };
  for (Workspace* ws : {&tls_work, &tls_stage2}) {
    if (ws->tev.size() < 2) continue;
    cudaEventSynchronize(ws->tev.back());
    for (size_t i = 1; i < ws->tev.size(); ++i) {
      float t = 0.f;
      if (cudaEventElapsedTime(&t, ws->tev[i - 1], ws->tev[i]) == cudaSuccess) acc[bucket(ws->tnames[i])] += t;
    }
  }
  int cnt = 0;
  for (int j = 0; j < 6 && cnt < *n; ++j, ++cnt) { names[cnt] = gptl[j]; ms[cnt] = acc[j]; }
  *n = cnt;
  return 0;
}

// sync the thread's stream and return the Brent failure count of the last zm_convr_batch_dev
int zm_sync_check(void* stream) {
  cudaStream_t s = (cudaStream_t)stream;      // NULL = the CUDA default stream
  TendPipe& tp = tls_pipe;
  if (tp.dev_nb > 1) {                        // last device call ran as sub-batches on the library's own streams
    CK(cudaStreamSynchronize(s));
    int fails = 0;
    for (int b = tp.dev_nb - 1; b >= 0; --b) {
      const int f = read_failures(tp.work[b], tp.work[b].stream);
      if (f < 0) return f;
      fails += f;
    }
    return fails;
  }
  return read_failures(tls_work, s);
}

int zm_convr_batch_dev(int nchunks, const int* ncol, const double* t, const double* qh, double* prec,
                       double* jctop, double* jcbot, const double* pblh, const double* zm,
                       const double* geos, const double* zi, double* qtnd, double* heat,
                       const double* pap, const double* paph, const double* dpp, double delt,
                       double* mcon, double* cme, double* cape, double* eurt, const double* tpert,
                       double* dlf, double* pflx, double* zdu, double* rprd, double* mu, double* md,
                       double* du, double* eu, double* ed, double* dp, double* dsubcld, int* jt,
                       int* maxg, int* ideep, int* lengath, double* ql, double* rliq,
                       const double* landfrac, double* dif, double* dnlf, double* dnif, double* rice,
                       void* stream) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  Workspace& ws = tls_work;
  if (ws.ensure(0)) return -100;
  tls_pipe.dev_nb = 0;
  cudaStream_t s = (cudaStream_t)stream;      // NULL = the CUDA default stream
  ConvrIn in{nchunks, ncol, t, qh, pap, paph, dpp, zm, zi, geos, pblh, tpert, landfrac, delt};
  ConvrOut o{prec, jctop, jcbot, qtnd, heat, mcon, cme, cape, eurt, dlf, pflx, zdu, rprd,
             mu, md, du, eu, ed, dp, dsubcld, jt, maxg, ideep, lengath, ql, rliq, dif, dnlf, dnif, rice};
  const OrgFields of = tls_org; tls_org = OrgFields{};       // one-shot
  in.org = g_params.zm_org ? of.org : nullptr;
  return convr_launch(ws, s, in, o, true, of.orgt, of.org2d);
}

int zm_convr_batch(int nchunks, const int* ncol, const double* t, const double* qh, double* prec,
                   double* jctop, double* jcbot, const double* pblh, const double* zm,
                   const double* geos, const double* zi, double* qtnd, double* heat,
                   const double* pap, const double* paph, const double* dpp, double delt, double* mcon,
                   double* cme, double* cape, double* eurt, const double* tpert, double* dlf,
                   double* pflx, double* zdu, double* rprd, double* mu, double* md, double* du,
                   double* eu, double* ed, double* dp, double* dsubcld, int* jt, int* maxg, int* ideep,
                   int* lengath, double* ql, double* rliq, const double* landfrac, double* dif,
                   double* dnlf, double* dnif, double* rice) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc;
  const size_t n2 = nc * L, n2p = nc * (L + 1);
  Workspace& st = tls_stage;
  size_t bytes = al(nchunks, 4) + 25 * al(n2, 8) + 4 * al(n2p, 8) + 13 * al(nc, 8) + 4 * al(nc, 4) + 8192;
  if (st.ensure(bytes)) return -100;
  Stager S(st);
  const OrgFields of = tls_org; tls_org = OrgFields{};       // one-shot
  const bool org_on = g_params.zm_org != 0;
  if (org_on && !(of.org && of.orgt && of.org2d)) {
    tls_err = "zm_org = 1: call zm_org_fields(org, orgt, org2d) before zm_convr_batch";
    return -8;
  }
  const int* d_ncol = S.in(ncol, nchunks);
  ConvrIn in{nchunks, d_ncol, S.in(t, n2), S.in(qh, n2), S.in(pap, n2), S.in(paph, n2p), S.in(dpp, n2),
             S.in(zm, n2), S.in(zi, n2p), S.in(geos, nc), S.in(pblh, nc), S.in(tpert, nc),
             S.in(landfrac, nc), delt};
  ConvrOut o;
  o.prec = S.out(prec, nc); o.jctop = S.out(jctop, nc); o.jcbot = S.out(jcbot, nc);
  o.qtnd = S.out(qtnd, n2); o.heat = S.out(heat, n2); o.mcon = S.out(mcon, n2p); o.cme = S.out(cme, n2);
  o.cape = S.out(cape, nc); o.eurt = S.out(eurt, n2); o.dlf = S.out(dlf, n2); o.pflx = S.out(pflx, n2p);
  o.zdu = S.out(zdu, n2); o.rprd = S.out(rprd, n2); o.mu = S.out(mu, n2); o.md = S.out(md, n2);
  o.du = S.out(du, n2); o.eu = S.out(eu, n2); o.ed = S.out(ed, n2); o.dp = S.out(dp, n2);
  o.dsubcld = S.out(dsubcld, nc); o.jt = S.out(jt, nc); o.maxg = S.out(maxg, nc);
  o.ideep = S.out(ideep, nc); o.lengath = S.out(lengath, (size_t)nchunks); o.ql = S.out(ql, n2);
  o.rliq = S.out(rliq, nc); o.dif = S.out(dif, n2); o.dnlf = S.out(dnlf, n2); o.dnif = S.out(dnif, n2);
  o.rice = S.out(rice, nc);
  double *d_orgt = nullptr, *d_org2d = nullptr;
  if (org_on) { in.org = S.in(of.org, n2); d_orgt = S.out(of.orgt, n2); d_org2d = S.out(of.org2d, n2); }
  int rc = convr_launch(tls_work, st.stream, in, o, true, d_orgt, d_org2d);
  if (rc) return rc;
  if (S.flush()) return -100;
  return read_failures(tls_work, st.stream);
}

int zm_conv_evap_batch_dev(int nchunks, const int* ncol, const double* t, const double* pmid,
                           const double* pdel, const double* q, const double* landfrac, double* tend_s,
                           double* tend_s_snwprd, double* tend_s_snwevmlt, double* tend_q,
                           const double* prdprec, const double* cldfrc, double deltat, double* prec,
                           double* snow, double* ntprprd, double* ntsnprd, double* flxprec,
                           double* flxsnow, void* stream) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  Workspace& ws = tls_work;
  if (!ws.stream && ws.ensure(0)) return -100;
  cudaStream_t s = (cudaStream_t)stream;      // NULL = the CUDA default stream
  EvapArgs a{nchunks, ncol, t, pmid, pdel, q, landfrac, prdprec, cldfrc, tend_s, tend_s_snwprd,
             tend_s_snwevmlt, tend_q, prec, snow, ntprprd, ntsnprd, flxprec, flxsnow, deltat};
  return evap_launch(s, a);
}

int zm_conv_evap_batch(int nchunks, const int* ncol, const double* t, const double* pmid,
                       const double* pdel, const double* q, const double* landfrac, double* tend_s,
                       double* tend_s_snwprd, double* tend_s_snwevmlt, double* tend_q,
                       const double* prdprec, const double* cldfrc, double deltat, double* prec,
                       double* snow, double* ntprprd, double* ntsnprd, double* flxprec, double* flxsnow) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc;
  const size_t n2 = nc * L, n2p = nc * (L + 1);
  Workspace& st = tls_stage;
  if (st.ensure(al(nchunks, 4) + 12 * al(n2, 8) + 2 * al(n2p, 8) + 3 * al(nc, 8) + 4096)) return -100;
  Stager S(st);
  EvapArgs a;
  a.nchunks = nchunks; a.ncol = S.in(ncol, nchunks);
  a.t = S.in(t, n2); a.pmid = S.in(pmid, n2); a.pdel = S.in(pdel, n2); a.q = S.in(q, n2);
  a.landfrac = S.in(landfrac, nc); a.prdprec = S.in(prdprec, n2); a.cldfrc = S.in(cldfrc, n2);
  // tend_s / tend_q are intent(inout) in the reference but every (1:ncol, 1:pver) element is assigned
  a.tend_s = S.inout(tend_s, n2); a.tend_s_snwprd = S.inout(tend_s_snwprd, n2);
  a.tend_s_snwevmlt = S.inout(tend_s_snwevmlt, n2); a.tend_q = S.inout(tend_q, n2);
  a.prec = S.inout(prec, nc); a.snow = S.inout(snow, nc);
  a.ntprprd = S.inout(ntprprd, n2); a.ntsnprd = S.inout(ntsnprd, n2);
  a.flxprec = S.inout(flxprec, n2p); a.flxsnow = S.inout(flxsnow, n2p);
  a.deltat = deltat;
  int rc = evap_launch(st.stream, a);
  if (rc) return rc;
  return S.flush();
}

int zm_momtran_batch_dev(int nchunks, const int* ncol, const int* domomtran, const double* q, int ncnst,
                         const double* mu, const double* md, const double* du, const double* eu,
                         const double* ed, const double* dp, const double* dsubcld, const int* jt,
                         const int* mx, const int* ideep, const int* lengath, double* dqdt,
                         double* pguall, double* pgdall, double* icwu, double* icwd, double dt,
                         double* seten, void* stream) {
  NEED_INIT();
  (void)dsubcld;
  if (nchunks <= 0) return 0;
  if (ncnst != 2) { tls_err = "momtran: ncnst must be 2 (u,v), as at its only call site zm_conv_intr.F90:822"; return -6; }
  Workspace& ws = tls_work;
  if (!ws.stream && ws.ensure(0)) return -100;
  cudaStream_t s = (cudaStream_t)stream;      // NULL = the CUDA default stream
  MomArgs a;
  a.nchunks = nchunks; a.ncnst = ncnst; a.ncol = ncol; a.jt = jt; a.mx = mx; a.ideep = ideep;
  a.lengath = lengath; a.ktm = nullptr; a.kbm = nullptr; a.slots = nullptr; a.count = nullptr;
  a.domom[0] = domomtran[0]; a.domom[1] = domomtran[1];
  a.q = q; a.mu = mu; a.md = md; a.du = du; a.eu = eu; a.ed = ed; a.dp = dp;
  a.dqdt = dqdt; a.pguall = pguall; a.pgdall = pgdall; a.icwu = icwu; a.icwd = icwd; a.seten = seten;
  a.dt = dt;
  return momtran_launch(ws, s, a);
}

int zm_momtran_batch(int nchunks, const int* ncol, const int* domomtran, const double* q, int ncnst,
                     const double* mu, const double* md, const double* du, const double* eu,
                     const double* ed, const double* dp, const double* dsubcld, const int* jt,
                     const int* mx, const int* ideep, const int* lengath, double* dqdt, double* pguall,
                     double* pgdall, double* icwu, double* icwd, double dt, double* seten) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  if (ncnst != 2) { tls_err = "momtran: ncnst must be 2 (u,v)"; return -6; }
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc;
  const size_t n2 = nc * L, n3 = n2 * ncnst;
  Workspace& st = tls_stage;
  if (st.ensure(2 * al(nchunks, 4) + 7 * al(n2, 8) + 6 * al(n3, 8) + 3 * al(nc, 4) + al(nc, 8) + 4096)) return -100;
  Stager S(st);
  const int* d_ncol = S.in(ncol, nchunks);
  const int* d_len = S.in(lengath, nchunks);
  const double* d_q = S.in(q, n3);
  const double *d_mu = S.in(mu, n2), *d_md = S.in(md, n2), *d_du = S.in(du, n2), *d_eu = S.in(eu, n2),
               *d_ed = S.in(ed, n2), *d_dp = S.in(dp, n2);
  const int *d_jt = S.in(jt, nc), *d_mx = S.in(mx, nc), *d_id = S.in(ideep, nc);
  // dqdt(:,:,m) is only written for active m; icwu/icwd only for i <= ncol: stage as inout
  double* d_dqdt = S.inout(dqdt, n3);
  double* d_pgu = S.out(pguall, n3); double* d_pgd = S.out(pgdall, n3);
  double* d_icwu = S.inout(icwu, n3); double* d_icwd = S.inout(icwd, n3);
  double* d_seten = S.out(seten, n2);
  int rc = zm_momtran_batch_dev(nchunks, d_ncol, domomtran, d_q, ncnst, d_mu, d_md, d_du, d_eu, d_ed, d_dp,
                                dsubcld, d_jt, d_mx, d_id, d_len, d_dqdt, d_pgu, d_pgd, d_icwu, d_icwd, dt,
                                d_seten, (void*)st.stream);
  if (rc) return rc;
  return S.flush();
}

int zm_convtran_batch_dev(int nchunks, const int* doconvtran, const double* q, int ncnst, const double* mu,
                          const double* md, const double* du, const double* eu, const double* ed,
                          const double* dp, const double* dsubcld, const int* jt, const int* mx,
                          const int* ideep, const int* lengath, const double* fracis, double* dqdt,
                          const double* dpdry, double dt, const int* cnst_is_dry, void* stream) {
  NEED_INIT();
  (void)dsubcld; (void)dt;
  if (nchunks <= 0) return 0;
  Workspace& ws = tls_work;
  if (!ws.stream && ws.ensure(0)) return -100;
  cudaStream_t s = (cudaStream_t)stream;      // NULL = the CUDA default stream
  TranArgs a;
  a.nchunks = nchunks; a.ncnst = ncnst; a.nactive = 0; a.jt = jt; a.mx = mx; a.ideep = ideep;
  a.lengath = lengath; a.ktm = nullptr; a.kbm = nullptr; a.active = nullptr; a.is_dry = nullptr;
  a.q = q; a.fracis = fracis; a.mu = mu; a.md = md; a.du = du; a.eu = eu; a.ed = ed; a.dp = dp;
  a.dpdry = dpdry; a.dqdt = dqdt;
  return convtran_launch(ws, s, a, doconvtran, cnst_is_dry);
}

int zm_convtran_batch(int nchunks, const int* doconvtran, const double* q, int ncnst, const double* mu,
                      const double* md, const double* du, const double* eu, const double* ed,
                      const double* dp, const double* dsubcld, const int* jt, const int* mx,
                      const int* ideep, const int* lengath, const double* fracis, double* dqdt,
                      const double* dpdry, double dt, const int* cnst_is_dry) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc;
  const size_t n2 = nc * L, n3 = n2 * ncnst;
  Workspace& st = tls_stage;
  if (st.ensure(al(nchunks, 4) + 7 * al(n2, 8) + 3 * al(n3, 8) + 3 * al(nc, 4) + 4096)) return -100;
  Stager S(st);
  const int* d_len = S.in(lengath, nchunks);
  const double *d_q = S.in(q, n3), *d_fr = S.in(fracis, n3);
  const double *d_mu = S.in(mu, n2), *d_md = S.in(md, n2), *d_du = S.in(du, n2), *d_eu = S.in(eu, n2),
               *d_ed = S.in(ed, n2), *d_dp = S.in(dp, n2), *d_dpd = S.in(dpdry, n2);
  const int *d_jt = S.in(jt, nc), *d_mx = S.in(mx, nc), *d_id = S.in(ideep, nc);
  double* d_dqdt = S.inout(dqdt, n3);      // inactive constituents keep the caller's values
  int rc = zm_convtran_batch_dev(nchunks, doconvtran, d_q, ncnst, d_mu, d_md, d_du, d_eu, d_ed, d_dp,
                                 dsubcld, d_jt, d_mx, d_id, d_len, d_fr, d_dqdt, d_dpd, dt, cnst_is_dry,
                                 (void*)st.stream);
  if (rc) return rc;
  return S.flush();
}

// zm_conv_tend (zm_conv_intr.F90:390-951, microphysics/org/convtran1 parts excluded): zm_convr ->
// physics_update -> zm_conv_evap -> momtran, everything resident on the device.
}  // extern "C"
namespace {
// events the host-pointer API uses to overlap PCIe copies with the kernels
struct TendHooks { cudaEvent_t late_inputs; cudaEvent_t convr_done; };
int conv_tend_impl(Workspace& ws, int nchunks, const int* ncol, const double* t, const double* q, const double* u,
                           const double* v, const double* pmid, const double* pint, const double* pdel,
                           const double* zm, const double* zi, const double* phis, const double* pblh,
                           const double* tpert, const double* landfrac, const double* cld, double ztodt,
                           double* ptend_s, double* ptend_q, double* ptend_u, double* ptend_v, double* mcon,
                           double* cme, double* pflx, double* zdu, double* rliq, double* rice, double* jctop,
                           double* jcbot, double* prec, double* snow, double* ql, double* rprd,
                           double* evapcdp, double* flxprec, double* flxsnow, double* dlf, double* mu,
                           double* md, double* du, double* eu, double* ed, double* dp, double* dsubcld,
                           int* jt, int* maxg, int* ideep, int* lengath, double* cape, void* stream,
                           const TendHooks* hooks, const double* org = nullptr, double* orgt = nullptr,
                           double* org2d = nullptr, const Tran1Dev* tr1 = nullptr, const HistFields* hist = nullptr) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc;
  const size_t n2 = nc * L, n2p = nc * (L + 1);
  const HistFields H = hist ? *hist : HistFields{};
  if (ws.ensure(convr_work_bytes(nc, (int)L) + 19 * al(n2, 8) + 6 * al(2 * n2, 8) + chunk_bounds_bytes(nchunks, (int)nc) + 8192 +
                (H.any() ? 4 * al(n2, 8) + 4 * al(2 * n2, 8) : 0)))
    return -100;
  cudaStream_t s = (cudaStream_t)stream;      // NULL = the CUDA default stream
  // History fields (zm_conv_tend_hist_fields): an attached field is written where it is computed; heat, qtnd, tend_s
  // and seten are needed anyway and live in scratch otherwise.  eurt, dif, dnlf, dnif of zm_convr, zm_conv_evap's four
  // diagnostics and momtran's pguall / pgdall / icwu / icwd are not materialised unless attached; the kernels store
  // the last two groups as a whole, so an attached group gets scratch for its unattached members.
  auto own = [&](int j, size_t n) { return H.p[j] ? H.p[j] : ws.take<double>(n); };
  const bool hist_evap = H.p[H_TEND_S] || H.p[H_SNWPRD] || H.p[H_SNWEVMLT] || H.p[H_NTPRPRD] || H.p[H_NTSNPRD];
  const bool hist_mom = H.p[H_PGUALL] || H.p[H_PGDALL] || H.p[H_ICWU] || H.p[H_ICWD];
  double *heat = own(H_HEAT, n2), *qtnd = own(H_QTND, n2), *eurt = H.p[H_EURT], *dif = H.p[H_DIF],
         *dnlf = H.p[H_DNLF], *dnif = H.p[H_DNIF], *t1 = ws.take<double>(n2), *q1 = ws.take<double>(n2),
         *ev_s = own(H_TEND_S, n2), *ev_q_scratch = ws.take<double>(n2), *snwprd = nullptr, *snwevmlt = nullptr,
         *ntprprd = nullptr, *ntsnprd = nullptr, *seten = own(H_SETEN, n2);
  double *winds = ws.take<double>(2 * n2), *wtend = ws.take<double>(2 * n2), *pgu = nullptr, *pgd = nullptr,
         *icwu = nullptr, *icwd = nullptr;
  if (hist_evap) {
    snwprd = own(H_SNWPRD, n2); snwevmlt = own(H_SNWEVMLT, n2); ntprprd = own(H_NTPRPRD, n2); ntsnprd = own(H_NTSNPRD, n2);
  }
  if (hist_mom) {
    pgu = own(H_PGUALL, 2 * n2); pgd = own(H_PGDALL, 2 * n2); icwu = own(H_ICWU, 2 * n2); icwd = own(H_ICWD, 2 * n2);
  }
  // zm_conv_evap's tend_q IS evapcdp (zm_conv_intr.F90:764-769 passes ptend_loc%q(:,:,1), :796 outputs it): written in place
  double* ev_q = evapcdp ? evapcdp : ev_q_scratch;
  const bool do_mom = !g_params.cam3;          // zm_conv_intr.F90:808: momentum transport is non-cam3 physics
  // momtran reads state%u / state%v and writes ptend_u / ptend_v directly when they can take 16-byte stores
  const bool split_env = !(getenv("ZM_TEND_SPLIT_WINDS") && atoi(getenv("ZM_TEND_SPLIT_WINDS")) == 0);   // 0: round-2a glue
  const bool split = split_env && do_mom && !(n2 & 1) &&
                     (((uintptr_t)ptend_u | (uintptr_t)ptend_v | (uintptr_t)seten) & 15) == 0;
  ConvrIn in{nchunks, ncol, t, q, pmid, pint, pdel, zm, zi, phis, pblh, tpert, landfrac, 0.5 * ztodt};
  ConvrOut o{prec, jctop, jcbot, qtnd, heat, mcon, cme, cape, eurt, dlf, pflx, zdu, rprd,
             mu, md, du, eu, ed, dp, dsubcld, jt, maxg, ideep, lengath, ql, rliq, dif, dnlf, dnif, rice};
  o.mcon_kgm2s = split_env ? 1 : 0;            // unit conversion of zm_conv_intr.F90:693 inside the plume kernel
  in.org = g_params.zm_org ? org : nullptr;
  // split winds: ptend_u / ptend_v / seten are zero outside the convective columns momtran writes -- filled with
  // zm_convr's own outputs at the start of the step
  FillList xf{};
  auto xadd = [&](double* p, size_t n) { xf.p[xf.cnt] = p; xf.n[xf.cnt] = n; ++xf.cnt; };
  if (split) { xadd(ptend_u, n2); xadd(ptend_v, n2); xadd(seten, n2); }
  // momtran's diagnostics: pguall / pgdall are zero outside the convective columns; with cam3 (no momtran,
  // zm_conv_intr.F90:808) all five momtran fields return 0
  if (hist_mom) { xadd(pgu, 2 * n2); xadd(pgd, 2 * n2); }
  if (!do_mom) {
    if (H.p[H_SETEN]) xadd(seten, n2);
    if (hist_mom) { xadd(icwu, 2 * n2); xadd(icwd, 2 * n2); }
  }
  int rc = convr_launch(ws, s, in, o, false, orgt, org2d, xf.cnt ? &xf : nullptr);
  if (rc) return rc;
  if (hooks) {
    CK(cudaEventRecord(hooks->convr_done, s));            // zm_convr outputs are final from here on
    CK(cudaStreamWaitEvent(s, hooks->late_inputs, 0));    // u, v, cld have arrived
  }
  const int nper = (int)(pc * L);
  EvapArgs ea{nchunks, ncol, t1, pmid, pdel, q1, landfrac, rprd, cld, ev_s, snwprd, snwevmlt, ev_q,
              prec, snow, ntprprd, ntsnprd, flxprec, flxsnow, ztodt};
  // zm_conv_evap and momtran both depend only on zm_convr's outputs (zm_conv_intr.F90:764, 822): evap
  // (with the t, q half of the state update) goes to a side stream and overlaps momtran (which only waits for
  // the wind half); kept serial while per-kernel profiling is on
  const bool fork = !g_profile;
  // With the split winds nothing but zm_conv_evap needs the updated state: the kernel applies physics_update to its
  // own operands and stores heat + tend_s / qtnd + tend_q straight into ptend_s / ptend_q (k_conv_evap<true>); what is
  // left for the end of the step is ptend_s += seten.  ZM_TEND_FUSE_EVAP=0: separate state update and final sum.
  const bool fuse_evap = split && o.mcon_kgm2s && (((uintptr_t)ptend_s) & 15) == 0 &&
                         !(getenv("ZM_TEND_FUSE_EVAP") && atoi(getenv("ZM_TEND_FUSE_EVAP")) == 0);
  if (fuse_evap) {     // tend_s stays: k_conv_evap<true, true> also stores it and the four snow diagnostics
    ea.t = t; ea.q = q; ea.heat = heat; ea.qtnd = qtnd; ea.ps = ptend_s; ea.pq = ptend_q;
    if (!hist_evap) ea.tend_s = nullptr;
  }
  if (fork) {
    if (ws.ensure_side()) return -100;
    CK(cudaEventRecord(ws.ev_fork, s));
    CK(cudaStreamWaitEvent(ws.side, ws.ev_fork, 0));
    if (!fuse_evap) {
      k_state_update<1><<<1184, 256, 0, ws.side>>>((int)n2, nper, t, q, heat, qtnd, u, v, ztodt, t1, q1, winds);
      ++tls_launches;
    }
    if (do_mom && !split) {     // packed winds feed momtran only
      k_state_update<2><<<1184, 256, 0, s>>>((int)n2, nper, t, q, heat, qtnd, u, v, ztodt, t1, q1, winds);
      ++tls_launches;
    }
  } else if (!fuse_evap) {
    k_state_update<0><<<1184, 256, 0, s>>>((int)n2, nper, t, q, heat, qtnd, u, v, ztodt, t1, q1, winds);
    ++tls_launches;
  }
  tick(ws, s, "state_update");
  rc = evap_launch(fork ? ws.side : s, ea);
  if (rc) return rc;
  if (g_params.zm_org) {     // zm_conv_intr.F90:773-777 (needs evapcdp = ev_q)
    k_org_tend<<<1184, 256, 0, fork ? ws.side : s>>>(nchunks, ncol, org, ev_q, ztodt, orgt); ++tls_launches;
  }
  if (fork) CK(cudaEventRecord(ws.ev_join, ws.side));
  tick(ws, s, "zm_conv_evap");
  const bool do_tran1 = tr1 && tr1->nactive > 0;
  ChunkBounds cb;
  if (do_mom || do_tran1) {
    rc = chunk_bounds_enqueue(ws, s, nchunks, jt, maxg, lengath, cb);
    if (rc) return rc;
  }
  // convtran1 depends on zm_convr's outputs and the chunk bounds only (the constituents it moves are not touched by
  // the state update): with the fork it runs on a second side stream beside momtran and zm_conv_evap
  cudaStream_t tran_stream = s;
  if (fork && do_tran1) {
    if (ws.ensure_side2()) return -100;
    CK(cudaEventRecord(ws.ev_fork2, s));
    CK(cudaStreamWaitEvent(ws.side2, ws.ev_fork2, 0));
    tran_stream = ws.side2;
  }
  if (do_mom) {
    MomArgs ma;
    ma.nchunks = nchunks; ma.ncnst = 2; ma.ncol = ncol; ma.jt = jt; ma.mx = maxg; ma.ideep = ideep;
    ma.lengath = lengath; ma.ktm = nullptr; ma.kbm = nullptr; ma.domom[0] = 1; ma.domom[1] = 1;
    ma.q = winds; ma.mu = mu; ma.md = md; ma.du = du; ma.eu = eu; ma.ed = ed; ma.dp = dp;
    ma.dqdt = wtend; ma.pguall = pgu; ma.pgdall = pgd; ma.icwu = icwu; ma.icwd = icwd; ma.seten = seten;
    ma.dt = ztodt;
    if (split) { ma.q_u = u; ma.q_v = v; ma.dq_u = ptend_u; ma.dq_v = ptend_v; }
    if (hist_mom) { k_icw_init<<<1184, 256, 0, s>>>(nchunks, ncol, u, v, icwu, icwd); ++tls_launches; }
    rc = momtran_launch(ws, s, ma, false, &cb);
    if (rc) return rc;
  }
  tick(ws, s, "momtran");
  if (do_tran1) {
    // convtran1 (zm_conv_intr.F90:865-880) on state1%q: its constituents m >= 2 are the caller's (only q(:,:,1)
    // was updated); fake_dpdry = 0 (the transported species are moist; a zeroed array stands in if one is 'dry')
    double* fake_dpdry = ws.take<double>(n2);
    if (tr1->any_dry) CK(cudaMemsetAsync(fake_dpdry, 0, n2 * sizeof(double), tran_stream));
    TranArgs ta;
    ta.nchunks = nchunks; ta.ncnst = tr1->ncnst; ta.nactive = tr1->nactive; ta.jt = jt; ta.mx = maxg; ta.ideep = ideep;
    ta.lengath = lengath; ta.active = tr1->active; ta.is_dry = tr1->is_dry;
    ta.q = tr1->q; ta.fracis = tr1->fracis; ta.mu = mu; ta.md = md; ta.du = du; ta.eu = eu; ta.ed = ed; ta.dp = dp;
    ta.dpdry = fake_dpdry; ta.dqdt = tr1->dqdt;
    rc = convtran_enqueue(tran_stream, ta, cb);
    if (rc) return rc;
    if (tran_stream != s) CK(cudaEventRecord(ws.ev_join2, ws.side2));
    tick(ws, s, "convtran1");
  }
  if (tran_stream != s) CK(cudaStreamWaitEvent(s, ws.ev_join2, 0));
  if (fork) CK(cudaStreamWaitEvent(s, ws.ev_join, 0));
  if (fuse_evap) {
    k_add_seten<<<1184, 256, 0, s>>>(n2 / 2, (double2*)ptend_s, (const double2*)seten);
  } else {
    auto fin = !do_mom ? (o.mcon_kgm2s ? k_tend_finalize<0, false> : k_tend_finalize<0, true>)
               : split ? (o.mcon_kgm2s ? k_tend_finalize<2, false> : k_tend_finalize<2, true>)
                       : (o.mcon_kgm2s ? k_tend_finalize<1, false> : k_tend_finalize<1, true>);
    fin<<<1184, 256, 0, s>>>((int)n2, (int)n2p, nper, heat, qtnd, ev_s, ev_q, seten, wtend, ptend_s, ptend_q, ptend_u,
                             ptend_v, evapcdp ? evapcdp : ev_q, mcon);
  }
  ++tls_launches;
  tick(ws, s, "tend_finalize");
  CK(cudaGetLastError());
  return 0;
}
}  // namespace
extern "C" {

int zm_conv_tend_batch_dev(int nchunks, const int* ncol, const double* t, const double* q, const double* u,
                           const double* v, const double* pmid, const double* pint, const double* pdel,
                           const double* zm, const double* zi, const double* phis, const double* pblh,
                           const double* tpert, const double* landfrac, const double* cld, double ztodt,
                           double* ptend_s, double* ptend_q, double* ptend_u, double* ptend_v, double* mcon,
                           double* cme, double* pflx, double* zdu, double* rliq, double* rice, double* jctop,
                           double* jcbot, double* prec, double* snow, double* ql, double* rprd,
                           double* evapcdp, double* flxprec, double* flxsnow, double* dlf, double* mu,
                           double* md, double* du, double* eu, double* ed, double* dp, double* dsubcld,
                           int* jt, int* maxg, int* ideep, int* lengath, double* cape, void* stream) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  // Optionally cut the batch into sub-batches of whole chunks that run on their own (prioritised) streams:
  // every kernel of the path is latency-bound at low occupancy, so the passes of different sub-batches
  // fill each other's idle issue slots.  ZM_DEV_SUBBATCHES = 1 keeps everything on `stream`.
  TendPipe& tp = tls_pipe;
  int NB = 1;
  if (const char* e = getenv("ZM_DEV_SUBBATCHES")) NB = atoi(e);
  NB = NB < 1 ? 1 : (NB > TendPipe::MAXB ? TendPipe::MAXB : NB);
  while (NB > 1 && nchunks / NB < 128) --NB;
  tp.dev_nb = 0;
  const OrgFields of = tls_org; tls_org = OrgFields{};       // one-shot
  const Tran1Fields tf = tls_tran1; tls_tran1 = Tran1Fields{};   // one-shot
  const HistFields hf = tls_hist; tls_hist = HistFields{};       // one-shot
  const HistFields* hfp = hf.any() ? &hf : nullptr;
  Tran1Dev td{};
  const Tran1Dev* tdp = nullptr;
  if (tf.pcnst > 0) {
    const int n = tf.pcnst;
    if (tls_tmeta1.set(tls_tran1_flags.data(), tls_tran1_flags.data() + n, n)) return -100;
    td = Tran1Dev{n, tls_tmeta1.nactive, tls_tmeta1.active(), tls_tmeta1.dry(), tls_tmeta1.any_dry, tf.q, tf.fracis, tf.ptend_q};
    tdp = &td;
  }
  if (NB == 1 || g_profile) {
    auto direct = [&](Workspace& ws, void* on) {
      return conv_tend_impl(ws, nchunks, ncol, t, q, u, v, pmid, pint, pdel, zm, zi, phis, pblh, tpert, landfrac,
                            cld, ztodt, ptend_s, ptend_q, ptend_u, ptend_v, mcon, cme, pflx, zdu, rliq, rice, jctop,
                            jcbot, prec, snow, ql, rprd, evapcdp, flxprec, flxsnow, dlf, mu, md, du, eu, ed, dp,
                            dsubcld, jt, maxg, ideep, lengath, cape, on, nullptr, of.org, of.orgt, of.org2d, tdp, hfp);
    };
    static const bool use_graph = !(getenv("ZM_DEV_GRAPH") && atoi(getenv("ZM_DEV_GRAPH")) == 0);
    if (g_profile || !use_graph) { tls_graph.clear(); return direct(tls_work, stream); }
    Workspace& ws = tls_work;
    TendGraph& G = tls_graph;
    double zt = ztodt; const void* ztbits; std::memcpy(&ztbits, &zt, sizeof ztbits);
    std::vector<const void*> key = {ncol, t, q, u, v, pmid, pint, pdel, zm, zi, phis, pblh, tpert, landfrac, cld,
        ptend_s, ptend_q, ptend_u, ptend_v, mcon, cme, pflx, zdu, rliq, rice, jctop, jcbot, prec, snow, ql, rprd,
        evapcdp, flxprec, flxsnow, dlf, mu, md, du, eu, ed, dp, dsubcld, jt, maxg, ideep, lengath, cape,
        of.org, of.orgt, of.org2d, ztbits, (const void*)(size_t)nchunks, (const void*)(size_t)g_epoch,
        tf.q, tf.fracis, tf.ptend_q, (const void*)(size_t)tf.pcnst, (const void*)tls_tmeta1.d,
        (const void*)(size_t)(tdp ? tls_tmeta1.version : 0)};
    // attached history fields: a replay must write where this call asked, and attaching or detaching recaptures
    key.insert(key.end(), hf.p, hf.p + H_N);
    key.push_back((const void*)ws.dbuf); key.push_back((const void*)ws.dcap);
    cudaStream_t s = (cudaStream_t)stream;
    if (key == G.key) {
      if (!G.exec) {                                   // second identical call: capture on the library's own stream
        cudaGraph_t graph = nullptr;
        const long long l0 = tls_launches;
        bool ok = ws.stream && cudaStreamBeginCapture(ws.stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
        if (ok) {
          const int rc = direct(ws, (void*)ws.stream);
          const cudaError_t ee = cudaStreamEndCapture(ws.stream, &graph);
          ok = rc == 0 && ee == cudaSuccess && graph && cudaGraphInstantiate(&G.exec, graph, 0) == cudaSuccess;
          if (graph) cudaGraphDestroy(graph);
        }
        G.launches = tls_launches - l0;
        tls_launches = l0;                             // captured launches did not run
        if (!ok) { cudaGetLastError(); G.clear(); return direct(ws, stream); }
      }
      CK(cudaGraphLaunch(G.exec, s));
      tls_launches += G.launches;
      return 0;
    }
    G.clear();
    const int rc = direct(ws, stream);                 // first call with these arguments: run, remember
    if (rc == 0) {
      G.key = key;
      G.key[G.key.size() - 2] = (const void*)ws.dbuf;  // the arena may have been (re)allocated by this call
      G.key[G.key.size() - 1] = (const void*)ws.dcap;
    }
    return rc;
  }
  if (tp.init(NB)) return -100;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t pc = g_params.pcols, L = g_params.pver, s2 = pc * L, s2p = pc * (L + 1), s1 = pc;
  CK(cudaEventRecord(tp.in_ready[0], s));
  for (int b = 0; b < NB; ++b) {
    const int c0 = tp.first(b, nchunks, NB), nb = tp.first(b + 1, nchunks, NB) - c0;
    Workspace& ws = tp.work[b];
    ws.chunk0 = c0;
    CK(cudaStreamWaitEvent(ws.stream, tp.in_ready[0], 0));
    Tran1Dev tb = td;            // this sub-batch's slice of the constituent arrays
    if (tdp) {
      const size_t o3 = (size_t)c0 * s2 * td.ncnst;
      tb.q = td.q + o3; tb.fracis = td.fracis + o3; tb.dqdt = td.dqdt + o3;
    }
    const HistFields hb = hf.slice(c0, s2);
#define O2(x)  ((x) + (size_t)c0 * s2)
#define O2P(x) ((x) + (size_t)c0 * s2p)
#define O1(x)  ((x) + (size_t)c0 * s1)
    int rc = conv_tend_impl(ws, nb, ncol + c0, O2(t), O2(q), O2(u), O2(v), O2(pmid), O2P(pint), O2(pdel), O2(zm),
                            O2P(zi), O1(phis), O1(pblh), O1(tpert), O1(landfrac), O2(cld), ztodt, O2(ptend_s),
                            O2(ptend_q), O2(ptend_u), O2(ptend_v), O2P(mcon), O2(cme), O2P(pflx), O2(zdu), O1(rliq),
                            O1(rice), O1(jctop), O1(jcbot), O1(prec), O1(snow), O2(ql), O2(rprd), O2(evapcdp),
                            O2P(flxprec), O2P(flxsnow), O2(dlf), O2(mu), O2(md), O2(du), O2(eu), O2(ed), O2(dp),
                            O1(dsubcld), O1(jt), O1(maxg), O1(ideep), lengath + c0, O1(cape), (void*)ws.stream, nullptr,
                            of.org ? O2(of.org) : nullptr, of.orgt ? O2(of.orgt) : nullptr,
                            of.org2d ? O2(of.org2d) : nullptr, tdp ? &tb : nullptr, hfp ? &hb : nullptr);
#undef O2
#undef O2P
#undef O1
    if (rc) return rc;
    CK(cudaEventRecord(tp.done[b], ws.stream));
    CK(cudaStreamWaitEvent(s, tp.done[b], 0));
  }
  tp.dev_nb = NB;
  return 0;
}

// The host-pointer step behind zm_conv_tend_batch (g == NULL) and zm_conv_tend_batch_gathered (g != NULL: the
// (pcols,pver[p]) outputs are packed into records that go to g->rec instead of being copied back whole; their
// pointers are NULL here).
static int conv_tend_batch(int nchunks, const int* ncol, const double* t, const double* q, const double* u,
                           const double* v, const double* pmid, const double* pint, const double* pdel,
                           const double* zm, const double* zi, const double* phis, const double* pblh,
                           const double* tpert, const double* landfrac, const double* cld, double ztodt,
                           double* ptend_s, double* ptend_q, double* ptend_u, double* ptend_v, double* mcon,
                           double* cme, double* pflx, double* zdu, double* rliq, double* rice, double* jctop,
                           double* jcbot, double* prec, double* snow, double* ql, double* rprd, double* evapcdp,
                           double* flxprec, double* flxsnow, double* dlf, double* mu, double* md, double* du,
                           double* eu, double* ed, double* dp, double* dsubcld, int* jt, int* maxg, int* ideep,
                           int* lengath, double* cape, const GatheredOut* g) {
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc;
  const size_t n2 = nc * L, n2p = nc * (L + 1);
  Workspace& st = tls_stage;
  tls_mirror = PbufMirror{};                 // whatever happens below, the previous step's mirror is gone
  const HistFields hf = tls_hist; tls_hist = HistFields{};       // one-shot
  size_t hist_bytes = 0;                     // staging of the attached history fields
  for (int j = 0; j < H_N; ++j)
    if (hf.p[j]) hist_bytes += al(HistFields::is3d(j) ? 2 * n2 : n2, 8);
  if (st.ensure(al(nchunks, 4) + 27 * al(n2, 8) + 6 * al(n2p, 8) + 14 * al(nc, 8) + 4 * al(nc, 4) + 8192 +
                al(nc * (20 * L + 4), 8) + al((size_t)nchunks + 16, 4) + hist_bytes))
    return -100;
  Workspace& mw = tls_mirror_ws;
  if (mw.ensure(6 * al(n2, 8) + al(nc, 8) + 3 * al(nc, 4) + al(nchunks, 4) + 4096)) return -100;
  // The batch is cut into NB sub-batches of whole chunks (columns are independent).  Sub-batch b's inputs
  // travel host->device while sub-batch b-1 computes, and its outputs travel back while sub-batch b+1
  // computes: PCIe (both directions) and the SMs are busy at the same time.  Every array keeps ONE
  // device allocation for the whole batch (sub-batches are chunk slices of it), so the pbuf mirror that
  // zm_conv_tend_2_batch reads stays contiguous.
  TendPipe& tp = tls_pipe;
  const auto wall0 = std::chrono::steady_clock::now();
  auto wall_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count(); };
  const bool dbg = getenv("ZM_TEND_DEBUG") != nullptr;
  const int NB = tp.plan(nchunks);
  if (tp.init(NB)) return -100;
  const size_t s2 = pc * L, s2p = pc * (L + 1), s1 = pc;            // per-chunk strides
  // kind 0 in, 1 late in, 2 early out, 3 final out; per-column/per-chunk arrays are small and travel once for the
  // whole batch (4: in, before the first sub-batch; 5: out, after the last) instead of once per sub-batch
  struct Arr { const void* h; void* d; size_t stride, esz; int kind; };
  std::vector<Arr> arrs; arrs.reserve(64);
  // Return path of the 2-D outputs: dense (default) copies the arrays whole; ZM_TEND_RETURN=sparse moves only the
  // convective columns' records and scatters them on the host into the arrays worker threads zero-filled meanwhile.
  // The sparse path moves a third of the bytes over PCIe but writes the caller's arrays with CPU stores, and on a
  // host whose memory bandwidth is of the order of the PCIe rate (the B200 boxes of this project: 70-78 GB/s for a
  // parallel memset against 56 GB/s D2H) that costs more than it saves -- measured 11.7 against 8.2 ms per f09 step
  // (DESIGN.md section 5) -- so it is opt-in, for hosts with memory bandwidth to spare.
  // ZM_TEND_OUTPUTS_PREZEROED=1: the caller's arrays are all-zero on entry (as after physics_ptend_init), the
  // zero-fill is skipped.  The gathered entry point ignores ZM_TEND_RETURN: its records are its return path.
  const char* ret_env = getenv("ZM_TEND_RETURN");
  const bool sparse = !g && ret_env && !strcmp(ret_env, "sparse");
  const bool prezeroed = getenv("ZM_TEND_OUTPUTS_PREZEROED") && atoi(getenv("ZM_TEND_OUTPUTS_PREZEROED")) != 0;
  double* sf_host[SF_N] = {};               // caller's arrays of the sparse fields (NULL: not wanted)
  double* sf_dev[SF_N] = {};
  int sf_next = -1;                          // id of the sparse field the next dev() call stages
  bool to_mirror = false;                    // the pbuf fields go to the mirror arena
  auto dev = [&](const void* h, size_t stride, size_t esz, int kind, bool always = true) -> void* {
    void* d = (void*)(to_mirror ? mw : st).take<char>((size_t)nchunks * stride * esz);
    if (stride <= pc) kind = (kind <= 1) ? 4 : 5;
    if (sf_next >= 0) {
      sf_host[sf_next] = (double*)h; sf_dev[sf_next] = (double*)d;
      if (sparse && h) kind = 6;             // no dense copy: travels in the records
      sf_next = -1;
    }
    if (h || always) arrs.push_back({h, d, stride, esz, h ? kind : -1});
    return d;
  };
#define DIN(x, str)   (const double*)dev(x, str, 8, 0)
#define DLATE(x, str) (const double*)dev(x, str, 8, 1)
#define DOUTE(x, str) (double*)dev(x, str, 8, 2)
#define DOUTF(x, str) (double*)dev(x, str, 8, 3)
#define SPE(id, x, str) (sf_next = id, DOUTE(x, str))
#define SPF(id, x, str) (sf_next = id, DOUTF(x, str))
  const int* d_ncol = (const int*)dev(ncol, 1, 4, 0);
  const double *d_t = DIN(t, s2), *d_q = DIN(q, s2), *d_pmid = DIN(pmid, s2), *d_pint = DIN(pint, s2p),
               *d_pdel = DIN(pdel, s2), *d_zm = DIN(zm, s2), *d_zi = DIN(zi, s2p), *d_phis = DIN(phis, s1),
               *d_pblh = DIN(pblh, s1), *d_tpert = DIN(tpert, s1), *d_lf = DIN(landfrac, s1);
  const double *d_u = DLATE(u, s2), *d_v = DLATE(v, s2), *d_cld = DLATE(cld, s2);
  to_mirror = true;
  double *d_mu = SPE(SF_MU, mu, s2), *d_md = SPE(SF_MD, md, s2), *d_du = SPE(SF_DU, du, s2), *d_eu = SPE(SF_EU, eu, s2),
         *d_ed = SPE(SF_ED, ed, s2), *d_dp = SPE(SF_DP, dp, s2), *d_dsub = DOUTE(dsubcld, s1);
  // gathered: lengath returns per sub-batch, ahead of that sub-batch's records (below), not with the batch's end
  int *d_jt = (int*)dev(jt, s1, 4, 2), *d_maxg = (int*)dev(maxg, s1, 4, 2), *d_ideep = (int*)dev(ideep, s1, 4, 2),
      *d_len = (int*)dev(g ? nullptr : lengath, 1, 4, 2);
  to_mirror = false;
  const PbufMirror new_mirror{nchunks, d_mu, d_md, d_du, d_eu, d_ed, d_dp, d_dsub, d_jt, d_maxg, d_ideep, d_len};
  double *d_ps = SPF(SF_PS, ptend_s, s2), *d_pq = SPF(SF_PQ, ptend_q, s2), *d_pu = SPF(SF_PU, ptend_u, s2),
         *d_pv = SPF(SF_PV, ptend_v, s2), *d_mcon = SPF(SF_MCON, mcon, s2p), *d_cme = SPE(SF_CME, cme, s2),
         *d_pflx = SPE(SF_PFLX, pflx, s2p), *d_zdu = SPE(SF_ZDU, zdu, s2),
         *d_rliq = DOUTE(rliq, s1), *d_rice = DOUTE(rice, s1), *d_jctop = DOUTE(jctop, s1), *d_jcbot = DOUTE(jcbot, s1),
         *d_prec = DOUTF(prec, s1), *d_snow = DOUTF(snow, s1), *d_ql = SPE(SF_QL, ql, s2), *d_rprd = SPE(SF_RPRD, rprd, s2),
         *d_evap = SPF(SF_EVAP, evapcdp, s2), *d_fp = SPF(SF_FP, flxprec, s2p), *d_fs = SPF(SF_FS, flxsnow, s2p),
         *d_dlf = SPE(SF_DLF, dlf, s2), *d_cape = DOUTE(cape, s1);
  const OrgFields of = tls_org; tls_org = OrgFields{};       // one-shot
  const double* d_org = nullptr; double *d_orgt = nullptr, *d_org2d = nullptr;
  if (g_params.zm_org) {
    if (!(of.org && of.orgt && of.org2d)) {
      tls_err = "zm_org = 1: call zm_org_fields(org, orgt, org2d) before zm_conv_tend_batch";
      return -8;
    }
    d_org = DIN(of.org, s2); d_org2d = DOUTE(of.org2d, s2); d_orgt = DOUTF(of.orgt, s2);
  }
  // history fields travel whole, also under ZM_TEND_RETURN=sparse: zm_convr's as soon as the plume kernel is done,
  // zm_conv_evap's and momtran's at the end of the sub-batch
  HistFields dh;
  for (int j = 0; j < H_N; ++j)
    if (hf.p[j]) dh.p[j] = (double*)dev(hf.p[j], HistFields::is3d(j) ? 2 * s2 : s2, 8, j <= H_DNIF ? 2 : 3);
  const bool hist_on = hf.any();
#undef DIN
#undef DLATE
#undef DOUTE
#undef DOUTF
#undef SPE
#undef SPF
  // sparse return: record layout (fields the caller asked for), device record buffer sized for the worst case so
  // that a sub-batch's region does not depend on the counts of the others.  gathered: the 14 column-indexed fields,
  // then the pbuf fields if asked for.
  int sf_off[SF_N], rec_len = 0;
  for (int qf = 0; qf < SF_N; ++qf) {
    const int nlev = (qf >= SF_MCON && qf <= SF_FS) ? (int)L + 1 : (int)L;
    const bool packed = sparse ? sf_host[qf] != nullptr : (g && (qf < SF_MU || g->pbuf));
    if (packed) { sf_off[qf] = rec_len; rec_len += nlev; } else sf_off[qf] = -1;
  }
  double* d_rec = nullptr; int* d_base = nullptr;
  if (rec_len > 0) {
    d_rec = st.take<double>(nc * rec_len);
    d_base = st.take<int>((size_t)nchunks + TendPipe::MAXB + 1);
    if (sparse && tp.ensure_pinned(0, 2 * (nc + nchunks + 2 * TendPipe::MAXB))) return -100;
  }
  // convtran1 (zm_conv_intr.F90:865-880): only the slices of the transported constituents travel; on the device
  // they are stored compactly, (pcols,pver,nactive) per chunk
  const Tran1Fields tf = tls_tran1; tls_tran1 = Tran1Fields{};   // one-shot
  struct SArr { const char* h; char* d; size_t hpitch, dpitch, width; int kind; };   // one constituent slice, all chunks
  std::vector<SArr> sarrs;
  Tran1Dev td{};
  const Tran1Dev* tdp = nullptr;
  if (tf.pcnst > 0) {
    const int n = tf.pcnst;
    std::vector<int> act, dryc;
    for (int m = 1; m < n; ++m)
      if (tls_tran1_flags[m]) { act.push_back(m); dryc.push_back(tls_tran1_flags[n + m]); }
    const int na = (int)act.size();
    if (na > 0) {
      if (tls_tmeta1c.set_compact(dryc)) return -100;
      Workspace& s3 = tls_stage2;                  // constituent slices: their own staging arena
      if (s3.ensure(3 * al((size_t)nchunks * na * s2, 8) + 4096)) return -100;
      double* d_q3 = s3.take<double>((size_t)nchunks * na * s2);
      double* d_f3 = s3.take<double>((size_t)nchunks * na * s2);
      double* d_t3 = s3.take<double>((size_t)nchunks * na * s2);
      for (int j = 0; j < na; ++j) {
        const size_t ho = (size_t)act[j] * s2 * 8, dof = (size_t)j * s2 * 8;
        sarrs.push_back({(const char*)tf.q + ho, (char*)d_q3 + dof, (size_t)n * s2 * 8, (size_t)na * s2 * 8, s2 * 8, 1});
        sarrs.push_back({(const char*)tf.fracis + ho, (char*)d_f3 + dof, (size_t)n * s2 * 8, (size_t)na * s2 * 8, s2 * 8, 1});
        sarrs.push_back({(const char*)tf.ptend_q + ho, (char*)d_t3 + dof, (size_t)n * s2 * 8, (size_t)na * s2 * 8, s2 * 8, 3});
      }
      td = Tran1Dev{na, na, tls_tmeta1c.active(), tls_tmeta1c.dry(), tls_tmeta1c.any_dry, d_q3, d_f3, d_t3};
      tdp = &td;
    }
  }
  int rc = 0;
  // error paths: no copy into or out of the caller's buffers may still be in flight when the call returns
  auto drain = [&]() {
    cudaStreamSynchronize(tp.h2d); cudaStreamSynchronize(tp.d2h_early); cudaStreamSynchronize(tp.d2h_final);
    for (int b = 0; b < TendPipe::MAXB; ++b) if (tp.work[b].stream) cudaStreamSynchronize(tp.work[b].stream);
  };
#define CKP(call)                                                                                   \
  do {                                                                                              \
    cudaError_t _e = (call);                                                                        \
    if (_e != cudaSuccess) {                                                                        \
      tls_err = std::string("CUDA error ") + cudaGetErrorString(_e) + " in zm_conv_tend_batch (" #call ")"; \
      drain();                                                                                      \
      return -100;                                                                                  \
    }                                                                                               \
  } while (0)
  long long moved_h2d = 0, moved_d2h = 0;
  // zero-fill of the caller's arrays of the sparse fields by the worker threads, one counter per sub-batch
  HostPool* pool = (sparse && rec_len > 0) ? &host_pool() : nullptr;
  std::atomic<int> zero_left[TendPipe::MAXB];
  for (auto& z : zero_left) z.store(0);
  // anything that returns early must not leave worker tasks (which write the caller's arrays) behind
  struct PoolGuard { HostPool* p; ~PoolGuard() { if (p) p->wait_all(); } } pool_guard{pool};
  auto copy_kind = [&](int kind, int c0, int nb, cudaStream_t on) {
    for (auto& a : arrs) {
      if (a.kind != kind) continue;
      const size_t off = (size_t)c0 * a.stride * a.esz, bytes = (size_t)nb * a.stride * a.esz;
      ((kind <= 1 || kind == 4) ? moved_h2d : moved_d2h) += (long long)bytes;
      cudaError_t e = (kind <= 1 || kind == 4) ? cudaMemcpyAsync((char*)a.d + off, (const char*)a.h + off, bytes, cudaMemcpyHostToDevice, on)
                                  : cudaMemcpyAsync((char*)a.h + off, (char*)a.d + off, bytes, cudaMemcpyDeviceToHost, on);
      if (e != cudaSuccess) rc = -100;
    }
    for (auto& a : sarrs) {
      if (a.kind != kind) continue;
      (kind == 1 ? moved_h2d : moved_d2h) += (long long)(a.width * nb);
      const cudaError_t e = (kind == 1)
          ? cudaMemcpy2DAsync(a.d + (size_t)c0 * a.dpitch, a.dpitch, a.h + (size_t)c0 * a.hpitch, a.hpitch, a.width, nb, cudaMemcpyHostToDevice, on)
          : cudaMemcpy2DAsync((char*)a.h + (size_t)c0 * a.hpitch, a.hpitch, a.d + (size_t)c0 * a.dpitch, a.dpitch, a.width, nb, cudaMemcpyDeviceToHost, on);
      if (e != cudaSuccess) rc = -100;
    }
  };
  // Enqueue order on the host thread: inputs of sub-batch b+1 go out right after the kernels of sub-batch b
  // were launched, so neither the copy engine nor the SMs wait for the host to finish enqueueing.
  auto send_inputs = [&](int b) -> int {
    const int c0 = tp.sched_first[b], nb = tp.sched_first[b + 1] - c0;
    copy_kind(0, c0, nb, tp.h2d);
    CKP(cudaEventRecord(tp.in_ready[b], tp.h2d));
    copy_kind(1, c0, nb, tp.h2d);
    CKP(cudaEventRecord(tp.late_ready[b], tp.h2d));
    return 0;
  };
  if (pool && !prezeroed) {
    for (int b = 0; b < NB; ++b) {
      const int c0 = tp.sched_first[b], nb = tp.sched_first[b + 1] - c0;
      for (int qf = 0; qf < SF_N; ++qf) {
        if (sf_off[qf] < 0) continue;
        const size_t str = ((qf >= SF_MCON && qf <= SF_FS) ? s2p : s2);
        char* base = (char*)(sf_host[qf] + (size_t)c0 * str);
        const size_t bytes = (size_t)nb * str * 8, piece = 2u << 20;
        for (size_t o = 0; o < bytes; o += piece) {
          zero_left[b].fetch_add(1);
          const size_t n = bytes - o < piece ? bytes - o : piece;
          std::atomic<int>* cnt = &zero_left[b];
          pool->submit([base, o, n, cnt] { std::memset(base + o, 0, n); cnt->fetch_sub(1); });
        }
      }
    }
  }
  CKP(cudaEventRecord(tp.t0, tp.h2d));
  const double w_t0 = wall_ms();
  copy_kind(4, 0, nchunks, tp.h2d);
  if (send_inputs(0)) { drain(); return -100; }
  for (int b = 0; b < NB && rc == 0; ++b) {
    const int c0 = tp.sched_first[b], nb = tp.sched_first[b + 1] - c0;
    Workspace& ws = tp.work[b];
    ws.chunk0 = c0;
    if (!ws.stream && ws.ensure(0)) { drain(); return -100; }
    CKP(cudaStreamWaitEvent(ws.stream, tp.in_ready[b], 0));
    TendHooks hooks{tp.late_ready[b], tp.convr_done[b]};
    Tran1Dev tb = td;
    if (tdp) {
      const size_t o3 = (size_t)c0 * s2 * td.ncnst;
      tb.q = td.q + o3; tb.fracis = td.fracis + o3; tb.dqdt = td.dqdt + o3;
    }
    const HistFields hb = dh.slice(c0, s2);
#define O2(x)  ((x) + (size_t)c0 * s2)
#define O2P(x) ((x) + (size_t)c0 * s2p)
#define O1(x)  ((x) + (size_t)c0 * s1)
    rc = conv_tend_impl(ws, nb, d_ncol + c0, O2(d_t), O2(d_q), O2(d_u), O2(d_v), O2(d_pmid), O2P(d_pint), O2(d_pdel),
                        O2(d_zm), O2P(d_zi), O1(d_phis), O1(d_pblh), O1(d_tpert), O1(d_lf), O2(d_cld), ztodt,
                        O2(d_ps), O2(d_pq), O2(d_pu), O2(d_pv), O2P(d_mcon), O2(d_cme), O2P(d_pflx), O2(d_zdu),
                        O1(d_rliq), O1(d_rice), O1(d_jctop), O1(d_jcbot), O1(d_prec), O1(d_snow), O2(d_ql),
                        O2(d_rprd), O2(d_evap), O2P(d_fp), O2P(d_fs), O2(d_dlf), O2(d_mu), O2(d_md), O2(d_du),
                        O2(d_eu), O2(d_ed), O2(d_dp), O1(d_dsub), O1(d_jt), O1(d_maxg), O1(d_ideep), d_len + c0,
                        O1(d_cape), (void*)ws.stream, &hooks, d_org ? O2(d_org) : nullptr,
                        d_orgt ? O2(d_orgt) : nullptr, d_org2d ? O2(d_org2d) : nullptr, tdp ? &tb : nullptr,
                        hist_on ? &hb : nullptr);
#undef O2
#undef O2P
#undef O1
    if (rc) break;
    const double w_k = wall_ms();
    if (rec_len > 0) {  // the convective columns' records of this sub-batch
      SparseFields sf;
      sf.rec_len = rec_len;
      for (int qf = 0; qf < SF_N; ++qf) {
        sf.off[qf] = sf_off[qf];
        sf.d[qf] = sf_off[qf] < 0 ? nullptr : sf_dev[qf] + (size_t)c0 * ((qf >= SF_MCON && qf <= SF_FS) ? s2p : s2);
      }
      int* base_b = d_base + c0 + b;                       // nb + 1 entries
      k_lengath_scan<<<1, 256, 0, ws.stream>>>(nb, d_len + c0, base_b);
      k_pack_records<<<nb * (int)pc, 64, 0, ws.stream>>>(nb, d_len + c0, d_ideep + (size_t)c0 * s1, base_b, sf,
                                                         d_rec + (size_t)c0 * pc * rec_len);
      tls_launches += 2;
    }
    CKP(cudaEventRecord(tp.done[b], ws.stream));
    if (pool) {         // (count, lengath, ideep) of the sub-batch: what the host needs to size and scatter the records
      int* hs = tp.h_small + 2 * ((size_t)c0 * pc + c0 + 2 * b);
      CKP(cudaStreamWaitEvent(tp.d2h_final, tp.done[b], 0));
      CKP(cudaMemcpyAsync(hs, d_base + c0 + b + nb, sizeof(int), cudaMemcpyDeviceToHost, tp.d2h_final));
      CKP(cudaMemcpyAsync(hs + 2, d_len + c0, (size_t)nb * sizeof(int), cudaMemcpyDeviceToHost, tp.d2h_final));
      CKP(cudaMemcpyAsync(hs + 2 + nb, d_ideep + (size_t)c0 * s1, (size_t)nb * pc * sizeof(int), cudaMemcpyDeviceToHost, tp.d2h_final));
      CKP(cudaEventRecord(tp.small_back[b], tp.d2h_final));
      moved_d2h += (long long)(1 + nb + nb * pc) * 4;
    }
    if (b + 1 < NB && send_inputs(b + 1)) { drain(); return -100; }
    const double w_in = wall_ms();
    // device->host: zm_convr's outputs as soon as they are final, the rest when the sub-batch ends
    // one return stream, in the order results become final: by the time sub-batch b's zm_convr outputs are
    // across, its evap/momtran kernels have finished too
    CKP(cudaStreamWaitEvent(tp.d2h_early, tp.convr_done[b], 0));
    copy_kind(2, c0, nb, tp.d2h_early);
    CKP(cudaEventRecord(tp.early_back[b], tp.d2h_early));
    CKP(cudaStreamWaitEvent(tp.d2h_early, tp.done[b], 0));
    copy_kind(3, c0, nb, tp.d2h_early);
    CKP(cudaEventRecord(tp.final_back[b], tp.d2h_early));
    if (dbg) fprintf(stderr, "  sub-batch %d: kernels enqueued %.3f, next inputs enqueued %.3f, returns enqueued %.3f ms\n",
                     b, w_k, w_in, wall_ms());
  }
  if (rc == 0 && pool) {
    // records: as soon as a sub-batch's count is known its records are fetched (exact size) while the worker threads
    // scatter the previous sub-batch's
    size_t hoff = 0;                       // doubles into the pinned record staging
    size_t rec_off[TendPipe::MAXB]; int rec_cnt[TendPipe::MAXB];
    auto scatter = [&](int b) {
      const int c0 = tp.sched_first[b], nb = tp.sched_first[b + 1] - c0;
      const int* hs = tp.h_small + 2 * ((size_t)c0 * pc + c0 + 2 * b);
      const int* len = hs + 2; const int* idp = hs + 2 + nb;
      while (zero_left[b].load() > 0) std::this_thread::yield();
      const int ntask = pool->size() * 2, total = rec_cnt[b];
      const double* recs = tp.h_rec + rec_off[b];
      int ca = 0, j0 = 0;
      for (int tsk = 0; tsk < ntask && ca < nb; ++tsk) {
        const int want = (int)(((long long)total * (tsk + 1)) / ntask);
        int cb = ca, j1 = j0;
        while (cb < nb && (j1 < want || tsk == ntask - 1)) j1 += len[cb++];
        if (cb == ca) continue;
        double* const* hostp = sf_host; const int* offp = sf_off;
        const int pcl = (int)pc, Ll = (int)L, rl = rec_len;
        pool->submit([=] {
          int j = j0;
          for (int c = ca; c < cb; ++c)
            for (int slot = 0; slot < len[c]; ++slot, ++j) {
              const int i = idp[(size_t)c * pcl + slot] - 1;
              const double* r = recs + (size_t)j * rl;
              for (int qf = 0; qf < SF_N; ++qf) {
                if (offp[qf] < 0) continue;
                const int nlev = (qf >= SF_MCON && qf <= SF_FS) ? Ll + 1 : Ll;
                double* dst = hostp[qf] + ((size_t)(c0 + c) * nlev) * pcl + (qf >= SF_MU ? slot : i);
                const double* src = r + offp[qf];
                for (int k = 0; k < nlev; ++k) dst[(size_t)k * pcl] = src[k];
              }
            }
        });
        ca = cb; j0 = j1;
      }
    };
    for (int b = 0; b < NB && rc == 0; ++b) {
      const int c0 = tp.sched_first[b];
      if (cudaEventSynchronize(tp.small_back[b]) != cudaSuccess) { rc = -100; break; }
      rec_cnt[b] = tp.h_small[2 * ((size_t)c0 * pc + c0 + 2 * b)];
      rec_off[b] = hoff;
      const size_t n = (size_t)rec_cnt[b] * rec_len;
      if (hoff + n > tp.h_rec_cap) {       // grow the pinned staging: earlier records must be scattered first
        for (int p2 = 0; p2 < b; ++p2) cudaEventSynchronize(tp.rec_back[p2]);
        pool->wait_all();
        if (tp.ensure_pinned(nc * rec_len, 0)) { rc = -100; break; }
      }
      if (n && cudaMemcpyAsync(tp.h_rec + hoff, d_rec + (size_t)c0 * pc * rec_len, n * sizeof(double),
                               cudaMemcpyDeviceToHost, tp.d2h_early) != cudaSuccess) rc = -100;
      if (cudaEventRecord(tp.rec_back[b], tp.d2h_early) != cudaSuccess) rc = -100;
      moved_d2h += (long long)n * 8;
      hoff += n;
      if (b > 0) {
        if (cudaEventSynchronize(tp.rec_back[b - 1]) != cudaSuccess) { rc = -100; break; }
        scatter(b - 1);
      }
    }
    if (rc == 0) {
      if (cudaEventSynchronize(tp.rec_back[NB - 1]) != cudaSuccess) rc = -100;
      else scatter(NB - 1);
    }
  }
  if (rc == 0 && g) {
    // gathered: a sub-batch's lengath comes back as soon as its kernels are done, into the caller's array; its sum is
    // the sub-batch's record count, and exactly that many records go to their final place in the caller's buffer
    // (chunk after chunk, so the running sum is the exclusive prefix of lengath).  The host waits here only after
    // every sub-batch has been enqueued.  Lengath and records share d2h_final, which has waited for no later
    // sub-batch yet, so sub-batch b's records move while the sub-batches after it compute; d2h_early, behind every
    // sub-batch's wait, keeps the attachments and the per-column outputs.
    size_t hoff = 0;                       // doubles into g->rec
    for (int b = 0; b < NB && rc == 0; ++b) {
      const int c0 = tp.sched_first[b], nb = tp.sched_first[b + 1] - c0;
      if (cudaStreamWaitEvent(tp.d2h_final, tp.done[b], 0) != cudaSuccess ||
          cudaMemcpyAsync(lengath + c0, d_len + c0, (size_t)nb * sizeof(int), cudaMemcpyDeviceToHost,
                          tp.d2h_final) != cudaSuccess ||
          cudaEventRecord(tp.small_back[b], tp.d2h_final) != cudaSuccess ||
          cudaEventSynchronize(tp.small_back[b]) != cudaSuccess) { rc = -100; break; }
      moved_d2h += (long long)nb * sizeof(int);
      size_t cnt = 0;
      for (int c = c0; c < c0 + nb; ++c) cnt += (size_t)lengath[c];
      const size_t n = cnt * rec_len;
      if (n && cudaMemcpyAsync(g->rec + hoff, d_rec + (size_t)c0 * pc * rec_len, n * sizeof(double),
                               cudaMemcpyDeviceToHost, tp.d2h_final) != cudaSuccess) rc = -100;
      // zm_tend_trace's "remaining outputs on host" of this sub-batch: its records
      if (cudaEventRecord(tp.final_back[b], tp.d2h_final) != cudaSuccess) rc = -100;
      moved_d2h += (long long)n * 8;
      hoff += n;
    }
  }
  if (rc == 0) copy_kind(5, 0, nchunks, tp.d2h_early);
  // the Brent failure counters of all sub-batches ride back on the return stream (it has waited for every
  // sub-batch): one synchronisation instead of one per sub-batch
  int fail_cnt[TendPipe::MAXB][4] = {};
  if (rc == 0)
    for (int b = 0; b < NB; ++b)
      if (tp.work[b].last_count &&
          cudaMemcpyAsync(fail_cnt[b], tp.work[b].last_count, sizeof fail_cnt[b], cudaMemcpyDeviceToHost, tp.d2h_early) != cudaSuccess)
        rc = -100;
  const double w_enq = wall_ms();
  cudaError_t e1 = cudaStreamSynchronize(tp.d2h_early), e2 = cudaStreamSynchronize(tp.d2h_final),
              e3 = cudaStreamSynchronize(tp.h2d);
  if (dbg) fprintf(stderr, "zm_conv_tend_batch host thread: t0 recorded at %.3f ms, everything enqueued at %.3f ms, "
                           "streams drained at %.3f ms\n", w_t0, w_enq, wall_ms());
  for (int b = 0; b < NB; ++b)
    if (tp.work[b].stream && cudaStreamSynchronize(tp.work[b].stream) != cudaSuccess) rc = -100;
  if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) rc = -100;
  if (rc) {
    if (rc == -100 && tls_err.empty()) tls_err = std::string("CUDA error: ") + cudaGetErrorString(cudaGetLastError());
    drain();
    return rc;
  }
  int fails = 0;
  for (int b = NB - 1; b >= 0; --b) {        // first failing sub-batch's message wins
    if (fail_cnt[b][2] == 0) continue;
    const int f = read_failures(tp.work[b], tp.work[b].stream);      // fetches the details and formats the message
    if (f < 0) return f;
    fails += f;
  }
  if (fails == 0) tls_mirror = new_mirror;   // a failed step (the reference stops in endrun) leaves no mirror
  if (pool) pool->wait_all();
  tp.last_h2d = moved_h2d; tp.last_d2h = moved_d2h;
  return fails;
#undef CKP
}

int zm_conv_tend_batch(int nchunks, const int* ncol, const double* t, const double* q, const double* u,
                       const double* v, const double* pmid, const double* pint, const double* pdel,
                       const double* zm, const double* zi, const double* phis, const double* pblh,
                       const double* tpert, const double* landfrac, const double* cld, double ztodt,
                       double* ptend_s, double* ptend_q, double* ptend_u, double* ptend_v, double* mcon,
                       double* cme, double* pflx, double* zdu, double* rliq, double* rice, double* jctop,
                       double* jcbot, double* prec, double* snow, double* ql, double* rprd, double* evapcdp,
                       double* flxprec, double* flxsnow, double* dlf, double* mu, double* md, double* du,
                       double* eu, double* ed, double* dp, double* dsubcld, int* jt, int* maxg, int* ideep,
                       int* lengath, double* cape) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  return conv_tend_batch(nchunks, ncol, t, q, u, v, pmid, pint, pdel, zm, zi, phis, pblh, tpert, landfrac, cld, ztodt,
                         ptend_s, ptend_q, ptend_u, ptend_v, mcon, cme, pflx, zdu, rliq, rice, jctop, jcbot, prec, snow,
                         ql, rprd, evapcdp, flxprec, flxsnow, dlf, mu, md, du, eu, ed, dp, dsubcld, jt, maxg, ideep,
                         lengath, cape, nullptr);
}

int zm_conv_tend_batch_gathered(int nchunks, const int* ncol, const double* t, const double* q, const double* u,
                                const double* v, const double* pmid, const double* pint, const double* pdel,
                                const double* zm, const double* zi, const double* phis, const double* pblh,
                                const double* tpert, const double* landfrac, const double* cld, double ztodt,
                                double* rliq, double* rice, double* jctop, double* jcbot, double* prec, double* snow,
                                double* cape, double* dsubcld, int* jt, int* maxg, int* ideep, int* lengath,
                                int pbuf_in_records, double* rec, long long rec_cap) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  // argument checks come before anything else: a refused call writes nothing and leaves attachments and mirror alone
  if (!ideep || !lengath || !rec) {
    tls_err = "zm_conv_tend_batch_gathered: ideep, lengath and rec are required (non-NULL)";
    return -9;
  }
  const long long L = g_params.pver, rec_len = (pbuf_in_records ? 20 : 14) * L + 4;
  const long long need = (long long)nchunks * g_params.pcols * rec_len;
  if (rec_cap < need) {
    tls_err = "zm_conv_tend_batch_gathered: rec_cap = " + std::to_string(rec_cap) + " doubles, need nchunks*pcols*rec_len = " +
              std::to_string(need) + " (rec_len = " + std::to_string(rec_len) + ")";
    return -9;
  }
  const GatheredOut g{rec, pbuf_in_records != 0};
  return conv_tend_batch(nchunks, ncol, t, q, u, v, pmid, pint, pdel, zm, zi, phis, pblh, tpert, landfrac, cld, ztodt,
                         nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, rliq, rice, jctop, jcbot,
                         prec, snow, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                         nullptr, nullptr, nullptr, dsubcld, jt, maxg, ideep, lengath, cape, &g);
}

// bytes the calling thread's last zm_conv_tend_batch moved over PCIe (host->device, device->host)
int zm_tend_transfer_bytes(long long* h2d, long long* d2h) {
  if (h2d) *h2d = tls_pipe.last_h2d;
  if (d2h) *d2h = tls_pipe.last_d2h;
  return 0;
}

// zm_org = 1: attach org (in), orgt and org2d (out), shapes (pcols,pver) per chunk, for the NEXT zm_convr_batch /
// zm_conv_tend_batch [_dev] call of this thread (host pointers for the host-pointer entry points, device pointers
// for *_dev).  Replaces the pointer dummies org/orgt/org2d of zm_convr (zm_conv.F90:242, 421-423).
int zm_org_fields(const double* org, double* orgt, double* org2d) {
  tls_org = OrgFields{org, orgt, org2d};
  return 0;
}

// zm_conv_tend's history fields (zm_conv_intr.F90:676-857) for the NEXT zm_conv_tend_batch[_dev] call of this
// thread; any pointer may be NULL (not materialised, not copied)
int zm_conv_tend_hist_fields(double* heat, double* qtnd, double* eurt, double* dif, double* dnlf, double* dnif,
                             double* tend_s, double* tend_s_snwprd, double* tend_s_snwevmlt,
                             double* ntprprd, double* ntsnprd,
                             double* seten, double* pguall, double* pgdall, double* icwu, double* icwd) {
  HistFields h;
  double* const a[H_N] = {heat, qtnd, eurt, dif, dnlf, dnif, tend_s, tend_s_snwprd, tend_s_snwevmlt, ntprprd, ntsnprd,
                          seten, pguall, pgdall, icwu, icwd};
  std::copy(a, a + H_N, h.p);
  tls_hist = h;
  return 0;
}

// convtran1 of zm_conv_tend (zm_conv_intr.F90:865-880): attaches state%q, fracis and ptend_loc%q, all
// (pcols,pver,pcnst) per chunk, and the constituent flags (lq(2:) = cnst_is_convtran1(2:); cnst_get_type_byind)
// for the NEXT zm_conv_tend_batch[_dev] call of this thread.  pcnst <= 0 detaches.
int zm_convtran1_fields(int pcnst, const int* doconvtran, const int* cnst_is_dry, const double* q,
                        const double* fracis, double* ptend_q) {
  if (pcnst <= 0 || !doconvtran || !q || !fracis || !ptend_q) { tls_tran1 = Tran1Fields{}; return 0; }
  tls_tran1_flags.assign(2 * (size_t)pcnst, 0);
  for (int m = 0; m < pcnst; ++m) {
    tls_tran1_flags[m] = doconvtran[m] != 0;
    tls_tran1_flags[pcnst + m] = cnst_is_dry ? (cnst_is_dry[m] != 0) : 0;
  }
  tls_tran1 = Tran1Fields{pcnst, q, fracis, ptend_q};
  return 0;
}

// zm_conv_tend's history fields that involve arithmetic (zm_conv_intr.F90:685-688, 700-706, 721-729)
int zm_conv_tend_diag_batch_dev(int nchunks, const int* ncol, const double* ps, const double* pmid, const double* mu,
                                const double* md, const int* jt, const int* maxg, const int* ideep, const int* lengath,
                                double* freqzm, double* mu_out, double* md_out, double* pcont, double* pconb,
                                void* stream) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  k_tend_diag<<<nchunks, 128, (size_t)g_params.pcols * sizeof(int), (cudaStream_t)stream>>>(
      nchunks, ncol, ps, pmid, mu, md, jt, maxg, ideep, lengath, freqzm, mu_out, md_out, pcont, pconb);
  ++tls_launches;
  CK(cudaGetLastError());
  return 0;
}
// host pointers; mu, md, jt, maxg, ideep, lengath may be NULL: taken from the device pbuf mirror of this thread's
// last zm_conv_tend_batch
int zm_conv_tend_diag_batch(int nchunks, const int* ncol, const double* ps, const double* pmid, const double* mu,
                            const double* md, const int* jt, const int* maxg, const int* ideep, const int* lengath,
                            double* freqzm, double* mu_out, double* md_out, double* pcont, double* pconb) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc, n2 = nc * L;
  const bool from_mirror = !(mu && md && jt && maxg && ideep && lengath);
  const PbufMirror M = tls_mirror;
  if (from_mirror && (M.nchunks != nchunks || !M.mu)) {
    tls_err = "zm_conv_tend_diag_batch: no device mirror from a zm_conv_tend_batch call with the same nchunks on this thread";
    return -7;
  }
  Workspace& st = tls_stage2;
  if (st.ensure(al(nchunks, 4) * 2 + 5 * al(n2, 8) + 3 * al(nc, 4) + 4 * al(nc, 8) + 4096)) return -100;
  Stager S(st);
  const int* d_ncol = S.in(ncol, nchunks);
  const double *d_ps = S.in(ps, nc), *d_pmid = S.in(pmid, n2);
  const double *d_mu = from_mirror ? M.mu : S.in(mu, n2), *d_md = from_mirror ? M.md : S.in(md, n2);
  const int *d_jt = from_mirror ? M.jt : S.in(jt, nc), *d_mx = from_mirror ? M.maxg : S.in(maxg, nc),
            *d_id = from_mirror ? M.ideep : S.in(ideep, nc), *d_len = from_mirror ? M.lengath : S.in(lengath, nchunks);
  double *d_f = S.out(freqzm, nc), *d_muo = S.out(mu_out, n2), *d_mdo = S.out(md_out, n2), *d_pt = S.out(pcont, nc),
         *d_pb = S.out(pconb, nc);
  int rc = zm_conv_tend_diag_batch_dev(nchunks, d_ncol, d_ps, d_pmid, d_mu, d_md, d_jt, d_mx, d_id, d_len, d_f, d_muo,
                                       d_mdo, d_pt, d_pb, (void*)st.stream);
  if (rc) return rc;
  return S.flush();
}

// Timeline of this thread's last zm_conv_tend_batch call: for each sub-batch 6 times in ms since the first
// host->device copy was enqueued: inputs on device, late inputs on device, zm_convr done, sub-batch done,
// zm_convr outputs on host, remaining outputs on host.  Returns the number of sub-batches.
int zm_tend_trace(double* ms, int cap) {
  TendPipe& tp = tls_pipe;
  for (int b = 0; b < tp.last_nb && 6 * (b + 1) <= cap; ++b) {
    cudaEvent_t ev[6] = {tp.in_ready[b], tp.late_ready[b], tp.convr_done[b], tp.done[b], tp.early_back[b], tp.final_back[b]};
    for (int j = 0; j < 6; ++j) {
      float t = 0.f;
      if (cudaEventElapsedTime(&t, tp.t0, ev[j]) != cudaSuccess) { cudaGetLastError(); t = -1.f; }
      ms[6 * b + j] = t;
    }
  }
  return tp.last_nb;
}

// Per-rank budget terms for the global conservation check (device pointers; out6 on device):
// [0] sum pdel/g*ptend_q  [1] sum 1000*(prec+rliq)  [2] sum pdel/g*ptend_s
// [3] sum 1000*(latvap*(prec+rliq)+latice*snow)  [4] convective columns  [5] columns
int zm_conservation_dev(int nchunks, const int* ncol, const double* pdel, const double* ptend_q,
                        const double* ptend_s, const double* prec, const double* snow, const double* rliq,
                        const int* lengath, double* out6, void* stream) {
  NEED_INIT();
  static thread_local double* partial = nullptr;
  const int nb = ZM_CONS_BLOCKS;
  if (!partial) CK(cudaMalloc(&partial, (size_t)nb * 6 * sizeof(double)));
  Workspace& ws = tls_work;
  if (!ws.stream && ws.ensure(0)) return -100;
  cudaStream_t s = (cudaStream_t)stream;      // NULL = the CUDA default stream
  k_conservation_partial<<<nb, 256, 0, s>>>(nchunks, ncol, pdel, ptend_q, ptend_s, prec, snow, rliq, lengath, partial);
  k_conservation_final<<<1, 192, 0, s>>>(nb, partial, out6);
  tls_launches += 2;
  CK(cudaGetLastError());
  return 0;
}

// zm_conv_tend_2 (zm_conv_intr.F90:955-1028) on device arrays: dpdry gather (:1014-1017) + convtran (:1020-1024)
// with the pbuf fields zm_conv_tend_batch_dev left in the caller's device arrays.  Enqueue on the stream the tend
// step ran on (the scratch arena is shared and reused in stream order).
int zm_conv_tend_2_batch_dev(int nchunks, const int* doconvtran, const double* q, int pcnst, const double* pdeldry,
                             const double* fracis, double* ptend_q, double ztodt, const int* cnst_is_dry,
                             const double* mu, const double* md, const double* du, const double* eu,
                             const double* ed, const double* dp, const double* dsubcld, const int* jt,
                             const int* maxg, const int* ideep, const int* lengath, void* stream) {
  NEED_INIT();
  (void)dsubcld; (void)ztodt;
  if (nchunks <= 0) return 0;
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc, n2 = nc * L;
  cudaStream_t s = (cudaStream_t)stream;
  if (tls_tmeta.set(doconvtran, cnst_is_dry, pcnst)) return -100;
  if (tls_tmeta.nactive == 0) return 0;
  Workspace& ws = tls_work;
  if (ws.ensure(chunk_bounds_bytes(nchunks, (int)nc) + al(n2, 8) + 1024)) return -100;
  double* dpdry = ws.take<double>(n2);
  for (auto e : ws.tev) cudaEventDestroy(e);
  ws.tev.clear(); ws.tnames.clear();
  tick(ws, s, "start");
  k_dpdry_gather<<<1184, 256, 0, s>>>(nchunks, ideep, lengath, pdeldry, dpdry); ++tls_launches;
  TranArgs a;
  a.nchunks = nchunks; a.ncnst = pcnst; a.nactive = tls_tmeta.nactive; a.jt = jt; a.mx = maxg; a.ideep = ideep;
  a.lengath = lengath; a.active = tls_tmeta.active(); a.is_dry = tls_tmeta.dry();
  a.q = q; a.fracis = fracis; a.mu = mu; a.md = md; a.du = du; a.eu = eu; a.ed = ed; a.dp = dp;
  a.dpdry = dpdry; a.dqdt = ptend_q;
  ChunkBounds cb;
  if (chunk_bounds_enqueue(ws, s, nchunks, jt, maxg, lengath, cb)) return -100;
  const int rc = convtran_enqueue(s, a, cb);
  tick(ws, s, "convtran2");
  return rc;
}

// zm_conv_tend_2 (zm_conv_intr.F90:955-1028): convtran over the constituents flagged convtran2, with the
// mass-flux fields of this thread's last zm_conv_tend_batch taken from the device mirror.
int zm_conv_tend_2_batch(int nchunks, const int* doconvtran, const double* q, int pcnst, const double* pdeldry,
                         const double* fracis, double* ptend_q, double ztodt, const int* cnst_is_dry) {
  NEED_INIT();
  tls_t2_h2d = tls_t2_d2h = 0;
  if (nchunks <= 0) return 0;
  const PbufMirror M = tls_mirror;
  if (M.nchunks != nchunks || !M.mu) {
    tls_err = "zm_conv_tend_2_batch: no device mirror from a zm_conv_tend_batch call with the same nchunks on this thread";
    return -7;
  }
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc, n2 = nc * L, n3 = n2 * pcnst;
  Workspace& st = tls_stage2;
  if (st.ensure(2 * al(n2, 8) + 3 * al(n3, 8) + 4096)) return -100;
  Stager S(st);
  const double *d_q = S.in(q, n3), *d_fr = S.in(fracis, n3), *d_pdd = S.in(pdeldry, n2);
  double* d_dpdry = st.take<double>(n2);
  double* d_dqdt = S.inout(ptend_q, n3);
  tls_t2_h2d = (long long)(3 * n3 + n2) * (long long)sizeof(double);     // q, fracis, pdeldry, ptend_q (inout)
  // dpdry(i,:) = pdeldry(ideep(i),:)/100 for i <= lengath, else 0 (zm_conv_intr.F90:1014-1017)
  k_dpdry_gather<<<1184, 256, 0, st.stream>>>(nchunks, M.ideep, M.lengath, d_pdd, d_dpdry); ++tls_launches;
  for (auto e : st.tev) cudaEventDestroy(e);
  st.tev.clear(); st.tnames.clear();
  tick(st, st.stream, "start");
  int rc = zm_convtran_batch_dev(nchunks, doconvtran, d_q, pcnst, M.mu, M.md, M.du, M.eu, M.ed, M.dp, M.dsubcld,
                                 M.jt, M.maxg, M.ideep, M.lengath, d_fr, d_dqdt, d_dpdry, ztodt, cnst_is_dry,
                                 (void*)st.stream);
  if (rc) return rc;
  tick(st, st.stream, "convtran2");
  rc = S.flush();
  if (rc == 0) tls_t2_d2h = (long long)n3 * (long long)sizeof(double);
  return rc;
}

// zm_conv_tend_2 on the convective columns' records (include/zmconv_b200.h): the caller packs q, fracis (and pdeldry
// when a flagged constituent is dry) of the columns ideep(1:lengath) of the flagged constituents and scatters the
// returned tendencies itself; the mass-flux fields come from the device mirror as in zm_conv_tend_2_batch.
int zm_conv_tend_2_batch_gathered(int nchunks, const int* lengath, const int* doconvtran, int pcnst,
                                  const int* cnst_is_dry, const double* q_rec, const double* fracis_rec,
                                  const double* pdeldry_rec, double* dqdt_rec, long long rec_cap, double ztodt) {
  NEED_INIT();
  (void)ztodt;
  tls_t2_h2d = tls_t2_d2h = 0;
  if (nchunks <= 0) return 0;
  const PbufMirror M = tls_mirror;
  if (M.nchunks != nchunks || !M.mu) {
    tls_err = "zm_conv_tend_2_batch_gathered: no device mirror from a zm_conv_tend_batch call with the same nchunks on "
              "this thread";
    return -7;
  }
  if (!doconvtran || pcnst < 1) {
    tls_err = "zm_conv_tend_2_batch_gathered: doconvtran is required and pcnst must be >= 1";
    return -9;
  }
  // the active list of the layout: m = 2..pcnst (1-based) with doconvtran(m), ascending
  int nact = 0;
  bool any_dry = false;
  for (int m = 1; m < pcnst; ++m)
    if (doconvtran[m]) { ++nact; any_dry = any_dry || (cnst_is_dry && cnst_is_dry[m]); }
  if (nact == 0) return 0;
  if (!lengath || !q_rec || !fracis_rec || !dqdt_rec || (any_dry && !pdeldry_rec)) {
    tls_err = "zm_conv_tend_2_batch_gathered: lengath, q_rec, fracis_rec, dqdt_rec are required, and pdeldry_rec when a "
              "flagged constituent is dry";
    return -9;
  }
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc, n2 = nc * L;
  Workspace& st = tls_stage2;
  if (!st.stream && st.ensure(0)) return -100;
  // the caller's lengath must be the mirror's: the records were packed with it and the kernels address them with it
  std::vector<int> mlen(nchunks);
  CK(cudaMemcpyAsync(mlen.data(), M.lengath, nchunks * sizeof(int), cudaMemcpyDeviceToHost, st.stream));
  CK(cudaStreamSynchronize(st.stream));
  tls_t2_d2h = (long long)nchunks * (long long)sizeof(int);
  long long ncols = 0;
  for (int c = 0; c < nchunks; ++c) {
    if (lengath[c] != mlen[c]) {
      tls_err = "zm_conv_tend_2_batch_gathered: lengath(" + std::to_string(c + 1) + ") = " + std::to_string(lengath[c]) +
                " differs from the device mirror's " + std::to_string(mlen[c]);
      return -9;
    }
    ncols += mlen[c];
  }
  const long long nrec = ncols * (long long)L * nact;
  if (rec_cap < nrec) {
    tls_err = "zm_conv_tend_2_batch_gathered: rec_cap = " + std::to_string(rec_cap) + " doubles, need sum(lengath)*pver*nact = " +
              std::to_string(nrec);
    return -9;
  }
  if (nrec == 0) return 0;                   // no convective column anywhere: nothing to transport or write
  const size_t npd = any_dry ? (size_t)ncols * L : 0;
  if (st.ensure(al(nchunks + 1, 4) + 3 * al(nrec, 8) + al(npd, 8) + (any_dry ? al(n2, 8) : 0) +
                chunk_bounds_bytes(nchunks, (int)nc) + 4096)) return -100;
  if (tls_tmeta.set(doconvtran, cnst_is_dry, pcnst)) return -100;
  Stager S(st);
  const double *d_q = S.in(q_rec, nrec), *d_fr = S.in(fracis_rec, nrec);
  const double* d_pdd = any_dry ? S.in(pdeldry_rec, npd) : nullptr;
  double* d_dqdt = S.out(dqdt_rec, nrec);
  tls_t2_h2d = (long long)(2 * nrec + npd) * (long long)sizeof(double);
  int* d_base = st.take<int>(nchunks + 1);
  k_lengath_scan<<<1, 256, 0, st.stream>>>(nchunks, M.lengath, d_base); ++tls_launches;
  double* d_dpdry = nullptr;
  if (any_dry) {
    // dpdry(i,:) = pdeldry(ideep(i),:)/100 for i <= lengath, else 0 (zm_conv_intr.F90:1014-1017), slot layout
    d_dpdry = st.take<double>(n2);
    k_dpdry_gather_rec<<<1184, 256, 0, st.stream>>>(nchunks, M.lengath, d_base, d_pdd, d_dpdry); ++tls_launches;
  }
  for (auto e : st.tev) cudaEventDestroy(e);
  st.tev.clear(); st.tnames.clear();
  tick(st, st.stream, "start");
  TranArgs a;
  a.nchunks = nchunks; a.ncnst = pcnst; a.nactive = tls_tmeta.nactive; a.jt = M.jt; a.mx = M.maxg; a.ideep = M.ideep;
  a.lengath = M.lengath; a.active = tls_tmeta.active(); a.is_dry = tls_tmeta.dry();
  a.q = d_q; a.fracis = d_fr; a.mu = M.mu; a.md = M.md; a.du = M.du; a.eu = M.eu; a.ed = M.ed; a.dp = M.dp;
  a.dpdry = d_dpdry; a.dqdt = d_dqdt;
  ChunkBounds cb;
  if (chunk_bounds_enqueue(st, st.stream, nchunks, M.jt, M.maxg, M.lengath, cb)) return -100;
  int rc = convtran_enqueue_gathered(st.stream, a, d_base, cb);
  if (rc) return rc;
  tick(st, st.stream, "convtran2");
  rc = S.flush();
  if (rc == 0) tls_t2_d2h += nrec * (long long)sizeof(double);
  return rc;
}

// bytes the calling thread's last zm_conv_tend_2_batch[_gathered] moved over PCIe (host->device, device->host)
int zm_tend_2_transfer_bytes(long long* h2d, long long* d2h) {
  if (h2d) *h2d = tls_t2_h2d;
  if (d2h) *d2h = tls_t2_d2h;
  return 0;
}

// ---- N4 neighbours: geopotential_t, convect_diagnostics_calc ----------------------------------------
int zm_geopotential_t_batch_dev(int nchunks, const int* ncol, int dycore_lr, const double* piln,
                                const double* pmln, const double* pint, const double* pmid, const double* pdel,
                                const double* rpdel, const double* t, const double* q, const double* rair,
                                double gravit, const double* zvir, double* zi, double* zm, void* stream) {
  NEED_INIT();
  (void)pmln;
  if (nchunks <= 0) return 0;
  GeoArgs a{nchunks, dycore_lr, ncol, piln, pint, pmid, pdel, rpdel, t, q, rair, zvir, gravit, zi, zm};
  const int ncolpad = nchunks * g_params.pcols;
  k_geopotential_t<<<(ncolpad + 127) / 128, 128, 0, (cudaStream_t)stream>>>(a); ++tls_launches;
  CK(cudaGetLastError());
  return 0;
}
int zm_geopotential_t_batch(int nchunks, const int* ncol, int dycore_lr, const double* piln, const double* pmln,
                            const double* pint, const double* pmid, const double* pdel, const double* rpdel,
                            const double* t, const double* q, const double* rair, double gravit,
                            const double* zvir, double* zi, double* zm) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc, n2 = nc * L, n2p = nc * (L + 1);
  Workspace& st = tls_stage;
  if (st.ensure(al(nchunks, 4) + 8 * al(n2, 8) + 3 * al(n2p, 8) + 4096)) return -100;
  Stager S(st);
  const int* d_ncol = S.in(ncol, nchunks);
  const double *d_piln = S.in(piln, n2p), *d_pint = S.in(pint, n2p), *d_pmid = S.in(pmid, n2), *d_pdel = S.in(pdel, n2),
               *d_rpdel = S.in(rpdel, n2), *d_t = S.in(t, n2), *d_q = S.in(q, n2), *d_rair = S.in(rair, n2),
               *d_zvir = S.in(zvir, n2);
  double *d_zi = S.inout(zi, n2p), *d_zm = S.inout(zm, n2);
  int rc = zm_geopotential_t_batch_dev(nchunks, d_ncol, dycore_lr, d_piln, nullptr, d_pint, d_pmid, d_pdel, d_rpdel,
                                       d_t, d_q, d_rair, gravit, d_zvir, d_zi, d_zm, (void*)st.stream);
  if (rc) return rc;
  return S.flush();
}

// generalized-virtual-temperature branch (physics/geopotential.F90:248-310)
int zm_geopotential_t_gen_batch_dev(int nchunks, const int* ncol, int dycore_lr, int ncnst, int nspecies,
                                    const int* species_idx, const double* piln, const double* pmln,
                                    const double* pint, const double* pmid, const double* pdel, const double* rpdel,
                                    const double* t, const double* q3, const double* rair, double gravit,
                                    const double* zvir, double* zi, double* zm, void* stream) {
  NEED_INIT();
  (void)pmln;
  if (nchunks <= 0) return 0;
  if (ncnst < 1 || nspecies < 0) { tls_err = "geopotential_t: ncnst >= 1 and nspecies >= 0 required"; return -2; }
  GeoGenArgs a{nchunks, dycore_lr, ncnst, nspecies, ncol, species_idx, piln, pint, pmid, pdel, rpdel, t, q3, rair, zvir,
               gravit, zi, zm};
  const int ncolpad = nchunks * g_params.pcols;
  k_geopotential_t_gen<<<(ncolpad + 127) / 128, 128, 0, (cudaStream_t)stream>>>(a); ++tls_launches;
  CK(cudaGetLastError());
  return 0;
}
int zm_geopotential_t_gen_batch(int nchunks, const int* ncol, int dycore_lr, int ncnst, int nspecies,
                                const int* species_idx, const double* piln, const double* pmln, const double* pint,
                                const double* pmid, const double* pdel, const double* rpdel, const double* t,
                                const double* q3, const double* rair, double gravit, const double* zvir, double* zi,
                                double* zm) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  if (ncnst < 1 || nspecies < 0) { tls_err = "geopotential_t: ncnst >= 1 and nspecies >= 0 required"; return -2; }
  for (int s = 0; s < nspecies; ++s)
    if (species_idx[s] < 1 || species_idx[s] > ncnst) {
      tls_err = "geopotential_t: thermodynamic_active_species_idx outside 1..ncnst";
      return -2;
    }
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc, n2 = nc * L, n2p = nc * (L + 1);
  Workspace& st = tls_stage;
  if (st.ensure(al(nchunks, 4) + al((size_t)nspecies + 1, 4) + 7 * al(n2, 8) + al(n2 * ncnst, 8) + 3 * al(n2p, 8) + 4096))
    return -100;
  Stager S(st);
  const int* d_ncol = S.in(ncol, nchunks);
  const int* d_sp = nspecies ? S.in(species_idx, (size_t)nspecies) : nullptr;
  const double *d_piln = S.in(piln, n2p), *d_pint = S.in(pint, n2p), *d_pmid = S.in(pmid, n2), *d_pdel = S.in(pdel, n2),
               *d_rpdel = S.in(rpdel, n2), *d_t = S.in(t, n2), *d_q3 = S.in(q3, n2 * ncnst), *d_rair = S.in(rair, n2),
               *d_zvir = S.in(zvir, n2);
  double *d_zi = S.inout(zi, n2p), *d_zm = S.inout(zm, n2);
  int rc = zm_geopotential_t_gen_batch_dev(nchunks, d_ncol, dycore_lr, ncnst, nspecies, d_sp, d_piln, nullptr, d_pint,
                                           d_pmid, d_pdel, d_rpdel, d_t, d_q3, d_rair, gravit, d_zvir, d_zi, d_zm,
                                           (void*)st.stream);
  if (rc) return rc;
  return S.flush();
}

int zm_convect_diagnostics_batch_dev(int nchunks, const int* ncol, double* cmfmc, double* qc, double* qc2,
                                     double* rliq, double* rliq2, const double* pmid, const double* rprddp,
                                     double* cnt, double* cnb, double* cmfmc2, double* rprdsh, double* rprdtot,
                                     double* pcnt, double* pcnb, void* stream) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  CdiagArgs a{nchunks, ncol, cmfmc, qc, qc2, rliq, rliq2, cnt, cnb, cmfmc2, rprdsh, rprdtot, pcnt, pcnb, pmid, rprddp};
  const int ncolpad = nchunks * g_params.pcols;
  (void)ncolpad;
  k_convect_diagnostics<<<1184, 256, 0, (cudaStream_t)stream>>>(a); ++tls_launches;
  CK(cudaGetLastError());
  return 0;
}
int zm_convect_diagnostics_batch(int nchunks, const int* ncol, double* cmfmc, double* qc, double* qc2,
                                 double* rliq, double* rliq2, const double* pmid, const double* rprddp, double* cnt,
                                 double* cnb, double* cmfmc2, double* rprdsh, double* rprdtot, double* pcnt,
                                 double* pcnb) {
  NEED_INIT();
  if (nchunks <= 0) return 0;
  const size_t pc = g_params.pcols, L = g_params.pver, nc = (size_t)nchunks * pc, n2 = nc * L, n2p = nc * (L + 1);
  Workspace& st = tls_stage;
  if (st.ensure(al(nchunks, 4) + 6 * al(n2, 8) + 2 * al(n2p, 8) + 6 * al(nc, 8) + 4096)) return -100;
  Stager S(st);
  const int* d_ncol = S.in(ncol, nchunks);
  double *d_cmfmc = S.inout(cmfmc, n2p), *d_qc = S.inout(qc, n2), *d_qc2 = S.inout(qc2, n2),
         *d_rliq = S.inout(rliq, nc), *d_rliq2 = S.inout(rliq2, nc), *d_cnt = S.inout(cnt, nc),
         *d_cnb = S.inout(cnb, nc), *d_cmfmc2 = S.inout(cmfmc2, n2p), *d_rprdsh = S.inout(rprdsh, n2),
         *d_rprdtot = S.inout(rprdtot, n2), *d_pcnt = S.inout(pcnt, nc), *d_pcnb = S.inout(pcnb, nc);
  const double *d_pmid = S.in(pmid, n2), *d_rprddp = S.in(rprddp, n2);
  int rc = zm_convect_diagnostics_batch_dev(nchunks, d_ncol, d_cmfmc, d_qc, d_qc2, d_rliq, d_rliq2, d_pmid, d_rprddp,
                                            d_cnt, d_cnb, d_cmfmc2, d_rprdsh, d_rprdtot, d_pcnt, d_pcnb,
                                            (void*)st.stream);
  if (rc) return rc;
  return S.flush();
}

// ---- diagnostics ---------------------------------------------------------------------------------
int zm_math_eval_host(int id, int n, const double* x, const double* y, double* o) {
  for (int i = 0; i < n; ++i) {
    switch (id) {
      case 0: o[i] = zmm::log_(x[i]); break;
      case 1: o[i] = zmm::log10_(x[i]); break;
      case 2: o[i] = zmm::exp_(x[i]); break;
      case 3: o[i] = zmm::pow10_(x[i]); break;
      case 5: o[i] = zmm::log_hot(x[i]); break;
      case 6: o[i] = zmm::log10_hot(x[i]); break;
      case 7: o[i] = zmm::pow10_hot(x[i]); break;
      case 8: o[i] = zmm::div_rcp(x[i], y[i], 1.0 / y[i]); break;
      case 9: o[i] = x[i] / y[i]; break;
      case 10: case 12: o[i] = zmm::svp_water<false>(x[i]); break;
      case 11: o[i] = zmm::svp_water_formula(x[i]); break;
      default: o[i] = zmm::pow_(x[i], y[i]); break;
    }
  }
  return 0;
}

int zm_math_eval_dev(int id, int n, const double* x, const double* y, double* out) {
  Workspace& st = tls_stage;
  if (st.ensure(3 * al(n, 8) + 1024)) return -100;
  Stager S(st);
  const double* dx = S.in(x, n); const double* dy = S.in(y, n); double* d_o = S.out(out, n);
  k_math_eval<<<(n + 127) / 128, 128, 0, st.stream>>>(id, n, dx, dy, d_o); ++tls_launches;
  CK(cudaGetLastError());
  return S.flush();
}

int zm_thermo_eval_dev(int id, int n, const double* a, const double* b, const double* c, const double* d,
                       const double* e, double* out0, double* out1) {
  NEED_INIT();
  Workspace& st = tls_stage;
  if (st.ensure(7 * al(n, 8) + 1024)) return -100;
  Stager S(st);
  const double *da = S.in(a, n), *db = S.in(b, n), *dc = S.in(c, n), *dd = S.in(d, n), *de = S.in(e, n);
  double *o0 = S.out(out0, n), *o1 = S.out(out1, n);
  k_thermo_eval<<<(n + 127) / 128, 128, 0, st.stream>>>(id, n, da, db, dc, dd, de, o0, o1); ++tls_launches;
  CK(cudaGetLastError());
  return S.flush();
}

// cycles per dependent call, one warp (ZM_MICROBENCH_N results): 0 div,1 log,2 log10,3 pow10,4 exp,5 es(T),
// 6 enthalpy,7 entropy,8 ienthalpy,9 ientropy,10 pow,11 Goff-Gratch formula,12 DFMA,13 DADD,14 DMUL,15 div_hot,
// 16 log_hot,17 es(T) from shared memory,18 compare+select,19 F2I+I2F.  Writes min(cap, ZM_MICROBENCH_N) values.
int zm_microbench(long long* cycles, int cap, int n) {
  NEED_INIT();
  if (!cycles || cap <= 0) return 0;
  double* d = nullptr; long long* c = nullptr;
  cudaError_t e = cudaMalloc(&d, 32 * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&c, ZM_MICROBENCH_N * sizeof(long long));
  if (e == cudaSuccess) e = cudaMemset(c, 0, ZM_MICROBENCH_N * sizeof(long long));
  if (e == cudaSuccess) { k_microbench<<<1, 32>>>(d, c, n); ++tls_launches; e = cudaGetLastError(); }
  const int m = cap < ZM_MICROBENCH_N ? cap : ZM_MICROBENCH_N;
  if (e == cudaSuccess) e = cudaMemcpy(cycles, c, m * sizeof(long long), cudaMemcpyDeviceToHost);
  cudaFree(d); cudaFree(c);
  if (e != cudaSuccess) { tls_err = std::string("zm_microbench: ") + cudaGetErrorString(e); return -100; }
  return m;
}

double zm_fp64_peak_flops(int iters) {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1.0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int blocks = sms * 8, threads = 256;
  double* d = nullptr;
  if (cudaMalloc(&d, (size_t)blocks * threads * sizeof(double)) != cudaSuccess) return -1.0;
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  k_fp64_peak<<<blocks, threads>>>(d, iters / 10 + 1);
  float best = 1e30f;
  for (int r = 0; r < 5; ++r) {
    cudaEventRecord(e0);
    k_fp64_peak<<<blocks, threads>>>(d, iters);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    if (ms < best) best = ms;
  }
  tls_launches += 6;
  cudaFree(d); cudaEventDestroy(e0); cudaEventDestroy(e1);
  return 2.0 * 8.0 * (double)iters * blocks * threads / (best * 1e-3);
}

}  // extern "C"
