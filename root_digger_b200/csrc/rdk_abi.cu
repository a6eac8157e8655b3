// rdk_abi.cu -- the C ABI of include/rdk.h on top of the sm_100a kernels.
//
// Host-side responsibilities: partition memory in HBM, the P-matrix pool with
// slot renaming, recording of P-matrix updates / CLV operations into a program,
// launch of the three kernels (pmat_expm_nonrev, clv_program, tree_reduce),
// NCCL exchange of the per-shard tree nodes, and the error channel.
//
// There is deliberately no CPU implementation of the path in this file: if a
// CUDA call fails the entry point fails (RDK_FAILURE / NaN).
#include "../../include/rdk.h"
#include "rdk_kernels.cuh"
#include "rdk_support.cuh"

#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <vector>

using namespace rdk;

// ---------------------------------------------------------------------------
// error channel (replaces corax_errno / corax_errmsg)
// ---------------------------------------------------------------------------
static thread_local int  tl_errno = 0;
static thread_local char tl_errmsg[256] = {0};
static thread_local int  tl_device = -1;

extern "C" int  *rdk_errno_location(void) { return &tl_errno; }
extern "C" char *rdk_errmsg_location(void) { return tl_errmsg; }

static int fail(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(tl_errmsg, sizeof(tl_errmsg), fmt, ap);
  va_end(ap);
  tl_errno = code;
  return RDK_FAILURE;
}

#define CUDA_TRY(expr)                                                              \
  do {                                                                              \
    cudaError_t _e = (expr);                                                        \
    if (_e != cudaSuccess)                                                          \
      return fail(RDK_ERROR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                  __FILE__, __LINE__);                                              \
  } while (0)

extern "C" const rdk_state_t rdk_map_nt[256] = {
    0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,   // 0
    0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,   // 16
    0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  15, 0,  0,   // 32  '-'=45
    0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  15,  // 48  '?'=63
    0,  1,  14, 2,  13, 0,  0,  4,  11, 0,  0,  12, 0,  3,  15, 15,  // 64  @ABCDEFGHIJKLMNO
    0,  0,  5,  6,  8,  8,  7,  9,  15, 10, 0,  0,  0,  0,  0,  0,   // 80  PQRSTUVWXYZ
    0,  1,  14, 2,  13, 0,  0,  4,  11, 0,  0,  12, 0,  3,  15, 15,  // 96  `abcdefghijklmno
    0,  0,  5,  6,  8,  8,  7,  9,  15, 10, 0,  0,  0,  0,  0,  0,   // 112 pqrstuvwxyz
};

// ---------------------------------------------------------------------------
// NCCL, resolved lazily with dlopen so that the library has no link-time
// dependency on it (single-GPU use never touches NCCL)
// ---------------------------------------------------------------------------
struct Id128 {  // ncclUniqueId: 128 opaque bytes, passed by value
  char b[128];
};
namespace {
struct NcclApi {
  void *handle = nullptr;
  int (*GetUniqueId)(void *) = nullptr;
  int (*CommInitRank)(void **, int, Id128, int) = nullptr;
  int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
  int (*CommDestroy)(void *) = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
};
}  // namespace
static NcclApi    g_nccl;
static std::mutex g_nccl_mu;

static int load_nccl() {
  std::lock_guard<std::mutex> lk(g_nccl_mu);
  if (g_nccl.handle) return RDK_SUCCESS;
  const char *names[] = {"libnccl.so.2", "libnccl.so"};
  void       *h = nullptr;
  for (const char *n : names) {
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) return fail(RDK_ERROR_COMM, "cannot dlopen libnccl.so.2: %s", dlerror());
  g_nccl.GetUniqueId = (int (*)(void *))dlsym(h, "ncclGetUniqueId");
  g_nccl.CommInitRank = (int (*)(void **, int, Id128, int))dlsym(h, "ncclCommInitRank");
  g_nccl.AllReduce =
      (int (*)(const void *, void *, size_t, int, int, void *, cudaStream_t))dlsym(h, "ncclAllReduce");
  g_nccl.CommDestroy = (int (*)(void *))dlsym(h, "ncclCommDestroy");
  g_nccl.GetErrorString = (const char *(*)(int))dlsym(h, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy)
    return fail(RDK_ERROR_COMM, "libnccl is missing required symbols");
  g_nccl.handle = h;
  return RDK_SUCCESS;
}
// ncclDataType_t / ncclRedOp_t values (stable across NCCL 2.x)
static const int kNcclFloat64 = 8, kNcclUint64 = 5, kNcclSum = 0, kNcclMax = 2;

// ---------------------------------------------------------------------------
// engine state
// ---------------------------------------------------------------------------
namespace {

struct Ring {  // pinned host ring + device ring of equal size, bump-allocated
  char  *h = nullptr, *d = nullptr;
  size_t cap = 0, head = 0;
};

struct Engine {
  int          device = 0;
  cudaStream_t stream = nullptr;
  bool         own_stream = true;
  int          sm_count = 148;

  unsigned tips = 0, clv_buffers = 0, S = 0, prob_matrices = 0, scale_buffers = 0;
  // K: the rate categories the device works with = the partition's (Kreal) padded to the next
  // divisor of the warp size.  A padding category repeats category 0's rate with weight 0: its
  // values equal category 0's (so the all-entries-small rescaling test is unchanged) and its
  // term enters the site likelihood as fma(0, t, sum) = sum, bit for bit.
  unsigned K = 0, Kreal = 0;
  size_t   clv_elems = 0;   // S*K*4 doubles per CLV
  size_t   tip_stride = 0;  // bytes per tip row

  unsigned char          *d_tips = nullptr;
  std::vector<double *>   clv_ptr;   // per inner CLV buffer, lazily allocated
  std::vector<void *>     slabs;     // cudaMalloc'd slabs backing clv_ptr
  double                 *slab_cur = nullptr;
  unsigned                slab_left = 0;
  std::vector<unsigned *> sc_ptr;    // per scale buffer, lazily allocated (zero-filled) in slabs:
  std::vector<void *>     sc_slabs;  // the reference creates 2n-2 of them and uses n-1
  unsigned               *sc_cur = nullptr;
  unsigned                sc_left = 0;
  unsigned               *d_weights = nullptr;  // [S]
  unsigned long long     *d_hist = nullptr;     // [16]

  // P-matrix pool with slot renaming
  double               *d_pool = nullptr;
  unsigned              pool_slots = 0;
  std::vector<unsigned> pm_map;      // matrix index -> physical slot
  std::vector<unsigned> pm_free;     // free physical slots
  std::vector<unsigned> pm_retired;  // freed at the next flush

  // recorded work.  What a program must produce is not kept here: the call that records evaluations
  // hands it to flush (ProgramOutputs), and no rdk_* entry returns with an rEval operation recorded.
  std::vector<PmatEntry> pend_pm;
  std::vector<ROp>       pend_prog;
  unsigned long long     pend_bytes = 0;  // algorithmic bytes of pend_prog
  unsigned               pend_ops = 0, pend_evals = 0;
  // Lazily materialised evaluation.  A full evaluation whose only requested result is the root
  // log-likelihood (the closure BFGS calls 13 times per step, reference src/model.cpp:455-476,
  // 1488-1502) stores only the CLVs it reads back itself; the others exist in registers only.  The
  // recorded operations (with the P-matrix slots they used, held back from recycling) are kept:
  // the next program either rewrites every stale buffer without reading it (the next BFGS
  // evaluation: the kept program is dropped) or makes the engine replay the kept program with
  // all its stores first.  Semantics are those of eager execution.
  struct Lazy {
    bool                  active = false;
    std::vector<ROp>      ops;
    std::vector<char>     stale_clv, stale_sc;  // per index: the value in memory is not the current one
    std::vector<unsigned> held;                 // P-matrix slots retired while the program is kept
  } lazy;
  bool     lazy_enabled = true;
  unsigned full_streak = 0;  // consecutive flushed programs that were lazy-eligible full traversals

  Ring    ring;
  double *d_partials = nullptr;
  size_t  partials_cap = 0;  // doubles
  double *d_nodes = nullptr; // sharded: [slots][global_blocks]
  size_t  nodes_cap = 0;
  double *d_persite = nullptr;
  double *d_rows = nullptr;    // [rows_cap][S]: unweighted per-pattern values (rdk_partition_set_site_lnl_rows)
  unsigned rows_cap = 0;
  double *h_results = nullptr;  // pinned, device-visible
  size_t  results_cap = 0;      // doubles

  // shard / comm
  unsigned long long site_offset = 0, global_sites = 0;
  void              *comm = nullptr;
  int                nranks = 1, rank = 0;
  unsigned long long max_shard_sites = 0;  // largest shard of the layout (agreed over the communicator)

  // Lowered programs kept for the next traversal of the same structure (a BFGS closure re-records
  // the same operations with new P-matrices 13 times per step, a search step alternates one full
  // traversal and one sweep): key = the recorded operations without their P slots + everything
  // else the lowering looks at (the chunks, scratch sets and lazy decision of the program's
  // ProgramOutputs), compared exactly; value = the instructions, whose P slots are refreshed from
  // the operations recorded now.
  struct KeptProgram {
    std::vector<ROp>      ops;
    std::vector<unsigned> chunk_off;
    std::vector<char>     scratch_clv, scratch_sc;
    bool                  lazy = false;
    // the lowering
    bool                  grouped = false;
    std::vector<LInstr>   lowered, lowered_join;
    std::vector<unsigned> lchunk;
    LowerStats            lst;
    unsigned long long    last_use = 0;
  };
  std::vector<KeptProgram> kept_programs;
  unsigned long long       kept_clock = 0;

  // launch config
  int ctas_per_sm = 0, threads = 0, elems = 0;
  int subtree_groups = 0;  // 0: by the cost model, 1: never, n: always n (rdk_partition_set_subtree_groups)

  // optional per-launch timing of the program kernel (bench / profiling)
  bool                                            timing = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pool;
  size_t                                          ev_used = 0;

  rdk_stats_t stats{};
  std::mutex  mu;
};

Engine *eng(rdk_partition_t *p) { return reinterpret_cast<Engine *>(p->engine); }

// host wall time of a scope, added to one of the rdk_stats_t host_*_ns counters
struct HostTimer {
  unsigned long long                   *acc;
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  explicit HostTimer(unsigned long long *a) : acc(a) {}
  ~HostTimer() {
    *acc += (unsigned long long)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0)
                .count();
  }
};

unsigned next_pow2(unsigned long long n) {
  unsigned long long v = 1;
  while (v < n) v <<= 1;
  return (unsigned)v;
}

int dev_alloc(Engine *e, void **ptr, size_t bytes) {
  if (bytes == 0) bytes = 16;
  cudaError_t err = cudaMalloc(ptr, bytes);
  if (err != cudaSuccess)
    return fail(RDK_ERROR_MEM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(err));
  e->stats.device_bytes += bytes;
  return RDK_SUCCESS;
}

int ring_alloc(Engine *e, size_t bytes, char **h, char **d) {
  bytes = (bytes + 255) & ~size_t(255);
  if (bytes > e->ring.cap) {
    // grow: drain the stream, then replace both rings
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    size_t ncap = std::max(bytes * 2, e->ring.cap * 2);
    if (e->ring.h) cudaFreeHost(e->ring.h);
    if (e->ring.d) {
      cudaFree(e->ring.d);
      e->stats.device_bytes -= e->ring.cap;
    }
    e->ring.h = e->ring.d = nullptr;
    CUDA_TRY(cudaMallocHost((void **)&e->ring.h, ncap));
    if (!dev_alloc(e, (void **)&e->ring.d, ncap)) return RDK_FAILURE;
    e->ring.cap = ncap;
    e->ring.head = 0;
  }
  if (e->ring.head + bytes > e->ring.cap) {
    // wrap: everything enqueued so far must have consumed its staging data
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    e->ring.head = 0;
  }
  *h = e->ring.h + e->ring.head;
  *d = e->ring.d + e->ring.head;
  e->ring.head += bytes;
  return RDK_SUCCESS;
}

int ensure_clv(Engine *e, unsigned buf) {
  if (e->clv_ptr[buf]) return RDK_SUCCESS;
  if (e->slab_left == 0) {
    // slabs of up to 64 CLVs or ~1 GiB, whichever is smaller
    size_t   bytes_one = e->clv_elems * sizeof(double);
    if (bytes_one == 0) bytes_one = 32;
    unsigned n = (unsigned)std::max<size_t>(1, std::min<size_t>(64, (size_t(1) << 30) / bytes_one));
    unsigned missing = 0;
    for (double *q : e->clv_ptr)
      if (!q) ++missing;
    n = std::min(n, std::max(1u, missing));
    void *slab = nullptr;
    if (!dev_alloc(e, &slab, bytes_one * n)) return RDK_FAILURE;
    e->slabs.push_back(slab);
    e->slab_cur = reinterpret_cast<double *>(slab);
    e->slab_left = n;
  }
  e->clv_ptr[buf] = e->slab_cur;
  e->slab_cur += e->clv_elems ? e->clv_elems : 4;
  e->slab_left -= 1;
  return RDK_SUCCESS;
}

int ensure_scaler(Engine *e, int idx) {
  if (idx < 0 || e->sc_ptr[idx]) return RDK_SUCCESS;
  const size_t one = ((size_t)std::max(1u, e->S) + 63) & ~size_t(63);  // 256-byte multiples
  if (e->sc_left == 0) {
    unsigned missing = 0;
    for (unsigned *q : e->sc_ptr)
      if (!q) ++missing;
    unsigned n = (unsigned)std::max<size_t>(1, std::min<size_t>(256, (size_t(1) << 28) / (one * 4)));
    n = std::min(n, std::max(1u, missing));
    void *slab = nullptr;
    if (!dev_alloc(e, &slab, one * 4 * n)) return RDK_FAILURE;
    CUDA_TRY(cudaMemsetAsync(slab, 0, one * 4 * n, e->stream));
    e->sc_slabs.push_back(slab);
    e->sc_cur = reinterpret_cast<unsigned *>(slab);
    e->sc_left = n;
  }
  e->sc_ptr[idx] = e->sc_cur;
  e->sc_cur += one;
  e->sc_left -= 1;
  return RDK_SUCCESS;
}

// ---- program-kernel timing ----------------------------------------------------
// fold the recorded event pairs into the stats (waits for them to complete)
void harvest_events(Engine *e) {
  for (size_t i = 0; i < e->ev_used; ++i) {
    float ms = 0.f;
    if (cudaEventSynchronize(e->ev_pool[i].second) == cudaSuccess &&
        cudaEventElapsedTime(&ms, e->ev_pool[i].first, e->ev_pool[i].second) == cudaSuccess) {
      e->stats.program_time_ns += (unsigned long long)((double)ms * 1e6 + 0.5);
      e->stats.program_timed++;
    }
  }
  e->ev_used = 0;
}

std::pair<cudaEvent_t, cudaEvent_t> *next_event_pair(Engine *e) {
  if (e->ev_used == e->ev_pool.size()) {
    if (e->ev_pool.size() >= 256) harvest_events(e);
    else {
      cudaEvent_t a = nullptr, b = nullptr;
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return nullptr;
      e->ev_pool.emplace_back(a, b);
    }
  }
  return &e->ev_pool[e->ev_used++];
}

// ---- launches --------------------------------------------------------------
int launch_pmatrices(rdk_partition_t *p) {
  Engine *e = eng(p);
  if (e->pend_pm.empty()) return RDK_SUCCESS;
  PmatArgs a;
  memset(&a, 0, sizeof(a));
  a.n = (int)e->pend_pm.size();
  a.K = (int)e->K;
  for (int i = 0; i < 12; ++i) a.r[i] = p->subst_params[0][i];
  for (int i = 0; i < 4; ++i) a.pi[i] = p->frequencies[0][i];
  a.pinv = p->prop_invar[0];
  for (unsigned k = 0; k < e->K; ++k) a.rates[k] = p->rates[k < e->Kreal ? k : 0];
  a.pool = e->d_pool;
  if (a.n <= kPmatInline) {
    for (int i = 0; i < a.n; ++i) a.inl[i] = e->pend_pm[i];
  } else {
    char  *h, *d;
    size_t bytes = sizeof(PmatEntry) * e->pend_pm.size();
    if (!ring_alloc(e, bytes, &h, &d)) return RDK_FAILURE;
    memcpy(h, e->pend_pm.data(), bytes);
    CUDA_TRY(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, e->stream));
    e->stats.h2d_bytes += bytes;
    a.entries = reinterpret_cast<const PmatEntry *>(d);
  }
  int total = a.n * a.K;
  int block = 64, grid = (total + block - 1) / block;
  pmat_expm_nonrev_kernel<<<grid, block, 0, e->stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  e->stats.kernel_launches++;
  e->stats.pmatrix_launches++;
  e->stats.pmatrices += e->pend_pm.size();
  e->pend_pm.clear();
  return RDK_SUCCESS;
}

int ensure_partials(Engine *e, unsigned slots, unsigned stride) {
  size_t need = (size_t)slots * stride;
  if (need > e->partials_cap) {
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    if (e->d_partials) {
      cudaFree(e->d_partials);
      e->stats.device_bytes -= e->partials_cap * sizeof(double);
    }
    size_t ncap = std::max(need, e->partials_cap * 2);
    if (!dev_alloc(e, (void **)&e->d_partials, ncap * sizeof(double))) return RDK_FAILURE;
    e->partials_cap = ncap;
  }
  if (slots > e->results_cap) {
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    if (e->h_results) cudaFreeHost(e->h_results);
    size_t ncap = std::max<size_t>(slots, std::max<size_t>(64, e->results_cap * 2));
    CUDA_TRY(cudaHostAlloc((void **)&e->h_results, ncap * sizeof(double), cudaHostAllocMapped));
    e->results_cap = ncap;
  }
  return RDK_SUCCESS;
}

// Launch shape of the program kernel.  A warp's walk is one long dependent instruction stream, so
// a launch costs (passes) x (instructions) x (time per instruction), and the time per instruction
// of a warp carrying E elements per thread grows with the warps that share its SM.  Measured on
// B200 (full evaluations of cfg2-like shards, us per instruction and pass):
//   E = 1: 0.84 at 10 warps per SM, 1.18 at 21      E = 4: 1.36 at 5 warps per SM, 1.43 at 11
// i.e. roughly lat0 + slope x warps with (0.53, 0.031) for E = 1 and (1.31, 0.009) for E = 4
// (E = 2: 1.5 at 10 warps -- never the best, kept for experiments).  The cheapest
// (E, passes) wins; the chunks of a chunked program share the device (grid x chunks CTAs, all
// resident at once).
struct LaunchPlan {
  int    E, threads, grid;
  double cost;  // passes x relative time per instruction
};
const double kStepLat0[5] = {0, 0.53, 1.2, 0, 1.31};
const double kStepSlope[5] = {0, 0.031, 0.03, 0, 0.009};
LaunchPlan plan_launch_for(int sm_count, unsigned n_witer, unsigned n_chunks, int E, int threads_cap, int per_sm_cap) {
  const LaunchShape sh = launch_shape(E);
  int               threads = threads_cap ? std::min(threads_cap, sh.threads) : sh.threads;
  threads = std::max(64, threads);
  const int per_sm = per_sm_cap ? std::min(per_sm_cap, sh.ctas_per_sm) : sh.ctas_per_sm;
  int       grid = sm_count * per_sm;
  if (n_chunks > 1) grid = std::max(1, grid / (int)n_chunks);
  const int cons = threads / 32 - 1;
  // never more consumer warps than warp iterations
  const int max_grid = (int)((n_witer + (unsigned)cons - 1) / (unsigned)cons);
  grid = std::max(1, std::min(grid, max_grid));
  const unsigned per_cta = (n_witer + (unsigned)grid - 1) / (unsigned)grid;
  const unsigned per_warp = (per_cta + (unsigned)cons - 1) / (unsigned)cons;
  const unsigned passes = std::max(1u, (per_warp + (unsigned)E - 1) / (unsigned)E);
  LaunchPlan     pl{};
  pl.E = E;
  pl.threads = threads;
  pl.grid = grid;
  const double warps_per_sm =
      std::min<double>((double)cons * per_sm, (double)n_witer * n_chunks / ((double)sm_count * E * passes));
  pl.cost = passes * (kStepLat0[E] + kStepSlope[E] * warps_per_sm);
  return pl;
}
LaunchPlan plan_launch(const Engine *e, unsigned n_witer, unsigned n_chunks) {
  if (e->elems) return plan_launch_for(e->sm_count, n_witer, n_chunks, e->elems, e->threads, e->ctas_per_sm);
  LaunchPlan best{};
  best.cost = 1e300;
  for (int E : {4, 1}) {
    LaunchPlan pl = plan_launch_for(e->sm_count, n_witer, n_chunks, E, e->threads, e->ctas_per_sm);
    if (pl.cost < best.cost) best = pl;
  }
  return best;
}

// A shard is walked by ONE launch, or by TWO when its iterations do not fill the last E = 4 pass:
// whole E = 4 passes first, then the remaining iterations in the shape that suits them (a warp
// cannot drop elements in its last pass -- the instruction loop is compiled for E elements -- so a
// pass that is 20 % full would cost a full one).  Every element is walked by exactly one launch
// and the two are ordered on the stream, so the results do not depend on the split.
struct LaunchSeg {
  LaunchPlan pl;
  unsigned   it0, n_witer;
};
int plan_segments(const Engine *e, unsigned n_witer, unsigned n_chunks, int n_instr, LaunchSeg seg[2]) {
  seg[0].pl = plan_launch(e, n_witer, n_chunks);
  seg[0].it0 = 0;
  seg[0].n_witer = n_witer;
  if (e->elems || n_instr < 32 || seg[0].pl.E != 4) return 1;
  const LaunchShape sh = launch_shape(4);
  const unsigned    grid = (unsigned)std::max(1, e->sm_count * sh.ctas_per_sm / (int)n_chunks);
  const unsigned    cap = grid * (unsigned)(sh.threads / 32 - 1) * 4u;  // iterations of one full pass
  const unsigned    full = n_witer / cap, rest = n_witer - full * cap;
  if (full == 0 || rest == 0) return 1;
  const LaunchPlan a = plan_launch_for(e->sm_count, full * cap, n_chunks, 4, 0, 0);
  const LaunchPlan b = plan_launch(e, rest, n_chunks);
  if (a.cost + b.cost + 0.02 >= seg[0].pl.cost) return 1;
  seg[0].pl = a;
  seg[0].n_witer = full * cap;
  seg[1].pl = b;
  seg[1].it0 = full * cap;
  seg[1].n_witer = rest;
  return 2;
}

// relative time per instruction of a program of n_instr instructions walked over n_witer warp
// iterations in n_chunks chunks side by side, launched the way launch_lowered launches it
double program_cost(const Engine *e, unsigned n_witer, unsigned n_chunks, int n_instr) {
  LaunchSeg seg[2];
  const int n = plan_segments(e, n_witer, n_chunks, n_instr, seg);
  return seg[0].pl.cost + (n > 1 ? seg[1].pl.cost : 0.0);
}

// index -> device pointer translation of a lowered instruction
void to_device_instr(Engine *e, const LInstr &li, Instr *out) {
  Instr in;
  memset(&in, 0, sizeof(in));
  in.flags = li.flags;
  in.slot = li.slot;
  if (li.flags & fWrite) in.parent = e->clv_ptr[li.parent - e->tips];
  if (li.flags & fWriteS) in.pscale = e->sc_ptr[li.pscale];
  if (li.flags & fTip1)
    in.c1 = e->d_tips + (size_t)li.c1 * e->tip_stride;
  else if (!(li.flags & fNop))
    in.c1 = e->clv_ptr[li.c1 - e->tips];
  if (li.flags & fTip2)
    in.c2 = e->d_tips + (size_t)li.c2 * e->tip_stride;
  else if (li.flags & fLoadV2)
    in.c2 = e->clv_ptr[li.c2 - e->tips];
  if (li.flags & fCnt1) in.c1scale = e->sc_ptr[li.c1scale];
  if (li.flags & fCnt2M) in.c2scale = e->sc_ptr[li.c2scale];
  if (!(li.flags & (fLoadV | fNop))) {
    // the table each child reads: P of an inner child, T of a tip child (same pool slot)
    const size_t K = e->K;
    in.P1 = e->d_pool + (size_t)li.pm1 * K * kSlotDoubles + ((li.flags & fTip1) ? (size_t)kPTabDoubles * K : 0);
    in.P2 = e->d_pool + (size_t)li.pm2 * K * kSlotDoubles + ((li.flags & fTip2) ? (size_t)kPTabDoubles * K : 0);
  }
  *out = in;
}

int materialize_lazy(rdk_partition_t *p);

// copy a lowered program to the device and launch the program kernel over the whole shard
int launch_lowered(rdk_partition_t *p, ProgArgs &a, const std::vector<LInstr> &lowered,
                   const std::vector<unsigned> &lchunk, bool chunked) {
  Engine        *e = eng(p);
  const unsigned n_witer = a.n_witer;
  a.n_instr = (int)lowered.size();
  a.n_chunks = 0;
  a.prog = nullptr;
  if (chunked) {
    a.n_chunks = (unsigned)lchunk.size() - 1;
    for (size_t c = 0; c < lchunk.size(); ++c) a.chunk_off[c] = lchunk[c];
  }
  if (a.n_instr <= kProgInline && !chunked) {
    for (int i = 0; i < a.n_instr; ++i) to_device_instr(e, lowered[i], &a.inl[i]);
  } else {
    char  *h, *d;
    size_t bytes = sizeof(Instr) * lowered.size();
    if (!ring_alloc(e, bytes, &h, &d)) return RDK_FAILURE;
    Instr *hp = reinterpret_cast<Instr *>(h);
    for (size_t i = 0; i < lowered.size(); ++i) to_device_instr(e, lowered[i], &hp[i]);
    CUDA_TRY(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, e->stream));
    e->stats.h2d_bytes += bytes;
    a.prog = reinterpret_cast<const Instr *>(d);
  }
  if (a.nelem == 0 || a.n_instr == 0) return RDK_SUCCESS;
  LaunchSeg seg[2];
  const int n_seg = plan_segments(e, n_witer, chunked ? a.n_chunks : 1u, a.n_instr, seg);
  const bool rows = a.row_stride != 0;  // the ROWS variant (flush, RDK_SWEEP_ROWS)
  for (int g = 0; g < n_seg; ++g) {
    const LaunchPlan &pl = seg[g].pl;
    a.it0 = seg[g].it0;
    a.n_witer = seg[g].n_witer;
    cudaError_t lerr;
    switch (e->K) {
      case 1: lerr = launch_program<1>(a, pl.grid, pl.threads, pl.E, rows, e->stream); break;
      case 2: lerr = launch_program<2>(a, pl.grid, pl.threads, pl.E, rows, e->stream); break;
      case 4: lerr = launch_program<4>(a, pl.grid, pl.threads, pl.E, rows, e->stream); break;
      case 8: lerr = launch_program<8>(a, pl.grid, pl.threads, pl.E, rows, e->stream); break;
      case 16: lerr = launch_program<16>(a, pl.grid, pl.threads, pl.E, rows, e->stream); break;
      case 32: lerr = launch_program<32>(a, pl.grid, pl.threads, pl.E, rows, e->stream); break;
      default: return fail(RDK_ERROR_PARAM, "rate_cats must divide 32");
    }
    if (lerr != cudaSuccess) return fail(RDK_ERROR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(lerr));
    CUDA_TRY(cudaGetLastError());
    e->stats.kernel_launches++;
  }
  a.n_witer = n_witer;
  a.it0 = 0;
  return RDK_SUCCESS;
}

void release_lazy(Engine *e) {
  for (unsigned s : e->lazy.held) e->pm_free.push_back(s);
  e->lazy.held.clear();
  e->lazy.ops.clear();
  e->lazy.active = false;
}

// replay the kept program with all its stores: every buffer holds its current value afterwards
int materialize_lazy(rdk_partition_t *p) {
  Engine *e = eng(p);
  if (!e->lazy.active) return RDK_SUCCESS;
  ProgArgs a;
  memset(&a, 0, sizeof(a));
  a.nelem = e->S * e->K;
  a.n_witer = (a.nelem + 31) / 32;
  a.weights = e->d_weights;
  a.partial_stride = a.n_witer ? a.n_witer : 1;
  std::vector<LInstr>   lowered;
  std::vector<unsigned> lchunk;
  LowerOptions          lopt;
  lopt.tips = e->tips;
  lower_program(e->lazy.ops, std::vector<unsigned>(), lopt, lowered, lchunk, nullptr);
  e->stats.instructions += lowered.size();
  e->stats.materializations++;
  if (!launch_lowered(p, a, lowered, lchunk, false)) return RDK_FAILURE;
  if (a.nelem && !lowered.empty()) e->stats.program_launches++;
  std::fill(e->lazy.stale_clv.begin(), e->lazy.stale_clv.end(), 0);
  std::fill(e->lazy.stale_sc.begin(), e->lazy.stale_sc.end(), 0);
  release_lazy(e);
  e->full_streak = 0;
  return RDK_SUCCESS;
}

// does the pending program read a stale buffer, or leave one stale?  (every child reference counts
// as a read from memory: the lowering may forward it in registers, the test is conservative)
bool pending_needs_materialization(const Engine *e) {
  const auto       &L = e->lazy;
  std::vector<char> wc(L.stale_clv.size(), 0), ws(L.stale_sc.size(), 0);
  auto stale_c = [&](unsigned c) { return c != kNoClv && c < L.stale_clv.size() && L.stale_clv[c] && !wc[c]; };
  auto stale_s = [&](int s) { return s >= 0 && (size_t)s < L.stale_sc.size() && L.stale_sc[s] && !ws[s]; };
  for (const ROp &r : e->pend_prog) {
    if (stale_c(r.c1) || stale_s(r.c1scale)) return true;
    if (!(r.flags & rLoadOnly) && (stale_c(r.c2) || stale_s(r.c2scale))) return true;
    if (r.flags & rWrite) {
      if (r.parent < wc.size()) wc[r.parent] = 1;
      if (r.pscale >= 0 && (size_t)r.pscale < ws.size()) ws[r.pscale] = 1;
    }
  }
  for (size_t c = 0; c < wc.size(); ++c)
    if (L.stale_clv[c] && !wc[c]) return true;
  for (size_t s = 0; s < ws.size(); ++s)
    if (L.stale_sc[s] && !ws[s]) return true;
  return false;
}

// What a flushed program must produce besides the buffers its operations write.  It belongs to the
// one call that records evaluations and runs them (run_evals); every other flush passes none, and
// no operation recorded then carries rEval.
struct ProgramOutputs {
  unsigned slots = 0;           // eval slots: one partial sum per slot and warp iteration
  double  *persite = nullptr;   // per-pattern values of eval slot 0, or of every slot (row_stride)
  bool     unweighted = false;  // persite receives the values before the pattern weight
  size_t   row_stride = 0;      // != 0: eval slot s stores at persite + s * row_stride (the ROWS kernel)
  std::vector<unsigned> chunk_off;  // empty, or the n + 1 offsets of n >= 2 independent chunks
  // per index: the buffer's content after the program is not required (a sweep's scratch); empty: none
  std::vector<char> scratch_clv, scratch_sc;
  bool              lazy_ok = false;  // the program may be evaluated lazily (Engine::Lazy)
};

constexpr size_t kKeptPrograms = 8;    // entries (least recently used replaced)
constexpr size_t kKeptMinOps = 32;     // shorter programs are lowered every time

// same structure?  (P slots and positions excepted)
bool same_structure(const ROp &a, const ROp &b) {
  return a.parent == b.parent && a.pscale == b.pscale && a.c1 == b.c1 && a.c2 == b.c2 && a.c1scale == b.c1scale &&
         a.c2scale == b.c2scale && a.flags == b.flags && a.slot == b.slot;
}

Engine::KeptProgram *find_kept_program(Engine *e, const ProgramOutputs &out, bool lazy) {
  for (Engine::KeptProgram &k : e->kept_programs) {
    if (k.lazy != lazy || k.ops.size() != e->pend_prog.size() || k.chunk_off != out.chunk_off ||
        k.scratch_clv != out.scratch_clv || k.scratch_sc != out.scratch_sc)
      continue;
    bool same = true;
    for (size_t i = 0; same && i < k.ops.size(); ++i) same = same_structure(k.ops[i], e->pend_prog[i]);
    if (same) return &k;
  }
  return nullptr;
}

Engine::KeptProgram *new_kept_program(Engine *e) {
  if (e->kept_programs.size() < kKeptPrograms) {
    e->kept_programs.emplace_back();
    return &e->kept_programs.back();
  }
  Engine::KeptProgram *lru = &e->kept_programs[0];
  for (Engine::KeptProgram &k : e->kept_programs)
    if (k.last_use < lru->last_use) lru = &k;
  return lru;
}

// Subtree groups (rdk_lower.hpp, rdk.h rdk_partition_set_subtree_groups): should the pending program
// run as G groups of disjoint subtrees side by side + the operations that join them?  Decided by
// the launch cost model above: the longest group at the per-instruction time of a launch shared
// by G groups, plus the joining operations at that of a plain launch, against all operations in
// one plain launch.  cfg2 over 8 GPUs (12.5 k sites, 499 operations): 4 groups of <= 130
// operations at 1.41 us + ~20 joining ones, against 499 x 0.86 us.
bool choose_subtree_groups(const Engine *e, unsigned n_witer, std::vector<ROp> &grouped, std::vector<unsigned> &goff,
                           std::vector<ROp> &join) {
  const std::vector<ROp> &ops = e->pend_prog;
  const int               mode = e->subtree_groups;
  const size_t            n = ops.size();
  if (mode == 1 || n < 4 || n_witer == 0) return false;
  if (mode == 0 && (n < 48 || e->elems)) return false;
  static const unsigned kGroups[] = {2, 3, 4, 6, 8};
  // (costs as the programs would really be launched: whole E = 4 passes + the rest in its own shape)
  const double          flat = program_cost(e, n_witer, 1, (int)n);
  double                shared[17] = {0};
  if (mode == 0) {
    // a shard that keeps the device busy with one program gains nothing: skip the analysis
    double best_possible = 1e300;
    for (unsigned g : kGroups) {
      shared[g] = program_cost(e, n_witer, g, (int)(n / g));
      best_possible = std::min(best_possible, (double)n / g * shared[g]);
    }
    if (best_possible >= 0.85 * (double)n * flat) return false;
  }
  ForestInfo fi;
  if (!analyse_forest(ops, e->tips, fi)) return false;
  std::vector<int> group, best_group;
  unsigned         best_used = 0;
  if (mode >= 2) {
    unsigned longest = 0, n_join = 0;
    best_used = assign_subtree_groups(fi, (unsigned)mode, (unsigned)((n + mode - 1) / mode), best_group, longest, n_join);
  } else {
    double best_cost = 0.9 * (double)n * flat;
    for (unsigned g : kGroups)
      for (unsigned div : {1u, 2u}) {
        unsigned       longest = 0, n_join = 0;
        const unsigned cap = (unsigned)((n + g * div - 1) / (g * div));
        const unsigned used = assign_subtree_groups(fi, g, cap, group, longest, n_join);
        if (used < 2) continue;
        const double per = used == g ? shared[g] : program_cost(e, n_witer, used, (int)longest);
        const double cost = longest * per + n_join * flat + 5.0;  // + a launch and its tail, us
        if (cost < best_cost) {
          best_cost = cost;
          best_used = used;
          best_group.swap(group);
        }
      }
  }
  if (best_used < 2) return false;
  split_by_group(ops, best_group, best_used, grouped, goff, join);
  return true;
}

void clear_pending_ops(Engine *e) {
  e->pend_prog.clear();
  e->pend_ops = e->pend_evals = 0;
  e->pend_bytes = 0;
}

// launch recorded P-matrix work and the recorded program, which produces `out` (no host sync)
int flush(rdk_partition_t *p, const ProgramOutputs &out = {}) {
  Engine *e = eng(p);
  if (!launch_pmatrices(p)) return RDK_FAILURE;
  if (e->pend_prog.empty()) {
    for (unsigned s : e->pm_retired) e->pm_free.push_back(s);
    e->pm_retired.clear();
    return RDK_SUCCESS;
  }
  // a kept (lazily evaluated) program: superseded by this one, or replayed before it
  if (e->lazy.active) {
    if (pending_needs_materialization(e)) {
      if (!materialize_lazy(p)) return RDK_FAILURE;
    } else {
      release_lazy(e);  // every stale buffer is rewritten without being read: nothing to keep
    }
  }
  const unsigned nelem = e->S * e->K;
  const unsigned n_witer = (nelem + 31) / 32;
  ProgArgs       a;
  memset(&a, 0, sizeof(a));
  a.nelem = nelem;
  a.n_witer = n_witer;
  a.weights = e->d_weights;
  a.partial_stride = n_witer ? n_witer : 1;
  for (int i = 0; i < 4; ++i) a.pi[i] = p->frequencies[0][i];
  for (unsigned k = 0; k < e->K; ++k) a.w[k] = k < e->Kreal ? p->rate_weights[k] : 0.0;
  if (out.slots) {
    if (!ensure_partials(e, out.slots, a.partial_stride)) return RDK_FAILURE;
    a.partials = e->d_partials;
  }
  a.persite = out.persite;
  a.persite_unweighted = out.unweighted;
  a.row_stride = out.row_stride;
  // recorded operations -> the instructions the kernel walks (rdk_lower.hpp)
  HostTimer             lower_timer(&e->stats.host_lower_ns);  // lowering, pointer translation, enqueue
  const bool            chunked = !out.chunk_off.empty();
  const bool            scratch = !out.scratch_clv.empty() || !out.scratch_sc.empty();
  // Lazy only in a STREAK of such traversals (the second consecutive one onwards): that is the
  // signature of a BFGS closure -- 13 evaluations per step, reference src/model.cpp:1488-1502 --
  // whereas the single compute_lh before a sweep or a root move would only have to be replayed
  // (measured on B200, cfg2 search step: 9.06 ms with an always-lazy compute_lh against 8.03 ms).
  e->full_streak = out.lazy_ok ? e->full_streak + 1 : 0;
  const bool lazy = out.lazy_ok && e->full_streak >= 2 && e->lazy_enabled && !chunked && !scratch;
  for (size_t i = 0; i < e->pend_prog.size(); ++i) e->pend_prog[i].id = (unsigned)i;
  Engine::KeptProgram  scratch_entry;  // programs that are not kept are lowered into this one
  Engine::KeptProgram *kp = nullptr;
  const bool           keepable = e->pend_prog.size() >= kKeptMinOps;
  if (keepable) kp = find_kept_program(e, out, lazy);
  if (kp) {
    e->stats.programs_reused++;
  } else {
    kp = keepable ? new_kept_program(e) : &scratch_entry;
    LowerOptions lopt;
    lopt.tips = e->tips;
    lopt.scratch_clv = &out.scratch_clv;
    lopt.scratch_scaler = &out.scratch_sc;
    lopt.discard_writes = lazy;  // keep only the stores the program reads back itself
    // a long traversal on a small shard: disjoint subtrees side by side, then what joins them
    std::vector<ROp>      group_ops, join_ops;
    std::vector<unsigned> group_off;
    kp->lowered_join.clear();
    kp->grouped = !chunked && !scratch && nelem != 0 && choose_subtree_groups(e, n_witer, group_ops, group_off, join_ops);
    if (kp->grouped)
      lower_grouped(group_ops, group_off, join_ops, lopt, kp->lowered, kp->lchunk, kp->lowered_join, &kp->lst);
    else
      lower_program(e->pend_prog, out.chunk_off, lopt, kp->lowered, kp->lchunk, &kp->lst);
    if (keepable) {
      kp->ops = e->pend_prog;
      kp->chunk_off = out.chunk_off;
      kp->scratch_clv = out.scratch_clv;
      kp->scratch_sc = out.scratch_sc;
      kp->lazy = lazy;
    }
  }
  kp->last_use = ++e->kept_clock;
  // the P slots of the operations recorded NOW (a kept program carries those of its first run)
  for (std::vector<LInstr> *part : {&kp->lowered, &kp->lowered_join})
    for (LInstr &li : *part) {
      if (li.src == kNoSrc) continue;
      const ROp &r = e->pend_prog[li.src];
      li.pm1 = li.swapped ? r.pm2 : r.pm1;
      li.pm2 = li.swapped ? r.pm1 : r.pm2;
    }
  const bool                   grouped = kp->grouped;
  const std::vector<LInstr>   &lowered = kp->lowered, &lowered_join = kp->lowered_join;
  const std::vector<unsigned> &lchunk = kp->lchunk;
  const LowerStats            &lst = kp->lst;
  if (grouped) e->stats.grouped_programs++;
  e->stats.instructions += lowered.size() + lowered_join.size();
  e->stats.stores_elided += lst.stores_dropped;
  if (lazy) {
    // which buffers hold their current value in registers only
    auto &L = e->lazy;
    L.stale_clv.assign(e->tips + e->clv_buffers, 0);
    L.stale_sc.assign(e->scale_buffers, 0);
    bool any = false;
    for (const std::vector<LInstr> *part : {&lowered, &lowered_join})
      for (const LInstr &li : *part) {
        if (li.parent != kNoClv && li.parent < L.stale_clv.size()) {
          L.stale_clv[li.parent] = (li.flags & fWrite) ? 0 : 1;
        }
        if (li.pscale >= 0 && (size_t)li.pscale < L.stale_sc.size())
          L.stale_sc[li.pscale] = (li.flags & fWriteS) ? 0 : 1;
      }
    for (char c : L.stale_clv) any = any || c;
    for (char c : L.stale_sc) any = any || c;
    if (any) {
      L.ops.clear();
      for (const ROp &r : e->pend_prog) {
        if (r.flags & rLoadOnly) continue;
        ROp k = r;
        k.flags = r.flags & rWrite;
        if (k.flags) L.ops.push_back(k);
      }
      L.active = true;
      e->stats.lazy_evaluations++;
    }
  }
  const bool runs = nelem != 0 && lowered.size() + lowered_join.size() != 0;
  std::pair<cudaEvent_t, cudaEvent_t> *ev = (runs && e->timing) ? next_event_pair(e) : nullptr;
  if (ev) CUDA_TRY(cudaEventRecord(ev->first, e->stream));
  if (grouped) {
    ProgArgs ag = a;
    if (!launch_lowered(p, ag, lowered, lchunk, true)) return RDK_FAILURE;
    if (!lowered_join.empty() && !launch_lowered(p, a, lowered_join, std::vector<unsigned>(), false)) return RDK_FAILURE;
  } else {
    if (!launch_lowered(p, a, lowered, lchunk, chunked)) return RDK_FAILURE;
  }
  if (ev) CUDA_TRY(cudaEventRecord(ev->second, e->stream));
  if (runs) e->stats.program_launches++;
  e->stats.clv_ops += e->pend_ops;
  e->stats.root_evals += e->pend_evals;
  e->stats.algorithmic_bytes += e->pend_bytes;
  clear_pending_ops(e);
  for (unsigned s : e->pm_retired) e->pm_free.push_back(s);
  e->pm_retired.clear();
  return RDK_SUCCESS;
}

// reduce the partials of `slots` eval slots to h_results[0..slots) (+ sync)
int finish_evals(rdk_partition_t *p, unsigned slots) {
  Engine        *e = eng(p);
  const unsigned nelem = e->S * e->K;
  const unsigned n_witer = (nelem + 31) / 32;
  const unsigned stride = n_witer ? n_witer : 1;
  double        *d_out = nullptr;
  CUDA_TRY(cudaHostGetDevicePointer((void **)&d_out, e->h_results, 0));
  const bool sharded = e->global_sites != 0 && (e->comm != nullptr || e->global_sites != e->S);
  if (!sharded) {
    unsigned span = next_pow2(std::max(1u, n_witer));
    tree_reduce_kernel<<<dim3(1, slots), 256, 0, e->stream>>>(e->d_partials, stride, n_witer, span, 1u,
                                                             d_out, 1, 0);
    CUDA_TRY(cudaGetLastError());
    e->stats.kernel_launches++;
    e->stats.reduce_launches++;
  } else {
    // nodes of the global tree that cover RDK_SHARD_ALIGN sites each
    const unsigned span1 = RDK_SHARD_ALIGN * e->K / 32;
    const unsigned gblocks =
        (unsigned)((e->global_sites + RDK_SHARD_ALIGN - 1) / RDK_SHARD_ALIGN);
    const unsigned lblocks = (n_witer + span1 - 1) / span1;
    const unsigned boff = (unsigned)(e->site_offset / RDK_SHARD_ALIGN);
    size_t         need = (size_t)slots * gblocks;
    if (need > e->nodes_cap) {
      CUDA_TRY(cudaStreamSynchronize(e->stream));
      if (e->d_nodes) {
        cudaFree(e->d_nodes);
        e->stats.device_bytes -= e->nodes_cap * sizeof(double);
      }
      if (!dev_alloc(e, (void **)&e->d_nodes, need * sizeof(double))) return RDK_FAILURE;
      e->nodes_cap = need;
    }
    CUDA_TRY(cudaMemsetAsync(e->d_nodes, 0, need * sizeof(double), e->stream));
    if (lblocks) {
      const unsigned per_block = 256u / std::min(span1, 256u);  // nodes one block reduces
      tree_reduce_kernel<<<dim3((lblocks + per_block - 1) / per_block, slots), 256, 0, e->stream>>>(
          e->d_partials, stride, n_witer, span1, lblocks, e->d_nodes, gblocks, boff);
      CUDA_TRY(cudaGetLastError());
      e->stats.kernel_launches++;
      e->stats.reduce_launches++;
    }
    if (e->comm) {
      // every other shard contributes +0.0 to a node, so the sum is exact and
      // the result is independent of the number of shards
      int rc = g_nccl.AllReduce(e->d_nodes, e->d_nodes, need, kNcclFloat64, kNcclSum, e->comm,
                                e->stream);
      if (rc != 0)
        return fail(RDK_ERROR_COMM, "ncclAllReduce failed: %s",
                    g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
    }
    tree_reduce_kernel<<<dim3(1, slots), 256, 0, e->stream>>>(e->d_nodes, gblocks, gblocks,
                                                             next_pow2(gblocks), 1u, d_out, 1, 0);
    CUDA_TRY(cudaGetLastError());
    e->stats.kernel_launches++;
    e->stats.reduce_launches++;
  }
  {
    HostTimer wait_timer(&e->stats.host_wait_ns);
    CUDA_TRY(cudaStreamSynchronize(e->stream));
  }
  e->stats.d2h_bytes += sizeof(double) * slots;
  return RDK_SUCCESS;
}

// Run the recorded program with the evaluations `out` asks for and copy their values to
// results[0..out.slots).  If that fails, the recorded operations are dropped: a later flush would
// run their evaluations without outputs.  The recorded P-matrix updates stay, because the indices
// already name their new slots (as after eager execution).
int run_evals(rdk_partition_t *p, const ProgramOutputs &out, double *results) {
  Engine *e = eng(p);
  if (!flush(p, out) || !finish_evals(p, out.slots)) {
    clear_pending_ops(e);
    return RDK_FAILURE;
  }
  for (unsigned i = 0; i < out.slots; ++i) results[i] = e->h_results[i];
  return RDK_SUCCESS;
}

// translate a corax-shaped operation into a recorded operation (buffers allocated, P-matrix
// indices resolved to the physical pool slots they name NOW)
int make_rop(rdk_partition_t *p, const rdk_operation_t &op, unsigned flags, ROp *out) {
  Engine *e = eng(p);
  const unsigned nclv = e->tips + e->clv_buffers;
  if (op.parent_clv_index < e->tips || op.parent_clv_index >= nclv)
    return fail(RDK_ERROR_PARAM, "parent_clv_index %u out of range", op.parent_clv_index);
  if (op.child1_clv_index >= nclv || op.child2_clv_index >= nclv)
    return fail(RDK_ERROR_PARAM, "child clv index out of range");
  if (op.child1_matrix_index >= e->prob_matrices || op.child2_matrix_index >= e->prob_matrices)
    return fail(RDK_ERROR_PARAM, "matrix index out of range");
  auto bad_scaler = [&](int s) { return s != RDK_SCALE_BUFFER_NONE && (s < 0 || (unsigned)s >= e->scale_buffers); };
  if (bad_scaler(op.parent_scaler_index) || bad_scaler(op.child1_scaler_index) ||
      bad_scaler(op.child2_scaler_index))
    return fail(RDK_ERROR_PARAM, "scaler index out of range");
  ROp r;
  memset(&r, 0, sizeof(r));
  r.flags = flags;
  r.parent = op.parent_clv_index;
  if (!ensure_clv(e, op.parent_clv_index - e->tips)) return RDK_FAILURE;
  // reading an unwritten CLV: zeros
  if (op.child1_clv_index >= e->tips && !ensure_clv(e, op.child1_clv_index - e->tips)) return RDK_FAILURE;
  if (op.child2_clv_index >= e->tips && !ensure_clv(e, op.child2_clv_index - e->tips)) return RDK_FAILURE;
  r.c1 = op.child1_clv_index;
  r.c2 = op.child2_clv_index;
  r.pscale = op.parent_scaler_index;
  // without a parent scale buffer the children's counts are dropped (coraxlib semantics)
  const bool scaled = op.parent_scaler_index != RDK_SCALE_BUFFER_NONE;
  r.c1scale = scaled ? op.child1_scaler_index : -1;
  r.c2scale = scaled ? op.child2_scaler_index : -1;
  if (op.child1_clv_index < e->tips && op.child2_clv_index < e->tips && r.c1scale >= 0 && r.c2scale >= 0)
    return fail(RDK_ERROR_PARAM, "two tip children with scale buffers are not supported (tips carry no scaler, "
                                 "reference test/src/tree.cpp:157)");
  if (!ensure_scaler(e, r.pscale) || !ensure_scaler(e, r.c1scale) || !ensure_scaler(e, r.c2scale)) return RDK_FAILURE;
  r.pm1 = e->pm_map[op.child1_matrix_index];
  r.pm2 = e->pm_map[op.child2_matrix_index];
  *out = r;
  return RDK_SUCCESS;
}

// SURVEY 8d accounting for one CLV operation on this shard
unsigned long long op_bytes(const Engine *e, const ROp &r) {
  unsigned long long S = e->S, clv = 32ull * e->Kreal * S, b = 0;  // the partition's categories, not the padding
  b += (r.c1 < e->tips) ? S : clv;
  b += (r.c2 < e->tips) ? S : clv;
  if (r.flags & rWrite) b += clv;
  if (r.c1scale >= 0) b += 4 * S;
  if (r.c2scale >= 0) b += 4 * S;
  if ((r.flags & rWrite) && r.pscale >= 0) b += 4 * S;
  if (r.flags & rEval) b += 4 * S;  // pattern weights
  return b;
}

// record CLV operations in order; when one is refused, those before it stay recorded
int record_ops(rdk_partition_t *p, const rdk_operation_t *ops, unsigned count) {
  Engine *e = eng(p);
  for (unsigned i = 0; i < count; ++i) {
    ROp r;
    if (!make_rop(p, ops[i], rWrite, &r)) return RDK_FAILURE;
    e->pend_bytes += op_bytes(e, r);
    e->pend_prog.push_back(r);
    e->pend_ops++;
  }
  return RDK_SUCCESS;
}

// Record the evaluation of root CLV `clv` (scale buffer rs, -1: none) into eval slot `slot`: fused
// into the last recorded operation if that one writes this CLV (keep_root: it is then only
// evaluated in registers and stores nothing), else as an operation that loads the CLV.  Returns
// whether the evaluation was fused.
bool record_root_eval(Engine *e, unsigned clv, int rs, unsigned slot, bool keep_root) {
  e->pend_evals++;
  if (!e->pend_prog.empty()) {
    ROp &last = e->pend_prog.back();
    if ((last.flags & rWrite) && !(last.flags & rEval) && last.parent == clv && last.pscale == rs) {
      e->pend_bytes -= op_bytes(e, last);
      last.flags |= rEval;
      if (keep_root) last.flags &= ~rWrite;
      last.slot = slot;
      e->pend_bytes += op_bytes(e, last);
      return true;
    }
  }
  ROp r;
  memset(&r, 0, sizeof(r));
  r.flags = rLoadOnly | rEval;
  r.parent = kNoClv;
  r.pscale = -1;
  r.c1 = clv;
  r.c1scale = rs;
  r.c2 = kNoClv;
  r.c2scale = -1;
  r.slot = slot;
  e->pend_bytes += 32ull * e->Kreal * e->S + (rs >= 0 ? 4ull * e->S : 0) + 4ull * e->S;
  e->pend_prog.push_back(r);
  return false;
}

// record a P-matrix update with slot renaming; caller holds the mutex
int record_pmatrix(rdk_partition_t *p, unsigned matrix_index, double t) {
  Engine *e = eng(p);
  if (e->pm_free.empty() && e->lazy.active) {
    if (!materialize_lazy(p)) return RDK_FAILURE;  // releases the slots held for the kept program
  }
  if (e->pm_free.empty()) {
    // recycle: launch what is recorded so that retired slots become free
    if (!flush(p)) return RDK_FAILURE;
    if (e->pm_free.empty()) return fail(RDK_ERROR_MEM, "P-matrix pool exhausted");
  }
  unsigned slot = e->pm_free.back();
  e->pm_free.pop_back();
  (e->lazy.active ? e->lazy.held : e->pm_retired).push_back(e->pm_map[matrix_index]);
  e->pm_map[matrix_index] = slot;
  PmatEntry ent;
  ent.slot = slot;
  ent.pad = 0;
  ent.t = t;
  e->pend_pm.push_back(ent);
  return RDK_SUCCESS;
}

// P entries recorded so far were computed against the current parameters;
// launch them before a parameter changes
int params_about_to_change(rdk_partition_t *p) { return launch_pmatrices(p); }

}  // namespace

// ---------------------------------------------------------------------------
// device selection
// ---------------------------------------------------------------------------
extern "C" int rdk_device_count(void) {
  int         n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    fail(RDK_ERROR_CUDA, "cudaGetDeviceCount failed: %s", cudaGetErrorString(e));
    return 0;
  }
  return n;
}

extern "C" int rdk_set_device(int device) {
  CUDA_TRY(cudaSetDevice(device));
  tl_device = device;
  return RDK_SUCCESS;
}

extern "C" const char *rdk_version(void) { return "rdk-b200 0.1 (sm_100a)"; }

// ---------------------------------------------------------------------------
// partition life cycle
// ---------------------------------------------------------------------------
static int engine_init(rdk_partition_t *p, Engine *e) {
  if (tl_device >= 0) CUDA_TRY(cudaSetDevice(tl_device));
  CUDA_TRY(cudaGetDevice(&e->device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, e->device));
  e->sm_count = prop.multiProcessorCount;
  CUDA_TRY(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  e->tips = p->tips;
  e->clv_buffers = p->clv_buffers;
  e->S = p->sites;
  if (const char *env = getenv("RDK_LAZY")) e->lazy_enabled = atoi(env) != 0;
  if (const char *env = getenv("RDK_SUBTREE_GROUPS")) e->subtree_groups = std::max(0, std::min(kMaxChunks, atoi(env)));
  e->Kreal = p->rate_cats;
  e->K = 1;
  while (e->K < e->Kreal) e->K <<= 1;
  e->prob_matrices = p->prob_matrices;
  e->scale_buffers = p->scale_buffers;
  e->clv_elems = (size_t)e->S * e->K * 4;
  e->tip_stride = ((size_t)e->S + 127) & ~size_t(127);
  e->global_sites = 0;
  e->clv_ptr.assign(e->clv_buffers, nullptr);

  if (!dev_alloc(e, (void **)&e->d_tips, e->tip_stride * std::max(1u, e->tips))) return RDK_FAILURE;
  CUDA_TRY(cudaMemsetAsync(e->d_tips, 0, e->tip_stride * std::max(1u, e->tips), e->stream));
  e->sc_ptr.assign(e->scale_buffers, nullptr);
  if (!dev_alloc(e, (void **)&e->d_weights, sizeof(unsigned) * std::max(1u, e->S))) return RDK_FAILURE;
  if (!dev_alloc(e, (void **)&e->d_hist, sizeof(unsigned long long) * 16)) return RDK_FAILURE;
  if (!dev_alloc(e, (void **)&e->d_persite, sizeof(double) * std::max(1u, e->S))) return RDK_FAILURE;
  std::vector<unsigned> ones(std::max(1u, e->S), 1u);
  CUDA_TRY(cudaMemcpyAsync(e->d_weights, ones.data(), sizeof(unsigned) * ones.size(),
                           cudaMemcpyHostToDevice, e->stream));
  CUDA_TRY(cudaStreamSynchronize(e->stream));

  // P-matrix pool: every index has a slot, plus spare slots for renaming
  // two generations of every matrix, 4096 for the per-placement root branches of a sweep, and
  // room for the chunks of a chunked sweep to re-record the branches they walk
  e->pool_slots = e->prob_matrices * 2 + 4096 + std::min<unsigned>(e->prob_matrices * (unsigned)kMaxChunks, 32768u);
  size_t pool_bytes = sizeof(double) * kSlotDoubles * e->K * (size_t)e->pool_slots;
  if (!dev_alloc(e, (void **)&e->d_pool, pool_bytes)) return RDK_FAILURE;
  CUDA_TRY(cudaMemsetAsync(e->d_pool, 0, pool_bytes, e->stream));
  e->pm_map.resize(e->prob_matrices);
  for (unsigned i = 0; i < e->prob_matrices; ++i) e->pm_map[i] = i;
  for (unsigned s = e->pool_slots; s-- > e->prob_matrices;) e->pm_free.push_back(s);

  e->ring.cap = 0;
  char *h, *d;
  if (!ring_alloc(e, size_t(1) << 20, &h, &d)) return RDK_FAILURE;
  e->ring.head = 0;
  if (!ensure_partials(e, 1, std::max(1u, (e->S * e->K + 31) / 32))) return RDK_FAILURE;
  return RDK_SUCCESS;
}

extern "C" rdk_partition_t *rdk_partition_create(unsigned int tips, unsigned int clv_buffers,
                                                 unsigned int states, unsigned int sites,
                                                 unsigned int rate_matrices,
                                                 unsigned int prob_matrices,
                                                 unsigned int rate_cats,
                                                 unsigned int scale_buffers,
                                                 unsigned int attributes) {
  tl_errno = 0;
  if (states != 4) {
    fail(RDK_ERROR_PARAM, "only 4-state (DNA) partitions are supported, got %u states", states);
    return nullptr;
  }
  if (!(attributes & RDK_ATTRIB_NONREV)) {
    fail(RDK_ERROR_PARAM, "RDK_ATTRIB_NONREV is required (non-reversible engine)");
    return nullptr;
  }
  if (rate_matrices != 1) {
    fail(RDK_ERROR_PARAM, "exactly one rate matrix per partition is supported (model_t::_submodels)");
    return nullptr;
  }
  if (rate_cats == 0 || rate_cats > (unsigned)kMaxCats) {
    fail(RDK_ERROR_PARAM, "rate_cats must be in [1, %d] (got %u)", kMaxCats, rate_cats);
    return nullptr;
  }
  if ((unsigned long long)sites * rate_cats >= (1ull << 31)) {
    fail(RDK_ERROR_PARAM, "sites * rate_cats must be < 2^31 per shard");
    return nullptr;
  }
  rdk_partition_t *p = (rdk_partition_t *)calloc(1, sizeof(rdk_partition_t));
  if (!p) {
    fail(RDK_ERROR_MEM, "out of host memory");
    return nullptr;
  }
  p->tips = tips;
  p->clv_buffers = clv_buffers;
  p->states = states;
  p->sites = sites;
  p->rate_matrices = rate_matrices;
  p->prob_matrices = prob_matrices;
  p->rate_cats = rate_cats;
  p->scale_buffers = scale_buffers;
  p->attributes = attributes;
  p->subst_params = (double **)calloc(rate_matrices, sizeof(double *));
  p->frequencies = (double **)calloc(rate_matrices, sizeof(double *));
  for (unsigned i = 0; i < rate_matrices; ++i) {
    p->subst_params[i] = (double *)calloc(12, sizeof(double));
    p->frequencies[i] = (double *)calloc(4, sizeof(double));
    for (int j = 0; j < 12; ++j) p->subst_params[i][j] = 1.0;
    for (int j = 0; j < 4; ++j) p->frequencies[i][j] = 0.25;
  }
  p->rates = (double *)calloc(rate_cats, sizeof(double));
  p->rate_weights = (double *)calloc(rate_cats, sizeof(double));
  for (unsigned k = 0; k < rate_cats; ++k) {
    p->rates[k] = 1.0;
    p->rate_weights[k] = 1.0 / rate_cats;
  }
  p->prop_invar = (double *)calloc(rate_matrices, sizeof(double));
  p->pattern_weights = (unsigned *)calloc(sites ? sites : 1, sizeof(unsigned));
  for (unsigned s = 0; s < sites; ++s) p->pattern_weights[s] = 1;
  Engine *e = new Engine();
  p->engine = e;
  if (!engine_init(p, e)) {
    rdk_partition_destroy(p);
    return nullptr;
  }
  return p;
}

extern "C" void rdk_partition_destroy(rdk_partition_t *p) {
  if (!p) return;
  Engine *e = eng(p);
  if (e) {
    cudaSetDevice(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    if (e->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(e->comm);
    cudaFree(e->d_tips);
    for (void *s : e->slabs) cudaFree(s);
    for (void *q : e->sc_slabs) cudaFree(q);
    cudaFree(e->d_weights);
    cudaFree(e->d_hist);
    cudaFree(e->d_persite);
    cudaFree(e->d_rows);
    cudaFree(e->d_pool);
    cudaFree(e->d_partials);
    cudaFree(e->d_nodes);
    cudaFree(e->ring.d);
    if (e->ring.h) cudaFreeHost(e->ring.h);
    if (e->h_results) cudaFreeHost(e->h_results);
    for (auto &pr : e->ev_pool) {
      cudaEventDestroy(pr.first);
      cudaEventDestroy(pr.second);
    }
    if (e->stream && e->own_stream) cudaStreamDestroy(e->stream);
    delete e;
  }
  for (unsigned i = 0; i < p->rate_matrices; ++i) {
    free(p->subst_params[i]);
    free(p->frequencies[i]);
  }
  free(p->subst_params);
  free(p->frequencies);
  free(p->rates);
  free(p->rate_weights);
  free(p->prop_invar);
  free(p->pattern_weights);
  free(p);
}

// ---------------------------------------------------------------------------
// inputs
// ---------------------------------------------------------------------------
extern "C" int rdk_set_tip_states(rdk_partition_t *p, unsigned int tip_index, const rdk_state_t *map,
                                  const char *sequence) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  if (tip_index >= e->tips) return fail(RDK_ERROR_PARAM, "tip index %u out of range", tip_index);
  CUDA_TRY(cudaSetDevice(e->device));
  if (!flush(p)) return RDK_FAILURE;
  if (!materialize_lazy(p)) return RDK_FAILURE;  // a kept program would be replayed on the NEW tips
  char *h, *d;
  if (!ring_alloc(e, e->S ? e->S : 1, &h, &d)) return RDK_FAILURE;
  for (unsigned s = 0; s < e->S; ++s) {
    rdk_state_t st = map[(unsigned char)sequence[s]];
    if (!st) {
      tl_errno = RDK_ERROR_TIP_DATA;
      snprintf(tl_errmsg, sizeof(tl_errmsg), "Illegal state code in tip \"%c\"", sequence[s]);
      return RDK_FAILURE;
    }
    h[s] = (char)tip_code_of_mask((unsigned)(st & 15ull));
  }
  CUDA_TRY(cudaMemcpyAsync(e->d_tips + (size_t)tip_index * e->tip_stride, h, e->S,
                           cudaMemcpyHostToDevice, e->stream));
  e->stats.h2d_bytes += e->S;
  return RDK_SUCCESS;
}

extern "C" void rdk_set_pattern_weights(rdk_partition_t *p, const unsigned int *w) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  cudaSetDevice(e->device);
  flush(p);
  memcpy(p->pattern_weights, w, sizeof(unsigned) * e->S);
  char *h, *d;
  if (!ring_alloc(e, sizeof(unsigned) * (e->S ? e->S : 1), &h, &d)) return;
  memcpy(h, w, sizeof(unsigned) * e->S);
  cudaMemcpyAsync(e->d_weights, h, sizeof(unsigned) * e->S, cudaMemcpyHostToDevice, e->stream);
  e->stats.h2d_bytes += sizeof(unsigned) * e->S;
}

extern "C" void rdk_set_subst_params(rdk_partition_t *p, unsigned int idx, const double *params) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  if (idx >= p->rate_matrices) return;
  cudaSetDevice(e->device);
  params_about_to_change(p);
  memcpy(p->subst_params[idx], params, sizeof(double) * 12);
}

extern "C" void rdk_set_frequencies(rdk_partition_t *p, unsigned int idx, const double *f) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  if (idx >= p->rate_matrices) return;
  cudaSetDevice(e->device);
  flush(p);  // frequencies also enter recorded evaluations
  memcpy(p->frequencies[idx], f, sizeof(double) * 4);
}

extern "C" void rdk_set_category_rates(rdk_partition_t *p, const double *rates) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  cudaSetDevice(e->device);
  params_about_to_change(p);
  memcpy(p->rates, rates, sizeof(double) * e->Kreal);
}

extern "C" void rdk_set_category_weights(rdk_partition_t *p, const double *w) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  cudaSetDevice(e->device);
  flush(p);
  memcpy(p->rate_weights, w, sizeof(double) * e->Kreal);
}

extern "C" int rdk_update_invariant_sites(rdk_partition_t *p) {
  // Marks invariant columns for the +I likelihood term.  RootDigger never sets
  // a non-zero proportion (reference src/model.cpp:292-300, SURVEY B-5), and the
  // engine rejects a non-zero proportion below, so the marks are never read.
  (void)p;
  return RDK_SUCCESS;
}

extern "C" int rdk_update_invariant_sites_proportion(rdk_partition_t *p, unsigned int idx,
                                                     double prop_invar) {
  if (idx >= p->rate_matrices) return fail(RDK_ERROR_PARAM, "params index out of range");
  if (prop_invar != 0.0)
    return fail(RDK_ERROR_PARAM,
                "a non-zero proportion of invariant sites is not supported (RootDigger always "
                "passes 0.0)");
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  params_about_to_change(p);
  p->prop_invar[idx] = prop_invar;
  return RDK_SUCCESS;
}

// ---------------------------------------------------------------------------
// the hot path
// ---------------------------------------------------------------------------
extern "C" int rdk_update_prob_matrices(rdk_partition_t *p, const unsigned int *params_indices,
                                        const unsigned int *matrix_indices,
                                        const double *branch_lengths, unsigned int count) {
  Engine *e = eng(p);
  if (params_indices)
    for (unsigned k = 0; k < e->Kreal; ++k)
      if (params_indices[k] != 0) return fail(RDK_ERROR_PARAM, "params_indices must be all 0");
  for (unsigned i = 0; i < count; ++i) {
    if (matrix_indices[i] >= e->prob_matrices)
      return fail(RDK_ERROR_PARAM, "matrix index %u out of range", matrix_indices[i]);
    if (!(branch_lengths[i] >= 0.0) || !std::isfinite(branch_lengths[i]))
      return fail(RDK_ERROR_PARAM, "branch length must be finite and non-negative");
  }
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  HostTimer record_timer(&e->stats.host_record_ns);
  for (unsigned i = 0; i < count; ++i)
    if (!record_pmatrix(p, matrix_indices[i], branch_lengths[i])) return RDK_FAILURE;
  return RDK_SUCCESS;
}

extern "C" void rdk_update_clvs(rdk_partition_t *p, const rdk_operation_t *ops, unsigned int count) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  cudaSetDevice(e->device);
  HostTimer record_timer(&e->stats.host_record_ns);
  record_ops(p, ops, count);  // error left in rdk_errno
}

// rdk_compute_root_loglikelihood; `row` (device, [S]) optionally receives the unweighted values
static double root_loglikelihood(rdk_partition_t *p, unsigned int clv_index, int scaler_index,
                                 double *persite_lnl, double *row) {
  Engine *e = eng(p);
  const double nan = std::numeric_limits<double>::quiet_NaN();
  std::lock_guard<std::mutex> lk(e->mu);
  if (cudaSetDevice(e->device) != cudaSuccess) return nan;
  if (clv_index >= e->tips + e->clv_buffers || clv_index < e->tips) {
    fail(RDK_ERROR_PARAM, "root clv index %u out of range", clv_index);
    return nan;
  }
  if (scaler_index != RDK_SCALE_BUFFER_NONE && (scaler_index < 0 || (unsigned)scaler_index >= e->scale_buffers)) {
    fail(RDK_ERROR_PARAM, "root scaler index out of range");
    return nan;
  }
  if (!ensure_clv(e, clv_index - e->tips)) return nan;
  const int rs = scaler_index == RDK_SCALE_BUFFER_NONE ? -1 : scaler_index;
  if (!ensure_scaler(e, rs)) return nan;
  const bool fused = record_root_eval(e, clv_index, rs, 0, false);
  ProgramOutputs out;
  out.slots = 1;
  // a row of unweighted values takes the place of the weighted per-site output (never both)
  out.persite = row ? row : (persite_lnl ? e->d_persite : nullptr);
  out.unweighted = row != nullptr;
  // a traversal whose only requested result is this log-likelihood may keep its CLVs in registers
  if (fused && !out.persite) {
    size_t writes = 0;
    for (const ROp &r : e->pend_prog) writes += (r.flags & rWrite) ? 1 : 0;
    out.lazy_ok = writes >= 16;
  }
  if (e->S == 0 && e->global_sites == 0) {  // no sites at all: nothing to reduce
    if (flush(p, out)) return 0.0;
    clear_pending_ops(e);
    return nan;
  }
  double lnl;
  if (!run_evals(p, out, &lnl)) return nan;
  if (persite_lnl) {
    if (cudaMemcpy(persite_lnl, e->d_persite, sizeof(double) * e->S, cudaMemcpyDeviceToHost) !=
        cudaSuccess) {
      fail(RDK_ERROR_CUDA, "persite copy failed");
      return nan;
    }
    e->stats.d2h_bytes += sizeof(double) * e->S;
  }
  return lnl;
}

extern "C" double rdk_compute_root_loglikelihood(rdk_partition_t *p, unsigned int clv_index,
                                                 int scaler_index, const unsigned int *freqs_indices,
                                                 double *persite_lnl) {
  (void)freqs_indices;
  return root_loglikelihood(p, clv_index, scaler_index, persite_lnl, nullptr);
}

// ---------------------------------------------------------------------------
// root placement support: per-pattern rows and the RELL statistics (rdk_support.cu)
// ---------------------------------------------------------------------------
extern "C" int rdk_partition_set_site_lnl_rows(rdk_partition_t *p, unsigned int rows) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  CUDA_TRY(cudaStreamSynchronize(e->stream));
  if (e->d_rows) {
    cudaFree(e->d_rows);
    e->stats.device_bytes -= sizeof(double) * (size_t)e->rows_cap * std::max(1u, e->S);
    e->d_rows = nullptr;
    e->rows_cap = 0;
  }
  if (rows == 0) return RDK_SUCCESS;
  if (!dev_alloc(e, (void **)&e->d_rows, sizeof(double) * (size_t)rows * std::max(1u, e->S))) return RDK_FAILURE;
  e->rows_cap = rows;
  return RDK_SUCCESS;
}

extern "C" double rdk_compute_root_loglikelihood_row(rdk_partition_t *p, unsigned int clv_index,
                                                     int scaler_index, unsigned int row) {
  Engine *e = eng(p);
  if (row >= e->rows_cap) {
    fail(RDK_ERROR_PARAM, "site row %u out of range (%u rows reserved)", row, e->rows_cap);
    return std::numeric_limits<double>::quiet_NaN();
  }
  return root_loglikelihood(p, clv_index, scaler_index, nullptr, e->d_rows + (size_t)row * e->S);
}

extern "C" int rdk_partition_get_site_lnl_rows(rdk_partition_t *p, unsigned int first, unsigned int count,
                                               double *out) {
  Engine *e = eng(p);
  if ((unsigned long long)first + count > e->rows_cap) return fail(RDK_ERROR_PARAM, "site rows out of range");
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  if (!flush(p)) return RDK_FAILURE;
  CUDA_TRY(cudaMemcpyAsync(out, e->d_rows + (size_t)first * e->S, sizeof(double) * (size_t)count * e->S,
                           cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(cudaStreamSynchronize(e->stream));
  e->stats.d2h_bytes += sizeof(double) * (size_t)count * e->S;
  return RDK_SUCCESS;
}

extern "C" int rdk_partition_permute_site_lnl_rows(rdk_partition_t *p, unsigned int count,
                                                   const unsigned int *order) {
  Engine *e = eng(p);
  if (count > e->rows_cap) return fail(RDK_ERROR_PARAM, "site rows out of range");
  std::vector<char> seen(count, 0);
  for (unsigned r = 0; r < count; ++r) {
    if (order[r] >= count || seen[order[r]]) return fail(RDK_ERROR_PARAM, "order is not a permutation of the rows");
    seen[order[r]] = 1;
  }
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  if (!flush(p)) return RDK_FAILURE;
  if (e->S == 0) return RDK_SUCCESS;
  // cycle by cycle, in place, through the per-site scratch row (S doubles)
  const size_t bytes = sizeof(double) * e->S;
  auto row = [&](unsigned r) { return e->d_rows + (size_t)r * e->S; };
  std::fill(seen.begin(), seen.end(), 0);
  for (unsigned r0 = 0; r0 < count; ++r0) {
    if (seen[r0] || order[r0] == r0) continue;
    CUDA_TRY(cudaMemcpyAsync(e->d_persite, row(r0), bytes, cudaMemcpyDeviceToDevice, e->stream));
    unsigned r = r0;
    while (order[r] != r0) {
      seen[r] = 1;
      CUDA_TRY(cudaMemcpyAsync(row(r), row(order[r]), bytes, cudaMemcpyDeviceToDevice, e->stream));
      r = order[r];
    }
    seen[r] = 1;
    CUDA_TRY(cudaMemcpyAsync(row(r), e->d_persite, bytes, cudaMemcpyDeviceToDevice, e->stream));
  }
  CUDA_TRY(cudaStreamSynchronize(e->stream));
  return RDK_SUCCESS;
}

static int rell_entry(rdk_partition_t *const *parts, unsigned int n, const unsigned int *global_index,
                      unsigned int rows, unsigned long long replicates, unsigned long long seed, rdk_rell_out_t *out,
                      rdk_rell_ms_out_t *ms) {
  if (n == 0 || rows == 0) return fail(RDK_ERROR_PARAM, "rdk_rell_support: no partitions or no rows");
  if (replicates == 0 || replicates > kRellMaxReplicates)
    return fail(RDK_ERROR_PARAM, "rdk_rell_support: replicates must be in [1, 2^20]");
  std::vector<RellPartition> rp(n);
  RellShard                  shard;
  const int                  device = eng(parts[0])->device;
  for (unsigned i = 0; i < n; ++i) {
    Engine *e = eng(parts[i]);
    if (e->device != device) return fail(RDK_ERROR_PARAM, "rdk_rell_support: partitions on different devices");
    if (e->comm) {
      if (n != 1) return fail(RDK_ERROR_PARAM, "rdk_rell_support: a site shard must be the only partition");
      shard.comm = e->comm;
      shard.nranks = e->nranks;
      shard.rank = e->rank;
      shard.site_offset = e->site_offset;
      shard.allreduce = g_nccl.AllReduce;
    } else if (e->global_sites && (e->site_offset != 0 || e->S != e->global_sites)) {
      return fail(RDK_ERROR_PARAM, "rdk_rell_support: a site shard needs a communicator (rdk_partition_attach_comm)");
    }
    if (e->rows_cap < rows) return fail(RDK_ERROR_PARAM, "rdk_rell_support: partition %u holds %u rows, %u asked",
                                        i, e->rows_cap, rows);
    std::lock_guard<std::mutex> lk(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    if (!flush(parts[i])) return RDK_FAILURE;
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    rp[i].rows = e->d_rows;
    rp[i].weights = parts[i]->pattern_weights;
    rp[i].patterns = e->S;
    rp[i].global_index = global_index ? global_index[i] : i;
  }
  CUDA_TRY(cudaSetDevice(device));
  char msg[256];
  if (!rell_support(rp.data(), n, rows, replicates, seed, shard, out, ms, msg, sizeof(msg)))
    return fail(RDK_ERROR_CUDA, "%s", msg);
  return RDK_SUCCESS;
}

extern "C" int rdk_rell_support(rdk_partition_t *const *parts, unsigned int n, const unsigned int *global_index,
                                unsigned int rows, unsigned long long replicates, unsigned long long seed,
                                rdk_rell_out_t *out) {
  return rell_entry(parts, n, global_index, rows, replicates, seed, out, nullptr);
}

extern "C" int rdk_rell_support_ms(rdk_partition_t *const *parts, unsigned int n, const unsigned int *global_index,
                                   unsigned int rows, unsigned long long replicates, unsigned long long seed,
                                   rdk_rell_out_t *out, rdk_rell_ms_out_t *ms) {
  if (!ms || !ms->scales || !ms->scale_count || !ms->elw_fixed)
    return fail(RDK_ERROR_PARAM, "rdk_rell_support_ms: null scales or output arrays");
  if (ms->n_scales < 2 || ms->n_scales > 32)
    return fail(RDK_ERROR_PARAM, "rdk_rell_support_ms: %u scales, 2 to 32 are needed", ms->n_scales);
  for (unsigned k = 0; k < ms->n_scales; ++k) {
    if (ms->scales[k] < 100 || ms->scales[k] > 10000)
      return fail(RDK_ERROR_PARAM, "rdk_rell_support_ms: scale %u is outside [100, 10000] thousandths", ms->scales[k]);
    if (k && ms->scales[k] <= ms->scales[k - 1])
      return fail(RDK_ERROR_PARAM, "rdk_rell_support_ms: scales must be strictly ascending");
  }
  return rell_entry(parts, n, global_index, rows, replicates, seed, out, ms);
}

// ---------------------------------------------------------------------------
// fused extensions
// ---------------------------------------------------------------------------
extern "C" int rdk_root_loglikelihood_multi(rdk_partition_t *p, const rdk_operation_t *root_op,
                                            const unsigned int *params_indices,
                                            const unsigned int *freqs_indices,
                                            const double *branch_lengths, unsigned int count,
                                            double *out_lnl) {
  (void)params_indices;
  (void)freqs_indices;
  Engine *e = eng(p);
  if (count == 0) return RDK_SUCCESS;
  for (unsigned i = 0; i < 2 * count; ++i)
    if (!(branch_lengths[i] >= 0.0) || !std::isfinite(branch_lengths[i]))
      return fail(RDK_ERROR_PARAM, "branch length must be finite and non-negative");
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  if (!flush(p)) return RDK_FAILURE;
  if (e->pm_free.size() < 2 * (size_t)count)
    return fail(RDK_ERROR_PARAM, "too many candidates in one call (max %zu)", e->pm_free.size() / 2);
  ROp base;
  if (!make_rop(p, *root_op, 0, &base)) return RDK_FAILURE;
  std::vector<unsigned> used;
  for (unsigned b = 0; b < count; ++b) {
    unsigned s1 = e->pm_free.back();
    e->pm_free.pop_back();
    unsigned s2 = e->pm_free.back();
    e->pm_free.pop_back();
    used.push_back(s1);
    used.push_back(s2);
    PmatEntry e1{s1, 0, branch_lengths[2 * b]}, e2{s2, 0, branch_lengths[2 * b + 1]};
    e->pend_pm.push_back(e1);
    e->pend_pm.push_back(e2);
    ROp r = base;
    r.flags = rEval;  // no rWrite: partition state is left untouched
    r.pm1 = s1;
    r.pm2 = s2;
    r.slot = b;
    e->pend_bytes += op_bytes(e, r);
    e->pend_prog.push_back(r);
    e->pend_evals++;
  }
  ProgramOutputs out;
  out.slots = count;
  const int ok = run_evals(p, out, out_lnl);
  for (unsigned s : used) e->pm_free.push_back(s);
  return ok;
}

extern "C" int rdk_sweep_root_placements(rdk_partition_t *p, unsigned int placements,
                                         const unsigned int *params_indices,
                                         const unsigned int *freqs_indices,
                                         const unsigned int *pm_offsets,
                                         const unsigned int *matrix_indices,
                                         const double *branch_lengths,
                                         const unsigned int *op_offsets,
                                         const rdk_operation_t *operations,
                                         unsigned int root_clv_index, int root_scaler_index,
                                         double *out_lnl) {
  return rdk_sweep_root_placements_ex(p, placements, params_indices, freqs_indices, pm_offsets, matrix_indices,
                                      branch_lengths, op_offsets, operations, root_clv_index,
                                      root_scaler_index, 0u, out_lnl);
}

extern "C" int rdk_sweep_root_placements_ex(rdk_partition_t *p, unsigned int placements,
                                            const unsigned int *params_indices,
                                            const unsigned int *freqs_indices,
                                            const unsigned int *pm_offsets,
                                            const unsigned int *matrix_indices,
                                            const double *branch_lengths,
                                            const unsigned int *op_offsets,
                                            const rdk_operation_t *operations,
                                            unsigned int root_clv_index, int root_scaler_index,
                                            unsigned int flags, double *out_lnl) {
  const unsigned int one[2] = {0u, placements};
  return rdk_sweep_root_placements_chunks(p, placements, params_indices, freqs_indices, pm_offsets,
                                          matrix_indices, branch_lengths, op_offsets, operations,
                                          root_clv_index, root_scaler_index, flags, 1u, one, out_lnl);
}

extern "C" unsigned int rdk_sweep_chunk_hint(unsigned int sites, unsigned int rate_cats) {
  if (const char *env = getenv("RDK_SWEEP_CHUNKS")) {  // kernel experiments
    int v = atoi(env);
    if (v >= 1) return (unsigned)std::min(v, kMaxChunks);
  }
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const unsigned n_witer = (unsigned)(((unsigned long long)sites * rate_cats + 31) / 32);
  if (n_witer == 0) return 1;
  // the cost model of plan_launch: a sweep cut into C chunks walks 1/C of the placements (plus the
  // re-derivation of the directed CLVs on the path to a chunk's first placement, ~ the tree depth)
  // per CTA, on 1/C of the device
  unsigned best_c = 1;
  double   best = 1e300;
  for (unsigned c = 1; c <= (unsigned)kMaxChunks; ++c) {
    Engine probe;
    probe.sm_count = sms;
    LaunchSeg seg[2];
    const int n_seg = plan_segments(&probe, n_witer, c, 1 << 20, seg);
    double    cost = seg[0].pl.cost + (n_seg > 1 ? seg[1].pl.cost : 0.0);
    cost *= 1.0 / c + 0.02;
    if (cost < best * 0.9) {  // a chunk more must pay for itself
      best = cost;
      best_c = c;
    }
  }
  return best_c;
}

extern "C" int rdk_sweep_root_placements_chunks(rdk_partition_t *p, unsigned int placements,
                                                const unsigned int *params_indices,
                                                const unsigned int *freqs_indices,
                                                const unsigned int *pm_offsets,
                                                const unsigned int *matrix_indices,
                                                const double *branch_lengths,
                                                const unsigned int *op_offsets,
                                                const rdk_operation_t *operations,
                                                unsigned int root_clv_index, int root_scaler_index,
                                                unsigned int flags, unsigned int n_chunks,
                                                const unsigned int *chunk_offsets, double *out_lnl) {
  (void)params_indices;
  (void)freqs_indices;
  Engine *e = eng(p);
  if (placements == 0) return RDK_SUCCESS;
  if (root_clv_index < e->tips || root_clv_index >= e->tips + e->clv_buffers)
    return fail(RDK_ERROR_PARAM, "root clv index out of range");
  for (unsigned i = 0; i < pm_offsets[placements]; ++i) {
    if (matrix_indices[i] >= e->prob_matrices) return fail(RDK_ERROR_PARAM, "matrix index out of range");
    if (!(branch_lengths[i] >= 0.0) || !std::isfinite(branch_lengths[i]))
      return fail(RDK_ERROR_PARAM, "branch length must be finite and non-negative");
  }
  if ((flags & RDK_SWEEP_ROWS) && e->rows_cap < placements)
    return fail(RDK_ERROR_PARAM, "RDK_SWEEP_ROWS: %u placements, %u site rows reserved (rdk_partition_set_site_lnl_rows)",
                placements, e->rows_cap);
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  if (!flush(p)) return RDK_FAILURE;
  if (!ensure_clv(e, root_clv_index - e->tips)) return RDK_FAILURE;
  const int rs = root_scaler_index == RDK_SCALE_BUFFER_NONE ? -1 : root_scaler_index;
  if (!ensure_scaler(e, rs)) return RDK_FAILURE;
  // batches bounded by the spare P-matrix slots and the partial-sum buffer.  With a communicator
  // attached the ranks' values are added slot by slot, so every rank must cut the sweep at the
  // same placements: the bound is derived from the LARGEST shard of the layout (agreed when the
  // communicator was attached), never from the local site count.
  const unsigned long long s_ref = e->comm ? e->max_shard_sites : e->S;
  const size_t             ref_stride = (size_t)std::max<unsigned long long>(1, (s_ref * e->K + 31) / 32);
  unsigned max_slots = (unsigned)std::max<size_t>(1, std::min<size_t>(4096, (size_t(256) << 20) / (ref_stride * 8)));
  if (const char *env = getenv("RDK_SWEEP_MAX_SLOTS")) {  // tests: force several batches on a small case
    const int v = atoi(env);
    if (v >= 1) max_slots = std::min(max_slots, (unsigned)v);
  }
  // the chunks run side by side only when nothing they share is written (the root CLV is:
  // RDK_SWEEP_KEEP_ROOT must be set) and the whole sweep is one launch; otherwise they run
  // in order, which the contract always allows
  bool concurrent = n_chunks > 1 && n_chunks <= (unsigned)kMaxChunks && (flags & RDK_SWEEP_KEEP_ROOT) &&
                    placements <= max_slots && pm_offsets[placements] <= e->pm_free.size();
  if (concurrent) {
    if (chunk_offsets[0] != 0 || chunk_offsets[n_chunks] != placements)
      return fail(RDK_ERROR_PARAM, "chunk_offsets must run from 0 to the number of placements");
    for (unsigned c = 0; c < n_chunks; ++c)
      if (chunk_offsets[c] >= chunk_offsets[c + 1]) concurrent = false;  // an empty chunk: run in order
    // every placement must end in the root operation that is evaluated in registers
    for (unsigned q = 0; q < placements && concurrent; ++q) {
      if (op_offsets[q + 1] == op_offsets[q]) {
        concurrent = false;
        break;
      }
      const rdk_operation_t &last = operations[op_offsets[q + 1] - 1];
      if (last.parent_clv_index != root_clv_index || last.parent_scaler_index != root_scaler_index)
        concurrent = false;
    }
  }
  // ---- batches: cut where the eval slots or the spare P-matrix slots run out -----------------
  std::vector<unsigned> cuts{0};  // batch k = placements [cuts[k], cuts[k+1])
  {
    const size_t budget0 = e->pm_free.size();  // restored by every flush (retired slots return)
    unsigned     q = 0;
    while (q < placements) {
      size_t   budget = budget0;
      unsigned b = 0;
      while (q + b < placements && b < max_slots) {
        const size_t need = pm_offsets[q + b + 1] - pm_offsets[q + b];
        if (need > budget) break;
        budget -= need;
        ++b;
      }
      if (b == 0) return fail(RDK_ERROR_PARAM, "a placement needs more P-matrices than the pool holds");
      q += b;
      cuts.push_back(q);
    }
  }
  // RDK_SWEEP_DISCARD with several batches: a buffer written by batch k is scratch FOR THAT BATCH
  // unless a later batch reads it before writing it (backward pass over the whole sweep)
  const size_t                   n_batches = cuts.size() - 1;
  std::vector<std::vector<char>> scratch_clv(n_batches), scratch_sc(n_batches);
  if (flags & RDK_SWEEP_DISCARD) {
    std::vector<char> need_clv(e->tips + e->clv_buffers, 0), need_sc(e->scale_buffers, 0);
    for (size_t k = n_batches; k-- > 0;) {
      scratch_clv[k].resize(need_clv.size());
      scratch_sc[k].resize(need_sc.size());
      for (size_t x = 0; x < need_clv.size(); ++x) scratch_clv[k][x] = !need_clv[x];
      for (size_t x = 0; x < need_sc.size(); ++x) scratch_sc[k][x] = !need_sc[x];
      for (unsigned i = op_offsets[cuts[k + 1]]; i-- > op_offsets[cuts[k]];) {
        const rdk_operation_t &o = operations[i];
        if (o.parent_clv_index < need_clv.size()) need_clv[o.parent_clv_index] = 0;
        if (o.parent_scaler_index >= 0 && (size_t)o.parent_scaler_index < need_sc.size()) need_sc[o.parent_scaler_index] = 0;
        if (o.child1_clv_index < need_clv.size()) need_clv[o.child1_clv_index] = 1;
        if (o.child2_clv_index < need_clv.size()) need_clv[o.child2_clv_index] = 1;
        if (o.child1_scaler_index >= 0 && (size_t)o.child1_scaler_index < need_sc.size()) need_sc[o.child1_scaler_index] = 1;
        if (o.child2_scaler_index >= 0 && (size_t)o.child2_scaler_index < need_sc.size()) need_sc[o.child2_scaler_index] = 1;
      }
    }
  }
  // ---- batch k: one program whose eval slot s is placement cuts[k] + s ------------------------
  auto record_batch = [&](size_t k, ProgramOutputs &out) -> int {
    HostTimer record_timer(&e->stats.host_record_ns);
    size_t    pm_budget = e->pm_free.size();
    unsigned  next_chunk = 0;
    for (unsigned q = cuts[k]; q < cuts[k + 1]; ++q) {
      const size_t need = pm_offsets[q + 1] - pm_offsets[q];
      if (need > pm_budget) return fail(RDK_ERROR_MEM, "P-matrix pool smaller than planned");
      pm_budget -= need;
      if (concurrent && next_chunk < n_chunks && q == chunk_offsets[next_chunk]) {
        out.chunk_off.push_back((unsigned)e->pend_prog.size());
        ++next_chunk;
      }
      for (unsigned i = pm_offsets[q]; i < pm_offsets[q + 1]; ++i)
        if (!record_pmatrix(p, matrix_indices[i], branch_lengths[i])) return RDK_FAILURE;
      if (!record_ops(p, operations + op_offsets[q], op_offsets[q + 1] - op_offsets[q])) return RDK_FAILURE;
      record_root_eval(e, root_clv_index, rs, q - cuts[k], flags & RDK_SWEEP_KEEP_ROOT);
    }
    if (concurrent) out.chunk_off.push_back((unsigned)e->pend_prog.size());
    out.slots = cuts[k + 1] - cuts[k];
    if (flags & RDK_SWEEP_DISCARD) {
      out.scratch_clv = std::move(scratch_clv[k]);
      out.scratch_sc = std::move(scratch_sc[k]);
    }
    if (flags & RDK_SWEEP_ROWS) {  // eval slot s stores into the row of its placement
      out.persite = e->d_rows + (size_t)cuts[k] * e->S;
      out.unweighted = true;
      out.row_stride = e->S;
    }
    return RDK_SUCCESS;
  };
  for (size_t k = 0; k < n_batches; ++k) {
    ProgramOutputs out;
    if (!record_batch(k, out)) {
      clear_pending_ops(e);  // no evaluation outlives the call
      return RDK_FAILURE;
    }
    if (!run_evals(p, out, out_lnl + cuts[k])) return RDK_FAILURE;
  }
  return RDK_SUCCESS;
}

// ---------------------------------------------------------------------------
// empirical frequencies (device histogram, exact integers)
// ---------------------------------------------------------------------------
extern "C" double *rdk_msa_empirical_frequencies(rdk_partition_t *p) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  if (cudaSetDevice(e->device) != cudaSuccess) return nullptr;
  if (!flush(p)) return nullptr;
  unsigned long long hist[16];
  cudaMemsetAsync(e->d_hist, 0, sizeof(hist), e->stream);
  if (e->S > 0 && e->tips > 0) {
    size_t total = (size_t)e->tips * e->S;
    int    grid = (int)std::min<size_t>((total + 255) / 256, (size_t)e->sm_count * 8);
    tip_hist_kernel<<<grid, 256, 0, e->stream>>>(e->d_tips, e->tip_stride, e->tips, e->S, e->d_weights,
                                                 e->d_hist);
    e->stats.kernel_launches++;
  }
  if (e->comm) {
    int rc = g_nccl.AllReduce(e->d_hist, e->d_hist, 16, kNcclUint64, kNcclSum, e->comm, e->stream);
    if (rc != 0) {
      fail(RDK_ERROR_COMM, "ncclAllReduce failed");
      return nullptr;
    }
  }
  if (cudaMemcpyAsync(hist, e->d_hist, sizeof(hist), cudaMemcpyDeviceToHost, e->stream) != cudaSuccess ||
      cudaStreamSynchronize(e->stream) != cudaSuccess) {
    fail(RDK_ERROR_CUDA, "histogram read-back failed");
    return nullptr;
  }
  // f_j = sum over masks m containing j of H[m] / popcount(m), ascending m;
  // normalised by (total pattern weight) * tips = sum of all H[m]
  double *f = (double *)calloc(4, sizeof(double));
  double  total = 0.0;
  for (int m = 1; m < 16; ++m) total += (double)hist[m];
  for (int j = 0; j < 4; ++j) {
    double s = 0.0;
    for (int m = 1; m < 16; ++m)
      if (m & (1 << j)) s += (double)hist[m] / (double)__builtin_popcount(m);
    f[j] = s / total;
  }
  return f;
}

// ---------------------------------------------------------------------------
// sharding
// ---------------------------------------------------------------------------
extern "C" int rdk_partition_set_shard(rdk_partition_t *p, unsigned long long site_offset,
                                       unsigned long long global_sites) {
  Engine *e = eng(p);
  if (site_offset % RDK_SHARD_ALIGN != 0)
    return fail(RDK_ERROR_PARAM, "site_offset must be a multiple of %u", RDK_SHARD_ALIGN);
  if (site_offset + e->S > global_sites)
    return fail(RDK_ERROR_PARAM, "shard [%llu, %llu) exceeds global_sites %llu", site_offset,
                site_offset + e->S, global_sites);
  if ((RDK_SHARD_ALIGN * e->K) % 32 != 0) return fail(RDK_ERROR_PARAM, "unsupported rate_cats for sharding");
  std::lock_guard<std::mutex> lk(e->mu);
  e->site_offset = site_offset;
  e->global_sites = global_sites;
  return RDK_SUCCESS;
}

extern "C" int rdk_comm_unique_id(void *id_out) {
  if (!load_nccl()) return RDK_FAILURE;
  Id128 id;
  memset(&id, 0, sizeof(id));
  int rc = g_nccl.GetUniqueId(&id);
  if (rc != 0) return fail(RDK_ERROR_COMM, "ncclGetUniqueId failed (%d)", rc);
  memcpy(id_out, &id, sizeof(id));
  return RDK_SUCCESS;
}

extern "C" int rdk_partition_attach_comm(rdk_partition_t *p, int nranks, int rank, const void *id) {
  Engine *e = eng(p);
  if (!load_nccl()) return RDK_FAILURE;
  if (e->global_sites == 0)
    return fail(RDK_ERROR_PARAM, "call rdk_partition_set_shard before attaching a communicator");
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  Id128 uid;
  memcpy(&uid, id, sizeof(uid));
  void *comm = nullptr;
  int   rc = g_nccl.CommInitRank(&comm, nranks, uid, rank);
  if (rc != 0)
    return fail(RDK_ERROR_COMM, "ncclCommInitRank failed: %s",
                g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
  e->comm = comm;
  e->nranks = nranks;
  e->rank = rank;
  // agree on the largest shard of the layout: everything that sizes a batch of a collective
  // evaluation is derived from it, so that all ranks cut their work at the same places
  unsigned long long mine = e->S, agreed = 0;
  CUDA_TRY(cudaMemcpyAsync(e->d_hist, &mine, sizeof(mine), cudaMemcpyHostToDevice, e->stream));
  rc = g_nccl.AllReduce(e->d_hist, e->d_hist, 1, kNcclUint64, kNcclMax, e->comm, e->stream);
  if (rc != 0)
    return fail(RDK_ERROR_COMM, "ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
  CUDA_TRY(cudaMemcpyAsync(&agreed, e->d_hist, sizeof(agreed), cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(cudaStreamSynchronize(e->stream));
  e->max_shard_sites = agreed;
  return RDK_SUCCESS;
}

// ---------------------------------------------------------------------------
// plumbing / introspection
// ---------------------------------------------------------------------------
extern "C" int rdk_partition_flush(rdk_partition_t *p) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  return flush(p);
}

extern "C" int rdk_partition_sync(rdk_partition_t *p) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  if (!flush(p)) return RDK_FAILURE;
  CUDA_TRY(cudaStreamSynchronize(e->stream));
  return RDK_SUCCESS;
}

extern "C" int rdk_partition_set_stream(rdk_partition_t *p, void *cuda_stream) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  if (!flush(p)) return RDK_FAILURE;
  CUDA_TRY(cudaStreamSynchronize(e->stream));
  if (e->own_stream && e->stream) cudaStreamDestroy(e->stream);
  e->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  e->own_stream = false;
  return RDK_SUCCESS;
}

extern "C" void *rdk_partition_stream(rdk_partition_t *p) { return eng(p)->stream; }

extern "C" int rdk_get_clv(rdk_partition_t *p, unsigned int clv_index, double *out) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  if (clv_index >= e->tips + e->clv_buffers) return fail(RDK_ERROR_PARAM, "clv index out of range");
  if (!flush(p)) return RDK_FAILURE;
  if (e->lazy.active && clv_index < e->lazy.stale_clv.size() && e->lazy.stale_clv[clv_index] && !materialize_lazy(p))
    return RDK_FAILURE;
  size_t bytes = (size_t)e->S * e->Kreal * 4 * sizeof(double);  // corax layout [site][cat][state]
  if (clv_index < e->tips) {
    double *tmp = nullptr;
    CUDA_TRY(cudaMalloc((void **)&tmp, bytes ? bytes : 32));
    size_t n = (size_t)e->S * e->Kreal;
    if (n) {
      tip_expand_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(
          e->d_tips + (size_t)clv_index * e->tip_stride, e->S, (int)e->Kreal, tmp);
      e->stats.kernel_launches++;
    }
    cudaError_t err = cudaMemcpyAsync(out, tmp, bytes, cudaMemcpyDeviceToHost, e->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(e->stream);
    cudaFree(tmp);
    CUDA_TRY(err);
  } else {
    if (!ensure_clv(e, clv_index - e->tips)) return RDK_FAILURE;
    if (e->K == e->Kreal) {
      CUDA_TRY(cudaMemcpyAsync(out, e->clv_ptr[clv_index - e->tips], bytes, cudaMemcpyDeviceToHost, e->stream));
      CUDA_TRY(cudaStreamSynchronize(e->stream));
    } else {
      // drop the padding categories: a strided copy of Kreal * 32 bytes out of every K * 32
      CUDA_TRY(cudaMemcpy2DAsync(out, (size_t)e->Kreal * 32, e->clv_ptr[clv_index - e->tips], (size_t)e->K * 32,
                                 (size_t)e->Kreal * 32, e->S, cudaMemcpyDeviceToHost, e->stream));
      CUDA_TRY(cudaStreamSynchronize(e->stream));
    }
  }
  e->stats.d2h_bytes += bytes;
  return RDK_SUCCESS;
}

extern "C" int rdk_get_scale_buffer(rdk_partition_t *p, int scaler_index, unsigned int *out) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  if (scaler_index < 0 || (unsigned)scaler_index >= e->scale_buffers)
    return fail(RDK_ERROR_PARAM, "scaler index out of range");
  if (!flush(p)) return RDK_FAILURE;
  if (e->lazy.active && (size_t)scaler_index < e->lazy.stale_sc.size() && e->lazy.stale_sc[scaler_index] &&
      !materialize_lazy(p))
    return RDK_FAILURE;
  if (!ensure_scaler(e, scaler_index)) return RDK_FAILURE;
  CUDA_TRY(cudaMemcpyAsync(out, e->sc_ptr[scaler_index], sizeof(unsigned) * e->S,
                           cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(cudaStreamSynchronize(e->stream));
  return RDK_SUCCESS;
}

extern "C" int rdk_get_pmatrix(rdk_partition_t *p, unsigned int matrix_index, double *out) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  if (matrix_index >= e->prob_matrices) return fail(RDK_ERROR_PARAM, "matrix index out of range");
  if (!flush(p)) return RDK_FAILURE;
  std::vector<double> tmp((size_t)kPTabDoubles * e->K);
  CUDA_TRY(cudaMemcpyAsync(tmp.data(), e->d_pool + (size_t)e->pm_map[matrix_index] * e->K * kSlotDoubles,
                           sizeof(double) * kPTabDoubles * e->K, cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(cudaStreamSynchronize(e->stream));
  // device layout [cat][18 (16 used)] -> corax layout [cat][i][j]
  for (unsigned k = 0; k < e->Kreal; ++k)
    for (int ij = 0; ij < 16; ++ij) out[(size_t)k * 16 + ij] = tmp[(size_t)k * kPTabDoubles + ij];
  return RDK_SUCCESS;
}

extern "C" void rdk_partition_stats(rdk_partition_t *p, rdk_stats_t *out) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  cudaSetDevice(e->device);
  harvest_events(e);
  *out = e->stats;
}

extern "C" void rdk_partition_reset_stats(rdk_partition_t *p) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  unsigned long long dev = e->stats.device_bytes;
  cudaSetDevice(e->device);
  harvest_events(e);
  memset(&e->stats, 0, sizeof(e->stats));
  e->stats.device_bytes = dev;
}

extern "C" int rdk_partition_set_timing(rdk_partition_t *p, int enabled) {
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  harvest_events(e);
  e->timing = enabled != 0;
  return RDK_SUCCESS;
}

extern "C" int rdk_partition_set_lazy(rdk_partition_t *p, int enabled) {
  if (!p) return fail(RDK_ERROR_PARAM, "null partition");
  Engine *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  if (!flush(p)) return RDK_FAILURE;
  if (!enabled && !materialize_lazy(p)) return RDK_FAILURE;
  e->lazy_enabled = enabled != 0;
  return RDK_SUCCESS;
}

extern "C" int rdk_partition_set_subtree_groups(rdk_partition_t *p, int groups) {
  if (groups < 0 || groups > kMaxChunks) return fail(RDK_ERROR_PARAM, "groups must be 0 .. %d", kMaxChunks);
  Engine                     *e = eng(p);
  std::lock_guard<std::mutex> lk(e->mu);
  e->subtree_groups = groups;
  e->kept_programs.clear();  // the decision is part of a kept lowering
  return RDK_SUCCESS;
}

// introspection (pure host code, no CUDA call): what choose_subtree_groups decides for a program
// on a shard of `sites` x `rate_cats` on a device of `sm_count` SMs
extern "C" int rdk_debug_choose_subtree_groups(unsigned int tips, unsigned int n_ops, const int *ops,
                                               unsigned int sites, unsigned int rate_cats, int sm_count,
                                               unsigned int *longest, unsigned int *n_join) {
  Engine e;
  e.sm_count = sm_count > 0 ? sm_count : 148;
  e.tips = tips;
  e.pend_prog.resize(n_ops);
  for (unsigned i = 0; i < n_ops; ++i) {
    const int *f = ops + 10 * (size_t)i;
    ROp       &r = e.pend_prog[i];
    memset(&r, 0, sizeof(r));
    r.parent = (unsigned)f[0];
    r.pscale = f[1];
    r.c1 = (unsigned)f[2];
    r.c2 = (unsigned)f[3];
    r.c1scale = f[4];
    r.c2scale = f[5];
    r.pm1 = (unsigned)f[6];
    r.pm2 = (unsigned)f[7];
    r.flags = (unsigned)f[8];
    r.slot = (unsigned)f[9];
    r.id = i;
  }
  unsigned K = 1;
  while (K < rate_cats) K <<= 1;
  const unsigned        n_witer = (unsigned)(((unsigned long long)sites * K + 31) / 32);
  std::vector<ROp>      grouped, join;
  std::vector<unsigned> goff;
  if (!choose_subtree_groups(&e, n_witer, grouped, goff, join)) return 0;
  unsigned l = 0;
  for (size_t g = 0; g + 1 < goff.size(); ++g) l = std::max(l, goff[g + 1] - goff[g]);
  if (longest) *longest = l;
  if (n_join) *n_join = (unsigned)join.size();
  return (int)goff.size() - 1;
}

extern "C" int rdk_partition_set_tail_mode(rdk_partition_t *p, int mode) {
  // kept for ABI compatibility: the program kernel has a single tail rule now (slots without an
  // iteration of their own recompute the warp's last iteration)
  if (!p) return fail(RDK_ERROR_PARAM, "null partition");
  if (mode < 0 || mode > 2) return fail(RDK_ERROR_PARAM, "tail mode must be 0, 1 or 2");
  return RDK_SUCCESS;
}

extern "C" int rdk_partition_set_launch_config(rdk_partition_t *p, int ctas_per_sm,
                                               int threads_per_cta, int elems_per_thread) {
  Engine *e = eng(p);
  if (threads_per_cta != 0 && (threads_per_cta < 64 || threads_per_cta > 512 || threads_per_cta % 32))
    return fail(RDK_ERROR_PARAM, "threads_per_cta must be a multiple of 32 in [64,512] (one warp is the table producer)");
  if (elems_per_thread < 0 || elems_per_thread > 4)
    return fail(RDK_ERROR_PARAM, "elems_per_thread must be in [0,4]");
  if (ctas_per_sm < 0 || ctas_per_sm > 32) return fail(RDK_ERROR_PARAM, "ctas_per_sm out of range");
  std::lock_guard<std::mutex> lk(e->mu);
  e->ctas_per_sm = ctas_per_sm;
  e->threads = threads_per_cta;
  e->elems = elems_per_thread;
  e->kept_programs.clear();  // the subtree-group decision of a kept lowering depends on the launch shape
  return RDK_SUCCESS;
}
