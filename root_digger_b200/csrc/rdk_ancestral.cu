// rdk_ancestral.cu -- marginal ancestral states: the pre-order pass over outside vectors and the
// posterior of every internal node (rdk_marginal_ancestral_states, include/rdk.h; DESIGN.md
// section 11).
//
// One thread per (pattern, category), the K categories of a pattern in adjacent lanes of one warp
// (K divides 32), as in the program kernel.  A thread walks the whole tree for its element: the pass
// has no dependency between patterns, so ONE launch covers every node.  Per node it reads the two
// child CLVs (a tip through its branch's tip table), recomputes d_v = h1 o h2 with the post-order
// operation's own rescaling test, and reads o_v from a scratch buffer; it writes o_c1 and o_c2 for
// the inner children.  The visit order (ancestral_schedule: smaller subtree first) bounds the live
// outside vectors by ceil(log2 count) + 2.  Cross-category sums and the per-pattern rescaling tests
// are warp shuffles and ballots over the K lanes of the pattern.
#define RDK_PROGRAM_KERNEL_ONLY 1
#include "rdk_kernels.cuh"
#include "rdk_ancestral.cuh"

#include <algorithm>
#include <cstdio>
#include <cstring>

namespace rdk {
namespace {

constexpr unsigned           kAncMaxThreads = 256;
constexpr unsigned long long kAncTileBytes = 512ull << 20;  // outputs + scratch of one tile

struct AncArgs {
  const AncNode  *nodes;
  unsigned        n_nodes;
  unsigned        site0, S;     // this tile: patterns [site0, site0 + S) of the partition
  double          pi[4];
  double          w[kMaxCats];
  double         *scratch;      // [slot][S*K][4], tile-local
  unsigned       *tau;          // [slot][S]
  unsigned char  *map_state;    // [count][S]
  double         *map_prob;     // [count][S]
  double         *posterior;    // [n_full][S][4]
  double         *log_norm;     // [count][S] or null
};

__device__ __forceinline__ bool all_small(const double (&x)[4]) {
  return x[0] < RDK_SCALE_THRESHOLD && x[1] < RDK_SCALE_THRESHOLD && x[2] < RDK_SCALE_THRESHOLD &&
         x[3] < RDK_SCALE_THRESHOLD;
}

// h[j] = sum_l P[j][l] x[l], an FMA chain with l ascending (the CLV update's mat-vec); a tip child
// reads its branch's tip table, which holds the same values
template <int K>
__device__ __forceinline__ void half_product(const double *tab, const void *c, int tip, unsigned site, unsigned k,
                                             size_t e, double (&h)[4]) {
  if (tip) {
    const unsigned code = reinterpret_cast<const unsigned char *>(c)[site] & 15u;
    const double  *t = tab + (size_t)K * kPTabDoubles + ((size_t)code * K + k) * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) h[j] = t[j];
    return;
  }
  const double *P = tab + (size_t)k * kPTabDoubles;
  const double4 *xp = reinterpret_cast<const double4 *>(c) + e;
  const double4  x4 = *xp;
  const double   x[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    double acc = dmul(P[j * 4 + 0], x[0]);
    acc = dfma(P[j * 4 + 1], x[1], acc);
    acc = dfma(P[j * 4 + 2], x[2], acc);
    acc = dfma(P[j * 4 + 3], x[3], acc);
    h[j] = acc;
  }
}

// o_c[i] = sum_j (o_v[j] h_sib[j]) P[j][i]: the transposed product, an FMA chain with j ascending
template <int K>
__device__ __forceinline__ void outside_of_child(const double *tab, unsigned k, const double (&o)[4],
                                                 const double (&hs)[4], double (&oc)[4]) {
  const double *P = tab + (size_t)k * kPTabDoubles;
  double        s[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) s[j] = dmul(o[j], hs[j]);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    double acc = dmul(s[0], P[0 * 4 + i]);
    acc = dfma(s[1], P[1 * 4 + i], acc);
    acc = dfma(s[2], P[2 * 4 + i], acc);
    acc = dfma(s[3], P[3 * 4 + i], acc);
    oc[i] = acc;
  }
}

template <int K>
__global__ void __launch_bounds__(kAncMaxThreads) ancestral_kernel(const __grid_constant__ AncArgs a) {
  const unsigned lane = threadIdx.x & 31u;
  const size_t   e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // tile element = site * K + k
  const unsigned k = (unsigned)(e % K);
  const unsigned site = (unsigned)(e / K);                            // in the tile
  const bool     live = site < a.S;
  const unsigned gsite = a.site0 + site;                              // in the partition
  const size_t   ge = (size_t)a.site0 * K + e;
  const unsigned lane0 = lane & ~(unsigned)(K - 1);                    // first lane of this site
  const unsigned gmask = K == 32 ? 0xffffffffu : (((1u << K) - 1u) << lane0);
  const size_t   SK = (size_t)a.S * K;
  // every lane of the warp takes part in the shuffles; lanes past the last site work on zeros
  auto site_small = [&](bool small) {
    const unsigned b = __ballot_sync(0xffffffffu, small);
    return (b & gmask) == gmask;
  };

  for (unsigned n = 0; n < a.n_nodes; ++n) {
    const AncNode nd = a.nodes[n];
    double        o[4], h1[4], h2[4];
    unsigned      tau = 0;
    if (nd.in < 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) o[i] = a.pi[i];
    } else if (live) {
      const double4 v = reinterpret_cast<const double4 *>(a.scratch + (size_t)nd.in * SK * 4)[e];
      o[0] = v.x, o[1] = v.y, o[2] = v.z, o[3] = v.w;
      tau = a.tau[(size_t)nd.in * a.S + site];
    } else {
      o[0] = o[1] = o[2] = o[3] = 0.0;
    }
    unsigned s1 = 0, s2 = 0;
    if (live) {
      half_product<K>(nd.tab1, nd.c1, nd.tip1, gsite, k, ge, h1);
      half_product<K>(nd.tab2, nd.c2, nd.tip2, gsite, k, ge, h2);
      if (nd.sc1) s1 = nd.sc1[gsite];
      if (nd.sc2) s2 = nd.sc2[gsite];
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) h1[i] = h2[i] = 0.0;
    }

    // d_v, rescaled as the post-order operation rescaled it
    double d[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) d[i] = dmul(h1[i], h2[i]);
    unsigned sigma = 0;
    if (nd.scaled) {
      sigma = s1 + s2;
      if (site_small(all_small(d))) {
#pragma unroll
        for (int i = 0; i < 4; ++i) d[i] = dmul(d[i], RDK_SCALE_FACTOR);
        sigma += 1;
      }
    }

    // posterior: t[i] = sum_k w_k (o d), an FMA chain over k ascending, gathered from the site's lanes
    double p[4], t[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = dmul(o[i], d[i]);
#pragma unroll
    for (int i = 0; i < 4; ++i) t[i] = dmul(a.w[0], __shfl_sync(0xffffffffu, p[i], lane0));
#pragma unroll
    for (int kk = 1; kk < K; ++kk)
#pragma unroll
      for (int i = 0; i < 4; ++i) t[i] = dfma(a.w[kk], __shfl_sync(0xffffffffu, p[i], lane0 + kk), t[i]);
    if (live && k == 0) {
      const double Z = dadd(dadd(dadd(t[0], t[1]), t[2]), t[3]);
      double       post[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) post[i] = ddiv(t[i], Z);
      unsigned best = 0;
      double   top = post[0];
#pragma unroll
      for (int i = 1; i < 4; ++i)
        if (post[i] > top) best = (unsigned)i, top = post[i];
      const size_t row = (size_t)nd.op * a.S + site;
      a.map_state[row] = (unsigned char)best;
      a.map_prob[row] = top;
      if (a.log_norm) a.log_norm[row] = dadd(rd_log(Z), dmul((double)(sigma + tau), RDK_LOG_SCALE_THRESHOLD));
      if (nd.full >= 0)
        reinterpret_cast<double4 *>(a.posterior)[(size_t)nd.full * a.S + site] =
            make_double4(post[0], post[1], post[2], post[3]);
    }

    // outside vectors of the inner children (o is in registers: a child may take v's buffer)
    double oc1[4], oc2[4];
    if (nd.out1 >= 0) outside_of_child<K>(nd.tab1, k, o, h2, oc1);
    if (nd.out2 >= 0) outside_of_child<K>(nd.tab2, k, o, h1, oc2);
    if (nd.out1 >= 0) {
      unsigned tc = tau + s2;
      if (site_small(all_small(oc1))) {
#pragma unroll
        for (int i = 0; i < 4; ++i) oc1[i] = dmul(oc1[i], RDK_SCALE_FACTOR);
        tc += 1;
      }
      if (live) {
        reinterpret_cast<double4 *>(a.scratch + (size_t)nd.out1 * SK * 4)[e] = make_double4(oc1[0], oc1[1], oc1[2], oc1[3]);
        if (k == 0) a.tau[(size_t)nd.out1 * a.S + site] = tc;
      }
    }
    if (nd.out2 >= 0) {
      unsigned tc = tau + s1;
      if (site_small(all_small(oc2))) {
#pragma unroll
        for (int i = 0; i < 4; ++i) oc2[i] = dmul(oc2[i], RDK_SCALE_FACTOR);
        tc += 1;
      }
      if (live) {
        reinterpret_cast<double4 *>(a.scratch + (size_t)nd.out2 * SK * 4)[e] = make_double4(oc2[0], oc2[1], oc2[2], oc2[3]);
        if (k == 0) a.tau[(size_t)nd.out2 * a.S + site] = tc;
      }
    }
  }
}

template <int K>
void launch(const AncArgs &a, unsigned grid, unsigned threads, cudaStream_t st) {
  ancestral_kernel<K><<<grid, threads, 0, st>>>(a);
}

struct DeviceBuffers {  // what one call allocates, freed on every return path
  std::vector<void *> ptrs;
  unsigned long long  bytes = 0;
  ~DeviceBuffers() {
    for (void *p : ptrs) cudaFree(p);
  }
  cudaError_t alloc(void **p, size_t n) {
    n = std::max<size_t>(n, 16);
    cudaError_t err = cudaMalloc(p, n);
    if (err == cudaSuccess) {
      ptrs.push_back(*p);
      bytes += n;
    }
    return err;
  }
};

}  // namespace

int ancestral_schedule(const rdk_operation_t *ops, unsigned count, unsigned tips, unsigned clv_count,
                       std::vector<AncNode> &nodes, unsigned &scratch, char *msg, size_t msg_cap) {
  if (count == 0) {
    snprintf(msg, msg_cap, "no operations");
    return 0;
  }
  std::vector<int> op_of(clv_count, -1);  // inner clv index -> the operation that writes it
  std::vector<int> parent_op(count, -1);
  for (unsigned i = 0; i < count; ++i) {
    const rdk_operation_t &op = ops[i];
    const unsigned         c[3] = {op.parent_clv_index, op.child1_clv_index, op.child2_clv_index};
    for (unsigned v : c)
      if (v >= clv_count) {
        snprintf(msg, msg_cap, "operation %u: clv index %u out of range", i, v);
        return 0;
      }
    if (op.parent_clv_index < tips) {
      snprintf(msg, msg_cap, "operation %u writes a tip", i);
      return 0;
    }
    for (int side = 0; side < 2; ++side) {
      const unsigned ch = side ? op.child2_clv_index : op.child1_clv_index;
      if (ch < tips) continue;
      const int w = op_of[ch];
      if (w < 0 || parent_op[w] >= 0) {
        snprintf(msg, msg_cap, "operation %u: child clv %u is not the node of exactly one earlier operation", i, ch);
        return 0;
      }
      parent_op[w] = (int)i;
    }
    if (op_of[op.parent_clv_index] >= 0) {
      snprintf(msg, msg_cap, "operation %u: clv %u is written twice", i, op.parent_clv_index);
      return 0;
    }
    op_of[op.parent_clv_index] = (int)i;
  }
  for (unsigned i = 0; i + 1 < count; ++i)
    if (parent_op[i] < 0) {
      snprintf(msg, msg_cap, "operation %u: its node is no child of a later operation (not one rooted tree)", i);
      return 0;
    }
  // subtree sizes in operations (children come before their parent)
  std::vector<unsigned> size(count, 1);
  for (unsigned i = 0; i < count; ++i)
    if (parent_op[i] >= 0) size[parent_op[i]] += size[i];

  auto child_op = [&](unsigned i, int side) {
    const unsigned ch = side ? ops[i].child2_clv_index : ops[i].child1_clv_index;
    return ch < tips ? -1 : op_of[ch];
  };
  nodes.clear();
  nodes.reserve(count);
  std::vector<int>                  free_slots;
  unsigned                          slots = 0;
  auto                              take = [&]() {
    if (!free_slots.empty()) {
      const int s = free_slots.back();
      free_slots.pop_back();
      return s;
    }
    return (int)slots++;
  };
  std::vector<std::pair<int, int>> stack{{(int)count - 1, -1}};  // (operation, buffer of its o)
  while (!stack.empty()) {
    const auto [v, in] = stack.back();
    stack.pop_back();
    AncNode nd{};
    nd.op = (unsigned)v;
    nd.in = in;
    nd.full = -1;
    const int a = child_op((unsigned)v, 0), b = child_op((unsigned)v, 1);
    nd.out1 = nd.out2 = -1;
    if (a >= 0 && b >= 0) {
      // the smaller subtree is visited next and takes v's buffer; the larger one waits in a new one
      const bool a_first = size[a] <= size[b];
      const int  first_buf = in >= 0 ? in : take();
      const int  later_buf = take();
      nd.out1 = a_first ? first_buf : later_buf;
      nd.out2 = a_first ? later_buf : first_buf;
      stack.push_back({a_first ? b : a, later_buf});
      stack.push_back({a_first ? a : b, first_buf});
    } else if (a >= 0 || b >= 0) {
      const int buf = in >= 0 ? in : take();
      (a >= 0 ? nd.out1 : nd.out2) = buf;
      stack.push_back({a >= 0 ? a : b, buf});
    } else if (in >= 0) {
      free_slots.push_back(in);
    }
    nodes.push_back(nd);
  }
  scratch = slots;
  return 1;
}

int ancestral_pass(const AncPass &pass, const std::vector<AncNode> &nodes, rdk_ancestral_out_t *out, char *msg,
                   size_t msg_cap) {
#define ANC_TRY(expr)                                                         \
  do {                                                                        \
    cudaError_t err_ = (expr);                                                \
    if (err_ != cudaSuccess) {                                                \
      snprintf(msg, msg_cap, "%s: %s", #expr, cudaGetErrorString(err_));      \
      return 0;                                                               \
    }                                                                         \
  } while (0)
  const unsigned K = pass.K, S = pass.S;
  const unsigned threads = out->threads ? out->threads : 256u;
  if (threads % 32u || threads > kAncMaxThreads) {
    snprintf(msg, msg_cap, "threads per block must be a multiple of 32 up to %u, not %u", kAncMaxThreads, threads);
    return 0;
  }
  if (K == 0 || K > 32u || (32u % K) != 0u) {
    snprintf(msg, msg_cap, "%u device categories: not a divisor of 32", K);
    return 0;
  }
  // Patterns are independent: the pass walks the partition in tiles of T patterns so that the outputs
  // and the scratch it holds on the device stay within kAncTileBytes, whatever the alignment's size.
  const unsigned long long per_site = (unsigned long long)pass.count * (out->log_norm ? 17u : 9u) +
                                      32ull * out->n_full +
                                      (unsigned long long)std::max(1u, pass.scratch) * (32ull * K + 4ull);
  unsigned T = out->tile_sites;
  if (T == 0) T = (unsigned)std::max<unsigned long long>(256ull, kAncTileBytes / per_site);
  T = std::max(1u, std::min(T, std::max(1u, S)));
  DeviceBuffers buf;
  AncArgs       a;
  memset(&a, 0, sizeof(a));
  a.n_nodes = (unsigned)nodes.size();
  for (int i = 0; i < 4; ++i) a.pi[i] = pass.pi[i];
  for (unsigned k = 0; k < K; ++k) a.w[k] = pass.w[k];
  const size_t TK = (size_t)T * K;
  ANC_TRY(buf.alloc((void **)&a.nodes, sizeof(AncNode) * nodes.size()));
  ANC_TRY(buf.alloc((void **)&a.scratch, sizeof(double) * 4 * TK * std::max(1u, pass.scratch)));
  ANC_TRY(buf.alloc((void **)&a.tau, sizeof(unsigned) * (size_t)T * std::max(1u, pass.scratch)));
  ANC_TRY(buf.alloc((void **)&a.map_state, (size_t)pass.count * T));
  ANC_TRY(buf.alloc((void **)&a.map_prob, sizeof(double) * pass.count * T));
  ANC_TRY(buf.alloc((void **)&a.posterior, sizeof(double) * 4 * (size_t)out->n_full * T));
  if (out->log_norm) ANC_TRY(buf.alloc((void **)&a.log_norm, sizeof(double) * pass.count * T));
  ANC_TRY(cudaMemcpyAsync((void *)a.nodes, nodes.data(), sizeof(AncNode) * nodes.size(), cudaMemcpyHostToDevice,
                          pass.stream));
  cudaEvent_t ev[2] = {nullptr, nullptr};
  ANC_TRY(cudaEventCreate(&ev[0]));
  if (cudaEventCreate(&ev[1]) != cudaSuccess) {
    cudaEventDestroy(ev[0]);
    snprintf(msg, msg_cap, "cudaEventCreate failed");
    return 0;
  }
  struct Events {
    cudaEvent_t *ev;
    ~Events() {
      cudaEventDestroy(ev[0]);
      cudaEventDestroy(ev[1]);
    }
  } events{ev};
  double ms_total = 0.0;
  for (unsigned s0 = 0; s0 < S; s0 += T) {
    const unsigned tl = std::min(T, S - s0);
    a.site0 = s0;
    a.S = tl;
    const unsigned grid = (unsigned)(((size_t)tl * K + threads - 1) / threads);
    ANC_TRY(cudaEventRecord(ev[0], pass.stream));
    switch (K) {
      case 1: launch<1>(a, grid, threads, pass.stream); break;
      case 2: launch<2>(a, grid, threads, pass.stream); break;
      case 4: launch<4>(a, grid, threads, pass.stream); break;
      case 8: launch<8>(a, grid, threads, pass.stream); break;
      case 16: launch<16>(a, grid, threads, pass.stream); break;
      default: launch<32>(a, grid, threads, pass.stream); break;
    }
    ANC_TRY(cudaGetLastError());
    ANC_TRY(cudaEventRecord(ev[1], pass.stream));
    // the tile's rows into columns [s0, s0 + tl) of the caller's [row][S] arrays
    ANC_TRY(cudaMemcpy2DAsync(out->map_state + s0, S, a.map_state, tl, tl, pass.count, cudaMemcpyDeviceToHost,
                              pass.stream));
    ANC_TRY(cudaMemcpy2DAsync(out->map_prob + s0, sizeof(double) * S, a.map_prob, sizeof(double) * tl,
                              sizeof(double) * tl, pass.count, cudaMemcpyDeviceToHost, pass.stream));
    if (out->n_full)
      ANC_TRY(cudaMemcpy2DAsync(out->posterior + (size_t)4 * s0, 32 * (size_t)S, a.posterior, 32 * (size_t)tl,
                                32 * (size_t)tl, out->n_full, cudaMemcpyDeviceToHost, pass.stream));
    if (out->log_norm)
      ANC_TRY(cudaMemcpy2DAsync(out->log_norm + s0, sizeof(double) * S, a.log_norm, sizeof(double) * tl,
                                sizeof(double) * tl, pass.count, cudaMemcpyDeviceToHost, pass.stream));
    ANC_TRY(cudaStreamSynchronize(pass.stream));  // the next tile reuses the buffers
    float ms = 0.f;
    ANC_TRY(cudaEventElapsedTime(&ms, ev[0], ev[1]));
    ms_total += ms;
  }
  out->ms = ms_total;
  out->device_bytes = buf.bytes;
  out->scratch = pass.scratch;
  out->tile_sites = T;
  return 1;
#undef ANC_TRY
}

}  // namespace rdk
