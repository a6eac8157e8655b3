// rdk_support.cu -- the three kernels of rdk_rell_support (DESIGN.md section 10).
//
//   counts        c[b][p]: Philox4x64-10 draws of the original sites of a partition, mapped to
//                 their pattern by a binary search in the cumulative weights (integer atomics);
//                 replicates are processed in tiles so that c stays under kCountsBytes
//   accumulation  Z[b][r] += sum_p c[b][p] * q[r][p], q = rint(L * 2^e) converted on load, in
//                 shared-memory tiles, int128 accumulators (a term is < 2^32 * 2^52)
//   statistics    column sums over b, row maxima over r, then the KH / SH / BP counts per record
//   AU / ELW      (rdk_rell_support_ms) the ELW quotients on the unit-scale Z, summed by the column-sum
//                 kernels; then per further scale the same counts and accumulation, argmax and histogram
//
// Every sum is an exact integer, so the result does not depend on launch shape or tiling.
#include "rdk_support.cuh"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

namespace rdk {
namespace {

typedef __int128          i128;
typedef unsigned __int128 u128;

constexpr size_t kCountsBytes = size_t(256) << 20;  // bound of one counts tile
constexpr int    kTile = 32;                        // accumulation: 32 replicates x 32 records x 32 patterns
// ncclDataType_t / ncclRedOp_t values (stable across NCCL 2.x)
constexpr int kNcclInt64 = 4, kNcclUint64 = 5, kNcclSum = 0, kNcclMax = 2;

// Philox4x64-10 (Salmon et al., SC'11), the generator of numpy.random.Philox
__device__ __forceinline__ void philox4x64_10(unsigned long long c[4], unsigned long long k0, unsigned long long k1) {
#pragma unroll
  for (int round = 0; round < 10; ++round) {
    if (round) {
      k0 += 0x9E3779B97F4A7C15ull;
      k1 += 0xBB67AE8584CAA73Bull;
    }
    const unsigned long long m0 = 0xD2E7470EE14C6C93ull, m1 = 0xCA5A826395121157ull;
    const unsigned long long hi0 = __umul64hi(m0, c[0]), lo0 = m0 * c[0];
    const unsigned long long hi1 = __umul64hi(m1, c[2]), lo1 = m1 * c[2];
    const unsigned long long n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0;
    c[1] = lo1;
    c[2] = n2;
    c[3] = lo0;
  }
}

// max |L| (as the bit pattern of a non-negative double, which orders like the value) and the
// lowest row holding a non-finite value
__global__ void rell_scan_kernel(const double *rows, size_t count, unsigned patterns, unsigned long long *maxbits,
                                 unsigned *bad_row) {
  unsigned long long m = 0;
  unsigned           bad = ~0u;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
    const double v = rows[i];
    if (!isfinite(v))
      bad = min(bad, (unsigned)(i / patterns));
    else
      m = max(m, (unsigned long long)__double_as_longlong(fabs(v)));
  }
  for (int off = 16; off; off >>= 1) {
    m = max(m, __shfl_xor_sync(0xffffffffu, m, off));
    bad = min(bad, __shfl_xor_sync(0xffffffffu, bad, off));
  }
  if ((threadIdx.x & 31) == 0) {
    if (m) atomicMax(maxbits, m);
    if (bad != ~0u) atomicMin(bad_row, bad);
  }
}

// c[b][p] for replicates [b0, b0 + tile) of one partition: one thread = one Philox block = 4 of the
// `draws` draws (counter {j + 1, word, 0, 0}) over the partition's `sites` original sites; the draws
// that hit this shard's sites [lo, lo + cumw[patterns]) are counted (lo = 0 and every site here when the
// partition is not sharded).  rdk_rell_support draws `sites` times with word 0; the multiscale
// bootstrap draws (s sites + 500) / 1000 times with word s - 1000.
__global__ void rell_counts_kernel(unsigned long long seed, unsigned long long global_index, unsigned long long b0,
                                   unsigned tile, unsigned long long draws, unsigned long long word,
                                   unsigned long long sites, unsigned long long lo, const unsigned long long *cumw,
                                   unsigned patterns, unsigned *c) {
  const unsigned long long blocks = (draws + 3) / 4;
  const unsigned long long here = cumw[patterns];
  const unsigned long long total = blocks * tile;
  for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < total;
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long b = i / blocks, j4 = i - b * blocks;
    unsigned long long       x[4] = {j4 + 1, word, 0, 0};  // numpy increments the counter before each block
    philox4x64_10(x, seed, (global_index << 32) | (b0 + b));
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (j4 * 4 + u >= draws) break;
      const unsigned long long site = __umul64hi(x[u], sites) - lo;  // wraps below lo
      if (site >= here) continue;
      unsigned p = 0, hi = patterns;  // cumw[p] <= site < cumw[hi]
      while (hi - p > 1) {
        const unsigned mid = (p + hi) / 2;
        if (cumw[mid] <= site)
          p = mid;
        else
          hi = mid;
      }
      atomicAdd(c + b * patterns + p, 1u);
    }
  }
}

// Z[b][r] (+)= sum_p c[b][p] * rint(L[r][p] * 2^e) for b < nb, r < nr
__global__ void __launch_bounds__(256) rell_accumulate_kernel(const unsigned *c, const double *rows, unsigned patterns,
                                                              unsigned nb, unsigned nr, int e, int add, i128 *z,
                                                              size_t z_stride) {
  __shared__ unsigned  cs[kTile][kTile + 1];
  __shared__ long long qs[kTile][kTile + 1];
  const unsigned tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  const unsigned b_base = blockIdx.y * kTile, r_base = blockIdx.x * kTile;
  i128           acc[4] = {0, 0, 0, 0};
  for (unsigned p0 = 0; p0 < patterns; p0 += kTile) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const unsigned row = ty + 8 * i, p = p0 + tx;
      cs[row][tx] = (b_base + row < nb && p < patterns) ? c[(size_t)(b_base + row) * patterns + p] : 0u;
      qs[row][tx] = (r_base + row < nr && p < patterns)
                        ? __double2ll_rn(scalbn(rows[(size_t)(r_base + row) * patterns + p], e))
                        : 0ll;
    }
    __syncthreads();
#pragma unroll 8
    for (int pp = 0; pp < kTile; ++pp) {
      const long long q = qs[tx][pp];
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i] += (i128)cs[ty + 8 * i][pp] * q;
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const unsigned b = b_base + ty + 8 * i, r = r_base + tx;
    if (b < nb && r < nr) {
      i128 &dst = z[(size_t)b * z_stride + r];
      dst = add ? dst + acc[i] : acc[i];
    }
  }
}

// part[chunk][r] = sum over b in chunk of Z[b][r]
__global__ void rell_colsum_kernel(const i128 *z, unsigned nb, unsigned nr, unsigned chunk, i128 *part) {
  const unsigned r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nr) return;
  const unsigned b_end = min(nb, (blockIdx.y + 1) * chunk);
  i128           s = 0;
  for (unsigned b = blockIdx.y * chunk; b < b_end; ++b) s += z[(size_t)b * nr + r];
  part[(size_t)blockIdx.y * nr + r] = s;
}

__global__ void rell_colsum_final_kernel(const i128 *part, unsigned chunks, unsigned nr, i128 *colsum) {
  const unsigned r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nr) return;
  i128 s = 0;
  for (unsigned k = 0; k < chunks; ++k) s += part[(size_t)k * nr + r];
  colsum[r] = s;
}

__device__ __forceinline__ i128 shfl_xor_i128(i128 v, int off) {
  const unsigned long long lo = (unsigned long long)(u128)v, hi = (unsigned long long)((u128)v >> 64);
  const unsigned long long l2 = __shfl_xor_sync(0xffffffffu, lo, off), h2 = __shfl_xor_sync(0xffffffffu, hi, off);
  return (i128)(((u128)h2 << 64) | l2);
}

// one warp per replicate: max_r (B Z[b][r] - colsum[r]) and argmax_r Z[b][r] (lowest index on ties)
__global__ void rell_rowstat_kernel(const i128 *z, unsigned nb, unsigned nr, const i128 *colsum, i128 *rowmax,
                                    unsigned *argmax) {
  const unsigned b = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32, lane = threadIdx.x & 31;
  if (b >= nb) return;
  const i128 B = nb;
  bool       any = false;
  i128       mt = 0, mz = 0;
  unsigned   at = ~0u;
  for (unsigned r = lane; r < nr; r += 32) {
    const i128 v = z[(size_t)b * nr + r], t = B * v - colsum[r];
    if (!any || t > mt) mt = t;
    if (!any || v > mz) {
      mz = v;
      at = r;
    }
    any = true;
  }
  for (int off = 16; off; off >>= 1) {
    const i128     omt = shfl_xor_i128(mt, off), omz = shfl_xor_i128(mz, off);
    const unsigned oat = __shfl_xor_sync(0xffffffffu, at, off);
    if (oat != ~0u) {
      if (at == ~0u || omt > mt) mt = omt;
      if (at == ~0u || omz > mz || (omz == mz && oat < at)) {
        mz = omz;
        at = oat;
      }
    }
  }
  if (lane == 0) {
    rowmax[b] = mt;
    argmax[b] = at;
  }
}

// per record r over the replicates of chunk blockIdx.y: the BP, KH and SH counts
__global__ void rell_count_kernel(const i128 *z, unsigned nb, unsigned nr, unsigned chunk, unsigned best,
                                  const i128 *colsum, const i128 *o, const i128 *rowmax, const unsigned *argmax,
                                  unsigned *bp, unsigned *kh, unsigned *sh) {
  const unsigned r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nr) return;
  const i128     B = nb;
  const i128     sum_d = colsum[best] - colsum[r];
  const i128     kh_bound = B * (o[best] - o[r]) + sum_d;  // B D - sum D >= B delta
  const i128     sh_bound = B * (o[best] - o[r]);
  unsigned       nbp = 0, nkh = 0, nsh = 0;
  const unsigned b_end = min(nb, (blockIdx.y + 1) * chunk);
  for (unsigned b = blockIdx.y * chunk; b < b_end; ++b) {
    const i128 zr = z[(size_t)b * nr + r], zb = z[(size_t)b * nr + best];
    nbp += argmax[b] == r;
    nkh += B * (zb - zr) >= kh_bound;
    nsh += rowmax[b] - (B * zr - colsum[r]) >= sh_bound;
  }
  if (nbp) atomicAdd(bp + r, nbp);
  if (nkh) atomicAdd(kh + r, nkh);
  if (nsh) atomicAdd(sh + r, nsh);
}

// count[argmax[b]] += 1: the multiscale BP counts of one scale
__global__ void rell_hist_kernel(const unsigned *argmax, unsigned nb, unsigned *count) {
  const unsigned b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < nb) atomicAdd(count + argmax[b], 1u);
}

// ---- expected likelihood weights (DESIGN.md section 10, item 8)

// int128 -> double, rounded to nearest even: the top 64 bits with the rest folded into a sticky bit
// round as the whole value does (11 bits are dropped below the sticky bit's position)
__device__ double i128_to_double_rn(i128 v) {
  const bool neg = v < 0;
  const u128 a = neg ? -(u128)v : (u128)v;
  const unsigned long long hi = (unsigned long long)(a >> 64);
  double                   d;
  if (hi == 0) {
    d = __ull2double_rn((unsigned long long)a);
  } else {
    const int                sh = 64 - __clzll((long long)hi);
    const unsigned long long top = (unsigned long long)(a >> sh) | (((a << (128 - sh)) != 0) ? 1ull : 0ull);
    d = scalbn(__ull2double_rn(top), sh);
  }
  return neg ? -d : d;
}

// fdlibm e_exp.c on [-40, 0], every operation rounded on its own; rd_exp(0) == 1
__device__ double rd_exp(double x) {
  const double P1 = 1.66666666666666019037e-01, P2 = -2.77777777770155933842e-03, P3 = 6.61375632143793436117e-05,
               P4 = -1.65339022054652515390e-06, P5 = 4.13813679705723846039e-08;
  const double ln2hi = 6.93147180369123816490e-01, ln2lo = 1.90821492927058770002e-10,
               invln2 = 1.44269504088896338700e+00;
  const unsigned hx = (unsigned)__double2hiint(x) & 0x7fffffffu;
  double         hi = 0, lo = 0;
  int            k = 0;
  if (hx > 0x3fd62e42u) {    // |x| > ln2 / 2
    if (hx < 0x3ff0a2b2u) {  // |x| < 3 ln2 / 2
      hi = __dadd_rn(x, ln2hi);
      lo = -ln2lo;
      k = -1;
    } else {
      k = __double2int_rz(__dadd_rn(__dmul_rn(invln2, x), -0.5));
      const double t = (double)k;
      hi = __dadd_rn(x, -__dmul_rn(t, ln2hi));
      lo = __dmul_rn(t, ln2lo);
    }
    x = __dadd_rn(hi, -lo);
  } else if (hx < 0x3e300000u) {  // |x| < 2^-28
    return __dadd_rn(1.0, x);
  }
  const double t = __dmul_rn(x, x);
  double       p = __dadd_rn(P4, __dmul_rn(t, P5));
  p = __dadd_rn(P3, __dmul_rn(t, p));
  p = __dadd_rn(P2, __dmul_rn(t, p));
  p = __dadd_rn(P1, __dmul_rn(t, p));
  const double c = __dadd_rn(x, -__dmul_rn(t, p));
  if (k == 0) return __dadd_rn(1.0, -__dadd_rn(__ddiv_rn(__dmul_rn(x, c), __dadd_rn(c, -2.0)), -x));
  const double y = __dadd_rn(1.0, -__dadd_rn(__dadd_rn(lo, -__ddiv_rn(__dmul_rn(x, c), __dadd_rn(2.0, -c))), -hi));
  return __hiloint2double(__double2hiint(y) + k * (1 << 20), __double2loint(y));  // y 2^k, exact for k >= -1021
}

// Delta < -40 2^e, exactly (|Delta| < 2^85; e < 0 only when max |L| >= 2^52)
__device__ __forceinline__ bool elw_below_cut(i128 d, int e) {
  if (e >= 80) return false;
  if (e >= 0) return d < -((i128)40 << e);
  return d != 0 && (-e >= 6 || ((-d) << -e) > 40);
}

// u = rint(rd_exp(Delta 2^-e) 2^52), 0 below the cut; the record of the maximum gets 2^52
__device__ __forceinline__ unsigned long long elw_weight(i128 d, int e) {
  if (elw_below_cut(d, e)) return 0;
  return __double2ull_rn(scalbn(rd_exp(scalbn(i128_to_double_rn(d), -e)), 52));
}

// one warp per replicate: D_b = sum_r u_b[r], then Z[b][r] := floor(u_b[r] 2^40 / D_b) in place (the
// unit-scale statistics are done with Z); the column sums of those quotients are elw_fixed
__global__ void rell_elw_kernel(i128 *z, unsigned nb, unsigned nr, int e, const unsigned *argmax) {
  const unsigned b = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32, lane = threadIdx.x & 31;
  if (b >= nb) return;
  i128      *zb = z + (size_t)b * nr;
  const i128 m = zb[argmax[b]];
  u128       D = 0;
  for (unsigned r = lane; r < nr; r += 32) D += elw_weight(zb[r] - m, e);
  for (int off = 16; off; off >>= 1) D += (u128)shfl_xor_i128((i128)D, off);
  __syncwarp();  // every lane has read m before any lane writes
  for (unsigned r = lane; r < nr; r += 32) zb[r] = (i128)(((u128)elw_weight(zb[r] - m, e) << 40) / D);
}

// int128 <-> three int64 limbs v = l0 + l1 2^42 + l2 2^84 (l0, l1 in [0, 2^42)), so that an NCCL
// sum of the limbs over up to 2^21 ranks cannot overflow; limbs[k * n + i]
constexpr int kLimbBits = 42;
__global__ void rell_to_limbs_kernel(const i128 *v, size_t n, long long *limbs) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const i128 x = v[i];
    const i128 mask = ((i128)1 << kLimbBits) - 1;
    limbs[i] = (long long)(x & mask);
    limbs[n + i] = (long long)((x >> kLimbBits) & mask);
    limbs[2 * n + i] = (long long)(x >> (2 * kLimbBits));
  }
}

__global__ void rell_from_limbs_kernel(const long long *limbs, size_t n, i128 *v) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    v[i] = (i128)limbs[i] + (i128)limbs[n + i] * ((i128)1 << kLimbBits) +
           (i128)limbs[2 * n + i] * ((i128)1 << (2 * kLimbBits));
}

struct DeviceBuffers {
  std::vector<void *> ptrs;
  unsigned long long  bytes = 0;
  ~DeviceBuffers() {
    for (void *p : ptrs) cudaFree(p);
  }
  template <typename T> cudaError_t alloc(T **p, size_t count) {
    const size_t b = std::max<size_t>(16, count * sizeof(T));
    cudaError_t  err = cudaMalloc((void **)p, b);
    if (err == cudaSuccess) {
      ptrs.push_back(*p);
      bytes += b;
    }
    return err;
  }
};

struct Events {
  cudaEvent_t ev[8] = {};
  ~Events() {
    for (cudaEvent_t e : ev)
      if (e) cudaEventDestroy(e);
  }
};

}  // namespace

#define RELL_TRY(expr)                                                                             \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      snprintf(msg, msg_cap, "%s failed: %s", #expr, cudaGetErrorString(_e));                      \
      if (stream) cudaStreamDestroy(stream);                                                       \
      return 0;                                                                                    \
    }                                                                                              \
  } while (0)

int rell_support(const RellPartition *parts, unsigned int n, unsigned int rows, unsigned long long replicates,
                 unsigned long long seed, const RellShard &shard, rdk_rell_out_t *out, rdk_rell_ms_out_t *ms,
                 char *msg, size_t msg_cap) {
  cudaStream_t  stream = nullptr;
  DeviceBuffers buf;
  Events        ev;
  out->bad_row = ~0u;
  out->device_bytes = 0;
  const unsigned nb = (unsigned)replicates;
  RELL_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  for (cudaEvent_t &e : ev.ev) RELL_TRY(cudaEventCreate(&e));
  int dev = 0, sms = 148;
  RELL_TRY(cudaGetDevice(&dev));
  RELL_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));

  // ---- the fixed-point grid: e from max |L| over every partition, record and pattern
  unsigned long long *d_max = nullptr;
  unsigned           *d_bad = nullptr;
  RELL_TRY(buf.alloc(&d_max, 1));
  RELL_TRY(buf.alloc(&d_bad, 1));
  RELL_TRY(cudaMemsetAsync(d_max, 0, sizeof(unsigned long long), stream));
  RELL_TRY(cudaMemsetAsync(d_bad, 0xff, sizeof(unsigned), stream));
  for (unsigned g = 0; g < n; ++g) {
    const size_t count = (size_t)rows * parts[g].patterns;
    if (count == 0) continue;
    const unsigned grid = (unsigned)std::min<size_t>((count + 255) / 256, (size_t)sms * 8);
    rell_scan_kernel<<<grid, 256, 0, stream>>>(parts[g].rows, count, parts[g].patterns, d_max, d_bad);
    RELL_TRY(cudaGetLastError());
  }
  unsigned long long maxbits = 0;
  unsigned           bad = ~0u;
  RELL_TRY(cudaMemcpyAsync(&maxbits, d_max, sizeof(maxbits), cudaMemcpyDeviceToHost, stream));
  RELL_TRY(cudaMemcpyAsync(&bad, d_bad, sizeof(unsigned), cudaMemcpyDeviceToHost, stream));
  RELL_TRY(cudaStreamSynchronize(stream));

  // site shards, exchange 1 and 2: M (and the first non-finite record) is an all-reduce max; the
  // shard's first original site is the sum of the weight totals of the shards before it
  unsigned long long lo = 0, sites_all = 0;
  unsigned long long local_total = 0;
  if (n == 1)
    for (unsigned p = 0; p < parts[0].patterns; ++p) local_total += parts[0].weights[p];
  if (shard.comm) {
    const int                       R2 = 2 + 2 * shard.nranks;
    std::vector<unsigned long long> h(R2, 0);
    unsigned long long             *d_x = nullptr;
    RELL_TRY(buf.alloc(&d_x, R2));
    h[0] = maxbits;
    h[1] = ~(unsigned long long)bad;  // max of the complement = min
    RELL_TRY(cudaMemcpyAsync(d_x, h.data(), sizeof(unsigned long long) * 2, cudaMemcpyHostToDevice, stream));
    if (shard.allreduce(d_x, d_x, 2, kNcclUint64, kNcclMax, shard.comm, stream) != 0) {
      snprintf(msg, msg_cap, "ncclAllReduce (max) failed");
      cudaStreamDestroy(stream);
      return 0;
    }
    std::fill(h.begin(), h.end(), 0ull);
    h[2 + 2 * shard.rank] = shard.site_offset;
    h[3 + 2 * shard.rank] = local_total;
    RELL_TRY(cudaMemcpyAsync(d_x + 2, h.data() + 2, sizeof(unsigned long long) * 2 * shard.nranks,
                             cudaMemcpyHostToDevice, stream));
    if (shard.allreduce(d_x + 2, d_x + 2, 2 * shard.nranks, kNcclUint64, kNcclSum, shard.comm, stream) != 0) {
      snprintf(msg, msg_cap, "ncclAllReduce (sum) failed");
      cudaStreamDestroy(stream);
      return 0;
    }
    RELL_TRY(cudaMemcpyAsync(h.data(), d_x, sizeof(unsigned long long) * R2, cudaMemcpyDeviceToHost, stream));
    RELL_TRY(cudaStreamSynchronize(stream));
    maxbits = h[0];
    bad = (unsigned)~h[1];
    for (int r = 0; r < shard.nranks; ++r) {
      sites_all += h[3 + 2 * r];
      if (h[2 + 2 * r] < shard.site_offset) lo += h[3 + 2 * r];
    }
  }
  if (bad != ~0u) {
    out->bad_row = bad;
    snprintf(msg, msg_cap, "record %u has a site of likelihood 0 (non-finite log-likelihood)", bad);
    cudaStreamDestroy(stream);
    return 0;
  }
  double M;
  memcpy(&M, &maxbits, sizeof(M));
  int x = 0;
  if (M > 0) frexp(M, &x);
  const int e = M > 0 ? 52 - x : 0;
  out->exponent = e;

  // ---- per-partition inputs: cumulative weights, weights as a 1-row count matrix
  size_t max_patterns = 1;
  for (unsigned g = 0; g < n; ++g) max_patterns = std::max<size_t>(max_patterns, parts[g].patterns);
  const unsigned tile = (unsigned)std::max<unsigned long long>(
      1, std::min<unsigned long long>(out->replicate_tile ? out->replicate_tile : kCountsBytes / (4 * max_patterns),
                                      nb));
  std::vector<unsigned long long *> d_cumw(n);
  std::vector<unsigned *>           d_w(n);
  std::vector<unsigned long long>   sites(n);
  for (unsigned g = 0; g < n; ++g) {
    const unsigned                  P = parts[g].patterns;
    std::vector<unsigned long long> cw(P + 1, 0);
    for (unsigned p = 0; p < P; ++p) cw[p + 1] = cw[p] + parts[g].weights[p];
    sites[g] = shard.comm ? sites_all : cw[P];
    RELL_TRY(buf.alloc(&d_cumw[g], P + 1));
    RELL_TRY(buf.alloc(&d_w[g], P));
    RELL_TRY(cudaMemcpyAsync(d_cumw[g], cw.data(), sizeof(unsigned long long) * (P + 1), cudaMemcpyHostToDevice,
                             stream));
    RELL_TRY(cudaMemcpyAsync(d_w[g], parts[g].weights, sizeof(unsigned) * P, cudaMemcpyHostToDevice, stream));
    RELL_TRY(cudaStreamSynchronize(stream));  // cw leaves scope
  }

  unsigned *d_c = nullptr;
  i128     *d_z = nullptr, *d_o = nullptr;
  RELL_TRY(buf.alloc(&d_c, (size_t)tile * max_patterns));
  RELL_TRY(buf.alloc(&d_z, (size_t)nb * rows));
  RELL_TRY(buf.alloc(&d_o, rows));

  // ---- O[r] = sum_g sum_p w q (the weights are a count matrix of one replicate)
  const dim3 acc_threads(256);
  for (unsigned g = 0; g < n; ++g) {
    const dim3 grid((rows + kTile - 1) / kTile, 1);
    rell_accumulate_kernel<<<grid, acc_threads, 0, stream>>>(d_w[g], parts[g].rows, parts[g].patterns, 1, rows, e,
                                                             g > 0, d_o, rows);
    RELL_TRY(cudaGetLastError());
  }

  // ---- counts and accumulation, tile by tile, of the replicates at one scale (thousandths; the
  // counter word is s - 1000 mod 2^64, so scale 1000 is word 0 and N_g draws)
  float t_counts = 0, t_acc = 0, t_stats = 0, t_ms = 0;
  auto  resample = [&](unsigned scale, float &counts_ms, float &acc_ms) -> int {
    const unsigned long long word = (unsigned long long)scale - 1000ull;
    for (unsigned long long b0 = 0; b0 < nb; b0 += tile) {
      const unsigned nt = (unsigned)std::min<unsigned long long>(tile, nb - b0);
      for (unsigned g = 0; g < n; ++g) {
        const unsigned           P = parts[g].patterns;
        const unsigned long long draws = std::max<unsigned long long>(1, (scale * sites[g] + 500) / 1000);
        RELL_TRY(cudaEventRecord(ev.ev[0], stream));
        RELL_TRY(cudaMemsetAsync(d_c, 0, sizeof(unsigned) * (size_t)nt * std::max(1u, P), stream));
        if (sites[g]) {
          const unsigned long long work = (draws + 3) / 4 * nt;
          const unsigned grid = (unsigned)std::min<unsigned long long>((work + 255) / 256, (unsigned long long)sms * 16);
          rell_counts_kernel<<<grid, 256, 0, stream>>>(seed, parts[g].global_index, b0, nt, draws, word, sites[g], lo,
                                                       d_cumw[g], P, d_c);
          RELL_TRY(cudaGetLastError());
        }
        RELL_TRY(cudaEventRecord(ev.ev[1], stream));
        const dim3 grid((rows + kTile - 1) / kTile, (nt + kTile - 1) / kTile);
        rell_accumulate_kernel<<<grid, acc_threads, 0, stream>>>(d_c, parts[g].rows, P, nt, rows, e, g > 0,
                                                                 d_z + b0 * rows, rows);
        RELL_TRY(cudaGetLastError());
        RELL_TRY(cudaEventRecord(ev.ev[2], stream));
        RELL_TRY(cudaEventSynchronize(ev.ev[2]));
        float t = 0;
        RELL_TRY(cudaEventElapsedTime(&t, ev.ev[0], ev.ev[1]));
        counts_ms += t;
        RELL_TRY(cudaEventElapsedTime(&t, ev.ev[1], ev.ev[2]));
        acc_ms += t;
      }
    }
    return 1;
  };
  RELL_TRY(cudaEventRecord(ev.ev[6], stream));
  if (!resample(1000, t_counts, t_acc)) return 0;

  // site shards, exchange 3: Z and O summed over the ranks as 42-bit limbs (exact); Z_k again per scale
  long long *d_limbs = nullptr;
  auto       allreduce = [&](i128 *v, size_t cnt) -> int {
    const unsigned grid = (unsigned)std::min<size_t>((cnt + 255) / 256, (size_t)sms * 8);
    rell_to_limbs_kernel<<<grid, 256, 0, stream>>>(v, cnt, d_limbs);
    RELL_TRY(cudaGetLastError());
    if (shard.allreduce(d_limbs, d_limbs, 3 * cnt, kNcclInt64, kNcclSum, shard.comm, stream) != 0) {
      snprintf(msg, msg_cap, "ncclAllReduce (limbs) failed");
      cudaStreamDestroy(stream);
      return 0;
    }
    rell_from_limbs_kernel<<<grid, 256, 0, stream>>>(d_limbs, cnt, v);
    RELL_TRY(cudaGetLastError());
    return 1;
  };
  if (shard.comm) {
    RELL_TRY(buf.alloc(&d_limbs, 3 * ((size_t)nb * rows + rows)));
    if (!allreduce(d_z, (size_t)nb * rows) || !allreduce(d_o, rows)) return 0;
  }

  // ---- statistics
  std::vector<i128> o(rows);
  RELL_TRY(cudaMemcpyAsync(o.data(), d_o, sizeof(i128) * rows, cudaMemcpyDeviceToHost, stream));
  RELL_TRY(cudaStreamSynchronize(stream));
  unsigned best = 0;
  for (unsigned r = 1; r < rows; ++r)
    if (o[r] > o[best]) best = r;
  out->best = best;

  const unsigned chunk = 256, chunks = (nb + chunk - 1) / chunk;
  i128          *d_part = nullptr, *d_colsum = nullptr, *d_rowmax = nullptr;
  unsigned      *d_argmax = nullptr, *d_counts = nullptr;
  RELL_TRY(buf.alloc(&d_part, (size_t)chunks * rows));
  RELL_TRY(buf.alloc(&d_colsum, rows));
  RELL_TRY(buf.alloc(&d_rowmax, nb));
  RELL_TRY(buf.alloc(&d_argmax, nb));
  RELL_TRY(buf.alloc(&d_counts, (size_t)3 * rows));
  RELL_TRY(cudaEventRecord(ev.ev[3], stream));
  RELL_TRY(cudaMemsetAsync(d_counts, 0, sizeof(unsigned) * 3 * rows, stream));
  const dim3 col_grid((rows + 127) / 128, chunks);
  rell_colsum_kernel<<<col_grid, 128, 0, stream>>>(d_z, nb, rows, chunk, d_part);
  rell_colsum_final_kernel<<<(rows + 127) / 128, 128, 0, stream>>>(d_part, chunks, rows, d_colsum);
  rell_rowstat_kernel<<<(nb + 7) / 8, 256, 0, stream>>>(d_z, nb, rows, d_colsum, d_rowmax, d_argmax);
  rell_count_kernel<<<col_grid, 128, 0, stream>>>(d_z, nb, rows, chunk, best, d_colsum, d_o, d_rowmax, d_argmax,
                                                  d_counts, d_counts + rows, d_counts + 2 * rows);
  RELL_TRY(cudaGetLastError());
  RELL_TRY(cudaEventRecord(ev.ev[4], stream));
  RELL_TRY(cudaMemcpyAsync(out->bp_count, d_counts, sizeof(unsigned) * rows, cudaMemcpyDeviceToHost, stream));
  RELL_TRY(cudaMemcpyAsync(out->kh_count, d_counts + rows, sizeof(unsigned) * rows, cudaMemcpyDeviceToHost, stream));
  RELL_TRY(cudaMemcpyAsync(out->sh_count, d_counts + 2 * rows, sizeof(unsigned) * rows, cudaMemcpyDeviceToHost,
                           stream));
  RELL_TRY(cudaEventRecord(ev.ev[7], stream));
  RELL_TRY(cudaStreamSynchronize(stream));
  RELL_TRY(cudaEventElapsedTime(&t_stats, ev.ev[3], ev.ev[4]));
  RELL_TRY(cudaEventElapsedTime(&t_ms, ev.ev[6], ev.ev[7]));

  if (ms) {
    // ELW on the unit-scale Z (its argmax is still in d_argmax), then overwritten by the quotients
    float t_ms_counts = 0, t_ms_acc = 0, t_ms_stats = 0, t = 0;
    RELL_TRY(cudaEventRecord(ev.ev[3], stream));
    rell_elw_kernel<<<(nb + 7) / 8, 256, 0, stream>>>(d_z, nb, rows, e, d_argmax);
    rell_colsum_kernel<<<col_grid, 128, 0, stream>>>(d_z, nb, rows, chunk, d_part);
    rell_colsum_final_kernel<<<(rows + 127) / 128, 128, 0, stream>>>(d_part, chunks, rows, d_colsum);
    RELL_TRY(cudaGetLastError());
    RELL_TRY(cudaEventRecord(ev.ev[4], stream));
    std::vector<i128> elw(rows);
    RELL_TRY(cudaMemcpyAsync(elw.data(), d_colsum, sizeof(i128) * rows, cudaMemcpyDeviceToHost, stream));
    RELL_TRY(cudaStreamSynchronize(stream));
    RELL_TRY(cudaEventElapsedTime(&t, ev.ev[3], ev.ev[4]));
    t_ms_stats += t;
    for (unsigned r = 0; r < rows; ++r) ms->elw_fixed[r] = (unsigned long long)elw[r];  // < 2^60

    // the other scales: Z_k in the same buffer, argmax per replicate, histogram
    for (unsigned k = 0; k < ms->n_scales; ++k) {
      unsigned *count = ms->scale_count + (size_t)k * rows;
      if (ms->scales[k] == 1000) {
        memcpy(count, out->bp_count, sizeof(unsigned) * rows);
        continue;
      }
      if (!resample(ms->scales[k], t_ms_counts, t_ms_acc)) return 0;
      if (shard.comm && !allreduce(d_z, (size_t)nb * rows)) return 0;
      RELL_TRY(cudaEventRecord(ev.ev[3], stream));
      RELL_TRY(cudaMemsetAsync(d_counts, 0, sizeof(unsigned) * rows, stream));
      rell_rowstat_kernel<<<(nb + 7) / 8, 256, 0, stream>>>(d_z, nb, rows, d_colsum, d_rowmax, d_argmax);
      rell_hist_kernel<<<(nb + 255) / 256, 256, 0, stream>>>(d_argmax, nb, d_counts);
      RELL_TRY(cudaGetLastError());
      RELL_TRY(cudaEventRecord(ev.ev[4], stream));
      RELL_TRY(cudaMemcpyAsync(count, d_counts, sizeof(unsigned) * rows, cudaMemcpyDeviceToHost, stream));
      RELL_TRY(cudaStreamSynchronize(stream));
      RELL_TRY(cudaEventElapsedTime(&t, ev.ev[3], ev.ev[4]));
      t_ms_stats += t;
    }
    ms->ms[0] = t_ms_counts;
    ms->ms[1] = t_ms_acc;
    ms->ms[2] = t_ms_stats;
  }

  out->ms[0] = t_counts;
  out->ms[1] = t_acc;
  out->ms[2] = t_stats;
  out->ms[3] = t_ms;
  for (unsigned r = 0; r < rows; ++r) {
    out->lnl_fixed[r] = ldexp((double)o[r], -e);  // int128 -> double rounds once
    if (out->o_lo) out->o_lo[r] = (unsigned long long)(u128)o[r];
    if (out->o_hi) out->o_hi[r] = (long long)(o[r] >> 64);
  }
  out->device_bytes = buf.bytes;
  cudaStreamDestroy(stream);
  return 1;
}

}  // namespace rdk
