// rdk_support.cu -- the three kernels of rdk_rell_support (DESIGN.md section 10).
//
//   counts        c[b][p]: Philox4x64-10 draws of the original sites of a partition, mapped to
//                 their pattern by a binary search in the cumulative weights (integer atomics);
//                 replicates are processed in tiles so that c stays under kCountsBytes
//   accumulation  Z[b][r] += sum_p c[b][p] * q[r][p], q = rint(L * 2^e) converted on load, in
//                 shared-memory tiles, int128 accumulators (a term is < 2^32 * 2^52)
//   statistics    column sums over b, row maxima over r, then the KH / SH / BP counts per record
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

// c[b][p] for replicates [b0, b0 + tile) of one partition: one thread = one Philox block = 4 draws of
// the partition's `sites` original sites; the draws that hit this shard's sites [lo, lo + cumw[patterns])
// are counted (lo = 0 and every site here when the partition is not sharded)
__global__ void rell_counts_kernel(unsigned long long seed, unsigned long long global_index, unsigned long long b0,
                                   unsigned tile, unsigned long long sites, unsigned long long lo,
                                   const unsigned long long *cumw, unsigned patterns, unsigned *c) {
  const unsigned long long blocks = (sites + 3) / 4;
  const unsigned long long here = cumw[patterns];
  const unsigned long long total = blocks * tile;
  for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < total;
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long b = i / blocks, j4 = i - b * blocks;
    unsigned long long       x[4] = {j4 + 1, 0, 0, 0};  // numpy increments the counter before each block
    philox4x64_10(x, seed, (global_index << 32) | (b0 + b));
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (j4 * 4 + u >= sites) break;
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
                 unsigned long long seed, const RellShard &shard, rdk_rell_out_t *out, char *msg, size_t msg_cap) {
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

  // ---- counts and accumulation, tile by tile
  float t_counts = 0, t_acc = 0, t_stats = 0, t_ms = 0;
  RELL_TRY(cudaEventRecord(ev.ev[6], stream));
  for (unsigned long long b0 = 0; b0 < nb; b0 += tile) {
    const unsigned nt = (unsigned)std::min<unsigned long long>(tile, nb - b0);
    for (unsigned g = 0; g < n; ++g) {
      const unsigned P = parts[g].patterns;
      RELL_TRY(cudaEventRecord(ev.ev[0], stream));
      RELL_TRY(cudaMemsetAsync(d_c, 0, sizeof(unsigned) * (size_t)nt * std::max(1u, P), stream));
      if (sites[g]) {
        const unsigned long long work = (sites[g] + 3) / 4 * nt;
        const unsigned grid = (unsigned)std::min<unsigned long long>((work + 255) / 256, (unsigned long long)sms * 16);
        rell_counts_kernel<<<grid, 256, 0, stream>>>(seed, parts[g].global_index, b0, nt, sites[g], lo, d_cumw[g],
                                                     P, d_c);
        RELL_TRY(cudaGetLastError());
      }
      RELL_TRY(cudaEventRecord(ev.ev[1], stream));
      const dim3 grid((rows + kTile - 1) / kTile, (nt + kTile - 1) / kTile);
      rell_accumulate_kernel<<<grid, acc_threads, 0, stream>>>(d_c, parts[g].rows, P, nt, rows, e, g > 0,
                                                               d_z + b0 * rows, rows);
      RELL_TRY(cudaGetLastError());
      RELL_TRY(cudaEventRecord(ev.ev[2], stream));
      RELL_TRY(cudaEventSynchronize(ev.ev[2]));
      RELL_TRY(cudaEventElapsedTime(&t_ms, ev.ev[0], ev.ev[1]));
      t_counts += t_ms;
      RELL_TRY(cudaEventElapsedTime(&t_ms, ev.ev[1], ev.ev[2]));
      t_acc += t_ms;
    }
  }

  // site shards, exchange 3: Z and O summed over the ranks as 42-bit limbs (exact)
  if (shard.comm) {
    const size_t n_all = (size_t)nb * rows + rows;
    long long   *d_limbs = nullptr;
    RELL_TRY(buf.alloc(&d_limbs, 3 * n_all));
    const unsigned grid = (unsigned)std::min<size_t>((n_all + 255) / 256, (size_t)sms * 8);
    for (int pass = 0; pass < 2; ++pass) {  // Z, then O
      i128        *v = pass ? d_o : d_z;
      const size_t cnt = pass ? rows : (size_t)nb * rows;
      rell_to_limbs_kernel<<<grid, 256, 0, stream>>>(v, cnt, d_limbs);
      RELL_TRY(cudaGetLastError());
      if (shard.allreduce(d_limbs, d_limbs, 3 * cnt, kNcclInt64, kNcclSum, shard.comm, stream) != 0) {
        snprintf(msg, msg_cap, "ncclAllReduce (limbs) failed");
        cudaStreamDestroy(stream);
        return 0;
      }
      rell_from_limbs_kernel<<<grid, 256, 0, stream>>>(d_limbs, cnt, v);
      RELL_TRY(cudaGetLastError());
    }
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
