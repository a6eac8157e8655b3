// rdk_kernels.cuh -- sm_100a kernels of the RootDigger likelihood engine.
//
// Replaces the arithmetic behind corax_update_prob_matrices,
// corax_update_clvs and corax_compute_root_loglikelihood (call sites:
// reference src/model.cpp:367,432,842 / :402,440,461,851 / :406,441,466).
//
// Arithmetic contract (DESIGN.md "Arithmetic specification", v2): fp64; the 4x4
// mat-vec of the CLV update and the dot products of the root log-likelihood are
// explicit FMA chains (__fma_rn, j ascending); every other +,-,*,/ is
// individually rounded (round-to-nearest-even, no contraction), in the order
// written.  All arithmetic goes through the __d*_rn / __fma_rn intrinsics so the
// contract holds whatever -fmad says.
//
// 0.61 flop/B, no tensor cores (a 4x4 mat-vec is not a dense contraction).  Designed as a
// bandwidth problem -- coalesced 32-byte-per-thread accesses, never re-reading a CLV from HBM --
// and, with most CLV traffic forwarded in registers or found in L2, measured on B200 to be bound
// by instruction issue and the half-rate fp64 pipe instead (DESIGN.md section 5.1).
#pragma once
#include <cuda_runtime.h>
#include "rdk_lower.hpp"
#include <stdint.h>
#include <type_traits>

namespace rdk {

constexpr int kMaxCats = 32;  // rate categories handled by the fast path: K | 32

// ---------------------------------------------------------------------------
// individually rounded arithmetic
// ---------------------------------------------------------------------------
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }
// the 4x4 mat-vec of the CLV update and the root dot products are explicit FMA chains
// (arithmetic spec v2); everything else stays individually rounded
__device__ __forceinline__ double dfma(double a, double b, double c) { return __fma_rn(a, b, c); }

// 2^-256 underflow threshold, 2^256 rescale factor, ln(2^-256)
#define RDK_SCALE_THRESHOLD 0x1p-256
#define RDK_SCALE_FACTOR 0x1p+256
#define RDK_LOG_SCALE_THRESHOLD (-177.44567822334599)

// ---------------------------------------------------------------------------
// rd_log: software natural logarithm.  Reduction of x to 2^k (1+f) with
// sqrt(2)/2 <= 1+f < sqrt(2), then the degree-14 minimax in s = f/(2+f)
// (fdlibm / musl formulation), < 1 ulp.  Written with integer bit operations
// and individually rounded fp64 ops only, so that it produces the same bits on
// any IEEE-754 machine; libdevice's log() is NOT used because its result may
// differ from a host libm in the last bit, which would make root-branch
// derivatives (difference quotients with h = 1e-8, reference
// src/model.cpp:481-519) irreproducible.
// ---------------------------------------------------------------------------
// the constants live in constant memory: a DFMA / DMUL takes them as c[bank][offset] operands,
// where a literal would cost two moves into a uniform register pair each
static __constant__ double kLogConst[9] = {
    6.93147180369123816490e-01, 1.90821492927058770002e-10,  // ln2_hi, ln2_lo
    6.666666666666735130e-01,   3.999999999940941908e-01,    // Lg1, Lg2
    2.857142874366239149e-01,   2.222219843214978396e-01,    // Lg3, Lg4
    1.818357216161805012e-01,   1.531383769920937332e-01,    // Lg5, Lg6
    1.479819860511658591e-01};                               // Lg7
__device__ __forceinline__ double rd_log(double x) {
  const double ln2_hi = kLogConst[0], ln2_lo = kLogConst[1], Lg1 = kLogConst[2], Lg2 = kLogConst[3],
               Lg3 = kLogConst[4], Lg4 = kLogConst[5], Lg5 = kLogConst[6], Lg6 = kLogConst[7],
               Lg7 = kLogConst[8];
  uint64_t ix = (uint64_t)__double_as_longlong(x);
  uint32_t hx = (uint32_t)(ix >> 32);
  int      k = 0;
  if (hx < 0x00100000u || (hx >> 31)) {
    if ((ix << 1) == 0) return __longlong_as_double(0xfff0000000000000LL);  // -inf
    if (hx >> 31) return __longlong_as_double(0x7ff8000000000000LL);        // nan
    k -= 54;
    x = dmul(x, 0x1p54);
    ix = (uint64_t)__double_as_longlong(x);
    hx = (uint32_t)(ix >> 32);
  } else if (hx >= 0x7ff00000u) {
    return x;
  } else if (hx == 0x3ff00000u && (ix << 32) == 0) {
    return 0.0;
  }
  hx += 0x3ff00000u - 0x3fe6a09eu;
  k += (int)(hx >> 20) - 0x3ff;
  hx = (hx & 0x000fffffu) + 0x3fe6a09eu;
  ix = ((uint64_t)hx << 32) | (ix & 0xffffffffULL);
  x = __longlong_as_double((long long)ix);

  double f = dsub(x, 1.0);
  double hfsq = dmul(dmul(0.5, f), f);
  double s = ddiv(f, dadd(2.0, f));
  double z = dmul(s, s);
  double w = dmul(z, z);
  double t1 = dmul(w, dadd(Lg2, dmul(w, dadd(Lg4, dmul(w, Lg6)))));
  double t2 = dmul(z, dadd(Lg1, dmul(w, dadd(Lg3, dmul(w, dadd(Lg5, dmul(w, Lg7)))))));
  double R = dadd(t2, t1);
  double dk = (double)k;
  double r = dmul(s, dadd(hfsq, R));
  r = dadd(r, dmul(dk, ln2_lo));
  r = dsub(r, hfsq);
  r = dadd(r, f);
  r = dadd(r, dmul(dk, ln2_hi));
  return r;
}

// ---------------------------------------------------------------------------
// expm4: exp of a 4x4 matrix, Higham (2005) scaling and squaring with Pade
// approximants of degree 3/5/7/9/13.  One thread per matrix.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void mm4(const double* A, const double* B, double* C) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      double s = dmul(A[i * 4 + 0], B[0 * 4 + j]);
      s = dadd(s, dmul(A[i * 4 + 1], B[1 * 4 + j]));
      s = dadd(s, dmul(A[i * 4 + 2], B[2 * 4 + j]));
      s = dadd(s, dmul(A[i * 4 + 3], B[3 * 4 + j]));
      C[i * 4 + j] = s;
    }
}

__device__ __forceinline__ double norm1_4(const double* A) {
  double best = 0.0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    double s = fabs(A[0 * 4 + j]);
    s = dadd(s, fabs(A[1 * 4 + j]));
    s = dadd(s, fabs(A[2 * 4 + j]));
    s = dadd(s, fabs(A[3 * 4 + j]));
    if (s > best) best = s;
  }
  return best;
}

// X = M^-1 N, Gaussian elimination with partial pivoting (first maximal pivot)
__device__ inline void solve4(double* M, double* N, double* X) {
  for (int c = 0; c < 4; ++c) {
    int    piv = c;
    double best = fabs(M[c * 4 + c]);
    for (int r = c + 1; r < 4; ++r) {
      double v = fabs(M[r * 4 + c]);
      if (v > best) {
        best = v;
        piv = r;
      }
    }
    if (piv != c) {
      for (int j = 0; j < 4; ++j) {
        double t = M[c * 4 + j];
        M[c * 4 + j] = M[piv * 4 + j];
        M[piv * 4 + j] = t;
        t = N[c * 4 + j];
        N[c * 4 + j] = N[piv * 4 + j];
        N[piv * 4 + j] = t;
      }
    }
    for (int r = c + 1; r < 4; ++r) {
      double f = ddiv(M[r * 4 + c], M[c * 4 + c]);
      for (int j = c + 1; j < 4; ++j) M[r * 4 + j] = dsub(M[r * 4 + j], dmul(f, M[c * 4 + j]));
      for (int j = 0; j < 4; ++j) N[r * 4 + j] = dsub(N[r * 4 + j], dmul(f, N[c * 4 + j]));
    }
  }
  for (int r = 3; r >= 0; --r)
    for (int j = 0; j < 4; ++j) {
      double s = N[r * 4 + j];
      for (int q = r + 1; q < 4; ++q) s = dsub(s, dmul(M[r * 4 + q], X[q * 4 + j]));
      X[r * 4 + j] = ddiv(s, M[r * 4 + r]);
    }
}

__device__ inline void expm4(const double* Ain, double* E) {
  const double TH3 = 1.495585217958292e-2, TH5 = 2.539398330063230e-1,
               TH7 = 9.504178996162932e-1, TH9 = 2.097847961257068e0,
               TH13 = 5.371920351148152e0;
  double A[16], U[16], V[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) A[i] = Ain[i];
  double n1 = norm1_4(A);
  int    s = 0;
  int    deg = 13;
  if (n1 <= TH3)
    deg = 3;
  else if (n1 <= TH5)
    deg = 5;
  else if (n1 <= TH7)
    deg = 7;
  else if (n1 <= TH9)
    deg = 9;
  if (deg == 13) {
    while (n1 > TH13) {
      n1 = dmul(n1, 0.5);
      ++s;
    }
    // 2^-s, exact
    double sc = __longlong_as_double((long long)(uint64_t)(1023 - s) << 52);
#pragma unroll
    for (int i = 0; i < 16; ++i) A[i] = dmul(A[i], sc);
  }
  double A2[16], A4[16], A6[16];
  mm4(A, A, A2);
  if (deg == 13) {
    const double b0 = 64764752532480000., b1 = 32382376266240000., b2 = 7771770303897600.,
                 b3 = 1187353796428800., b4 = 129060195264000., b5 = 10559470521600.,
                 b6 = 670442572800., b7 = 33522128640., b8 = 1323241920., b9 = 40840800.,
                 b10 = 960960., b11 = 16380., b12 = 182., b13 = 1.;
    double W1[16], Z1[16], W[16], T[16];
    mm4(A2, A2, A4);
    mm4(A4, A2, A6);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      double t = dmul(b13, A6[i]);
      t = dadd(t, dmul(b11, A4[i]));
      t = dadd(t, dmul(b9, A2[i]));
      W1[i] = t;
      t = dmul(b12, A6[i]);
      t = dadd(t, dmul(b10, A4[i]));
      t = dadd(t, dmul(b8, A2[i]));
      Z1[i] = t;
    }
    mm4(A6, W1, T);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      double id = (i % 5 == 0) ? 1.0 : 0.0;
      double t = dmul(b7, A6[i]);
      t = dadd(t, dmul(b5, A4[i]));
      t = dadd(t, dmul(b3, A2[i]));
      t = dadd(t, dmul(b1, id));
      W[i] = dadd(T[i], t);
    }
    mm4(A, W, U);
    mm4(A6, Z1, T);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      double id = (i % 5 == 0) ? 1.0 : 0.0;
      double t = dmul(b6, A6[i]);
      t = dadd(t, dmul(b4, A4[i]));
      t = dadd(t, dmul(b2, A2[i]));
      t = dadd(t, dmul(b0, id));
      V[i] = dadd(T[i], t);
    }
  } else {
    double A8[16], W[16];
    if (deg >= 5) mm4(A2, A2, A4);
    if (deg >= 7) mm4(A4, A2, A6);
    if (deg >= 9) mm4(A6, A2, A8);
    for (int i = 0; i < 16; ++i) {
      double id = (i % 5 == 0) ? 1.0 : 0.0;
      double w, v;
      if (deg == 3) {
        w = dmul(1., A2[i]);
        v = dmul(12., A2[i]);
        W[i] = dadd(w, dmul(60., id));
        V[i] = dadd(v, dmul(120., id));
      } else if (deg == 5) {
        w = dmul(1., A4[i]);
        w = dadd(w, dmul(420., A2[i]));
        v = dmul(30., A4[i]);
        v = dadd(v, dmul(3360., A2[i]));
        W[i] = dadd(w, dmul(15120., id));
        V[i] = dadd(v, dmul(30240., id));
      } else if (deg == 7) {
        w = dmul(1., A6[i]);
        w = dadd(w, dmul(1512., A4[i]));
        w = dadd(w, dmul(277200., A2[i]));
        v = dmul(56., A6[i]);
        v = dadd(v, dmul(25200., A4[i]));
        v = dadd(v, dmul(1995840., A2[i]));
        W[i] = dadd(w, dmul(8648640., id));
        V[i] = dadd(v, dmul(17297280., id));
      } else {
        w = dmul(1., A8[i]);
        w = dadd(w, dmul(3960., A6[i]));
        w = dadd(w, dmul(2162160., A4[i]));
        w = dadd(w, dmul(302702400., A2[i]));
        v = dmul(90., A8[i]);
        v = dadd(v, dmul(110880., A6[i]));
        v = dadd(v, dmul(30270240., A4[i]));
        v = dadd(v, dmul(2075673600., A2[i]));
        W[i] = dadd(w, dmul(8821612800., id));
        V[i] = dadd(v, dmul(17643225600., id));
      }
    }
    mm4(A, W, U);
  }
  double M[16], N[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    M[i] = dsub(V[i], U[i]);
    N[i] = dadd(V[i], U[i]);
  }
  solve4(M, N, E);
  for (int q = 0; q < s; ++q) {
    double T[16];
    mm4(E, E, T);
#pragma unroll
    for (int i = 0; i < 16; ++i) E[i] = T[i];
  }
}

// Q_ij = r_(ij) pi_j (12 r's row-major off-diagonal), diagonal = -row sum,
// normalised to unit mean rate -sum_i pi_i Q_ii = 1 (SURVEY Appendix A-2).
__device__ inline void build_q_nonrev(const double* r, const double* pi, double* Q) {
  int k = 0;
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j)
      if (i != j) Q[i * 4 + j] = dmul(r[k++], pi[j]);
  for (int i = 0; i < 4; ++i) {
    double s = 0.0;
    bool   first = true;
    for (int j = 0; j < 4; ++j) {
      if (j == i) continue;
      if (first) {
        s = Q[i * 4 + j];
        first = false;
      } else
        s = dadd(s, Q[i * 4 + j]);
    }
    Q[i * 4 + i] = -s;
  }
  double mu = dmul(pi[0], -Q[0]);
  mu = dadd(mu, dmul(pi[1], -Q[5]));
  mu = dadd(mu, dmul(pi[2], -Q[10]));
  mu = dadd(mu, dmul(pi[3], -Q[15]));
  for (int i = 0; i < 16; ++i) Q[i] = ddiv(Q[i], mu);
}

// ---------------------------------------------------------------------------
// Tip states are stored on the device as 4-bit CODES, a permutation of the
// 4-bit state masks chosen so that the unambiguous states A,C,G,T get codes
// 0..3 (they then hit distinct shared-memory banks in the tip tables).
// ---------------------------------------------------------------------------
__host__ __device__ __forceinline__ unsigned tip_mask_of_code(unsigned code) {
  // code: 0  1  2  3  4  5  6  7  8  9  10 11 12 13 14 15
  // mask: 1  2  4  8  3  5  6  7  9  10 11 12 13 14 15 0
  return (unsigned)((0x0FEDCBA976538421ULL >> (4 * code)) & 15ULL);
}
__host__ __device__ __forceinline__ unsigned tip_code_of_mask(unsigned mask) {
  // mask: 0  1  2  3  4  5  6  7  8  9  10 11 12 13 14 15
  // code: 15 0  1  4  2  5  6  7  3  8  9  10 11 12 13 14
  return (unsigned)((0xEDCBA9837652410FULL >> (4 * mask)) & 15ULL);
}

// ---------------------------------------------------------------------------
// pmat_expm_nonrev: one thread per (branch entry, rate category).
// Replaces corax_update_prob_matrices.  A pool slot holds, for one branch,
//   P : [cat][i*4+j (+2 pad)]   18*K doubles  (the transition matrices; the pad
//                               makes a category's row start 144 B apart so that the
//                               128-bit shared-memory reads of a warp's K categories
//                               fall into distinct banks)
//   T : [tip code][cat][i]      64*K doubles  (tip lookup table)
// T[code][k][i] = ((P_i0 c_0 + P_i1 c_1) + P_i2 c_2) + P_i3 c_3 with c the 0/1
// vector of the tip state: exactly the expression a tip child contributes to a
// CLV update, evaluated once per branch instead of once per site.
// The slot layout IS the shared-memory layout: the program kernel moves P or T
// with one bulk async copy.
// ---------------------------------------------------------------------------
constexpr int kPTabDoubles = 18;    // per category
constexpr int kTipTabDoubles = 64;  // per category
constexpr int kTabDoubles = 64;     // per category: the larger of the two
constexpr int kSlotDoubles = kPTabDoubles + kTipTabDoubles;  // per category

struct PmatEntry {
  unsigned slot;  // physical slot in the P-matrix pool
  unsigned pad;
  double   t;  // branch length
};

constexpr int kPmatInline = 16;
struct PmatArgs {
  const PmatEntry* entries;  // used when n > kPmatInline
  int              n;
  int              K;
  double           r[12];
  double           pi[4];
  double           pinv;
  double           rates[kMaxCats];
  double*          pool;
  PmatEntry        inl[kPmatInline];
};

#ifndef RDK_PROGRAM_KERNEL_ONLY
__global__ void __launch_bounds__(64) pmat_expm_nonrev_kernel(const __grid_constant__ PmatArgs a) {
  int tid = blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= a.n * a.K) return;
  int       e = tid / a.K, k = tid - e * a.K;
  PmatEntry ent = (a.n <= kPmatInline) ? a.inl[e] : a.entries[e];
  double    Q[16], A[16], E[16];
  double    r[12], pi[4];
  for (int i = 0; i < 12; ++i) r[i] = a.r[i];
  for (int i = 0; i < 4; ++i) pi[i] = a.pi[i];
  build_q_nonrev(r, pi, Q);
  double c = ddiv(dmul(a.rates[k], ent.t), dsub(1.0, a.pinv));
  for (int i = 0; i < 16; ++i) A[i] = dmul(Q[i], c);
  expm4(A, E);
  double* slot = a.pool + (size_t)ent.slot * a.K * kSlotDoubles;
  double* out = slot + (size_t)k * kPTabDoubles;
  for (int i = 0; i < 16; ++i) out[i] = E[i];
  out[16] = out[17] = 0.0;
  double* tab = slot + (size_t)a.K * kPTabDoubles;
  for (int i = 0; i < 4; ++i)
    for (unsigned code = 0; code < 16; ++code) {
      unsigned m = tip_mask_of_code(code);
      double   x = dmul(E[i * 4 + 0], (m & 1u) ? 1.0 : 0.0);
      x = dadd(x, dmul(E[i * 4 + 1], (m & 2u) ? 1.0 : 0.0));
      x = dadd(x, dmul(E[i * 4 + 2], (m & 4u) ? 1.0 : 0.0));
      x = dadd(x, dmul(E[i * 4 + 3], (m & 8u) ? 1.0 : 0.0));
      tab[((size_t)code * a.K + k) * 4 + i] = x;
    }
}

#endif  // RDK_PROGRAM_KERNEL_ONLY

// ---------------------------------------------------------------------------
// The likelihood program kernel.
//
// A "program" is a list of instructions executed in order for every
// (site, category) element.  Elements are independent of each other (the
// dependency between a parent CLV and its children is per site), so each warp
// owns a contiguous range of elements and walks the WHOLE program on it with
// no grid synchronisation: a full post-order traversal (n-1 CLV operations +
// the root log-likelihood), a root move, or an entire placement sweep is ONE
// launch.
//
// Thread mapping: element e = site*K + k; lane l of warp iteration `it` handles
// e = 32*it + l, so a warp access is 32 consecutive 32-byte (4 x fp64) vectors =
// 1 KiB contiguous per CLV.  Every thread carries E elements through each
// instruction.
//
// What a warp keeps between instructions is ONE CLV value per element in
// registers, `v` (rdk_lower.hpp): an instruction computes r = A(c1) o B(v),
// with A a mat-vec on the CLV c1 that was LOADED while the previous instruction
// computed, or a tip-table lookup, and B a mat-vec on v or a tip lookup.  A
// regular operation leaves r in v (and stores it if a later instruction or the
// caller reads it from memory); a placement evaluation (fEval) consumes r in
// registers and leaves v as it was, so that the directed CLV it was computed
// from is still there for the descent into the subtree.
//
// Tables.  The last warp of a CTA is the PRODUCER: it walks the program ahead of
// the other (consumer) warps and fills a ring of kDepth slots in shared memory,
// one slot per instruction = the 64-byte instruction itself + the two tables it
// reads (P: 18K doubles of an inner child's branch, T: 64K doubles of a tip
// child's branch), moved with cp.async.bulk and completed on the slot's `full`
// mbarrier; a consumer warp that has finished an instruction arrives on the
// slot's `empty` mbarrier.  The consumers of a CTA therefore drift up to kDepth
// instructions apart, no warp ever waits for a table it asked for itself, and
// there is no CTA-wide barrier after the prologue.
// ---------------------------------------------------------------------------
struct alignas(16) Instr {
  double*              parent;   // fWrite: where r is stored
  const void*          c1;       // tip row (fTip1) or the inner CLV A loads
  const void*          c2;       // tip row (fTip2); the CLV loaded into v beforehand (fLoadV2)
  unsigned*            pscale;   // fWriteS
  const unsigned*      c1scale;  // fCnt1
  const unsigned*      c2scale;  // fCnt2M
  const double*        P1;       // the table A reads (in its branch's pool slot)   -- producer only
  const double*        P2;       // the table B reads                               -- producer only
  unsigned             flags;
  unsigned             slot;     // eval slot (row of the partial-sum buffer)
  unsigned             pad[2];
};
static_assert(sizeof(Instr) == 80, "Instr layout");

constexpr int kProgInline = 8;
constexpr int kMaxChunks = 16;  // independent sub-programs one launch can run side by side
struct ProgArgs {
  const Instr*    prog;  // null: the program is inl[0..n_instr)
  int             n_instr;
  unsigned        nelem;    // sites * K on this shard
  unsigned        n_witer;  // warp iterations (32 elements each) THIS launch walks ...
  unsigned        it0;      // ... starting at this one (a shard is walked by one or two launches)
  const unsigned* weights;  // pattern weights [sites]
  double*         partials; // [slots][partial_stride], one value per warp iteration
  unsigned        partial_stride;
  double*         persite;  // optional, eval slot 0 only (the ROWS variant: every eval slot, see row_stride)
  unsigned        persite_unweighted;  // persite receives the values before the pattern weight
  double          pi[4];
  double          w[kMaxCats];
  // n_chunks > 1: the program is n_chunks INDEPENDENT sub-programs (chunk c = instructions
  // [chunk_off[c], chunk_off[c+1]) of prog); blockIdx.y selects the one a CTA walks, so a
  // small shard fills the device with (site range) x (chunk) warps instead of leaving a
  // handful of warps per SM to walk one long chain
  unsigned        n_chunks;
  unsigned        chunk_off[kMaxChunks + 1];
  Instr           inl[kProgInline];
  // the ROWS variant of the kernel (placement sweeps that capture per-pattern rows): eval slot s
  // stores its UNWEIGHTED values at persite + s * row_stride.  Last, so that the fields the other
  // variants read keep their offsets.
  size_t          row_stride;
};

// the table ring of one CTA
template <int K>
struct Ring {
  // 8 slots, fewer for K = 16 / 32 so that the ring stays at about 66 KB of shared memory (a slot
  // holds two K-sized tables); depths 4 / 8 / 16 measured the same on B200: the ring is not the
  // limiter (DESIGN.md section 5.1)
  static constexpr int      kDepth = K <= 8 ? 8 : (K == 16 ? 4 : 2);
  static constexpr int      kLogDepth = kDepth == 8 ? 3 : (kDepth == 4 ? 2 : 1);
  static constexpr unsigned kTabBytes = kTabDoubles * K * 8;      // one child's table (the larger kind)
  static constexpr unsigned kPBytes = kPTabDoubles * K * 8;       // P of an inner child
  static constexpr unsigned kInstrBytes = 128;                    // the instruction, padded
  static constexpr unsigned kSlotBytes = kInstrBytes + 2 * kTabBytes;
  static constexpr unsigned kSmemBytes = kDepth * kSlotBytes + 2 * kDepth * 8;
};

struct d4 {
  double v[4];
};

__device__ __forceinline__ d4 ld_clv(const void* base, unsigned e) {
  // one 256-bit load per element (sm_100 LDG.E.256): a warp access covers 1 KiB
  // contiguous with every 32-byte sector used by exactly one lane.  L2-coherent
  // (.cg): a CLV is read once per instruction, by one warp.
  const char* q = reinterpret_cast<const char*>(base) + (size_t)e * 32u;
  d4          r;
  asm volatile("ld.global.cg.v4.f64 {%0,%1,%2,%3}, [%4];\n"
               : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3])
               : "l"(q));
  return r;
}
__device__ __forceinline__ void st_clv(double* base, unsigned e, const d4& x) {
  char* q = reinterpret_cast<char*>(base) + (size_t)e * 32u;
  asm volatile("st.global.cg.v4.f64 [%0], {%1,%2,%3,%4};\n" ::"l"(q), "d"(x.v[0]), "d"(x.v[1]), "d"(x.v[2]),
               "d"(x.v[3])
               : "memory");
}

// ---- mbarrier + bulk async copy (one elected thread moves a whole table) ----
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
      "selp.u32 %0, 1, 0, P1;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// high word of a double as a signed integer: for the likelihood values (finite, >= 0, or a
// negative rounding residue) x < 2^-256  <=>  hi(x) < hi(2^-256), exactly (the low word of
// 2^-256 is zero) -- the underflow test then runs on the integer pipe, not the fp64 pipe
__device__ __forceinline__ int hi_word(double x) { return __double2hiint(x); }
constexpr int kScaleThresholdHi = (1023 - 256) << 20;

// back-off of the producer warp while its ring is full (200 / 1000 / 4000 ns measured the same on B200)
constexpr unsigned kProducerSleepNs = 200;

// ROWS: every evaluation stores its unweighted per-pattern values into the row of its eval slot
// (a compile-time variant, so that the instantiations without it compile to the code they had)
template <int K, int E, int MAXT, int MINB, bool ROWS = false>
__global__ void __launch_bounds__(MAXT, MINB) clv_program_kernel(const __grid_constant__ ProgArgs a) {
  static_assert(32 % K == 0, "K must divide the warp size");
  using R = Ring<K>;
  constexpr unsigned D = R::kDepth;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned long long* const s_full = reinterpret_cast<unsigned long long*>(smem_raw + D * R::kSlotBytes);
  unsigned long long* const s_empty = s_full + D;

  const unsigned tid = threadIdx.x;
  unsigned       lane;  // (volatile: kept in a register instead of being re-read from SR_TID in the loop)
  asm volatile("mov.u32 %0, %%laneid;\n" : "=r"(lane));
  const unsigned wib = tid >> 5;
  const unsigned n_cons = (blockDim.x >> 5) - 1u;  // consumer warps; warp n_cons is the producer

  const Instr* prog = a.prog;
  unsigned     n_instr = (unsigned)a.n_instr;
  const bool   inline_prog = a.prog == nullptr;  // <= kProgInline instructions, in the launch arguments
  if (a.n_chunks > 1) {
    prog += a.chunk_off[blockIdx.y];
    n_instr = a.chunk_off[blockIdx.y + 1] - a.chunk_off[blockIdx.y];
  }

  // the CTA's range of warp iterations, split evenly over its consumer warps; every warp of the
  // CTA runs the same number of passes (the ring is walked in lock step, kDepth apart at most)
  const unsigned c_begin = a.it0 + (unsigned)(((unsigned long long)a.n_witer * blockIdx.x) / gridDim.x);
  const unsigned c_end = a.it0 + (unsigned)(((unsigned long long)a.n_witer * (blockIdx.x + 1)) / gridDim.x);
  const unsigned c_len = c_end - c_begin;
  const unsigned passes = ((c_len + n_cons - 1) / n_cons + E - 1) / E;
  const unsigned total = passes * n_instr;  // instructions this CTA's ring carries

  if (tid == 0) {
#pragma unroll
    for (unsigned s = 0; s < D; ++s) {
      mbar_init(&s_full[s], 1);
      mbar_init(&s_empty[s], n_cons);
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();

  if (wib == n_cons) {
    // ------------------------------- producer warp -------------------------------------
    // lane l takes instructions j = base + l: it reads its instruction from global memory (or
    // the launch arguments) ahead of time, then the lanes fill their slots in order
    for (unsigned base = 0; base < total; base += 32u) {
      const unsigned j = base + lane;
      int4           w0 = make_int4(0, 0, 0, 0), w1 = w0, w2 = w0, w3 = w0, w4 = w0;
      if (j < total) {
        const unsigned idx = j % n_instr;
        const int4*    src = reinterpret_cast<const int4*>(inline_prog ? &a.inl[idx] : &prog[idx]);
        w0 = src[0];
        w1 = src[1];
        w2 = src[2];
        w3 = src[3];
        w4 = src[4];
      }
      const unsigned cnt = min(32u, total - base);
      for (unsigned t = 0; t < cnt; ++t) {
        if (lane == t) {
          const unsigned s = j & (D - 1u);
          // the producer runs kDepth instructions ahead: it is nearly always waiting here, and a
          // busy wait would take issue slots from the consumer warps of its sub-partition
          while (!mbar_try_wait(&s_empty[s], ((j >> R::kLogDepth) & 1u) ^ 1u)) __nanosleep(kProducerSleepNs);
          unsigned char* slot = smem_raw + s * R::kSlotBytes;
          int4*          dst = reinterpret_cast<int4*>(slot);
          dst[0] = w0;
          dst[1] = w1;
          dst[2] = w2;
          dst[3] = w3;
          dst[4] = w4;
          const unsigned fl = (unsigned)w4.x;
          unsigned       b1 = 0, b2 = 0;
          if (!(fl & (fLoadV | fNop))) {
            b1 = (fl & fTip1) ? R::kTabBytes : R::kPBytes;
            b2 = (fl & fTip2) ? R::kTabBytes : R::kPBytes;
          }
          // the arrive releases the plain stores above to the consumers that acquire the barrier
          mbar_expect_tx(&s_full[s], b1 + b2);
          if (b1) {
            const unsigned long long p1 = ((unsigned long long)(unsigned)w3.y << 32) | (unsigned)w3.x;
            bulk_g2s(slot + R::kInstrBytes, reinterpret_cast<const void*>(p1), b1, &s_full[s]);
          }
          if (b2) {
            const unsigned long long p2 = ((unsigned long long)(unsigned)w3.w << 32) | (unsigned)w3.z;
            bulk_g2s(slot + R::kInstrBytes + R::kTabBytes, reinterpret_cast<const void*>(p2), b2, &s_full[s]);
          }
        }
        __syncwarp();
      }
    }
    return;
  }

  // --------------------------------- consumer warps --------------------------------------
  constexpr unsigned SPW = 32 / K;  // sites per warp iteration
  const unsigned     k = lane % K;
  const unsigned     sl = lane / K;
  const unsigned     lane0 = lane - k;  // the k == 0 lane of this lane's site
  unsigned           gmask = 0;         // the K lanes that hold this lane's site
#pragma unroll
  for (int j = 0; j < K; ++j) gmask |= 1u << (j + lane0);

  const unsigned it_begin = c_begin + (unsigned)(((unsigned long long)c_len * wib) / n_cons);
  const unsigned it_end = c_begin + (unsigned)(((unsigned long long)c_len * (wib + 1)) / n_cons);
  const unsigned last_site = a.nelem / K - 1;

  auto slot_of = [&](unsigned j) -> const unsigned char* { return smem_raw + (j & (D - 1u)) * R::kSlotBytes; };
  auto wait_full = [&](unsigned j) { mbar_wait(&s_full[j & (D - 1u)], (j >> R::kLogDepth) & 1u); };
  auto release = [&](unsigned j) {
    __syncwarp();
    if (lane == 0) mbar_arrive(&s_empty[j & (D - 1u)]);
  };

  d4       v[E];     // the CLV value carried from instruction to instruction
  unsigned vcnt[E];  // its scaler counts
  d4       c1r[E];   // the loaded child-1 CLV of the instruction about to run
  unsigned m1[E], m2n[E], cnt1[E];  // its tip codes / child-1 scaler counts
#pragma unroll
  for (int u = 0; u < E; ++u) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[u].v[i] = c1r[u].v[i] = 0.0;
    vcnt[u] = cnt1[u] = 0;
    m1[u] = m2n[u] = 15u;  // code 15: all-zero table row
  }

  unsigned jg = 0;  // position in the CTA's instruction stream (all passes)
  for (unsigned pass = 0; pass < passes; ++pass) {
    if (!(it_begin + pass * E < it_end)) {
      // no iteration of its own in this pass: keep the ring protocol going
      for (unsigned ii = 0; ii < n_instr; ++ii, ++jg) {
        wait_full(jg);
        release(jg);
      }
      continue;
    }
    // slots without an iteration of their own (the warp's last pass) redundantly recompute the
    // warp's last iteration and store the identical values (same thread: no race); lanes
    // without a site of their own (tail of the partition) do the same with the last site
    unsigned it[E], e[E], site[E], wgt[E];
#pragma unroll
    for (int u = 0; u < E; ++u) {
      const unsigned i0 = it_begin + pass * E + u;
      it[u] = i0 < it_end ? i0 : it_end - 1;
      unsigned st = it[u] * SPW + sl;
      if (st > last_site) st = last_site;
      site[u] = st;
      e[u] = st * K + k;
      wgt[u] = __ldg(a.weights + st);
    }

    // issue the global loads of one instruction's operands
    auto load_operands = [&](const Instr& in) __attribute__((always_inline)) {
      const unsigned fl = in.flags;
      if (fl & fTip1) {
        const unsigned char* t = reinterpret_cast<const unsigned char*>(in.c1);
#pragma unroll
        for (int u = 0; u < E; ++u) m1[u] = __ldg(t + site[u]);
      } else if (!(fl & fNop)) {
        const void* g = in.c1;
#pragma unroll
        for (int u = 0; u < E; ++u) c1r[u] = ld_clv(g, e[u]);
      }
      if (fl & fTip2) {
        const unsigned char* t = reinterpret_cast<const unsigned char*>(in.c2);
#pragma unroll
        for (int u = 0; u < E; ++u) m2n[u] = __ldg(t + site[u]);
      }
#pragma unroll
      for (int u = 0; u < E; ++u) cnt1[u] = 0;
      if (fl & fCnt1) {
        const unsigned* s1 = in.c1scale;
#pragma unroll
        for (int u = 0; u < E; ++u) cnt1[u] = __ldcg(s1 + site[u]);
      }
    };

    // fLoadV2: v := the CLV child 2 of `in` (issued at the very end of the previous instruction:
    // v is dead by then, and the previous instruction's stores precede it in program order)
    auto load_v = [&](const Instr& in) __attribute__((always_inline)) {
      const unsigned fl = in.flags;
      if (fl & fLoadV2) {
        const void* g = in.c2;
#pragma unroll
        for (int u = 0; u < E; ++u) v[u] = ld_clv(g, e[u]);
#pragma unroll
        for (int u = 0; u < E; ++u) vcnt[u] = 0;
        if (fl & fCnt2M) {
          const unsigned* s2 = in.c2scale;
#pragma unroll
          for (int u = 0; u < E; ++u) vcnt[u] = __ldcg(s2 + site[u]);
        }
      }
    };

    // 2^256 rescaling of the values of one instruction (SURVEY A-3): a site is rescaled when all
    // its K*4 values are below 2^-256
    auto rescale = [&](d4(&r)[E], unsigned(&cnt)[E]) __attribute__((always_inline)) {
      // the test runs on the integer pipe (hi_word); a ballot per slot tells every lane which
      // sites of the warp iteration are all-small.  The multiplication itself is rare: it sits
      // behind a WARP-UNIFORM branch (any site of any slot), so the common case costs no
      // predicated fp64 work at all.
      int mx[E], mn = 0x7fffffff;
#pragma unroll
      for (int u = 0; u < E; ++u) {
        mx[u] = max(max(hi_word(r[u].v[0]), hi_word(r[u].v[1])), max(hi_word(r[u].v[2]), hi_word(r[u].v[3])));
        mn = min(mn, mx[u]);
      }
      if (!__any_sync(0xffffffffu, mn < kScaleThresholdHi)) return;  // no (site, category) of the warp is all-small
      unsigned m[E], any = 0;
#pragma unroll
      for (int u = 0; u < E; ++u) {
        m[u] = __ballot_sync(0xffffffffu, mx[u] < kScaleThresholdHi);
        unsigned t = m[u];  // bit at a site's first lane <=> all K lanes of the site are set
#pragma unroll
        for (int sft = 1; sft < K; sft <<= 1) t &= t >> sft;
        any |= t;
      }
      constexpr unsigned kSiteBase = K == 1 ? 0xffffffffu : (K == 2 ? 0x55555555u : (K == 4 ? 0x11111111u : (K == 8 ? 0x01010101u : (K == 16 ? 0x00010001u : 1u))));
      if (any & kSiteBase) {
#pragma unroll
        for (int u = 0; u < E; ++u) {
          if ((m[u] & gmask) == gmask) {
#pragma unroll
            for (int i = 0; i < 4; ++i) r[u].v[i] = dmul(r[u].v[i], RDK_SCALE_FACTOR);
            cnt[u] += 1;
          }
        }
      }
    };

    // root log-likelihood of the values r (SURVEY A-4) into eval slot in.slot
    auto evaluate = [&](const Instr& in, const unsigned fl, const d4(&r)[E], const unsigned(&cnt)[E])
                        __attribute__((always_inline)) {
      // every lane of a site gathers the K category terms in category order
      double term[E];
#pragma unroll
      for (int u = 0; u < E; ++u) {
        double t = dmul(a.pi[0], r[u].v[0]);
        t = dfma(a.pi[1], r[u].v[1], t);
        t = dfma(a.pi[2], r[u].v[2], t);
        t = dfma(a.pi[3], r[u].v[3], t);
        double tm = dmul(a.w[0], __shfl_sync(0xffffffffu, t, lane0));
#pragma unroll
        for (int kk = 1; kk < K; ++kk) {
          double tk = __shfl_sync(0xffffffffu, t, lane0 + kk);
          tm = dfma(a.w[kk], tk, tm);
        }
        term[u] = tm;
      }
      const unsigned eslot = in.slot;
      if constexpr (E <= K) {
        // the K lanes of a site hold the same term: lane k takes the logarithm of the
        // site of slot u = k, so that ONE pass through rd_log serves all E slots
        double   x = term[0];
        unsigned cn = cnt[0], st = site[0], iw = it[0], wg = wgt[0];
#pragma unroll
        for (int u = 1; u < E; ++u)
          if (k == (unsigned)u) {
            x = term[u];
            cn = cnt[u];
            st = site[u];
            iw = it[u];
            wg = wgt[u];
          }
        double l = 0.0;
        if (k < (unsigned)E && iw * SPW + sl <= last_site) {
          l = rd_log(x);
          if (fl & fEvalScaler) l = dadd(l, dmul((double)cn, RDK_LOG_SCALE_THRESHOLD));
          const double lw = dmul(l, (double)wg);
          if constexpr (ROWS) a.persite[(size_t)eslot * a.row_stride + st] = l;
          else if (a.persite && eslot == 0) a.persite[st] = a.persite_unweighted ? l : lw;
          l = lw;
        }
        // canonical tree over the 32/K sites of a warp iteration (the lanes of equal k)
#pragma unroll
        for (int off2 = 1; off2 < (int)SPW; off2 <<= 1) l = dadd(l, __shfl_xor_sync(0xffffffffu, l, off2 * K));
        if (sl == 0 && k < (unsigned)E) a.partials[(size_t)eslot * a.partial_stride + iw] = l;
      } else {
#pragma unroll
        for (int u = 0; u < E; ++u) {
          double l = 0.0;
          if (k == 0 && it[u] * SPW + sl <= last_site) {
            l = rd_log(term[u]);
            if (fl & fEvalScaler) l = dadd(l, dmul((double)cnt[u], RDK_LOG_SCALE_THRESHOLD));
            const double lw = dmul(l, (double)wgt[u]);
            if constexpr (ROWS) a.persite[(size_t)eslot * a.row_stride + site[u]] = l;
            else if (a.persite && eslot == 0) a.persite[site[u]] = a.persite_unweighted ? l : lw;
            l = lw;
          }
#pragma unroll
          for (int off2 = 1; off2 < (int)SPW; off2 <<= 1) l = dadd(l, __shfl_xor_sync(0xffffffffu, l, off2 * K));
          if (lane == 0) a.partials[(size_t)eslot * a.partial_stride + it[u]] = l;
        }
      }
    };

    // pipeline prologue: the operands of the pass's first instruction
    wait_full(jg);
    load_operands(*reinterpret_cast<const Instr*>(slot_of(jg)));
    load_v(*reinterpret_cast<const Instr*>(slot_of(jg)));

    for (unsigned ii = 0; ii < n_instr; ++ii, ++jg) {
      const unsigned char* slot = slot_of(jg);
      const Instr&         in = *reinterpret_cast<const Instr*>(slot);
      const unsigned       fl = in.flags;
      const unsigned char* tab1 = slot + R::kInstrBytes;
      const unsigned char* tab2 = tab1 + R::kTabBytes;
      const bool           main_op = !(fl & (fLoadV | fNop));

      d4       y[E];     // B(child 2), then (placement evaluations) r
      unsigned cnt[E];   // scaler counts of r
      unsigned m2c[E];   // this instruction's child-2 tip codes (m2n is reloaded below)
#pragma unroll
      for (int u = 0; u < E; ++u) {
        m2c[u] = m2n[u];
        cnt[u] = cnt1[u] + ((fl & fCnt2V) ? vcnt[u] : 0u);
      }

      // ---- phase 1: y = A(child 1); c1r / m1 are dead afterwards ---------------------------
      // child-1 term first: its operands are dead before the second mat-vec, so the next
      // instruction's loads fly longer; the other order measured 8.69 vs 8.46 ms on B200
      // (DESIGN.md section 5.1)
      if (main_op) {
        if (fl & fTip1) {
#pragma unroll
          for (int u = 0; u < E; ++u) {
            const double2* t = reinterpret_cast<const double2*>(tab1 + (m1[u] * K + k) * 32u);
            const double2  lo = t[0], hi = t[1];
            y[u].v[0] = lo.x;
            y[u].v[1] = lo.y;
            y[u].v[2] = hi.x;
            y[u].v[3] = hi.y;
          }
        } else {
          const double2* p = reinterpret_cast<const double2*>(tab1 + k * (kPTabDoubles * 8));
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const double2 p01 = p[i * 2], p23 = p[i * 2 + 1];
#pragma unroll
            for (int u = 0; u < E; ++u) {
              double s = dmul(p01.x, c1r[u].v[0]);
              s = dfma(p01.y, c1r[u].v[1], s);
              s = dfma(p23.x, c1r[u].v[2], s);
              s = dfma(p23.y, c1r[u].v[3], s);
              y[u].v[i] = s;
            }
          }
        }
      } else if (fl & fLoadV) {
#pragma unroll
        for (int u = 0; u < E; ++u) {
          v[u] = c1r[u];
          vcnt[u] = cnt1[u];
        }
      }

      // ---- the operands of the next instruction of this pass (c1r, m1, cnt1 are dead now) ---
      if (ii + 1 < n_instr) {
        wait_full(jg + 1);
        load_operands(*reinterpret_cast<const Instr*>(slot_of(jg + 1)));
      }

      // ---- phase 2: r = y o B(child 2), in place ------------------------------------------
      const bool keep_v = (fl & fEval) != 0;
      if (main_op) {
        if (fl & fTip2) {
#pragma unroll
          for (int u = 0; u < E; ++u) {
            const double2* t = reinterpret_cast<const double2*>(tab2 + (m2c[u] * K + k) * 32u);
            const double2  lo = t[0], hi = t[1];
            y[u].v[0] = dmul(y[u].v[0], lo.x);
            y[u].v[1] = dmul(y[u].v[1], lo.y);
            y[u].v[2] = dmul(y[u].v[2], hi.x);
            y[u].v[3] = dmul(y[u].v[3], hi.y);
          }
        } else {
          const double2* p = reinterpret_cast<const double2*>(tab2 + k * (kPTabDoubles * 8));
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const double2 p01 = p[i * 2], p23 = p[i * 2 + 1];
#pragma unroll
            for (int u = 0; u < E; ++u) {
              double s = dmul(p01.x, v[u].v[0]);
              s = dfma(p01.y, v[u].v[1], s);
              s = dfma(p23.x, v[u].v[2], s);
              s = dfma(p23.y, v[u].v[3], s);
              y[u].v[i] = dmul(y[u].v[i], s);
            }
          }
        }
      }

      // ---- rescale, store, evaluate -----------------------------------------------------
      if (main_op) {
        if (fl & fScale) rescale(y, cnt);
        if (keep_v) {
          evaluate(in, fl, y, cnt);
        } else {
          if (fl & fWrite) {
            double* par = in.parent;
#pragma unroll
            for (int u = 0; u < E; ++u) st_clv(par, e[u], y[u]);
          }
          if ((fl & fWriteS) && k == 0) {
            unsigned* ps = in.pscale;
#pragma unroll
            for (int u = 0; u < E; ++u) __stcg(ps + site[u], cnt[u]);
          }
#pragma unroll
          for (int u = 0; u < E; ++u) {
            v[u] = y[u];
            vcnt[u] = cnt[u];
          }
        }
      }
      if (fl & fEvalV) evaluate(in, fl, v, vcnt);
      if (ii + 1 < n_instr) load_v(*reinterpret_cast<const Instr*>(slot_of(jg + 1)));
      release(jg);
    }
  }
}

// Launch of the program kernel for K rate categories: one explicit specialisation per K,
// each in its own translation unit (rdk_program_inst.cu).  `threads` counts the producer warp.
// Returns the CUDA status of the launch configuration (the launch itself is checked by the
// caller with cudaGetLastError).
// rows != 0 launches the ROWS variant (ProgArgs::row_stride).
template <int K>
cudaError_t launch_program(const ProgArgs& a, int grid, int threads, int E, bool rows, cudaStream_t st);
template <> cudaError_t launch_program<1>(const ProgArgs&, int, int, int, bool, cudaStream_t);
template <> cudaError_t launch_program<2>(const ProgArgs&, int, int, int, bool, cudaStream_t);
template <> cudaError_t launch_program<4>(const ProgArgs&, int, int, int, bool, cudaStream_t);
template <> cudaError_t launch_program<8>(const ProgArgs&, int, int, int, bool, cudaStream_t);
template <> cudaError_t launch_program<16>(const ProgArgs&, int, int, int, bool, cudaStream_t);
template <> cudaError_t launch_program<32>(const ProgArgs&, int, int, int, bool, cudaStream_t);
// the launch shapes the kernel is compiled for, per elements-per-thread E: threads per CTA
// (producer warp included) and CTAs per SM
struct LaunchShape {
  int threads, ctas_per_sm;
};
constexpr LaunchShape launch_shape(int E) {
  return E == 4 ? LaunchShape{384, 1} : (E == 3 ? LaunchShape{512, 1} : (E == 2 ? LaunchShape{320, 2} : LaunchShape{512, 2}));
}

#ifndef RDK_PROGRAM_KERNEL_ONLY
// ---------------------------------------------------------------------------
// Canonical reduction: balanced binary tree over contiguous halves of the
// zero-padded (to a power of two) GLOBAL site index space.  The program kernel
// produced the tree nodes that cover one warp iteration (32/K sites); this
// kernel continues the same tree.
//   in : [slots][in_stride], n_in valid leaves per slot, leaf index offset
//        `leaf0` within the padded tree (sharded partitions)
//   out: [slots][out_stride]; out[slot][b] = tree node over leaves
//        [b*span, (b+1)*span) (span = power of two), b < n_nodes
// A node is reduced by R = min(span, 256) threads (each folds span / R consecutive
// leaves with the same tree first); a block holds 256 / R nodes, blockIdx.y = slot.
// With span >= n_in and one node per slot this yields the final sum.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) tree_reduce_kernel(const double* __restrict__ in,
                                                           unsigned in_stride, unsigned n_in,
                                                           unsigned span, unsigned n_nodes,
                                                           double* __restrict__ out,
                                                           unsigned out_stride, unsigned out_offset) {
  __shared__ double sm[256];
  const unsigned R = span < 256u ? span : 256u;  // power of two
  const unsigned L = span / R;                   // power of two
  const unsigned slot = blockIdx.y, t = threadIdx.x;
  const unsigned b = blockIdx.x * (256u / R) + t / R;  // the node this thread works on
  const unsigned tr = t % R;
  const double*  p = in + (size_t)slot * in_stride;
  double         res = 0.0;
  if (b < n_nodes) {
    const unsigned long long base = (unsigned long long)b * span + (unsigned long long)tr * L;
    if (base < n_in) {
      double st[32];
      int    top = 0;
      for (unsigned i = 0; i < L; ++i) {
        unsigned long long idx = base + i;
        double             s = idx < n_in ? p[idx] : 0.0;
        for (unsigned j = i; j & 1u; j >>= 1) s = dadd(st[--top], s);
        st[top++] = s;
      }
      res = st[0];
    }
  }
  sm[t] = res;
  __syncthreads();
  for (unsigned w = 1; w < R; w <<= 1) {
    if ((tr % (2 * w)) == 0) sm[t] = dadd(sm[t], sm[t + w]);
    __syncthreads();
  }
  if (tr == 0 && b < n_nodes) out[(size_t)slot * out_stride + out_offset + b] = sm[0 + t];
}

// ---------------------------------------------------------------------------
// Weighted histogram of tip state masks (exact integer arithmetic), the input
// of the empirical base frequencies (corax_msa_empirical_frequencies).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) tip_hist_kernel(const unsigned char* __restrict__ tips,
                                                        size_t tip_stride, unsigned ntips,
                                                        unsigned sites,
                                                        const unsigned* __restrict__ weights,
                                                        unsigned long long* __restrict__ hist) {
  __shared__ unsigned long long sh[16];
  if (threadIdx.x < 16) sh[threadIdx.x] = 0;
  __syncthreads();
  unsigned long long local[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) local[i] = 0;
  const size_t total = (size_t)ntips * sites;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    unsigned tip = (unsigned)(idx / sites), s = (unsigned)(idx - (size_t)tip * sites);
    unsigned m = tip_mask_of_code(tips[(size_t)tip * tip_stride + s] & 15u);
    unsigned w = weights[s];
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (m == (unsigned)i) local[i] += w;
  }
#pragma unroll
  for (int i = 0; i < 16; ++i)
    if (local[i]) atomicAdd(&sh[i], local[i]);
  __syncthreads();
  if (threadIdx.x < 16 && sh[threadIdx.x]) atomicAdd(&hist[threadIdx.x], sh[threadIdx.x]);
}

// expand a tip's byte masks to a full 0/1 CLV (rdk_get_clv on a tip index)
__global__ void tip_expand_kernel(const unsigned char* __restrict__ tip, unsigned sites, int K,
                                  double* __restrict__ out) {
  size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (size_t)sites * K) return;
  unsigned m = tip_mask_of_code(tip[e / K] & 15u);
  for (int j = 0; j < 4; ++j) out[e * 4 + j] = ((m >> j) & 1u) ? 1.0 : 0.0;
}

#endif  // RDK_PROGRAM_KERNEL_ONLY

}  // namespace rdk
