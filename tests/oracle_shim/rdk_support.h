/*
 * tests/oracle_shim/rdk_support.h -- TEST INFRASTRUCTURE.
 *
 * The root placement support entries of include/rdk.h (rdk_partition_set_site_lnl_rows,
 * rdk_compute_root_loglikelihood_row, rdk_partition_get_site_lnl_rows, rdk_rell_support)
 * restated over the CPU oracle with plain loops and __int128, so that the oracle-backed host
 * (tests/_build/librd_host_oracle.so) runs model_t::placement_support on a machine without a
 * GPU and the parity tests compare the CUDA engine with it.  Included by the host sources only
 * when they are compiled against the oracle (RD_BACKEND_ORACLE).  Never part of the product.
 */
#ifndef RDK_SUPPORT_ORACLE_H_
#define RDK_SUPPORT_ORACLE_H_
#include "rdk.h"

#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <vector>

#ifndef RDK_ERROR_PARAM
#define RDK_ERROR_PARAM 1
#endif

typedef struct rdk_rell_out_t {
  unsigned int        replicate_tile;
  int                 exponent;
  unsigned int        best;
  unsigned int        bad_row;
  double             *lnl_fixed;
  unsigned long long *o_lo;
  long long          *o_hi;
  unsigned int       *bp_count;
  unsigned int       *kh_count;
  unsigned int       *sh_count;
  double              ms[4];
  unsigned long long  device_bytes;
} rdk_rell_out_t;

namespace rdk_support_oracle {
typedef __int128          i128;
typedef unsigned __int128 u128;

inline std::map<const rdo_partition_t *, std::vector<double>> &rows_of() {
  static std::map<const rdo_partition_t *, std::vector<double>> rows;
  return rows;
}

inline int refuse(const char *what) {
  rdo_errno = RDK_ERROR_PARAM;
  snprintf(rdo_errmsg, sizeof(rdo_errmsg), "%s", what);
  return RDO_FAILURE;
}

inline void philox4x64_10(unsigned long long c[4], unsigned long long k0, unsigned long long k1) {
  for (int round = 0; round < 10; ++round) {
    if (round) {
      k0 += 0x9E3779B97F4A7C15ull;
      k1 += 0xBB67AE8584CAA73Bull;
    }
    const u128 p0 = (u128)0xD2E7470EE14C6C93ull * c[0], p1 = (u128)0xCA5A826395121157ull * c[2];
    const unsigned long long n0 = (unsigned long long)(p1 >> 64) ^ c[1] ^ k0;
    const unsigned long long n2 = (unsigned long long)(p0 >> 64) ^ c[3] ^ k1;
    c[0] = n0;
    c[1] = (unsigned long long)p1;
    c[2] = n2;
    c[3] = (unsigned long long)p0;
  }
}
}  // namespace rdk_support_oracle

static inline int rdk_partition_set_site_lnl_rows(rdo_partition_t *p, unsigned int rows) {
  auto &all = rdk_support_oracle::rows_of();
  if (rows == 0)
    all.erase(p);
  else
    all[p].assign((size_t)rows * p->sites, 0.0);
  return RDO_SUCCESS;
}

/* the unweighted values are those of the same evaluation with every pattern weight 1 (l * 1 == l) */
static inline double rdk_compute_root_loglikelihood_row(rdo_partition_t *p, unsigned int clv_index, int scaler_index,
                                                        unsigned int row) {
  auto &all = rdk_support_oracle::rows_of();
  auto  it = all.find(p);
  if (it == all.end() || (size_t)(row + 1) * p->sites > it->second.size()) {
    rdk_support_oracle::refuse("site row out of range");
    return NAN;
  }
  std::vector<unsigned int> freqs(p->rate_cats, 0u), keep(p->pattern_weights, p->pattern_weights + p->sites);
  for (unsigned s = 0; s < p->sites; ++s) p->pattern_weights[s] = 1;
  rdo_compute_root_loglikelihood(p, clv_index, scaler_index, freqs.data(), it->second.data() + (size_t)row * p->sites);
  memcpy(p->pattern_weights, keep.data(), sizeof(unsigned) * p->sites);
  return rdo_compute_root_loglikelihood(p, clv_index, scaler_index, freqs.data(), nullptr);
}

static inline int rdk_partition_get_site_lnl_rows(rdo_partition_t *p, unsigned int first, unsigned int count,
                                                  double *out) {
  auto &all = rdk_support_oracle::rows_of();
  auto  it = all.find(p);
  if (it == all.end() || (size_t)(first + count) * p->sites > it->second.size())
    return rdk_support_oracle::refuse("site rows out of range");
  memcpy(out, it->second.data() + (size_t)first * p->sites, sizeof(double) * count * p->sites);
  return RDO_SUCCESS;
}

/* the definition of include/rdk.h, item by item */
static inline int rdk_rell_support(rdo_partition_t *const *parts, unsigned int n, const unsigned int *global_index,
                                   unsigned int rows, unsigned long long replicates, unsigned long long seed,
                                   rdk_rell_out_t *out) {
  using namespace rdk_support_oracle;
  out->bad_row = ~0u;
  out->device_bytes = 0;
  if (n == 0 || rows == 0) return refuse("rdk_rell_support: no partitions or no rows");
  if (replicates == 0 || replicates > (1ull << 20)) return refuse("rdk_rell_support: replicates must be in [1, 2^20]");
  const unsigned            B = (unsigned)replicates;
  std::vector<const double *> L(n);
  double                    M = 0;
  for (unsigned g = 0; g < n; ++g) {
    auto it = rows_of().find(parts[g]);
    if (it == rows_of().end() || it->second.size() < (size_t)rows * parts[g]->sites)
      return refuse("rdk_rell_support: a partition holds fewer rows than asked");
    L[g] = it->second.data();
    for (unsigned r = 0; r < rows; ++r)
      for (unsigned s = 0; s < parts[g]->sites; ++s) {
        const double v = L[g][(size_t)r * parts[g]->sites + s];
        if (!std::isfinite(v)) {
          if (r < out->bad_row) out->bad_row = r;
        } else if (std::fabs(v) > M) {
          M = std::fabs(v);
        }
      }
  }
  if (out->bad_row != ~0u) {
    rdo_errno = RDK_ERROR_PARAM;
    snprintf(rdo_errmsg, sizeof(rdo_errmsg), "record %u has a site of likelihood 0 (non-finite log-likelihood)",
             out->bad_row);
    return RDO_FAILURE;
  }
  int x = 0;
  if (M > 0) frexp(M, &x);
  const int e = M > 0 ? 52 - x : 0;
  out->exponent = e;
  std::vector<i128> Z((size_t)B * rows, 0), O(rows, 0);
  for (unsigned g = 0; g < n; ++g) {
    const unsigned                  P = parts[g]->sites;
    const unsigned long long        gi = global_index ? global_index[g] : g;
    std::vector<long long>          q((size_t)rows * P);
    std::vector<unsigned long long> cumw(P + 1, 0);
    for (size_t i = 0; i < q.size(); ++i) q[i] = llrint(ldexp(L[g][i], e));
    for (unsigned p = 0; p < P; ++p) cumw[p + 1] = cumw[p] + parts[g]->pattern_weights[p];
    const unsigned long long N = cumw[P];
    for (unsigned r = 0; r < rows; ++r)
      for (unsigned p = 0; p < P; ++p) O[r] += (i128)parts[g]->pattern_weights[p] * q[(size_t)r * P + p];
    std::vector<unsigned> c(P);
    for (unsigned b = 0; b < B; ++b) {
      std::fill(c.begin(), c.end(), 0u);
      for (unsigned long long j4 = 0; j4 * 4 < N; ++j4) {
        unsigned long long xs[4] = {j4 + 1, 0, 0, 0};
        philox4x64_10(xs, seed, (gi << 32) | b);
        for (unsigned u = 0; u < 4 && j4 * 4 + u < N; ++u) {
          const unsigned long long site = (unsigned long long)(((u128)xs[u] * N) >> 64);
          unsigned                 lo = 0, hi = P;
          while (hi - lo > 1) {
            const unsigned mid = (lo + hi) / 2;
            if (cumw[mid] <= site)
              lo = mid;
            else
              hi = mid;
          }
          c[lo]++;
        }
      }
      for (unsigned r = 0; r < rows; ++r) {
        i128 s = 0;
        for (unsigned p = 0; p < P; ++p) s += (i128)c[p] * q[(size_t)r * P + p];
        Z[(size_t)b * rows + r] += s;
      }
    }
  }
  unsigned best = 0;
  for (unsigned r = 1; r < rows; ++r)
    if (O[r] > O[best]) best = r;
  out->best = best;
  std::vector<i128> colsum(rows, 0);
  for (unsigned b = 0; b < B; ++b)
    for (unsigned r = 0; r < rows; ++r) colsum[r] += Z[(size_t)b * rows + r];
  for (unsigned r = 0; r < rows; ++r) out->bp_count[r] = out->kh_count[r] = out->sh_count[r] = 0;
  const i128 Bi = B;
  for (unsigned b = 0; b < B; ++b) {
    const i128 *z = &Z[(size_t)b * rows];
    unsigned    top = 0;
    i128        mt = Bi * z[0] - colsum[0];
    for (unsigned r = 1; r < rows; ++r) {
      if (z[r] > z[top]) top = r;
      const i128 t = Bi * z[r] - colsum[r];
      if (t > mt) mt = t;
    }
    out->bp_count[top]++;
    for (unsigned r = 0; r < rows; ++r) {
      const i128 d = z[best] - z[r], sum_d = colsum[best] - colsum[r], delta = O[best] - O[r];
      if (Bi * d - sum_d >= Bi * delta) out->kh_count[r]++;
      if (mt - (Bi * z[r] - colsum[r]) >= Bi * delta) out->sh_count[r]++;
    }
  }
  for (unsigned r = 0; r < rows; ++r) {
    out->lnl_fixed[r] = ldexp((double)O[r], -e);
    if (out->o_lo) out->o_lo[r] = (unsigned long long)(u128)O[r];
    if (out->o_hi) out->o_hi[r] = (long long)(O[r] >> 64);
  }
  for (double &t : out->ms) t = 0;
  return RDO_SUCCESS;
}
#endif
