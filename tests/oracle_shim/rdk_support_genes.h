/*
 * tests/oracle_shim/rdk_support_genes.h -- TEST INFRASTRUCTURE.
 *
 * rdk_rell_support_genes of include/rdk.h (gene and gene-then-site resampling, DESIGN.md section 10
 * items 11-14) restated over the CPU oracle with plain loops and __int128, next to rdk_rell_support in
 * rdk_support.h.  Included by the host sources only when they are compiled against the oracle
 * (RD_BACKEND_ORACLE).  Never part of the product.
 */
#ifndef RDK_SUPPORT_GENES_ORACLE_H_
#define RDK_SUPPORT_GENES_ORACLE_H_
#include "rdk_support.h"

#define RDK_RELL_GENE      1u
#define RDK_RELL_GENE_SITE 2u
typedef struct rdk_rell_gene_out_t {
  unsigned int        sampling;
  double             *partition_lnl_fixed;
  unsigned long long *o_lo;
  long long          *o_hi;
  double              draws_ms;
} rdk_rell_gene_out_t;

/* the definition of include/rdk.h: items 1-5 with items 11-14's replicates */
static inline int rdk_rell_support_genes(rdo_partition_t *const *parts, unsigned int n,
                                         const unsigned int *global_index, unsigned int rows,
                                         unsigned long long replicates, unsigned long long seed, rdk_rell_out_t *out,
                                         rdk_rell_gene_out_t *genes) {
  using namespace rdk_support_oracle;
  out->bad_row = ~0u;
  out->device_bytes = 0;
  if (!genes || !genes->partition_lnl_fixed) return refuse("rdk_rell_support_genes: null output arrays");
  if (genes->sampling != RDK_RELL_GENE && genes->sampling != RDK_RELL_GENE_SITE)
    return refuse("rdk_rell_support_genes: unknown sampling mode");
  if (n < 2) return refuse("rdk_rell_support_genes: at least 2 partitions are needed");
  if (rows == 0) return refuse("rdk_rell_support: no partitions or no rows");
  if (replicates == 0 || replicates > (1ull << 20)) return refuse("rdk_rell_support: replicates must be in [1, 2^20]");
  const unsigned              B = (unsigned)replicates;
  std::vector<const double *> L(n);
  std::vector<unsigned long long> N(n, 0);
  double                      M = 0;
  unsigned long long          n_max = 0;
  for (unsigned g = 0; g < n; ++g) {
    auto it = rows_of().find(parts[g]);
    if (it == rows_of().end() || it->second.size() < (size_t)rows * parts[g]->sites)
      return refuse("rdk_rell_support: a partition holds fewer rows than asked");
    L[g] = it->second.data();
    for (unsigned p = 0; p < parts[g]->sites; ++p) N[g] += parts[g]->pattern_weights[p];
    if (N[g] > n_max) n_max = N[g];
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
  if ((unsigned long long)n * n_max >= (1ull << 32))
    return refuse("rdk_rell_support_genes: partitions x sites (the largest) reach 2^32");
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

  // item 11: m[b][i]
  std::vector<unsigned> m((size_t)B * n, 0);
  for (unsigned b = 0; b < B; ++b)
    for (unsigned j4 = 0; j4 * 4 < n; ++j4) {
      unsigned long long xs[4] = {j4 + 1ull, 0, 1, 0};
      philox4x64_10(xs, seed, b);
      for (unsigned u = 0; u < 4 && j4 * 4 + u < n; ++u) m[(size_t)b * n + (unsigned)(((u128)xs[u] * n) >> 64)]++;
    }

  // O_i, then Z per item 12 or 13
  std::vector<i128> Z((size_t)B * rows, 0), O(rows, 0), Oi((size_t)n * rows, 0);
  for (unsigned g = 0; g < n; ++g) {
    const unsigned                  P = parts[g]->sites;
    const unsigned long long        gi = global_index ? global_index[g] : g;
    std::vector<long long>          q((size_t)rows * P);
    std::vector<unsigned long long> cumw(P + 1, 0);
    for (size_t i = 0; i < q.size(); ++i) q[i] = llrint(ldexp(L[g][i], e));
    for (unsigned p = 0; p < P; ++p) cumw[p + 1] = cumw[p] + parts[g]->pattern_weights[p];
    for (unsigned r = 0; r < rows; ++r) {
      for (unsigned p = 0; p < P; ++p) Oi[(size_t)g * rows + r] += (i128)parts[g]->pattern_weights[p] * q[(size_t)r * P + p];
      O[r] += Oi[(size_t)g * rows + r];
    }
    std::vector<unsigned> c(P);
    for (unsigned b = 0; b < B; ++b) {
      const unsigned long long mb = m[(size_t)b * n + g];
      if (genes->sampling == RDK_RELL_GENE) {
        for (unsigned r = 0; r < rows; ++r) Z[(size_t)b * rows + r] += (i128)mb * Oi[(size_t)g * rows + r];
        continue;
      }
      const unsigned long long draws = mb * N[g];
      std::fill(c.begin(), c.end(), 0u);
      for (unsigned long long j4 = 0; j4 * 4 < draws; ++j4) {
        unsigned long long xs[4] = {j4 + 1, 0, 0, 0};
        philox4x64_10(xs, seed, (gi << 32) | b);
        for (unsigned u = 0; u < 4 && j4 * 4 + u < draws; ++u) {
          const unsigned long long site = (unsigned long long)(((u128)xs[u] * N[g]) >> 64);
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

  // items 4-5 over this Z
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
  for (size_t i = 0; i < Oi.size(); ++i) {
    genes->partition_lnl_fixed[i] = ldexp((double)Oi[i], -e);
    if (genes->o_lo) genes->o_lo[i] = (unsigned long long)(u128)Oi[i];
    if (genes->o_hi) genes->o_hi[i] = (long long)(Oi[i] >> 64);
  }
  for (double &t : out->ms) t = 0;
  genes->draws_ms = 0;
  return RDO_SUCCESS;
}
#endif
