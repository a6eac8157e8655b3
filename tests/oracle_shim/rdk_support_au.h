/*
 * tests/oracle_shim/rdk_support_au.h -- TEST INFRASTRUCTURE.
 *
 * rdk_rell_support_ms of include/rdk.h (the multiscale RELL counts of the AU test and the expected
 * likelihood weights, DESIGN.md section 10 items 6-8) restated over the CPU oracle with plain loops,
 * __int128 and one rounded double operation per step, next to rdk_rell_support in rdk_support.h.
 * Included by the host sources only when they are compiled against the oracle (RD_BACKEND_ORACLE).
 * Never part of the product.
 */
#ifndef RDK_SUPPORT_AU_ORACLE_H_
#define RDK_SUPPORT_AU_ORACLE_H_
#include "rdk_support.h"

#include <algorithm>
#include <cstdint>

typedef struct rdk_rell_ms_out_t {
  const unsigned int *scales;
  unsigned int        n_scales;
  unsigned int       *scale_count;
  unsigned long long *elw_fixed;
  double              ms[3];
} rdk_rell_ms_out_t;

namespace rdk_support_oracle {

/* Z[b][r] at one scale (thousandths): N' = max(1, (s N_g + 500) / 1000) draws of Philox counter
 * {j + 1, s - 1000, 0, 0}, each mapped to a site (x N_g) >> 64 and to its pattern */
inline std::vector<i128> multiscale_z(rdo_partition_t *const *parts, unsigned n, const unsigned *global_index,
                                      unsigned rows, unsigned B, unsigned long long seed, int e, unsigned scale) {
  std::vector<i128> Z((size_t)B * rows, 0);
  for (unsigned g = 0; g < n; ++g) {
    const unsigned                  P = parts[g]->sites;
    const unsigned long long        gi = global_index ? global_index[g] : g;
    const double                   *L = rows_of().find(parts[g])->second.data();
    std::vector<long long>          q((size_t)rows * P);
    std::vector<unsigned long long> cumw(P + 1, 0);
    for (size_t i = 0; i < q.size(); ++i) q[i] = llrint(ldexp(L[i], e));
    for (unsigned p = 0; p < P; ++p) cumw[p + 1] = cumw[p] + parts[g]->pattern_weights[p];
    const unsigned long long N = cumw[P];
    if (N == 0) continue;
    const unsigned long long draws = std::max<unsigned long long>(1, (scale * N + 500) / 1000);
    const unsigned long long word = (unsigned long long)scale - 1000ull;
    std::vector<unsigned>    c(P);
    for (unsigned b = 0; b < B; ++b) {
      std::fill(c.begin(), c.end(), 0u);
      for (unsigned long long j4 = 0; j4 * 4 < draws; ++j4) {
        unsigned long long xs[4] = {j4 + 1, word, 0, 0};
        philox4x64_10(xs, seed, (gi << 32) | b);
        for (unsigned u = 0; u < 4 && j4 * 4 + u < draws; ++u) {
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
  return Z;
}

/* fdlibm e_exp.c on [-40, 0] (the host is built with -ffp-contract=off: one rounding per operation) */
inline double rd_exp(double x) {
  const double P1 = 1.66666666666666019037e-01, P2 = -2.77777777770155933842e-03, P3 = 6.61375632143793436117e-05,
               P4 = -1.65339022054652515390e-06, P5 = 4.13813679705723846039e-08;
  const double ln2hi = 6.93147180369123816490e-01, ln2lo = 1.90821492927058770002e-10,
               invln2 = 1.44269504088896338700e+00;
  uint64_t bits;
  memcpy(&bits, &x, sizeof(bits));
  const uint32_t hx = (uint32_t)(bits >> 32) & 0x7fffffffu;
  double         hi = 0, lo = 0;
  int            k = 0;
  if (hx > 0x3fd62e42u) {
    if (hx < 0x3ff0a2b2u) {
      hi = x + ln2hi;
      lo = -ln2lo;
      k = -1;
    } else {
      k = (int)(invln2 * x - 0.5);
      const double t = k;
      hi = x - t * ln2hi;
      lo = t * ln2lo;
    }
    x = hi - lo;
  } else if (hx < 0x3e300000u) {
    return 1.0 + x;
  }
  const double t = x * x;
  const double c = x - t * (P1 + t * (P2 + t * (P3 + t * (P4 + t * P5))));
  if (k == 0) return 1.0 - ((x * c) / (c - 2.0) - x);
  const double y = 1.0 - ((lo - (x * c) / (2.0 - c)) - hi);
  return ldexp(y, k);
}

/* Delta < -40 2^e, exactly */
inline bool elw_below_cut(i128 d, int e) {
  if (e >= 80) return false;
  if (e >= 0) return d < -((i128)40 << e);
  return d != 0 && (-e >= 6 || ((-d) << -e) > 40);
}

inline unsigned long long elw_weight(i128 d, int e) {
  if (elw_below_cut(d, e)) return 0;
  return (unsigned long long)rint(ldexp(rd_exp(ldexp((double)d, -e)), 52));
}
}  // namespace rdk_support_oracle

/* the definition of include/rdk.h: rdk_rell_support, then items 6-8 */
static inline int rdk_rell_support_ms(rdo_partition_t *const *parts, unsigned int n, const unsigned int *global_index,
                                      unsigned int rows, unsigned long long replicates, unsigned long long seed,
                                      rdk_rell_out_t *out, rdk_rell_ms_out_t *ms) {
  using namespace rdk_support_oracle;
  if (!ms || !ms->scales || !ms->scale_count || !ms->elw_fixed)
    return refuse("rdk_rell_support_ms: null scales or output arrays");
  if (ms->n_scales < 2 || ms->n_scales > 32) return refuse("rdk_rell_support_ms: 2 to 32 scales are needed");
  for (unsigned k = 0; k < ms->n_scales; ++k) {
    if (ms->scales[k] < 100 || ms->scales[k] > 10000)
      return refuse("rdk_rell_support_ms: a scale is outside [100, 10000] thousandths");
    if (k && ms->scales[k] <= ms->scales[k - 1]) return refuse("rdk_rell_support_ms: scales must be strictly ascending");
  }
  if (rdk_rell_support(parts, n, global_index, rows, replicates, seed, out) != RDO_SUCCESS) return RDO_FAILURE;
  const unsigned B = (unsigned)replicates;
  const int      e = out->exponent;
  for (unsigned k = 0; k < ms->n_scales; ++k) {
    unsigned *count = ms->scale_count + (size_t)k * rows;
    for (unsigned r = 0; r < rows; ++r) count[r] = 0;
    const std::vector<i128> Z = multiscale_z(parts, n, global_index, rows, B, seed, e, ms->scales[k]);
    for (unsigned b = 0; b < B; ++b) {
      const i128 *z = &Z[(size_t)b * rows];
      unsigned    top = 0;
      for (unsigned r = 1; r < rows; ++r)
        if (z[r] > z[top]) top = r;
      count[top]++;
    }
  }
  const std::vector<i128> Z = multiscale_z(parts, n, global_index, rows, B, seed, e, 1000);
  std::vector<u128>       acc(rows, 0);
  for (unsigned b = 0; b < B; ++b) {
    const i128 *z = &Z[(size_t)b * rows];
    i128        m = z[0];
    for (unsigned r = 1; r < rows; ++r)
      if (z[r] > m) m = z[r];
    u128 D = 0;
    for (unsigned r = 0; r < rows; ++r) D += elw_weight(z[r] - m, e);
    for (unsigned r = 0; r < rows; ++r) acc[r] += ((u128)elw_weight(z[r] - m, e) << 40) / D;
  }
  for (unsigned r = 0; r < rows; ++r) ms->elw_fixed[r] = (unsigned long long)acc[r];
  for (double &t : ms->ms) t = 0;
  return RDO_SUCCESS;
}
#endif
