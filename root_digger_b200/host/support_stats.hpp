// support_stats.hpp -- the approximately unbiased (AU) test's fit from multiscale bootstrap counts
// (DESIGN.md section 10, item 7): host fp64, the same code for every backend.
#ifndef RD_SUPPORT_STATS_HPP_
#define RD_SUPPORT_STATS_HPP_

#include <cmath>
#include <stdexcept>
#include <string>
#include <vector>

namespace rd {

// scales of the multiscale bootstrap in thousandths: 2 to 32, strictly ascending, in [100, 10000]
inline void check_au_scales(const unsigned *scales, size_t n) {
  if (n < 2 || n > 32)
    throw std::invalid_argument("AU scales: " + std::to_string(n) + " given, 2 to 32 are needed");
  for (size_t k = 0; k < n; ++k) {
    if (scales[k] < 100 || scales[k] > 10000)
      throw std::invalid_argument("AU scales: " + std::to_string(scales[k]) +
                                  " thousandths is outside [100, 10000]");
    if (k && scales[k] <= scales[k - 1]) throw std::invalid_argument("AU scales must be strictly ascending");
  }
}

// the standard normal quantile, Wichura's AS241 (PPND16), for 0 < p < 1
inline double ppnd16(double p) {
  const double q = p - 0.5;
  if (std::fabs(q) <= 0.425) {
    const double r = 0.180625 - q * q;
    return q *
           (((((((2.5090809287301226727e+3 * r + 3.3430575583588128105e+4) * r + 6.7265770927008700853e+4) * r +
                4.5921953931549871457e+4) * r + 1.3731693765509461125e+4) * r + 1.9715909503065514427e+3) * r +
             1.3314166789178437745e+2) * r + 3.3871328727963666080e+0) /
           (((((((5.2264952788528545610e+3 * r + 2.8729085735721942674e+4) * r + 3.9307895800092710610e+4) * r +
                2.1213794301586595867e+4) * r + 5.3941960214247511077e+3) * r + 6.8718700749205790830e+2) * r +
             4.2313330701600911252e+1) * r + 1.0);
  }
  double r = std::sqrt(-std::log(q < 0 ? p : 1.0 - p)), v;
  if (r <= 5.0) {
    r -= 1.6;
    v = (((((((7.74545014278341407640e-4 * r + 2.27238449892691845833e-2) * r + 2.41780725177450611770e-1) * r +
             1.27045825245236838258e+0) * r + 3.64784832476320460504e+0) * r + 5.76949722146069140550e+0) * r +
          4.63033784615654529590e+0) * r + 1.42343711074968357734e+0) /
        (((((((1.05075007164441684324e-9 * r + 5.47593808499534494600e-4) * r + 1.51986665636164571966e-2) * r +
             1.48103976427480074590e-1) * r + 6.89767334985100004550e-1) * r + 1.67638483018380384940e+0) * r +
          2.05319162663775882187e+0) * r + 1.0);
  } else {
    r -= 5.0;
    v = (((((((2.01033439929228813265e-7 * r + 2.71155556874348757815e-5) * r + 1.24266094738807843860e-3) * r +
             2.65321895265761230930e-2) * r + 2.96560571828504891230e-1) * r + 1.78482653991729133580e+0) * r +
          5.46378491116411436990e+0) * r + 6.65790464350110377720e+0) /
        (((((((2.04426310338993978564e-15 * r + 1.42151175831644588870e-7) * r + 1.84631831751005468180e-5) * r +
             7.86869131145613259100e-4) * r + 1.48753612908506148525e-2) * r + 1.36929880922735805310e-1) * r +
          5.99832206555887937690e-1) * r + 1.0);
  }
  return q < 0 ? -v : v;
}

struct au_fit_t {
  double   p_au = 0, d = 0, c = 0, rss = 0;
  unsigned used = 0;
};

// Shimodaira's two-parameter fit (Syst. Biol. 51:492, 2002) without the iterated threshold
// refinement of CONSEL / IQ-TREE: over the scales with 0 < n_k < B, z_k = -PPND16(n_k / B) is fitted
// as d a_k + c / a_k, a_k = sqrt(s_k / 1000), by weighted least squares with weights
// B phi(z_k)^2 / (p_k (1 - p_k)) (closed-form normal equations, sums in ascending scale order);
// p_AU = 1 - Phi(d - c).  Fewer than two usable scales: p_AU is the pooled BP, d = c = rss = 0.
inline au_fit_t au_fit(const unsigned *count, const unsigned *scales, size_t n, unsigned long long B) {
  au_fit_t             out;
  std::vector<double>  z, a, b, w;
  unsigned long long   pooled = 0;
  for (size_t k = 0; k < n; ++k) {
    pooled += count[k];
    if (count[k] == 0 || count[k] >= B) continue;
    const double p = (double)count[k] / (double)B;
    const double zk = -ppnd16(p);
    const double phi = std::exp(-zk * zk / 2.0) * 0.3989422804014327;
    const double ak = std::sqrt(scales[k] / 1000.0);
    z.push_back(zk);
    a.push_back(ak);
    b.push_back(1.0 / ak);
    w.push_back((double)B * phi * phi / (p * (1.0 - p)));
  }
  out.used = (unsigned)z.size();
  if (out.used < 2) {
    out.p_au = (double)pooled / ((double)n * (double)B);
    return out;
  }
  double saa = 0, sab = 0, sbb = 0, saz = 0, sbz = 0;
  for (size_t k = 0; k < z.size(); ++k) {
    saa += w[k] * a[k] * a[k];
    sab += w[k] * a[k] * b[k];
    sbb += w[k] * b[k] * b[k];
    saz += w[k] * a[k] * z[k];
    sbz += w[k] * b[k] * z[k];
  }
  const double det = saa * sbb - sab * sab;
  out.d = (sbb * saz - sab * sbz) / det;
  out.c = (saa * sbz - sab * saz) / det;
  for (size_t k = 0; k < z.size(); ++k) {
    const double res = z[k] - out.d * a[k] - out.c * b[k];
    out.rss += w[k] * res * res;
  }
  out.p_au = 0.5 * std::erfc((out.d - out.c) * std::sqrt(0.5));
  return out;
}

}  // namespace rd

#endif
