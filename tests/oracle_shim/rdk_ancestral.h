/*
 * tests/oracle_shim/rdk_ancestral.h -- TEST INFRASTRUCTURE.
 *
 * rdk_marginal_ancestral_states (include/rdk.h; DESIGN.md section 11) restated over the oracle's
 * public arrays (clv, pmatrix, scale_buffer, frequencies, rate_weights) with plain loops, in the
 * order of the definition: operations in reverse order (every parent before its children), one
 * outside vector per inner node, every product and sum as written there.  Tips are the oracle's 0/1
 * CLVs, whose FMA chains equal the engine's tip tables bit for bit.
 */
#ifndef RDK_ANCESTRAL_SHIM_H_
#define RDK_ANCESTRAL_SHIM_H_
#include "rdk.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define RDO_LOG_SCALE_THRESHOLD_SHIM (-177.44567822334599) /* ln 2^-256, as rd_oracle.c */

typedef struct rdk_ancestral_out_t {
  const unsigned int *full_ops;
  unsigned int        n_full;
  unsigned int        threads;
  unsigned int        tile_sites;
  unsigned char      *map_state;
  double             *map_prob;
  double             *posterior;
  double             *log_norm;
  double              ms;
  unsigned long long  device_bytes;
  unsigned int        scratch;
} rdk_ancestral_out_t;

/* h[k][j] = sum_l P[k][j][l] x[k][l], FMA chain l ascending */
static inline void rdk_anc_half(const double *P, const double *x, unsigned K, double *h) {
  for (unsigned k = 0; k < K; ++k)
    for (int j = 0; j < 4; ++j) {
      const double *pr = P + k * 16 + j * 4;
      const double *xr = x + k * 4;
      double        acc = pr[0] * xr[0];
      acc = fma(pr[1], xr[1], acc);
      acc = fma(pr[2], xr[2], acc);
      acc = fma(pr[3], xr[3], acc);
      h[k * 4 + j] = acc;
    }
}

/* o_c[k][i] = sum_j (o[k][j] hs[k][j]) P[k][j][i], FMA chain j ascending; rescaled when every entry
 * is below 2^-256.  Returns whether it was rescaled. */
static inline int rdk_anc_outside(const double *P, const double *o, const double *hs, unsigned K, double *oc) {
  int small = 1;
  for (unsigned k = 0; k < K; ++k) {
    double s[4];
    for (int j = 0; j < 4; ++j) s[j] = o[k * 4 + j] * hs[k * 4 + j];
    for (int i = 0; i < 4; ++i) {
      const double *pk = P + k * 16;
      double        acc = s[0] * pk[0 * 4 + i];
      acc = fma(s[1], pk[1 * 4 + i], acc);
      acc = fma(s[2], pk[2 * 4 + i], acc);
      acc = fma(s[3], pk[3 * 4 + i], acc);
      oc[k * 4 + i] = acc;
      if (!(acc < 0x1p-256)) small = 0;
    }
  }
  if (small)
    for (unsigned q = 0; q < K * 4; ++q) oc[q] = oc[q] * 0x1p+256;
  return small;
}

static inline int rdk_marginal_ancestral_states(rdo_partition_t *p, const rdo_operation_t *ops, unsigned int count,
                                                const unsigned int *freqs_indices, rdk_ancestral_out_t *out) {
  if (!p || !ops || !out || count == 0 || !out->map_state || !out->map_prob ||
      (out->n_full && (!out->full_ops || !out->posterior))) {
    snprintf(rdo_errmsg, sizeof(rdo_errmsg), "rdk_marginal_ancestral_states: missing arguments");
    rdo_errno = 1;
    return RDO_FAILURE;
  }
  const unsigned K = p->rate_cats, S = p->sites, n_clv = p->tips + p->clv_buffers;
  const size_t   span = (size_t)K * 4;
  const double  *pi = p->frequencies[freqs_indices ? freqs_indices[0] : 0];
  int           *full_row = (int *)malloc(sizeof(int) * count);
  double       **o = (double **)calloc(n_clv, sizeof(double *));  /* outside vector per inner node */
  unsigned     **tau = (unsigned **)calloc(n_clv, sizeof(unsigned *));
  double        *h1 = (double *)malloc(sizeof(double) * span), *h2 = (double *)malloc(sizeof(double) * span);
  double        *d = (double *)malloc(sizeof(double) * span);
  for (unsigned i = 0; i < count; ++i) full_row[i] = -1;
  for (unsigned f = 0; f < out->n_full; ++f) full_row[out->full_ops[f]] = (int)f;
  const unsigned root = ops[count - 1].parent_clv_index;
  o[root] = (double *)malloc(sizeof(double) * span * (S ? S : 1));
  tau[root] = (unsigned *)calloc(S ? S : 1, sizeof(unsigned));
  for (unsigned s = 0; s < S; ++s)
    for (unsigned k = 0; k < K; ++k)
      for (int i = 0; i < 4; ++i) o[root][s * span + k * 4 + i] = pi[i];
  for (unsigned n = count; n-- > 0;) {
    const rdo_operation_t *op = &ops[n];
    const unsigned         v = op->parent_clv_index, c1 = op->child1_clv_index, c2 = op->child2_clv_index;
    const double          *P1 = p->pmatrix[op->child1_matrix_index], *P2 = p->pmatrix[op->child2_matrix_index];
    const unsigned *s1b = op->child1_scaler_index < 0 ? NULL : p->scale_buffer[op->child1_scaler_index];
    const unsigned *s2b = op->child2_scaler_index < 0 ? NULL : p->scale_buffer[op->child2_scaler_index];
    if (c1 >= p->tips) {
      o[c1] = (double *)malloc(sizeof(double) * span * (S ? S : 1));
      tau[c1] = (unsigned *)malloc(sizeof(unsigned) * (S ? S : 1));
    }
    if (c2 >= p->tips) {
      o[c2] = (double *)malloc(sizeof(double) * span * (S ? S : 1));
      tau[c2] = (unsigned *)malloc(sizeof(unsigned) * (S ? S : 1));
    }
    for (unsigned s = 0; s < S; ++s) {
      const double *ov = o[v] + s * span;
      const unsigned sc1 = s1b ? s1b[s] : 0u, sc2 = s2b ? s2b[s] : 0u;
      rdk_anc_half(P1, p->clv[c1] + s * span, K, h1);
      rdk_anc_half(P2, p->clv[c2] + s * span, K, h2);
      /* d_v with the post-order operation's own rescaling test */
      int small = 1;
      for (size_t q = 0; q < span; ++q) {
        d[q] = h1[q] * h2[q];
        if (!(d[q] < 0x1p-256)) small = 0;
      }
      unsigned sigma = 0;
      if (op->parent_scaler_index >= 0) {
        sigma = sc1 + sc2;
        if (small) {
          for (size_t q = 0; q < span; ++q) d[q] = d[q] * 0x1p+256;
          sigma += 1;
        }
      }
      double t[4];
      for (int i = 0; i < 4; ++i) {
        t[i] = p->rate_weights[0] * (ov[i] * d[i]);
        for (unsigned k = 1; k < K; ++k) t[i] = fma(p->rate_weights[k], ov[k * 4 + i] * d[k * 4 + i], t[i]);
      }
      const double Z = ((t[0] + t[1]) + t[2]) + t[3];
      double       post[4];
      for (int i = 0; i < 4; ++i) post[i] = t[i] / Z;
      unsigned best = 0;
      for (unsigned i = 1; i < 4; ++i)
        if (post[i] > post[best]) best = i;
      const size_t row = (size_t)n * S + s;
      out->map_state[row] = (unsigned char)best;
      out->map_prob[row] = post[best];
      if (out->log_norm) out->log_norm[row] = rdo_log(Z) + (double)(sigma + tau[v][s]) * RDO_LOG_SCALE_THRESHOLD_SHIM;
      if (full_row[n] >= 0)
        for (int i = 0; i < 4; ++i) out->posterior[((size_t)full_row[n] * S + s) * 4 + i] = post[i];
      if (c1 >= p->tips) tau[c1][s] = tau[v][s] + sc2 + (unsigned)rdk_anc_outside(P1, ov, h2, K, o[c1] + s * span);
      if (c2 >= p->tips) tau[c2][s] = tau[v][s] + sc1 + (unsigned)rdk_anc_outside(P2, ov, h1, K, o[c2] + s * span);
    }
    free(o[v]);
    free(tau[v]);
    o[v] = NULL;
    tau[v] = NULL;
  }
  out->ms = 0.0;
  out->device_bytes = 0;
  out->scratch = 0;
  free(full_row);
  free(o);
  free(tau);
  free(h1);
  free(h2);
  free(d);
  return RDO_SUCCESS;
}
#endif
