/*
 * tests/oracle_shim/rdk_sweep_rows.h -- TEST INFRASTRUCTURE.
 *
 * The row capture of the placement sweep (RDK_SWEEP_ROWS of rdk_sweep_root_placements_ex /
 * _chunks) and rdk_partition_permute_site_lnl_rows, restated over the CPU oracle so that the
 * oracle-backed host (tests/_build/librd_host_oracle.so) runs model_t::branch_support on a machine
 * without a GPU.  The flag is restated as the call sequence it stands for: placement q ends in
 * rdk_compute_root_loglikelihood_row(root, row q) instead of rdk_compute_root_loglikelihood.  The
 * sweep entries of tests/oracle_shim/rdk.h are wrapped, under their rdk_* names, by the ones below.
 * Included by the host sources only when they are compiled against the oracle (RD_BACKEND_ORACLE),
 * after rdk_support.h.  Never part of the product.
 */
#ifndef RDK_SWEEP_ROWS_ORACLE_H_
#define RDK_SWEEP_ROWS_ORACLE_H_
#include "rdk.h"
#include "rdk_support.h"

#include <cstring>
#include <vector>

#define RDK_SWEEP_ROWS 4u

namespace rdk_sweep_rows_oracle {
inline int sweep_rows(rdo_partition_t *p, unsigned int placements, const unsigned int *params_indices,
                      const unsigned int *pm_offsets, const unsigned int *matrix_indices, const double *branch_lengths,
                      const unsigned int *op_offsets, const rdo_operation_t *operations, unsigned int root_clv_index,
                      int root_scaler_index, double *out_lnl) {
  auto it = rdk_support_oracle::rows_of().find(p);
  if (it == rdk_support_oracle::rows_of().end() || it->second.size() < (size_t)placements * p->sites)
    return rdk_support_oracle::refuse("RDK_SWEEP_ROWS: fewer site rows reserved than placements");
  for (unsigned int q = 0; q < placements; ++q) {
    if (rdo_update_prob_matrices(p, params_indices, matrix_indices + pm_offsets[q], branch_lengths + pm_offsets[q],
                                 pm_offsets[q + 1] - pm_offsets[q]) != RDO_SUCCESS)
      return RDO_FAILURE;
    rdo_update_clvs(p, operations + op_offsets[q], op_offsets[q + 1] - op_offsets[q]);
    out_lnl[q] = rdk_compute_root_loglikelihood_row(p, root_clv_index, root_scaler_index, q);
  }
  return RDO_SUCCESS;
}

inline int sweep_ex(rdo_partition_t *p, unsigned int placements, const unsigned int *params_indices,
                    const unsigned int *freqs_indices, const unsigned int *pm_offsets, const unsigned int *matrix_indices,
                    const double *branch_lengths, const unsigned int *op_offsets, const rdo_operation_t *operations,
                    unsigned int root_clv_index, int root_scaler_index, unsigned int flags, double *out_lnl) {
  if (flags & RDK_SWEEP_ROWS)
    return sweep_rows(p, placements, params_indices, pm_offsets, matrix_indices, branch_lengths, op_offsets,
                      operations, root_clv_index, root_scaler_index, out_lnl);
  return rdk_sweep_root_placements_ex(p, placements, params_indices, freqs_indices, pm_offsets, matrix_indices,
                                      branch_lengths, op_offsets, operations, root_clv_index, root_scaler_index, flags,
                                      out_lnl);
}

/* chunks may always run in order (include/rdk.h) */
inline int sweep_chunks(rdo_partition_t *p, unsigned int placements, const unsigned int *params_indices,
                        const unsigned int *freqs_indices, const unsigned int *pm_offsets,
                        const unsigned int *matrix_indices, const double *branch_lengths,
                        const unsigned int *op_offsets, const rdo_operation_t *operations, unsigned int root_clv_index,
                        int root_scaler_index, unsigned int flags, unsigned int n_chunks,
                        const unsigned int *chunk_offsets, double *out_lnl) {
  if (flags & RDK_SWEEP_ROWS)
    return sweep_rows(p, placements, params_indices, pm_offsets, matrix_indices, branch_lengths, op_offsets,
                      operations, root_clv_index, root_scaler_index, out_lnl);
  return rdk_sweep_root_placements_chunks(p, placements, params_indices, freqs_indices, pm_offsets, matrix_indices,
                                          branch_lengths, op_offsets, operations, root_clv_index, root_scaler_index,
                                          flags, n_chunks, chunk_offsets, out_lnl);
}
}  // namespace rdk_sweep_rows_oracle

/* from here on the host's calls reach the wrappers above */
#define rdk_sweep_root_placements_ex rdk_sweep_rows_oracle::sweep_ex
#define rdk_sweep_root_placements_chunks rdk_sweep_rows_oracle::sweep_chunks

/* row r afterwards holds what row order[r] held (order: a permutation of 0..count-1) */
static inline int rdk_partition_permute_site_lnl_rows(rdo_partition_t *p, unsigned int count,
                                                      const unsigned int *order) {
  auto &all = rdk_support_oracle::rows_of();
  auto  it = all.find(p);
  if (it == all.end() || (size_t)count * p->sites > it->second.size())
    return rdk_support_oracle::refuse("site rows out of range");
  std::vector<char> seen(count, 0);
  for (unsigned r = 0; r < count; ++r) {
    if (order[r] >= count || seen[order[r]]) return rdk_support_oracle::refuse("order is not a permutation of the rows");
    seen[order[r]] = 1;
  }
  const std::vector<double> before(it->second.begin(), it->second.begin() + (size_t)count * p->sites);
  for (unsigned r = 0; r < count; ++r)
    memcpy(it->second.data() + (size_t)r * p->sites, before.data() + (size_t)order[r] * p->sites,
           sizeof(double) * p->sites);
  return RDO_SUCCESS;
}
#endif
