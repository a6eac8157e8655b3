// rdk_support.cuh -- RELL bootstrap proportions and KH / SH tests over per-pattern
// log-likelihood rows (rdk_rell_support, include/rdk.h; DESIGN.md section 10).
#ifndef RDK_SUPPORT_CUH_
#define RDK_SUPPORT_CUH_

#include "../../include/rdk.h"

#include <cuda_runtime.h>

#include <cstddef>

namespace rdk {

constexpr unsigned long long kRellMaxReplicates = 1ull << 20;

// one partition's inputs: rows [rows][patterns] on the device, weights on the host
struct RellPartition {
  const double       *rows;
  const unsigned int *weights;
  unsigned int        patterns;
  unsigned int        global_index;
};

// A site shard: this process holds global patterns [site_offset, site_offset + patterns) of the one
// partition; `allreduce` is ncclAllReduce on the shard's communicator (data type / operation codes
// of nccl.h).  Every rank must call rell_support with the same rows, replicates and seed.
typedef int (*rell_allreduce_fn)(const void *send, void *recv, size_t count, int datatype, int op, void *comm,
                                 cudaStream_t stream);
struct RellShard {
  void              *comm = nullptr;  // null: not sharded
  int                nranks = 1, rank = 0;
  unsigned long long site_offset = 0;
  rell_allreduce_fn  allreduce = nullptr;
};

// runs on the current device; returns 0 with a message in msg on failure.  ms (validated by the
// caller; null for rdk_rell_support) adds the multiscale counts and the ELW of rdk_rell_support_ms.
int rell_support(const RellPartition *parts, unsigned int n, unsigned int rows, unsigned long long replicates,
                 unsigned long long seed, const RellShard &shard, rdk_rell_out_t *out, rdk_rell_ms_out_t *ms,
                 char *msg, size_t msg_cap);

}  // namespace rdk

#endif
