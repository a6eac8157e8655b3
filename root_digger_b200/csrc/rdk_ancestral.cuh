// rdk_ancestral.cuh -- marginal ancestral states of the rooted tree (rdk_marginal_ancestral_states,
// include/rdk.h; DESIGN.md section 11).
#ifndef RDK_ANCESTRAL_CUH_
#define RDK_ANCESTRAL_CUH_

#include "../../include/rdk.h"

#include <cuda_runtime.h>

#include <cstddef>
#include <vector>

namespace rdk {

// One internal node v of the pre-order pass.  The order of the visits only decides which scratch
// buffers hold the outside vectors; every value is that of the definition.
struct AncNode {
  unsigned op;              // position of v's operation: the output row
  int      in;              // scratch buffer holding o_v, -1 at the root (o = pi)
  int      out1, out2;      // scratch buffer receiving o_c1 / o_c2, -1 for a tip child
  int      full;            // row of the full posterior, -1 for none
  // filled in by the caller (device pointers)
  const double       *tab1, *tab2;  // the children's pool slots: P [cat][18], then the tip table
  const void         *c1, *c2;      // inner child CLV [site][cat][4], or tip row (1-byte codes)
  const unsigned int *sc1, *sc2;    // the children's scale buffers, or null
  int                 tip1, tip2;
  int                 scaled;       // v's operation has a scale buffer: d_v takes its rescaling test
};

// Validates that ops[0..count) are the post-order operations of one rooted tree over clv indices
// >= tips for inner nodes, and lays out the pass: every node once, parents before children, the
// smaller child subtree first.  Returns the visits and the number of scratch buffers (at most
// ceil(log2 count) + 2); 0 with a message on failure.
int ancestral_schedule(const rdk_operation_t *ops, unsigned count, unsigned tips, unsigned clv_count,
                       std::vector<AncNode> &nodes, unsigned &scratch, char *msg, size_t msg_cap);

struct AncPass {
  unsigned     S = 0, K = 0;  // patterns, device categories (a divisor of 32)
  double       pi[4] = {0, 0, 0, 0};
  double       w[32] = {0};   // category weights, 0 for padding categories
  unsigned     scratch = 0;
  unsigned     count = 0;     // operations
  cudaStream_t stream = nullptr;
};

// Runs the pass on the current device and stream and copies the outputs to out's host arrays.
int ancestral_pass(const AncPass &pass, const std::vector<AncNode> &nodes, rdk_ancestral_out_t *out, char *msg,
                   size_t msg_cap);

}  // namespace rdk

#endif
