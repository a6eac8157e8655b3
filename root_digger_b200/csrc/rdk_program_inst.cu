// rdk_program_inst.cu -- the instantiations of clv_program_kernel for ONE number of rate
// categories (compiled once per K with -DRDK_INST_K=K: the translation units build in
// parallel, which is what keeps the library's build time short).
#define RDK_PROGRAM_KERNEL_ONLY 1
#include "rdk_kernels.cuh"

#ifndef RDK_INST_K
#error "compile with -DRDK_INST_K=<rate categories>"
#endif

namespace rdk {
namespace {

template <int K, int E, bool ROWS>
cudaError_t launch_inst(const ProgArgs &a, int grid, int threads, cudaStream_t st) {
  constexpr LaunchShape shape = launch_shape(E);
  const size_t          smem = Ring<K>::kSmemBytes;  // the table ring + its mbarriers
  static bool           configured = false;          // per template instantiation
  if (!configured) {
    cudaError_t err = cudaFuncSetAttribute(clv_program_kernel<K, E, shape.threads, shape.ctas_per_sm, ROWS>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    configured = true;
  }
  if (threads > shape.threads) threads = shape.threads;
  clv_program_kernel<K, E, shape.threads, shape.ctas_per_sm, ROWS>
      <<<dim3((unsigned)grid, a.n_chunks > 1 ? a.n_chunks : 1u), threads, smem, st>>>(a);
  return cudaSuccess;
}

template <bool ROWS>
cudaError_t launch_e(const ProgArgs &a, int grid, int threads, int E, cudaStream_t st) {
  constexpr int K = RDK_INST_K;
  switch (E) {
    case 1: return launch_inst<K, 1, ROWS>(a, grid, threads, st);
    case 2: return launch_inst<K, 2, ROWS>(a, grid, threads, st);
    case 3: return launch_inst<K, 3, ROWS>(a, grid, threads, st);
    default: return launch_inst<K, 4, ROWS>(a, grid, threads, st);
  }
}

}  // namespace

// elements per thread E trades registers (occupancy) for fewer per-instruction preambles per
// element (rdk_abi.cu picks it from the shard size); `rows` selects the variant that stores every
// evaluation's per-pattern row (placement sweeps with RDK_SWEEP_ROWS)
template <>
cudaError_t launch_program<RDK_INST_K>(const ProgArgs &a, int grid, int threads, int E, bool rows, cudaStream_t st) {
  return rows ? launch_e<true>(a, grid, threads, E, st) : launch_e<false>(a, grid, threads, E, st);
}

}  // namespace rdk
