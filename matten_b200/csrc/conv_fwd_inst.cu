// Explicit instantiation of the fused conv forward kernel for one (dtype, HP) pair;
// compiled once per pair (see matten_b200/build.py) so the 65 CG types build in parallel.
#include "conv_fwd.cuh"

#ifndef MT_INST_T
#error "compile with -DMT_INST_T=float|double -DMT_INST_HP=8|16|32|64|0"
#endif

namespace mt {

template <typename T, int HP>
int launch_conv_fwd(const ConvFwdParams& p, int grid, int threads, size_t smem, cudaStream_t st);

template <>
int launch_conv_fwd<MT_INST_T, MT_INST_HP>(const ConvFwdParams& p, int grid, int threads, size_t smem,
                                           cudaStream_t st) {
  static thread_local size_t configured = 0;  // per host thread; cudaFuncSetAttribute is cheap
  if (smem > configured) {
    MT_CUDA_OK(cudaFuncSetAttribute(conv_fwd_kernel<MT_INST_T, MT_INST_HP>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  conv_fwd_kernel<MT_INST_T, MT_INST_HP><<<grid, threads, smem, st>>>(p);
  MT_LAUNCH_OK();
  return MT_OK;
}

}  // namespace mt
