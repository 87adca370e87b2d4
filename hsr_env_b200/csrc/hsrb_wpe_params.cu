// Warp-per-environment action kernel with per-environment parameters (hsrb_wpe.cuh: hsrb_wpe_params_kernel_t), in its own
// translation unit with the flags of hsrb_wpe.cu: the instances without parameters keep their code.
#define HSR_COMPACT 1
#define HSRB_WPE_IMPL 1
#include "hsrb_wpe.cuh"

cudaError_t hsrb_wpe_params_prepare(const Plan&) {
  cudaError_t e = cudaFuncSetAttribute(hsrb_wpe_params_kernel_t<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(hsrb_wpe_params_kernel_t<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  return e;
}

cudaError_t hsrb_wpe_params_launch(const Plan& p, const KArgs& a, cudaStream_t s) {
  if (p.lock) hsrb_wpe_params_kernel_t<true><<<p.grid, p.threads, p.smem, s>>>(a, *p.fam);
  else hsrb_wpe_params_kernel_t<false><<<p.grid, p.threads, p.smem, s>>>(a, *p.fam);
  return cudaGetLastError();
}
