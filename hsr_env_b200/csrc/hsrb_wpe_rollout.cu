// Warp-per-environment action kernel with the action loop of hsrb_rollout (hsrb_wpe.cuh: hsrb_wpe_rollout_kernel_t and
// hsrb_wpe_rollout_params_kernel_t, phase-locked), in its own translation unit with the flags of hsrb_wpe.cu: the
// instances hsrb_step launches keep their code.
#define HSR_COMPACT 1
#define HSRB_WPE_IMPL 1
#include "hsrb_wpe.cuh"

cudaError_t hsrb_wpe_rollout_prepare() {
  cudaError_t e = cudaFuncSetAttribute(hsrb_wpe_rollout_kernel_t<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(hsrb_wpe_rollout_params_kernel_t<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  return e;
}

cudaError_t hsrb_wpe_rollout_launch(const Plan& p, const KArgs& a, int nact, cudaStream_t s) {
  if (a.params) hsrb_wpe_rollout_params_kernel_t<true><<<p.grid, p.threads, p.smem, s>>>(a, *p.fam, nact);
  else hsrb_wpe_rollout_kernel_t<true><<<p.grid, p.threads, p.smem, s>>>(a, *p.fam, nact);
  return cudaGetLastError();
}
