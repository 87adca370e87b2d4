// Phase-locked general action kernel with per-environment parameters (hsrb_kernels.cuh: hsrb_step_lock_kernel<true>).
#define HSRB_STEP_LOCK_IMPL 1
#include "hsrb_kernels.cuh"

cudaError_t hsrb_step_lock_params_prepare() {
  return cudaFuncSetAttribute(hsrb_step_lock_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

cudaError_t hsrb_step_lock_params_launch(const Plan& p, const KArgs& a, cudaStream_t s) {
  hsrb_step_lock_kernel<true><<<p.grid, p.threads, p.smem, s>>>(a);
  return cudaGetLastError();
}
