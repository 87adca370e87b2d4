// Phase-locked general action kernel with the action loop of hsrb_rollout (hsrb_kernels.cuh: hsrb_step_lock_rollout_kernel),
// with and without per-environment parameters, in its own translation unit with the flags of hsrb_step_lock.cu.
#define HSRB_STEP_LOCK_IMPL 1
#include "hsrb_kernels.cuh"

cudaError_t hsrb_step_lock_rollout_prepare() {
  cudaError_t e = cudaFuncSetAttribute(hsrb_step_lock_rollout_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(hsrb_step_lock_rollout_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  return e;
}

cudaError_t hsrb_step_lock_rollout_launch(const Plan& p, const KArgs& a, int nact, cudaStream_t s) {
  if (a.params) hsrb_step_lock_rollout_kernel<true><<<p.grid, p.threads, p.smem, s>>>(a, nact);
  else hsrb_step_lock_rollout_kernel<false><<<p.grid, p.threads, p.smem, s>>>(a, nact);
  return cudaGetLastError();
}
