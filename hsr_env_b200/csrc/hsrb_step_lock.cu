// Phase-locked general action kernel (hsrb_kernels.cuh: hsrb_step_lock_kernel): launch helpers.
#define HSRB_STEP_LOCK_IMPL 1
#include "hsrb_kernels.cuh"

cudaError_t hsrb_step_lock_prepare(const Plan& p, int* bps) {
  cudaError_t e = cudaFuncSetAttribute(hsrb_step_lock_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = hsrb_step_lock_params_prepare();
  if (e == cudaSuccess) e = hsrb_step_lock_rollout_prepare();
  if (e != cudaSuccess) return e;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(bps, hsrb_step_lock_kernel<false>, p.threads, p.smem);
}

cudaError_t hsrb_step_lock_launch(const Plan& p, const KArgs& a, cudaStream_t s) {
  if (a.params) return hsrb_step_lock_params_launch(p, a, s);
  hsrb_step_lock_kernel<false><<<p.grid, p.threads, p.smem, s>>>(a);
  return cudaGetLastError();
}
