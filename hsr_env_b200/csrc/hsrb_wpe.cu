// Warp-per-environment action kernel (hsrb_wpe.cuh): launch helpers.
#define HSR_COMPACT 1
#define HSRB_WPE_IMPL 1
#include "hsrb_wpe.cuh"

// occupancy of the free-running instance for both: the plan's layout is the same whichever p.lock launches
cudaError_t hsrb_wpe_prepare(const Plan& p, int* bps) {
  cudaError_t e = cudaFuncSetAttribute(hsrb_wpe_kernel_t<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(hsrb_wpe_kernel_t<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = hsrb_wpe_params_prepare(p);
  if (e == cudaSuccess) e = hsrb_wpe_rollout_prepare();
  if (e != cudaSuccess) return e;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(bps, hsrb_wpe_kernel_t<false>, p.threads, p.smem);
}

cudaError_t hsrb_wpe_launch(const Plan& p, const KArgs& a, cudaStream_t s) {
  if (a.params) return hsrb_wpe_params_launch(p, a, s);
  if (p.lock) hsrb_wpe_kernel_t<true><<<p.grid, p.threads, p.smem, s>>>(a, *p.fam);
  else hsrb_wpe_kernel_t<false><<<p.grid, p.threads, p.smem, s>>>(a, *p.fam);
  return cudaGetLastError();
}

#if defined(WPE_CHAIN_CLOCKS)
// experiment hook (not part of include/hsrb.h): out[0..31] = cycles, out[32..63] = occurrences per chain section; resets
extern "C" int hsrb_debug_chain_clocks(unsigned long long* out) {
  unsigned long long z[32] = {0};
  cudaDeviceSynchronize();
  if (cudaMemcpyFromSymbol(out, wpe::wpe_ck_cyc, sizeof(z)) != cudaSuccess) return -1;
  if (cudaMemcpyFromSymbol(out + 32, wpe::wpe_ck_cnt, sizeof(z)) != cudaSuccess) return -1;
  cudaMemcpyToSymbol(wpe::wpe_ck_cyc, z, sizeof(z)); cudaMemcpyToSymbol(wpe::wpe_ck_cnt, z, sizeof(z));
  return 0;
}
#endif
