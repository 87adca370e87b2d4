// Action-kernel instantiations of hsrb_push.cuh: G = 8 / 16 / 32 lanes per environment, NV = 8 (one block) and 2 (none).
#define HSR_COMPACT 1
#include "hsrb_push.cuh"

template <int G, int NV>
static cudaError_t prepare_t(const Plan& p, int* bps) {
  cudaError_t e = cudaFuncSetAttribute(hsrb_push_kernel<G, NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);   // per function, not per handle: handles with different layouts share it
  if (e != cudaSuccess) return e;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(bps, hsrb_push_kernel<G, NV>, p.threads, p.smem);
}

template <int G, int NV>
static cudaError_t launch_t(const Plan& p, const KArgs& a, cudaStream_t s) {
  hsrb_push_kernel<G, NV><<<p.grid, p.threads, p.smem, s>>>(a, *p.fam);
  return cudaGetLastError();
}

cudaError_t hsrb_push_prepare(const Plan& p, int* bps) {
  const bool blk = p.fam->nv == 8;
  switch (p.lanes) {
    case 8: return blk ? prepare_t<8, 8>(p, bps) : prepare_t<8, 2>(p, bps);
    case 16: return blk ? prepare_t<16, 8>(p, bps) : prepare_t<16, 2>(p, bps);
    default: return blk ? prepare_t<32, 8>(p, bps) : prepare_t<32, 2>(p, bps);
  }
}

cudaError_t hsrb_push_launch(const Plan& p, const KArgs& a, cudaStream_t s) {
  const bool blk = p.fam->nv == 8;
  switch (p.lanes) {
    case 8: return blk ? launch_t<8, 8>(p, a, s) : launch_t<8, 2>(p, a, s);
    case 16: return blk ? launch_t<16, 8>(p, a, s) : launch_t<16, 2>(p, a, s);
    default: return blk ? launch_t<32, 8>(p, a, s) : launch_t<32, 2>(p, a, s);
  }
}
