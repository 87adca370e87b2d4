// The transition-derivative kernels (hsrb_fd.cuh): the run kernel, one instance per lanes-per-environment layout of the
// general path with and without per-environment parameters, and the kernel that forms A and B.  Built with the flags of
// hsrb_step_g*.cu (IEEE division and square root): the stages of the runs are then compiled as those of the MODE_DEBUG
// instance, and a run's x' has the bits of hsrb_debug_substep on its perturbed input.
#include "hsrb_fd.cuh"

namespace {
template <int G>
cudaError_t prepare_g(const Plan& p, int* bps) {   // per function and device
  cudaError_t e = cudaFuncSetAttribute(hsrb_fd_kernel<G, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(hsrb_fd_kernel<G, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(bps, hsrb_fd_kernel<G, false>, 32, p.smem);
  return e;
}
template <int G>
cudaError_t launch_g(const FdArgs& f, int grid, size_t smem, cudaStream_t s) {
  if (f.k.params) hsrb_fd_kernel<G, true><<<grid, 32, smem, s>>>(f);
  else hsrb_fd_kernel<G, false><<<grid, 32, smem, s>>>(f);
  return cudaGetLastError();
}
}  // namespace

cudaError_t hsrb_fd_prepare(const Plan& p, int* bps) {
  switch (p.lanes) {
    case 4: return prepare_g<4>(p, bps);
    case 8: return prepare_g<8>(p, bps);
    case 16: return prepare_g<16>(p, bps);
    default: return prepare_g<32>(p, bps);
  }
}

// the run kernel on `grid` one-warp blocks, then the forming kernel
cudaError_t hsrb_fd_launch(const Plan& p, const FdArgs& f, int grid, cudaStream_t s) {
  cudaError_t e;
  switch (p.lanes) {
    case 4: e = launch_g<4>(f, grid, p.smem, s); break;
    case 8: e = launch_g<8>(f, grid, p.smem, s); break;
    case 16: e = launch_g<16>(f, grid, p.smem, s); break;
    default: e = launch_g<32>(f, grid, p.smem, s); break;
  }
  if (e != cudaSuccess) return e;
  const long long threads = (long long)f.k.n * (2 * f.k.m.nv + f.k.m.nu + 1);
  const unsigned blocks = (unsigned)((threads + 127) / 128);
  if (f.centered) hsrb_fd_form_kernel<true><<<blocks, 128, 0, s>>>(f);
  else hsrb_fd_form_kernel<false><<<blocks, 128, 0, s>>>(f);
  return cudaGetLastError();
}
