// The episode kernel (hsrb_episode.cuh), one instance per lanes-per-environment layout of the general path.  Built with
// IEEE division and square root, as the lean reset instance of hsrb_step_g*.cu: reset draws and the quaternion
// normalisation are then bit-identical to hsrb_reset's.
#include "hsrb_episode.cuh"

namespace {
__global__ void episode_clear_kernel(const unsigned char* __restrict__ mask, int n, int* age, float* ret, int* sub) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n || (mask && !mask[e])) return;
  age[e] = 0; ret[e] = 0.f; sub[e] = 0;
}
template <int G>
cudaError_t prepare_g() {   // per function and device
  return cudaFuncSetAttribute(hsrb_episode_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}
template <int G>
cudaError_t launch_g(const EpArgs& a, int grid, size_t smem, cudaStream_t s) {
  hsrb_episode_kernel<G><<<grid, 32, smem, s>>>(a);
  return cudaGetLastError();
}
}  // namespace

cudaError_t hsrb_episode_prepare(const Plan& p) {
  switch (p.lanes) {
    case 4: return prepare_g<4>();
    case 8: return prepare_g<8>();
    case 16: return prepare_g<16>();
    default: return prepare_g<32>();
  }
}

cudaError_t hsrb_episode_launch(const Plan& p, const EpArgs& a, cudaStream_t s) {   // one warp per block (p.threads)
  switch (p.lanes) {
    case 4: return launch_g<4>(a, p.grid, p.smem, s);
    case 8: return launch_g<8>(a, p.grid, p.smem, s);
    case 16: return launch_g<16>(a, p.grid, p.smem, s);
    default: return launch_g<32>(a, p.grid, p.smem, s);
  }
}

cudaError_t hsrb_episode_clear(const unsigned char* mask, int n, int* age, float* ret, int* sub, cudaStream_t s) {
  episode_clear_kernel<<<(n + 255) / 256, 256, 0, s>>>(mask, n, age, ret, sub);
  return cudaGetLastError();
}
