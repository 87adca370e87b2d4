// The contact query kernel (hsrb_contacts.cuh), one instance per lanes-per-environment layout of the general path, with and
// without per-environment parameters.  Built with the flags of hsrb_step_g*.cu (IEEE division and square root): its
// stages are then compiled as those of the MODE_DEBUG instance, and its contacts and forces are hsrb_debug_substep's bits.
#include "hsrb_contacts.cuh"

namespace {
template <int G>
cudaError_t prepare_g() {   // per function and device
  cudaError_t e = cudaFuncSetAttribute(hsrb_contacts_kernel<G, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(hsrb_contacts_kernel<G, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  return e;
}
template <int G>
cudaError_t launch_g(const ConArgs& c, int grid, size_t smem, cudaStream_t s) {
  if (c.k.params) hsrb_contacts_kernel<G, true><<<grid, 32, smem, s>>>(c);
  else hsrb_contacts_kernel<G, false><<<grid, 32, smem, s>>>(c);
  return cudaGetLastError();
}
}  // namespace

cudaError_t hsrb_contacts_prepare(const Plan& p) {
  switch (p.lanes) {
    case 4: return prepare_g<4>();
    case 8: return prepare_g<8>();
    case 16: return prepare_g<16>();
    default: return prepare_g<32>();
  }
}

cudaError_t hsrb_contacts_launch(const Plan& p, const ConArgs& c, cudaStream_t s) {   // one warp per block (p.threads)
  switch (p.lanes) {
    case 4: return launch_g<4>(c, p.grid, p.smem, s);
    case 8: return launch_g<8>(c, p.grid, p.smem, s);
    case 16: return launch_g<16>(c, p.grid, p.smem, s);
    default: return launch_g<32>(c, p.grid, p.smem, s);
  }
}
