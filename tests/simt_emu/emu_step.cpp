// TEST INFRASTRUCTURE: runs hsr_env_b200/csrc/hsrb_kernels.cuh (the GENERAL CUDA action kernel, unchanged source) on the
// CPU through the SIMT emulator (simt_emu.h).  Build: tests/simt_emu/build.py (build_general).  Never linked into the product.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#define HSRB_STEP_LOCK_IMPL 1
#include "../../hsr_env_b200/csrc/hsrb_kernels.cuh"

namespace {
template <int G>
void run(const KArgs& a, int grid, size_t smem) {
  emu::launch(grid, 32, smem, [&]() { hsrb_step_kernel<G>(a); });
}
}  // namespace

// ncon_max / nefc_max > 0 replace the model's capacities (as hsrb_config does on the device)
extern "C" int emu_general_step(const void* blob, size_t bytes, int G, int n, int nsub, int ncon_max, int nefc_max,
                                const double* qpos, const double* qvel,
                                const double* warm, const double* ctrl, double* qpos_o, double* qvel_o, double* warm_o,
                                int* taken, unsigned char* flags, long long* stats_out) {
  HostModel<float> hm;
  std::string err;
  if (!hm.parse(blob, bytes, err)) { fprintf(stderr, "emu_general_step: %s\n", err.c_str()); return -1; }
  const ModelT<float>& m = hm.m;
  const int S = m.nq + 2 * m.nv + 3, nobs = m.nq + m.nv;
  std::vector<float> state((size_t)n * S, 0.f), c32((size_t)n * (m.nu > 0 ? m.nu : 1)), obs((size_t)n * nobs), reward(n);
  std::vector<unsigned char> done(n), succ(n), bad(n);
  std::vector<int> tk(n);
  std::vector<unsigned long long> stats(ST_COUNT, 0);
  for (int e = 0; e < n; e++) {
    float* st = state.data() + (size_t)e * S;
    for (int i = 0; i < m.nq; i++) st[i] = (float)qpos[(size_t)e * m.nq + i];
    for (int i = 0; i < m.nv; i++) { st[m.nq + i] = (float)qvel[(size_t)e * m.nv + i]; st[m.nq + m.nv + i] = (float)warm[(size_t)e * m.nv + i]; }
    for (int i = 0; i < m.nu; i++) c32[(size_t)e * m.nu + i] = (float)ctrl[(size_t)e * m.nu + i];
  }
  KArgs a;
  memset(&a, 0, sizeof(a));
  a.m = m;
  if (ncon_max > 0) a.m.ncon_max = ncon_max;
  if (nefc_max > 0) a.m.nefc_max = nefc_max;
  a.n = n; a.S = S; a.nsub = nsub; a.mode = MODE_STEP;
  a.ws_bytes = (unsigned)ws_carve<float>(a.m, nullptr, nullptr);
  a.state = state.data(); a.ctrl = c32.data(); a.obs = obs.data(); a.reward = reward.data(); a.done = done.data();
  a.success = succ.data(); a.taken = tk.data(); a.bad = bad.data(); a.stats = stats.data();
  if (G == 0) {   // the phase-locked kernel: one warp per environment, 3 warps per block
    const int wpb = 3;
    emu::launch((n + wpb - 1) / wpb, 32 * wpb, (size_t)a.ws_bytes * wpb + lock_tail_bytes(), [&]() { hsrb_step_lock_kernel(a); });
  }
  const int gpb = G ? 32 / G : 1;
  const int grid = (n + gpb - 1) / gpb;
  const size_t smem = (size_t)a.ws_bytes * gpb;
  if (G == 4) run<4>(a, grid, smem); else if (G == 8) run<8>(a, grid, smem); else if (G == 16) run<16>(a, grid, smem);
  else if (G == 32) run<32>(a, grid, smem); else if (G != 0) return -3;
  for (int e = 0; e < n; e++) {
    const float* st = state.data() + (size_t)e * S;
    for (int i = 0; i < m.nq; i++) qpos_o[(size_t)e * m.nq + i] = st[i];
    for (int i = 0; i < m.nv; i++) { qvel_o[(size_t)e * m.nv + i] = st[m.nq + i]; warm_o[(size_t)e * m.nv + i] = st[m.nq + m.nv + i]; }
    taken[e] = tk[e]; flags[e] = bad[e];
  }
  if (stats_out) for (int i = 0; i < ST_COUNT; i++) stats_out[i] = (long long)stats[i];
  return 0;
}
