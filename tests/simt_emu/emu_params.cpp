// TEST INFRASTRUCTURE: the action kernels' instances with per-environment parameters (hsr_core.h EnvScale) and their
// instances without, on the CPU through the SIMT emulator (simt_emu.h), plus the reset draw of the parameters.  Build:
// tests/test_env_params_emu.py.  Never linked into the product.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#define HSRB_STEP_LOCK_IMPL 1
#define HSRB_WPE_IMPL 1
#include "../../hsr_env_b200/csrc/hsrb_wpe.cuh"

namespace {
template <int G, bool PARAMS>
void run_general(const KArgs& a, int grid, size_t smem) {
  emu::launch(grid, 32, smem, [&]() { hsrb_step_kernel<G, true, PARAMS>(a); });
}
template <int G>
void run_g(const KArgs& a, bool params, int grid, size_t smem) {
  if (params) run_general<G, true>(a, grid, smem); else run_general<G, false>(a, grid, smem);
}
}  // namespace

// kernel: 4 / 8 / 16 / 32 the general kernel with that many lanes per environment, 0 the phase-locked general kernel
// (3 warps per block), -1 / -2 the warp-per-environment kernel free-running / phase-locked (one block of `wpb` warps).
// params [n, PRM_COUNT] or null: the instance without parameters.
extern "C" int emu_params_step(const void* blob, size_t bytes, int kernel, int wpb, int n, int nsub, const double* qpos,
                               const double* qvel, const double* warm, const double* ctrl, const float* params, double* qpos_o,
                               double* qvel_o, double* warm_o, unsigned char* flags) {
  HostModel<float> hm;
  std::string err;
  if (!hm.parse(blob, bytes, err)) { fprintf(stderr, "emu_params_step: %s\n", err.c_str()); return -1; }
  const ModelT<float>& m = hm.m;
  const int S = m.nq + 2 * m.nv + 3, nobs = m.nq + m.nv;
  std::vector<float> state((size_t)n * S, 0.f), c32((size_t)n * (m.nu > 0 ? m.nu : 1)), obs((size_t)n * nobs), reward(n);
  std::vector<float> prm(params ? params : (const float*)nullptr, params ? params + (size_t)n * PRM_COUNT : (const float*)nullptr);
  std::vector<unsigned char> done(n), succ(n), bad(n);
  std::vector<int> tk(n), work(n);
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
  a.cfg.qidx0 = 0; a.cfg.qidx1 = 2;
  a.n = n; a.S = S; a.nsub = nsub; a.mode = MODE_STEP;
  a.state = state.data(); a.ctrl = c32.data(); a.obs = obs.data(); a.reward = reward.data(); a.done = done.data();
  a.success = succ.data(); a.taken = tk.data(); a.bad = bad.data(); a.stats = stats.data();
  a.params = params ? prm.data() : nullptr;
  if (kernel < 0) {
    PushInfo fi;
    PushTables tb;
    char why[128];
    if (!push_fill_info(hm.m, fi, tb, why, sizeof(why))) { fprintf(stderr, "emu_params_step: %s\n", why); return -2; }
    tb.point(fi, (const unsigned char*)tb.tab.data());
    a.m.ncon_max = WPE_MAXCON; a.m.nefc_max = WPE_MAXROW;
    a.ws_bytes = (unsigned)wpe::slice_bytes();
    a.work = work.data();
    const size_t smem = (size_t)a.ws_bytes * wpb + wpe::shared_tail(a.m);
    emu::launch(1, 32 * wpb, smem, [&]() {   // one block: each warp runs n / wpb environments of the grid-stride loop
      if (kernel == -1) { if (params) hsrb_wpe_params_kernel_t<false>(a, fi); else hsrb_wpe_kernel_t<false>(a, fi); }
      else { if (params) hsrb_wpe_params_kernel_t<true>(a, fi); else hsrb_wpe_kernel_t<true>(a, fi); }
    });
  } else if (kernel == 0) {
    a.ws_bytes = (unsigned)ws_carve<float>(a.m, nullptr, nullptr);
    const int w = 3;
    emu::launch((n + w - 1) / w, 32 * w, (size_t)a.ws_bytes * w + lock_tail_bytes(), [&]() {
      if (params) hsrb_step_lock_kernel<true>(a); else hsrb_step_lock_kernel<false>(a);
    });
  } else {
    a.ws_bytes = (unsigned)ws_carve<float>(a.m, nullptr, nullptr);
    const int gpb = 32 / kernel;
    const int grid = (n + gpb - 1) / gpb;
    const size_t smem = (size_t)a.ws_bytes * gpb;
    const bool p = params != nullptr;
    if (kernel == 4) run_g<4>(a, p, grid, smem); else if (kernel == 8) run_g<8>(a, p, grid, smem);
    else if (kernel == 16) run_g<16>(a, p, grid, smem); else if (kernel == 32) run_g<32>(a, p, grid, smem); else return -3;
  }
  for (int e = 0; e < n; e++) {
    const float* st = state.data() + (size_t)e * S;
    for (int i = 0; i < m.nq; i++) qpos_o[(size_t)e * m.nq + i] = st[i];
    for (int i = 0; i < m.nv; i++) { qvel_o[(size_t)e * m.nv + i] = st[m.nq + i]; warm_o[(size_t)e * m.nv + i] = st[m.nq + m.nv + i]; }
    flags[e] = bad[e];
  }
  return 0;
}

// hsr_core.h sample_env_params: the multipliers a reset of global environment env_id at `episode` draws
extern "C" void emu_env_params(const float* lo, const float* hi, unsigned long long seed, unsigned env_id, unsigned episode,
                               float* out4) {
  hsr::sample_env_params(lo, hi, seed, env_id, episode, out4);
}

// MODE_RESET of the lean general instance (hsrb_reset) for n environments at their first episode, with (lo / hi given) or
// without parameter draws: state_o [n, S], params_o [n, PRM_COUNT] (1.0 where nothing was drawn)
extern "C" int emu_params_reset(const void* blob, size_t bytes, int n, unsigned long long seed, unsigned long long env_off,
                                const float* goal_lohi, const float* block_lohi, const float* lo, const float* hi,
                                float* state_o, float* params_o) {
  HostModel<float> hm;
  std::string err;
  if (!hm.parse(blob, bytes, err)) { fprintf(stderr, "emu_params_reset: %s\n", err.c_str()); return -1; }
  const ModelT<float>& m = hm.m;
  const int S = m.nq + 2 * m.nv + 3, nobs = m.nq + m.nv;
  std::vector<float> state((size_t)n * S, 0.f), obs((size_t)n * nobs);
  std::vector<unsigned> episode(n, 0);
  std::vector<unsigned long long> stats(ST_COUNT, 0);
  for (size_t i = 0; i < (size_t)n * PRM_COUNT; i++) params_o[i] = 1.f;
  KArgs a;
  memset(&a, 0, sizeof(a));
  a.m = m;
  a.cfg.qidx0 = 0; a.cfg.qidx1 = 2;
  a.cfg.has_goal = goal_lohi ? 1 : 0; a.cfg.has_block = block_lohi ? 1 : 0;
  for (int k = 0; k < 3; k++) { a.cfg.goal_lo[k] = goal_lohi ? goal_lohi[k] : 0.f; a.cfg.goal_hi[k] = goal_lohi ? goal_lohi[3 + k] : 0.f; }
  for (int k = 0; k < 4; k++) { a.cfg.block_lo[k] = block_lohi ? block_lohi[k] : 0.f; a.cfg.block_hi[k] = block_lohi ? block_lohi[4 + k] : 0.f; }
  a.n = n; a.S = S; a.mode = MODE_RESET; a.seed = seed; a.env_off = env_off;
  a.state = state.data(); a.episode = episode.data(); a.obs = obs.data(); a.stats = stats.data();
  a.ws_bytes = (unsigned)ws_carve<float>(a.m, nullptr, nullptr);
  if (lo && hi) {
    a.params = params_o; a.prm_draw = 1;
    for (int k = 0; k < PRM_COUNT; k++) { a.prm_lo[k] = lo[k]; a.prm_hi[k] = hi[k]; }
  }
  emu::launch((n + 3) / 4, 32, (size_t)a.ws_bytes * 4, [&]() { hsrb_step_kernel<8, false>(a); });
  memcpy(state_o, state.data(), sizeof(float) * state.size());
  return 0;
}
