// TEST INFRASTRUCTURE: the rollout instances of the phase-locked action kernels (hsrb_rollout: K actions per environment in
// one launch) against K launches of the step instances, on the CPU through the SIMT emulator (simt_emu.h).  Build:
// tests/test_rollout_emu.py.  Never linked into the product.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#define HSRB_STEP_LOCK_IMPL 1
#define HSRB_WPE_IMPL 1
#include "../../hsr_env_b200/csrc/hsrb_wpe.cuh"

// kernel -2: the phase-locked warp-per-environment kernel (one block of `wpb` warps, so that each warp runs several
// environments of the grid-stride loop); 0: the phase-locked general kernel (3 warps per block).  rollout = 1: one launch
// of the rollout instance for the K actions; 0: K launches of the step instance on slice k of every array, as hsrb_rollout
// falls back to.  state [n, S] is updated in place; ctrl [K, n, nu]; params [n, PRM_COUNT] or null; geofence > 0 turns the
// goal test on (the goal point is each environment's mocap in state).  Outputs: obs [K, n, nq+nv], reward / done / taken /
// bad [K, n], stats [ST_COUNT]; wpe kernel: sep [wpb, 4 * WPE_MAXPAIR] the separating-direction cache of each warp's slice
// at the end of the launch (of the last launch of the K: the last action of the warp's last environment), which the
// outputs cannot show (the cache only saves work): the last action must start from an empty cache in both forms.
extern "C" int emu_rollout(const void* blob, size_t bytes, int kernel, int wpb, int rollout, int n, int K, int nsub,
                           float geofence, float* state, const float* ctrl, const float* params, float* obs, float* reward,
                           unsigned char* done, int* taken, unsigned char* bad, unsigned long long* stats, float* sep) {
  HostModel<float> hm;
  std::string err;
  if (!hm.parse(blob, bytes, err)) { fprintf(stderr, "emu_rollout: %s\n", err.c_str()); return -1; }
  const ModelT<float>& m = hm.m;
  const size_t nobs = (size_t)(m.nq + m.nv);
  std::vector<float> prm(params ? params : (const float*)nullptr, params ? params + (size_t)n * PRM_COUNT : (const float*)nullptr);
  std::vector<int> work(n);
  KArgs a;
  memset(&a, 0, sizeof(a));
  a.m = m;
  a.cfg.qidx0 = 0; a.cfg.qidx1 = 2;
  a.cfg.has_goal = geofence > 0.f ? 1 : 0; a.cfg.geofence = geofence;
  a.n = n; a.S = m.nq + 2 * m.nv + 3; a.nsub = nsub; a.mode = MODE_STEP;
  a.state = state; a.ctrl = ctrl; a.obs = obs; a.reward = reward; a.done = done; a.taken = taken; a.bad = bad; a.stats = stats;
  a.params = params ? prm.data() : nullptr;
  const bool P = params != nullptr;
  if (kernel == -2) {
    PushInfo fi;
    PushTables tb;
    char why[128];
    if (!push_fill_info(hm.m, fi, tb, why, sizeof(why))) { fprintf(stderr, "emu_rollout: %s\n", why); return -2; }
    tb.point(fi, (const unsigned char*)tb.tab.data());
    a.m.ncon_max = WPE_MAXCON; a.m.nefc_max = WPE_MAXROW;
    a.ws_bytes = (unsigned)wpe::slice_bytes();
    a.work = work.data();
    const size_t smem = (size_t)a.ws_bytes * wpb + wpe::shared_tail(a.m);
    // lane 0 of each warp, once the kernel returned (no other warp serves this environment's jobs after its last substep)
    const auto save_sep = [&]() {
      if ((threadIdx.x & 31) == 0) memcpy(sep + (threadIdx.x >> 5) * 4 * WPE_MAXPAIR, wpe::slice(threadIdx.x >> 5).sep, sizeof(float) * 4 * WPE_MAXPAIR);
    };
    if (rollout) {
      emu::launch(1, 32 * wpb, smem, [&]() {
        if (P) hsrb_wpe_rollout_params_kernel_t<true>(a, fi, K); else hsrb_wpe_rollout_kernel_t<true>(a, fi, K);
        save_sep();
      });
    } else {
      for (int k = 0; k < K; k++) {
        KArgs b = a;
        const size_t r = (size_t)k * n;
        b.ctrl = ctrl + r * m.nu; b.obs = obs + r * nobs; b.reward = reward + r; b.done = done + r; b.taken = taken + r; b.bad = bad + r;
        emu::launch(1, 32 * wpb, smem, [&]() {
          if (P) hsrb_wpe_params_kernel_t<true>(b, fi); else hsrb_wpe_kernel_t<true>(b, fi);
          save_sep();
        });
      }
    }
  } else if (kernel == 0) {
    a.ws_bytes = (unsigned)ws_carve<float>(a.m, nullptr, nullptr);
    const int w = 3;
    const int grid = (n + w - 1) / w;
    const size_t smem = (size_t)a.ws_bytes * w + lock_tail_bytes();
    if (rollout) {
      emu::launch(grid, 32 * w, smem, [&]() {
        if (P) hsrb_step_lock_rollout_kernel<true>(a, K); else hsrb_step_lock_rollout_kernel<false>(a, K);
      });
    } else {
      for (int k = 0; k < K; k++) {
        KArgs b = a;
        const size_t r = (size_t)k * n;
        b.ctrl = ctrl + r * m.nu; b.obs = obs + r * nobs; b.reward = reward + r; b.done = done + r; b.taken = taken + r; b.bad = bad + r;
        emu::launch(grid, 32 * w, smem, [&]() {
          if (P) hsrb_step_lock_kernel<true>(b); else hsrb_step_lock_kernel<false>(b);
        });
      }
    }
  } else {
    return -3;
  }
  return 0;
}
