// TEST INFRASTRUCTURE: runs hsr_env_b200/csrc/hsrb_episode.cuh (the episode kernel, unchanged source) on the CPU through
// the SIMT emulator (simt_emu.h).  Build: tests/simt_emu/emu_episode.py.  Never linked into the product.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../hsr_env_b200/csrc/hsrb_episode.cuh"

namespace {
template <int G>
void run(const EpArgs& a, int grid, size_t smem) {
  emu::launch(grid, 32, smem, [&]() { hsrb_episode_kernel<G>(a); });
}
}  // namespace

// One episode-kernel launch on n environments.  The reset configuration is the part of EnvCfg reset_lane0 reads: goal
// point space (has_goal, goal_lohi[6]), block space (has_block, block_lohi[8], min_sep, qidx0 / qidx1) and nstart start
// spaces (adr, width, lo[7], hi[7]).  state[n, nq + 2 nv + 3], episode, age, ret, sub are read and written in place; the
// step outputs (term, reward, taken, bad) are inputs; counters[8] accumulate.
extern "C" int emu_episode(const void* blob, size_t bytes, int G, int grid, int n, unsigned long long seed, unsigned long long env_off,
                           int has_goal, const double* goal_lohi, int has_block, const double* block_lohi, double min_sep, int qidx0,
                           int qidx1, int nstart, const int* adr, const int* width, const double* lo, const double* hi,
                           int max_steps, int autoreset, float* state, unsigned* episode, int* age, float* ret, int* sub,
                           const unsigned char* term, const float* reward, const int* taken, const unsigned char* bad,
                           unsigned char* trunc, float* final_obs, float* obs, int* ep_len, float* ep_ret, int* ep_sub,
                           unsigned long long* counters) {
  HostModel<float> hm;
  std::string err;
  if (!hm.parse(blob, bytes, err)) { fprintf(stderr, "emu_episode: %s\n", err.c_str()); return -1; }
  if (G != 4 && G != 8 && G != 16 && G != 32) return -3;
  EpArgs e;
  memset(&e, 0, sizeof(e));
  KArgs& k = e.k;
  k.m = hm.m;
  EnvCfg<float>& c = k.cfg;
  c.has_goal = has_goal; c.has_block = has_block; c.min_sep = (float)min_sep; c.qidx0 = qidx0; c.qidx1 = qidx1;
  for (int i = 0; i < 3; i++) { c.goal_lo[i] = (float)goal_lohi[i]; c.goal_hi[i] = (float)goal_lohi[3 + i]; }
  for (int i = 0; i < 4; i++) { c.block_lo[i] = (float)block_lohi[i]; c.block_hi[i] = (float)block_lohi[4 + i]; }
  c.nstart = nstart;
  for (int s = 0; s < nstart; s++) {
    c.start_adr[s] = adr[s]; c.start_width[s] = width[s];
    for (int i = 0; i < 7; i++) { c.start_lo[s][i] = (float)lo[7 * s + i]; c.start_hi[s][i] = (float)hi[7 * s + i]; }
  }
  k.n = n; k.S = hm.m.nq + 2 * hm.m.nv + 3; k.seed = seed; k.env_off = env_off;
  k.ws_bytes = (unsigned)ws_carve<float>(k.m, nullptr, nullptr);
  k.state = state; k.episode = episode; k.obs = obs;
  e.max_steps = max_steps; e.autoreset = autoreset;
  e.terminated = term; e.reward = reward; e.taken = taken; e.bad = bad;
  e.age = age; e.ret = ret; e.sub = sub;
  e.truncated = trunc; e.final_obs = final_obs; e.ep_length = ep_len; e.ep_return = ep_ret; e.ep_substeps = ep_sub;
  e.counters = counters;
  const size_t smem = (size_t)k.ws_bytes * (32 / G);
  if (G == 4) run<4>(e, grid, smem); else if (G == 8) run<8>(e, grid, smem); else if (G == 16) run<16>(e, grid, smem);
  else run<32>(e, grid, smem);
  return 0;
}
