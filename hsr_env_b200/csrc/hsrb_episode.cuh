// The episode kernel: gym.wrappers.TimeLimit and the caller's `if done: env.reset()` on the device
// (/root/reference/hsr/__init__.py:22, /root/reference/hsr/control.py:73-75), run after an action kernel.
//
// Per environment: terminated = success of the step, age += 1, truncated = age >= max_steps && !terminated (max_steps 0:
// no limit), done = terminated | truncated.  The step's qpos | qvel go to final_obs; the episode's length and summed
// reward go to ep_length / ep_return where done; the cumulative counters (EP_*) are warp-aggregated.  With autoreset the
// done environments are reset in the same launch with the stages MODE_RESET of hsrb_step_kernel runs (reset_lane0,
// kinematics_trig, kinematics_lane0, between load_state and store_state): the same Philox draw as hsrb_reset(mask =
// done), so both loops give the same bits, parameter draws included.  Environments that are not reset load and store no
// state.
//
// Layout: the lean launch of the general path (configure() in hsrb_api.cu): G lanes per environment, one warp per block,
// 32 / G workspaces of ws_bytes in shared memory (only the reset stages use them), a grid-stride loop.
#pragma once
#include "hsrb_kernels.cuh"

enum { EP_EPISODES = 0, EP_SUCCESSES, EP_TRUNCATIONS, EP_LENGTH, EP_SUBSTEPS, EP_BAD, EP_RESETS, EP_ACTIONS, EP_COUNT };

struct EpArgs {
  KArgs k;                        // model, goals / starts, n, S, ws_bytes, seed, env_off, state, episode; k.obs = new obs
  int max_steps, autoreset;
  // the step that was taken (outputs of the action kernel); reward / taken / bad may be null (read as 0)
  const unsigned char* terminated; const float* reward; const int* taken; const unsigned char* bad;
  // per-environment episode accumulators: actions since the last reset, summed reward and substeps of the running episode
  int* age; float* ret; int* sub;
  // outputs (nullable)
  unsigned char* truncated; float* final_obs; int* ep_length; float* ep_return; int* ep_substeps;
  unsigned long long* counters;   // [EP_COUNT]
};

__device__ __forceinline__ unsigned long long ep_warp_sum(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int G>
__global__ void __launch_bounds__(32) hsrb_episode_kernel(const __grid_constant__ EpArgs a) {
  HSRB_DYN_SMEM(smem);
  const KArgs& k = a.k;
  DevGrp<G> g;
  const int gpb = 32 / G;
  const int gi = threadIdx.x / G;
  WS<float> w;
  ws_carve<float>(k.m, &w, smem + (size_t)gi * k.ws_bytes);
  const int nobs = k.m.nq + k.m.nv;
  // env0 is the same for all lanes of the warp: the warp stays converged at the ballots and shuffles below
  for (int env0 = blockIdx.x * gpb; env0 < k.n; env0 += gridDim.x * gpb) {
    const int env = env0 + gi;
    const bool valid = env < k.n;
    bool term = false, trunc = false, bad = false;
    int age = 0, sub = 0;
    if (valid) {
      term = a.terminated[env] != 0;
      age = a.age[env] + 1;
      trunc = a.max_steps > 0 && age >= a.max_steps && !term;
      bad = a.bad && a.bad[env] != 0;
      sub = a.sub[env] + (a.taken ? a.taken[env] : 0);
    }
    const bool done = term || trunc;
    const bool reset = done && a.autoreset;
    g.sync();   // every lane of the group has read age / sums before lane 0 overwrites them
    if (valid && a.final_obs)
      for (int i = g.lane; i < nobs; i += G) a.final_obs[(size_t)env * nobs + i] = k.state[(size_t)env * k.S + i];
    if (valid && g.lane == 0) {
      const float ret = a.ret[env] + (a.reward ? a.reward[env] : 0.f);
      if (a.truncated) a.truncated[env] = trunc ? 1 : 0;
      if (done) {
        if (a.ep_length) a.ep_length[env] = age;
        if (a.ep_return) a.ep_return[env] = ret;
        if (a.ep_substeps) a.ep_substeps[env] = sub;
      }
      a.age[env] = reset ? 0 : age;
      a.ret[env] = reset ? 0.f : ret;
      a.sub[env] = reset ? 0 : sub;
    }
    if (valid && reset) {
      // MujocoEnv.reset + HSREnv.reset_model (mujoco_env.py:83-85, env.py:158-177), as MODE_RESET of hsrb_step_kernel
      load_state<G>(k, w, g, env);
      g.sync();
      if (g.lane == 0) {
        const unsigned ep = k.episode[env];
        k.episode[env] = ep + 1;
        reset_lane0(k.m, k.cfg, w, k.seed, (uint32_t)(k.env_off + (unsigned long long)env), ep);
        reset_params(k, env, ep);
      }
      g.sync();
      kinematics_trig(k.m, w, g);
      if (g.lane == 0) kinematics_lane0(k.m, w);  // sim.forward(): normalises free-joint quaternions in qpos
      g.sync();
      store_state<G>(k, w, g, env);
      if (k.obs) for (int i = g.lane; i < nobs; i += G) k.obs[(size_t)env * nobs + i] = w.qpos[i];
      g.sync();
    }
    // one contribution per environment (lane 0 of its group), summed over the warp, one atomic per counter and warp
    const bool lead = valid && g.lane == 0;
    const unsigned c_done = __popc(__ballot_sync(0xffffffffu, lead && done));
    const unsigned c_term = __popc(__ballot_sync(0xffffffffu, lead && term));
    const unsigned c_trunc = __popc(__ballot_sync(0xffffffffu, lead && trunc));
    const unsigned c_bad = __popc(__ballot_sync(0xffffffffu, lead && bad));
    const unsigned c_reset = __popc(__ballot_sync(0xffffffffu, lead && reset));
    const unsigned c_act = __popc(__ballot_sync(0xffffffffu, lead));
    const unsigned long long s_len = ep_warp_sum(lead && done ? (unsigned long long)age : 0ull);
    const unsigned long long s_sub = ep_warp_sum(lead && done ? (unsigned long long)sub : 0ull);
    if ((threadIdx.x & 31) == 0) {
      unsigned long long* c = a.counters;
      if (c_done) atomicAdd(c + EP_EPISODES, (unsigned long long)c_done);
      if (c_term) atomicAdd(c + EP_SUCCESSES, (unsigned long long)c_term);
      if (c_trunc) atomicAdd(c + EP_TRUNCATIONS, (unsigned long long)c_trunc);
      if (s_len) atomicAdd(c + EP_LENGTH, s_len);
      if (s_sub) atomicAdd(c + EP_SUBSTEPS, s_sub);
      if (c_bad) atomicAdd(c + EP_BAD, (unsigned long long)c_bad);
      if (c_reset) atomicAdd(c + EP_RESETS, (unsigned long long)c_reset);
      atomicAdd(c + EP_ACTIONS, (unsigned long long)c_act);
    }
  }
}

// host side (hsrb_episode.cu), in the general kernel's plan p: p.lanes picks G; prepare sets the shared-memory limit
cudaError_t hsrb_episode_prepare(const Plan& p);
cudaError_t hsrb_episode_launch(const Plan& p, const EpArgs& a, cudaStream_t s);
// the environments in `mask` (null = all) start new episodes: their ages and sums restart at 0 (hsrb_reset)
cudaError_t hsrb_episode_clear(const unsigned char* mask, int n, int* age, float* ret, int* sub, cudaStream_t s);
