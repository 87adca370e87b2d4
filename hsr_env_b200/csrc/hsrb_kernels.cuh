// Kernel-side definitions shared by the per-G translation units (hsrb_step_g*.cu) and the API TU (hsrb_api.cu).
//
// One persistent kernel per action: a group of G lanes of a warp owns one environment, loads its state
// (qpos, qvel, qacc_warmstart, mocap, ctrl) from HBM once, keeps state, kinematics, contacts, constraint
// Jacobian and solver vectors in its slice of shared memory for all <=300 substeps, and writes state, obs,
// reward, done and substep counts back once.  No tensor cores: the per-environment systems are 8x8..26x26.
//
// Replaces HSREnv.step's loop over sim.step()  (/root/reference/hsr/env.py:115-135).
#pragma once
#include <cuda_runtime.h>

#include "hsr_core.h"

using namespace hsr;

// dynamic shared memory of the block (the SIMT emulator of tests/simt_emu substitutes a host buffer)
#if defined(HSRB_SIMT_EMU)
#define HSRB_DYN_SMEM(name) unsigned char* name = emu::dyn_smem
#else
#define HSRB_DYN_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
#endif

enum { ST_SUBSTEPS = 0, ST_ITERS, ST_NARROW, ST_LSEVAL, ST_CONTACTS, ST_ROWS, ST_LAUNCHES, ST_BAD, ST_FLOPS, ST_PHASE0, ST_COUNT = ST_PHASE0 + PH_COUNT };

struct KArgs {
  ModelT<float> m;
  EnvCfg<float> cfg;
  int n, S, nsub, mode;
  unsigned opts;           // experiment switches (HSRB_OPTS): bit 0 = no separating-direction cache in the fast kernel
  unsigned ws_bytes;
  unsigned long long seed, env_off;
  float* state;            // [N,S]: qpos nq | qvel nv | qacc_warmstart nv | mocap 3
  unsigned* episode;       // [N]
  const float* ctrl;       // [N,nu]
  const unsigned char* mask;
  float* obs; float* reward; unsigned char* done; unsigned char* success; int* taken; unsigned char* bad;
  float* body_xpos; float* gripper;
  double* dump; unsigned dump_stride;
  unsigned long long* stats;
  const int* order;        // wpe kernel: environment of launch slot r (heaviest first), or null = identity
  int* work;               // wpe kernel: [N] work estimate of this action per environment (the next launch's sort key)
  // per-environment parameters (hsrb_set_env_params): [N, PRM_COUNT] multipliers, or null: the model as it is, and the
  // instances without parameters.  prm_draw: resets redraw the reset environments' rows ~ U[prm_lo, prm_hi)
  float* params;
  int prm_draw;
  float prm_lo[PRM_COUNT], prm_hi[PRM_COUNT];
};

// the scale policy of an instance (hsr_core.h): PARAMS = false reads the model as it is
template <bool PARAMS> struct ScaleOf { typedef NoScale type; };
template <> struct ScaleOf<true> { typedef EnvScale type; };
__device__ __forceinline__ void load_scale(NoScale&, const KArgs&, int) {}
__device__ __forceinline__ void load_scale(EnvScale& sc, const KArgs& a, int env) {
  for (int k = 0; k < PRM_COUNT; k++) sc.s[k] = a.params[(size_t)env * PRM_COUNT + k];
}
// lane 0 of a reset: the environment's parameter draw (hsr_core.h sample_env_params), same key and episode as reset_lane0
__device__ __forceinline__ void reset_params(const KArgs& a, int env, unsigned ep) {
  if (a.prm_draw)
    sample_env_params(a.prm_lo, a.prm_hi, a.seed, (uint32_t)(a.env_off + (unsigned long long)env), ep,
                      a.params + (size_t)env * PRM_COUNT);
}

enum { MODE_STEP = 0, MODE_DEBUG = 1, MODE_FORWARD = 2, MODE_RESET = 3 };

template <int G>
__device__ __forceinline__ void load_state(const KArgs& a, WS<float>& w, const DevGrp<G>& g, int env) {
  const float* st = a.state + (size_t)env * a.S;
  int n0 = a.m.nq + 2 * a.m.nv;
  for (int i = g.lane; i < n0; i += G) w.qpos[i] = st[i];  // qpos|qvel|warm are contiguous in the workspace
  for (int i = g.lane; i < 3; i += G) w.mocap[i] = st[n0 + i];
  for (int i = g.lane; i < WI_COUNT; i += G) w.wi[i] = 0;
  for (int i = g.lane; i < 4 * a.m.npair; i += G) w.sep[i] = 0.f;   // no cached separating directions
}
template <int G>
__device__ __forceinline__ void store_state(const KArgs& a, WS<float>& w, const DevGrp<G>& g, int env) {
  float* st = a.state + (size_t)env * a.S;
  int n0 = a.m.nq + 2 * a.m.nv;
  for (int i = g.lane; i < n0; i += G) st[i] = w.qpos[i];
  for (int i = g.lane; i < 3; i += G) st[n0 + i] = w.mocap[i];
}

// The action kernel.  blockDim.x = 32 (one warp), 32/G environments per block, grid-stride over environments.
// FULL = false: the same kernel without the STEP / DEBUG modes (reset and forward launches): a few KB of code instead of
// several hundred, which matters when it runs between two action kernels on a cold L2 (bench.py flushes L2 between timed
// steps: the masked reset through the full kernel's binary cost 1.4-2.6 ms of instruction fetch from DRAM, 0.03 ms warm).
// Only the lean instance draws parameters at reset.  PARAMS = true (FULL only): STEP / DEBUG with a.params.
template <int G, bool FULL = true, bool PARAMS = false>
__global__ void __launch_bounds__(32) hsrb_step_kernel(const __grid_constant__ KArgs a) {
  HSRB_DYN_SMEM(smem);
  DevGrp<G> g;
  const int gpb = 32 / G;
  const int gi = threadIdx.x / G;
  WS<float> w;
  ws_carve<float>(a.m, &w, smem + (size_t)gi * a.ws_bytes);
  const int nobs = a.m.nq + a.m.nv;
  for (int env = blockIdx.x * gpb + gi; env < a.n; env += gridDim.x * gpb) {
    load_state<G>(a, w, g, env);
    for (int i = g.lane; i < a.m.nu; i += G) w.ctrl[i] = a.ctrl ? a.ctrl[(size_t)env * a.m.nu + i] : 0.f;
    g.sync();
    bool success = false;
    int taken = 0;
    typename ScaleOf<PARAMS>::type sc;
    load_scale(sc, a, env);
    if (FULL && a.mode == MODE_STEP) {
      taken = env_action(a.m, a.cfg, w, g, a.nsub, success, sc);
    } else if (FULL && a.mode == MODE_DEBUG) {
      forward(a.m, w, g, sc);
      euler_solve(a.m, w, g, sc);
      if (g.lane == 0) euler_lane0(a.m, w);
      g.sync();
      if (g.lane == 0) debug_dump(a.m, w, a.dump + (size_t)env * a.dump_stride);
      success = goal_reached(a.m, a.cfg, w);
      taken = 1;
    } else if (a.mode == MODE_RESET) {
      // MujocoEnv.reset + HSREnv.reset_model (mujoco_env.py:83-85, env.py:158-177) for the masked environments
      // environments outside the mask keep their state bit for bit (only their observation is emitted)
      if (!a.mask || a.mask[env]) {
        if (g.lane == 0) {
          unsigned ep = a.episode[env];
          a.episode[env] = ep + 1;
          reset_lane0(a.m, a.cfg, w, a.seed, (uint32_t)(a.env_off + (unsigned long long)env), ep);
          if (!FULL) reset_params(a, env, ep);
        }
        g.sync();
        kinematics_trig(a.m, w, g);
        if (g.lane == 0) kinematics_lane0(a.m, w);  // sim.forward(): normalises free-joint quaternions in qpos
        g.sync();
      }
    } else {  // MODE_FORWARD: body positions of the current state (data.get_body_xpos, env.py:144,180,184)
      kinematics_trig(a.m, w, g);
      if (g.lane == 0) kinematics_lane0(a.m, w);
      g.sync();
      if (a.body_xpos)
        for (int i = g.lane; i < a.m.nbody * 3; i += G) a.body_xpos[(size_t)env * a.m.nbody * 3 + i] = (float)w.xpos[i];
      if (a.gripper && g.lane < 3) {
        GT s = 0;
        for (int k = 0; k < 2; k++) {
          int b = a.m.finger_body[k];
          const GT* R = w.xmat + 9 * b;
          const float* p = a.m.finger_pos + 3 * k;
          s += w.xpos[3 * b + g.lane] + R[3 * g.lane] * (GT)p[0] + R[3 * g.lane + 1] * (GT)p[1] + R[3 * g.lane + 2] * (GT)p[2];
        }
        a.gripper[(size_t)env * 3 + g.lane] = (float)(0.5 * s);
      }
      success = goal_reached(a.m, a.cfg, w);
    }
    store_state<G>(a, w, g, env);
    if (a.obs) for (int i = g.lane; i < nobs; i += G) a.obs[(size_t)env * nobs + i] = w.qpos[i];
    if (g.lane == 0) {
      int flags = w.wi[WI_FLAGS];
      if (a.reward) a.reward[env] = success ? 1.0f : 0.0f;
      if (a.done) a.done[env] = success ? 1 : 0;
      if (a.success) a.success[env] = success ? 1 : 0;
      if (a.taken) a.taken[env] = taken;
      if (a.bad) a.bad[env] = (unsigned char)flags;
      if (a.mode <= MODE_DEBUG) {
      atomicAdd(a.stats + ST_SUBSTEPS, (unsigned long long)taken);
      atomicAdd(a.stats + ST_ITERS, (unsigned long long)w.wi[WI_ITER]);
      atomicAdd(a.stats + ST_NARROW, (unsigned long long)w.wi[WI_NARROW]);
      atomicAdd(a.stats + ST_LSEVAL, (unsigned long long)w.wi[WI_LSEVAL]);
      atomicAdd(a.stats + ST_CONTACTS, (unsigned long long)w.wi[WI_SUMCON]);
      atomicAdd(a.stats + ST_ROWS, (unsigned long long)w.wi[WI_SUMEFC]);
      atomicAdd(a.stats + ST_FLOPS, (unsigned long long)w.wi[WI_KFLOP]);
#ifdef HSRB_PHASE_CLOCKS
      for (int k = 0; k < PH_COUNT; k++) atomicAdd(a.stats + ST_PHASE0 + k, (unsigned long long)w.wi[WI_PHASE0 + k]);
#endif
      if (flags) atomicAdd(a.stats + ST_BAD, 1ull);
      }
    }
    g.sync();
  }
}

// ------------------------------------------------------------------------------------------------ phase-locked general kernel
// The action kernel of the general path for STEP launches: one WARP per environment (32 lanes), a block of several warps
// that run the phases of a substep together (team barriers: the warps share the instruction cache instead of thrashing it)
// and share ONE queue of convex-convex narrowphase jobs: any warp refines any environment's candidate pair (the owner's
// poses, the serving warp's registers), so an environment with ten hull pairs near contact (the gripper on the pan,
// configs[2]) no longer refines them one after the other.  Same arithmetic as hsrb_step_kernel<32>: the stages are the
// functions of hsr_core.h, bitwise.
#define HSRB_LOCK_MAXWARPS 12
struct LockQueue {
  int cnt[4];                                    // [0] long jobs, [1] quick jobs, [2] next to serve
  int jobs[HSRB_LOCK_MAXWARPS * HSR_MAXJOBS];    // (owner warp << 16) | (slot << 8) | pair
};
__host__ __device__ inline size_t lock_tail_bytes() { return sizeof(LockQueue) + 16; }

#if defined(HSRB_STEP_LOCK_IMPL)   // defined by the translation units that own the kernel (hsrb_step_lock*.cu, the emulated build)
#define LOCK_ROLLOUT 0
#define LOCK_ENTRY hsrb_step_lock_kernel
#include "hsrb_step_lock_kernel.cuh"
#undef LOCK_ENTRY
#undef LOCK_ROLLOUT
// the open-loop rollout instances (hsrb_rollout: K actions per environment in one launch; hsrb_step_lock_rollout.cu)
#define LOCK_ROLLOUT 1
#define LOCK_ENTRY hsrb_step_lock_rollout_kernel
#include "hsrb_step_lock_kernel.cuh"
#undef LOCK_ENTRY
#undef LOCK_ROLLOUT
#endif  // HSRB_STEP_LOCK_IMPL

// Launch configuration of one action kernel for one handle, worked out by hsrb_api.cu (configure) on first use.  Every
// kernel translation unit exports the same two entry points: X_prepare(p, &bps) sets the kernel's shared-memory limit
// and returns the resident blocks per SM at p.threads / p.smem; X_launch(p, a, s) launches the template instance p and
// a.mode call for.
struct PushInfo;
struct Plan {
  bool ready;
  int lanes, threads, grid, bps;   // lanes per environment, threads per block, blocks, resident blocks per SM
  unsigned ws;                     // shared-memory bytes of one environment's workspace (KArgs::ws_bytes)
  size_t smem;                     // dynamic shared memory of a block
  int ncon_max, nefc_max;          // contacts / constraint rows the kernel holds per environment
  const PushInfo* fam;             // push / wpe kernels: constants of the sliding-base family
  bool lock;                       // wpe kernel: the phase-locked instance
  cudaError_t (*launch)(const Plan& p, const KArgs& a, cudaStream_t s);
  // hsrb_rollout: nact STEP actions in one launch, or null where the kernel has no instance with the action loop (the
  // rollout then launches `launch` once per action)
  cudaError_t (*rollout)(const Plan& p, const KArgs& a, int nact, cudaStream_t s);
};

cudaError_t hsrb_step_lock_prepare(const Plan& p, int* bps);
cudaError_t hsrb_step_lock_launch(const Plan& p, const KArgs& a, cudaStream_t s);
// the instances with per-environment parameters live in translation units of their own (hsrb_step_lock_params.cu,
// hsrb_step_g*_params.cu): a function the two instances of one unit share is inlined differently than when one calls it
cudaError_t hsrb_step_lock_params_prepare();
cudaError_t hsrb_step_lock_params_launch(const Plan& p, const KArgs& a, cudaStream_t s);
// the instances with the action loop (hsrb_step_lock_rollout.cu): nact actions in one launch
cudaError_t hsrb_step_lock_rollout_prepare();
cudaError_t hsrb_step_lock_rollout_launch(const Plan& p, const KArgs& a, int nact, cudaStream_t s);

// per-G entry points of hsrb_step_kernel, one translation unit each (parallel compilation)
#define HSRB_DECL_G(G)                                                                    \
  cudaError_t hsrb_step##G##_prepare(const Plan& p, int* bps);                           \
  cudaError_t hsrb_step##G##_launch(const Plan& p, const KArgs& a, cudaStream_t s);      \
  cudaError_t hsrb_step##G##_params_prepare();                                           \
  cudaError_t hsrb_step##G##_params_launch(const Plan& p, const KArgs& a, cudaStream_t s);
HSRB_DECL_G(4) HSRB_DECL_G(8) HSRB_DECL_G(16) HSRB_DECL_G(32)

#define HSRB_DEFINE_G(G)                                                                                               \
  cudaError_t hsrb_step##G##_prepare(const Plan& p, int* bps) {                                                        \
    cudaError_t e = cudaFuncSetAttribute(hsrb_step_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024); /* per function, shared by all handles */ \
    if (e == cudaSuccess) e = cudaFuncSetAttribute(hsrb_step_kernel<G, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024); \
    if (e == cudaSuccess) e = hsrb_step##G##_params_prepare();                                                        \
    if (e != cudaSuccess) return e;                                                                                    \
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(bps, hsrb_step_kernel<G>, p.threads, p.smem);                 \
  }                                                                                                                    \
  cudaError_t hsrb_step##G##_launch(const Plan& p, const KArgs& a, cudaStream_t s) {                                   \
    if (a.mode == MODE_RESET || a.mode == MODE_FORWARD) hsrb_step_kernel<G, false><<<p.grid, p.threads, p.smem, s>>>(a); /* the lean instance */ \
    else if (a.params) return hsrb_step##G##_params_launch(p, a, s); /* STEP / DEBUG with parameters */             \
    else hsrb_step_kernel<G><<<p.grid, p.threads, p.smem, s>>>(a);                                                     \
    return cudaGetLastError();                                                                                         \
  }
// the STEP / DEBUG instance with per-environment parameters
#define HSRB_DEFINE_G_PARAMS(G)                                                                                        \
  cudaError_t hsrb_step##G##_params_prepare() {                                                                        \
    return cudaFuncSetAttribute(hsrb_step_kernel<G, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024); \
  }                                                                                                                    \
  cudaError_t hsrb_step##G##_params_launch(const Plan& p, const KArgs& a, cudaStream_t s) {                            \
    hsrb_step_kernel<G, true, true><<<p.grid, p.threads, p.smem, s>>>(a);                                              \
    return cudaGetLastError();                                                                                         \
  }
