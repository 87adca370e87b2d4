// libhsrb.so - C ABI of the batched physics backend (include/hsrb.h).
//
// Host side of the action kernel: owns the device copy of the model blob, the resident per-environment
// state [N, S] (qpos | qvel | qacc_warmstart | mocap_pos), the episode counters that key the Philox reset
// streams, and the launch configuration.  Everything is asynchronous on the caller's stream; no entry point
// throws; errors come back as negative codes with a thread-local message.
//
// Replaces mujoco_py.load_model_from_path / MjSim / sim.step / sim.reset / sim.forward / get_state /
// set_state as used by /root/reference/hsr/mujoco_env.py:33-34,83-94 and /root/reference/hsr/env.py:115-177.
#include <cuda_runtime.h>
#include <cub/device/device_radix_sort.cuh>

#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>

#include "../../include/hsrb.h"
#include "hsrb_wpe.cuh"
#include "hsrb_episode.cuh"
#include "hsrb_contacts.cuh"
#include "hsrb_fd.cuh"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) return fail(-2, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

// Experiment switches (INTEGRATION.md), read from the environment once, when the handle is created
struct Knobs {
  unsigned opts = 0;          // HSRB_OPTS: KArgs::opts
  bool wpe_lock = true;       // HSRB_WPE_LOCK=0: free-running warps instead of the phase-locked wpe kernel
  unsigned wpe_teams = 2;     // HSRB_WPE_TEAMS=1|2|4: teams per block of the phase-locked wpe kernel
  bool wpe_sort = true;       // HSRB_WPE_SORT=0: identity launch order of the wpe kernel instead of the work-sorted one
  int wpe_wpb = 0;            // HSRB_WPE_WPB: warps per block of the wpe kernel (0: derived from the batch size)
  bool general_lock = true;   // HSRB_GENERAL_LOCK=0: one-warp-per-block general kernel for STEP launches
};

Knobs read_knobs() {
  Knobs k;
  const auto off = [](const char* name) { const char* v = getenv(name); return v && v[0] == '0'; };
  if (const char* o = getenv("HSRB_OPTS")) k.opts = (unsigned)strtoul(o, nullptr, 0);
  k.wpe_lock = !off("HSRB_WPE_LOCK");
  if (const char* t = getenv("HSRB_WPE_TEAMS")) k.wpe_teams = (unsigned)atoi(t);
  k.wpe_sort = !off("HSRB_WPE_SORT");
  if (const char* w = getenv("HSRB_WPE_WPB")) k.wpe_wpb = atoi(w);
  k.general_lock = !off("HSRB_GENERAL_LOCK");
  return k;
}

__global__ void fill_iota(int* p, int n) { const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = i; }

// Work-sorted launch order of the warp-per-environment kernel (hsrb_wpe_kernel_t): the kernel writes a work estimate per
// environment, a radix sort (cub, descending, stable: ties keep the environment order) turns it into the order of the next
// launch (slot r -> block r % grid, warp r / grid: the heaviest warps of every block form team 0).  Results do not depend
// on it.
struct SortBufs {
  int *work = nullptr, *work_sorted = nullptr, *iota = nullptr, *order = nullptr;
  void* tmp = nullptr;
  size_t tmp_bytes = 0;
  bool valid = false;   // order holds the order of the previous launch
  int alloc(int n, cudaStream_t s) {
    if (work) return 0;
    const size_t nb = sizeof(int) * (size_t)n;
    CU(cudaMalloc(&work, nb)); CU(cudaMalloc(&work_sorted, nb)); CU(cudaMalloc(&iota, nb)); CU(cudaMalloc(&order, nb));
    CU(cudaMemsetAsync(work, 0, nb, s));
    fill_iota<<<(n + 255) / 256, 256, 0, s>>>(iota, n);
    CU(cub::DeviceRadixSort::SortPairsDescending(nullptr, tmp_bytes, work, work_sorted, iota, order, n, 0, 24, s));
    CU(cudaMalloc(&tmp, tmp_bytes));
    return 0;
  }
  int update(int n, cudaStream_t s) {   // the next launch's order
    CU(cub::DeviceRadixSort::SortPairsDescending(tmp, tmp_bytes, work, work_sorted, iota, order, n, 0, 24, s));
    valid = true;
    return 0;
  }
  void free() { cudaFree(work); cudaFree(work_sorted); cudaFree(iota); cudaFree(order); cudaFree(tmp); }
};

// Episode loop (hsrb_step_episode), allocated on first use: ages and sums of the running episodes, cumulative counters,
// and stand-ins for the step outputs the caller does not want
struct EpisodeBufs {
  int *age = nullptr, *sub = nullptr;
  float* ret = nullptr;
  unsigned long long* counters = nullptr;
  unsigned char *term = nullptr, *bad = nullptr;
  float* reward = nullptr;
  int* taken = nullptr;
  int lanes = 0;   // layout the episode kernel was prepared for
  int alloc(int n_envs, cudaStream_t s) {   // zeroed on the caller's stream
    if (age) return 0;
    const size_t n = (size_t)n_envs;
    CU(cudaMalloc(&age, sizeof(int) * n)); CU(cudaMalloc(&sub, sizeof(int) * n)); CU(cudaMalloc(&ret, sizeof(float) * n));
    CU(cudaMalloc(&counters, sizeof(unsigned long long) * EP_COUNT));
    CU(cudaMalloc(&term, n)); CU(cudaMalloc(&bad, n));
    CU(cudaMalloc(&reward, sizeof(float) * n)); CU(cudaMalloc(&taken, sizeof(int) * n));
    CU(cudaMemsetAsync(age, 0, sizeof(int) * n, s)); CU(cudaMemsetAsync(sub, 0, sizeof(int) * n, s));
    CU(cudaMemsetAsync(ret, 0, sizeof(float) * n, s));
    CU(cudaMemsetAsync(counters, 0, sizeof(unsigned long long) * EP_COUNT, s));
    return 0;
  }
  void free() {
    cudaFree(age); cudaFree(sub); cudaFree(ret); cudaFree(counters); cudaFree(term); cudaFree(bad); cudaFree(reward); cudaFree(taken);
  }
};

__global__ void fill_f32(float* p, size_t n, float v) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// Per-environment parameters (hsrb_set_env_params, hsrb_set_env_param_ranges), allocated on first use.  A handle that
// never calls those functions launches the instances without parameters.
struct ParamBufs {
  float* d = nullptr;        // [N, PRM_COUNT] multipliers, 1.0 until set or drawn
  bool on = false;           // STEP / DEBUG launches pass d: the instances with parameters
  bool draw = false;         // resets redraw the reset environments' rows ~ U[lo, hi)
  float lo[PRM_COUNT], hi[PRM_COUNT];
  int alloc(int n, cudaStream_t s) {
    if (d) return 0;
    const size_t cnt = (size_t)n * PRM_COUNT;
    CU(cudaMalloc(&d, sizeof(float) * cnt));
    return nominal(n, s);
  }
  int nominal(int n, cudaStream_t s) {
    const size_t cnt = (size_t)n * PRM_COUNT;
    fill_f32<<<(unsigned)((cnt + 255) / 256), 256, 0, s>>>(d, cnt, 1.f);
    CU(cudaGetLastError());
    return 0;
  }
  void free() { cudaFree(d); }
};

// The action kernels.  K_GENERAL (hsrb_step_kernel<G>) also runs every reset, forward and debug launch; the others
// run STEP launches only.  A new kernel is one more entry here, its configure_* function and one line in select().
enum Kernel { K_GENERAL, K_LOCK, K_PUSH, K_WPE, K_COUNT };
const int kPathCode[K_COUNT] = {1, 1, 2, 3};   // what hsrb_set_path and hsrb_launch_info report

}  // namespace

struct hsrb {
  HostModel<float> hm;      // host copy (pointers into hm.buf)
  ModelT<float> dm;         // same table with device pointers
  unsigned char* d_model = nullptr;
  EnvCfg<float> cfg;
  int n = 0, device = 0, S = 0, num_sm = 0;
  unsigned long long seed = 0, env_off = 0;
  float* d_state = nullptr;
  unsigned* d_episode = nullptr;
  unsigned long long* d_stats = nullptr;
  long long launches = 0;
  Knobs knobs;
  int lanes_req = 0;        // hsrb_config's lanes per environment (0: the plan's choice)
  int path = 0;             // hsrb_set_path
  Plan plan[K_COUNT];       // launch configuration per kernel, worked out on first use
  // sliding base + at most one free box (hsrb_push.cuh, hsrb_wpe.cuh)
  PushInfo fast;
  PushTables fast_tab;
  unsigned char* d_fast_tab = nullptr;
  bool fast_ok = false, wpe_ok = false;
  char fast_why[128] = "";
  SortBufs sort;
  EpisodeBufs ep;
  ParamBufs prm;
  int con_lanes = 0;        // layout the contact query kernel was prepared for (hsrb_contacts)
  int fd_lanes = 0, fd_bps = 0;   // layout the transition-derivative kernels were prepared for, its resident blocks per SM
  size_t fd_smem = 0;             // ... and the shared memory of a block fd_bps holds for
  float* d_fd = nullptr;    // hsrb_transition_fd scratch, fd_words 4-byte words
  size_t fd_words = 0;
  // scratch for the host-buffer entry point
  float *d_ctrl = nullptr, *d_obs = nullptr, *d_reward = nullptr;
  unsigned char* d_done = nullptr;
  int* d_taken = nullptr;
};

namespace {

// The kernel a STEP launch of the handle runs.  The fast kernels take the sliding-base family in its env_wrapper goal form
// only (one block against the goal point); among them, auto (path 0) and path 3 take the warp-per-environment kernel,
// phase-locked, two teams per block - measured on B200, round 2, TimeLimit workload: 48.4 M substeps/s at 4096 envs
// (lock-step 8-lane kernel 34.6 M, free-running warps 32.9 M), 65.8 M at 131072 envs (52.3 M / 53.2 M).  A goal list
// under path 3 runs the general kernel; under path 2 it is an error.  Per-environment parameters (hsrb_set_env_params) have
// instances in every kernel but the lock-step 8-lane one: under path 2 they are an error as well.
int select(const hsrb* h, Kernel* k) {
  const bool fast = h->fast_ok && h->path != 1 && h->cfg.ngoal == 0;
  if (fast && h->wpe_ok && h->path != 2) *k = K_WPE;
  else if (fast && h->prm.on && h->path == 2)
    return fail(-3, "per-environment parameters are not available in the lock-step fast kernel (path 2, kernel='lockstep')");
  else if (fast && !h->prm.on) *k = K_PUSH;
  else if (h->path == 2) return fail(-3, "fast path not available for this model: %s", h->fast_why);
  else if (h->knobs.general_lock && h->hm.m.npair <= 256 && !h->lanes_req) *k = K_LOCK;
  else *k = K_GENERAL;
  return 0;
}

// Choose lanes-per-environment and the grid: as many lanes per env as keeps every environment resident in
// one wave (more lanes = shorter dependent chain per substep), otherwise fewer lanes / a grid-stride loop.
int configure_general(const hsrb* h, Plan& p) {
  p.ws = (unsigned)ws_carve<float>(h->dm, nullptr, nullptr);
  p.ncon_max = h->dm.ncon_max; p.nefc_max = h->dm.nefc_max;
  p.threads = 32;
  // lanes per environment: the widest layout that holds every environment in one wave; if none does, shared memory
  // decides how many environments an SM holds (one warp per block, 32/G workspaces per block), and among the layouts
  // within 10 % of the best residency the narrowest one wins: the single-lane stages (kinematics, bias forces, Euler)
  // then run for 32/G environments at once.  Measured on B200 (tools/sweep_lanes.py): C3 (nv = 13, 16384 envs)
  // G = 8: 3.5 M substeps/s against 2.6 M (G = 4, one block per SM) and 1.1 M (G = 32); C5 (nv = 26): G = 32 0.53 M
  // against 0.29 M (G = 16)
  const struct { int G; cudaError_t (*prepare)(const Plan&, int*); cudaError_t (*launch)(const Plan&, const KArgs&, cudaStream_t); } cands[4] = {
      {32, hsrb_step32_prepare, hsrb_step32_launch}, {16, hsrb_step16_prepare, hsrb_step16_launch},
      {8, hsrb_step8_prepare, hsrb_step8_launch}, {4, hsrb_step4_prepare, hsrb_step4_launch}};
  int best = -1;
  long long res[4] = {0, 0, 0, 0};
  int bpsv[4] = {0, 0, 0, 0};
  long long resmax = 0;
  for (int k = 0; k < 4; k++) {
    const int G = cands[k].G;
    if (h->lanes_req && G != h->lanes_req) continue;
    p.smem = (size_t)p.ws * (32 / G);
    if (p.smem > 227 * 1024) continue;
    int bps = 0;
    if (cands[k].prepare(p, &bps) != cudaSuccess || bps <= 0) { cudaGetLastError(); continue; }
    bpsv[k] = bps;
    res[k] = (long long)bps * h->num_sm * (32 / G);
    if (res[k] > resmax) resmax = res[k];
  }
  for (int k = 0; k < 4 && best < 0; k++)
    if (res[k] >= h->n) best = k;
  for (int k = 3; k >= 0 && best < 0; k--)
    if (res[k] > 0 && res[k] * 10 >= resmax * 9) best = k;
  if (best < 0) return fail(-3, "no launch configuration fits: workspace %u bytes per environment", p.ws);
  p.lanes = cands[best].G;
  p.launch = cands[best].launch;
  p.bps = bpsv[best];
  p.smem = (size_t)p.ws * (32 / p.lanes);
  const int gpb = 32 / p.lanes;
  const int need = (h->n + gpb - 1) / gpb;
  const int cap = p.bps * h->num_sm;
  p.grid = need < cap ? need : cap;
  if (p.grid < 1) p.grid = 1;
  return 0;
}

// STEP launches of the general path: one warp per environment, as many warps per block as shared memory holds
int configure_lock(const hsrb* h, Plan& p) {
  p.ws = (unsigned)ws_carve<float>(h->dm, nullptr, nullptr);
  p.ncon_max = h->dm.ncon_max; p.nefc_max = h->dm.nefc_max;
  p.lanes = 32;
  p.launch = hsrb_step_lock_launch;
  p.rollout = hsrb_step_lock_rollout_launch;
  const size_t tail = lock_tail_bytes();
  int wpb = (int)((227 * 1024 - tail) / p.ws);
  if (wpb < 1) return fail(-3, "no launch configuration fits: workspace %u bytes per environment", p.ws);
  if (wpb > HSRB_LOCK_MAXWARPS) wpb = HSRB_LOCK_MAXWARPS;
  const int need_w = (h->n + h->num_sm - 1) / h->num_sm;
  if (wpb > need_w) wpb = need_w;
  p.threads = 32 * wpb;
  p.smem = (size_t)p.ws * wpb + tail;
  CU(hsrb_step_lock_prepare(p, &p.bps));
  if (p.bps < 1) return fail(-3, "phase-locked general kernel does not fit on an SM (%zu bytes of shared memory)", p.smem);
  const int need = (h->n + wpb - 1) / wpb;
  const int cap = p.bps * h->num_sm;
  p.grid = need < cap ? need : cap;
  return 0;
}

int configure_push(const hsrb* h, Plan& p) {
  p.ws = (unsigned)push::carve(h->dm, nullptr, nullptr);
  p.ncon_max = PUSH_MAXCON; p.nefc_max = 2 + PUSH_ROWS;
  p.fam = &h->fast;
  p.launch = hsrb_push_launch;
  // lanes per environment: the caller's choice (hsrb_config) when it is one this kernel has, else 8
  const int G = (h->lanes_req == 8 || h->lanes_req == 16 || h->lanes_req == 32) ? h->lanes_req : 8;
  p.lanes = G;
  const int epw = 32 / G;
  // warps per block so that all environments are resident in one wave when they fit: n / (envs per warp) / SMs
  int warps_needed = (h->n + epw - 1) / epw;
  int wpb = (warps_needed + h->num_sm - 1) / h->num_sm;
  if (wpb < 1) wpb = 1;
  const int wpb_max = G == 16 ? 14 : 8;   // __launch_bounds__ of the kernel (hsrb_push.cuh)
  if (wpb == 7 && wpb_max >= 8) wpb = 8;   // two warps on each of the four schedulers: 128 blocks x 32 envs beat 147 x 28 (measured +2 %)
  if (wpb > wpb_max) wpb = wpb_max;
  // shared memory: at most 227 KB per block
  const size_t tail = push::shared_tail(h->dm);
  while (wpb > 1 && (size_t)p.ws * (wpb * epw) + tail > 227 * 1024) wpb--;
  p.threads = 32 * wpb;
  p.smem = (size_t)p.ws * (p.threads / G) + tail;
  CU(hsrb_push_prepare(p, &p.bps));
  if (p.bps < 1) return fail(-3, "fast kernel does not fit on an SM (%zu bytes of shared memory)", p.smem);
  const int epb = p.threads / G;
  const int need = (h->n + epb - 1) / epb;
  const int cap = p.bps * h->num_sm;
  p.grid = need < cap ? need : cap;
  return 0;
}

int configure_wpe(const hsrb* h, Plan& p) {
  p.ws = (unsigned)wpe::slice_bytes();
  p.ncon_max = WPE_MAXCON; p.nefc_max = WPE_MAXROW;
  p.fam = &h->fast;
  p.lock = h->knobs.wpe_lock;
  p.lanes = 32;
  p.launch = hsrb_wpe_launch;
  if (p.lock) p.rollout = hsrb_wpe_rollout_launch;   // the free-running variant has no instance with the action loop
  const size_t tail = wpe::shared_tail(h->dm);
  // one warp per environment; all environments resident in one wave when they fit (warps per block = n / SMs),
  // otherwise the most warps shared memory and the register file hold, and a grid-stride loop over the environments
  int wpb = (h->n + h->num_sm - 1) / h->num_sm;
  if (wpb < 1) wpb = 1;
  if (wpb > WPE_MAXWARPS) wpb = WPE_MAXWARPS;
  if (h->knobs.wpe_wpb >= 1 && h->knobs.wpe_wpb <= WPE_MAXWARPS) wpb = h->knobs.wpe_wpb;
  while (wpb > 1 && (size_t)p.ws * wpb + tail > 227 * 1024) wpb--;
  p.threads = 32 * wpb;
  p.smem = (size_t)p.ws * wpb + tail;
  CU(hsrb_wpe_prepare(p, &p.bps));
  if (p.bps < 1) return fail(-3, "warp-per-environment kernel does not fit on an SM (%zu bytes of shared memory)", p.smem);
  const int need = (h->n + wpb - 1) / wpb;
  const int cap = p.bps * h->num_sm;
  p.grid = need < cap ? need : cap;
  if (wpb > 1 && p.grid < cap && 2 * p.grid > cap) p.grid = cap;   // 4096 envs: 148 blocks of 27-28 instead of 147 of 28 + an idle SM
  return 0;
}

// the plan of kernel k, worked out on first use
int configure(hsrb* h, Kernel k, const Plan** out) {
  Plan& p = h->plan[k];
  if (!p.ready) {
    Plan q = Plan();
    const int rc = k == K_WPE ? configure_wpe(h, q) : k == K_PUSH ? configure_push(h, q) : k == K_LOCK ? configure_lock(h, q)
                                                                                         : configure_general(h, q);
    if (rc) return rc;
    q.ready = true;
    p = q;
  }
  *out = &p;
  return 0;
}

KArgs base_args(hsrb* h) {
  KArgs a;
  memset(&a, 0, sizeof(a));
  a.m = h->dm; a.cfg = h->cfg; a.n = h->n; a.S = h->S;
  a.seed = h->seed; a.env_off = h->env_off; a.state = h->d_state; a.episode = h->d_episode; a.stats = h->d_stats;
  a.opts = h->knobs.opts;
  if (h->prm.on) {
    a.params = h->prm.d; a.prm_draw = h->prm.draw;
    for (int k = 0; k < PRM_COUNT; k++) { a.prm_lo[k] = h->prm.lo[k]; a.prm_hi[k] = h->prm.hi[k]; }
  }
  return a;
}

// nact > 0: a STEP launch of nact actions through the plan's rollout instance (hsrb_rollout; the caller checked there is one)
int run(hsrb* h, KArgs& a, void* stream, int nact = 0) {
  cudaStream_t s = (cudaStream_t)stream;
  Kernel k = K_GENERAL;
  if (a.mode == MODE_STEP) { const int rc = select(h, &k); if (rc) return rc; }
  const Plan* p = nullptr;
  int rc = configure(h, k, &p);
  if (rc) return rc;
  a.ws_bytes = p->ws;
  a.m.ncon_max = p->ncon_max; a.m.nefc_max = p->nefc_max;
  const bool sorted = k == K_WPE && h->knobs.wpe_sort;
  if (k == K_WPE && !(a.opts & 0xf0u)) a.opts |= (h->knobs.wpe_teams & 15u) << 4;
  if (sorted) {
    if ((rc = h->sort.alloc(h->n, s))) return rc;
    a.work = h->sort.work; a.order = h->sort.valid ? h->sort.order : nullptr;
  }
  // (the work-sorted launch order was tried on the phase-locked general kernel too: no gain on configs[2] / [4], 2.80 vs
  // 2.88 and 1.28 vs 1.35 M substeps/s - configs[2] resets every environment before every action, configs[4] runs four
  // warps per block)
  CU(nact ? p->rollout(*p, a, nact, s) : p->launch(*p, a, s));
  if (sorted && (rc = h->sort.update(h->n, s))) return rc;
  h->launches++;
  return 0;
}

// the episode kernel on the outputs of the step before it, in the lean launch layout of the general path
int run_episode(hsrb* h, int max_steps, int autoreset, const unsigned char* term, const float* reward, const int* taken,
                const unsigned char* bad, float* obs, unsigned char* truncated, float* final_obs, int* ep_length, float* ep_return,
                int* ep_substeps, void* stream) {
  int rc = h->ep.alloc(h->n, (cudaStream_t)stream);
  if (rc) return rc;
  const Plan* p = nullptr;
  rc = configure(h, K_GENERAL, &p);
  if (rc) return rc;
  if (h->ep.lanes != p->lanes) {
    CU(hsrb_episode_prepare(*p));
    h->ep.lanes = p->lanes;
  }
  EpArgs e;
  memset(&e, 0, sizeof(e));
  e.k = base_args(h);
  e.k.ws_bytes = p->ws;
  e.k.obs = obs;
  e.max_steps = max_steps; e.autoreset = autoreset;
  e.terminated = term; e.reward = reward; e.taken = taken; e.bad = bad;
  e.age = h->ep.age; e.ret = h->ep.ret; e.sub = h->ep.sub;
  e.truncated = truncated; e.final_obs = final_obs; e.ep_length = ep_length; e.ep_return = ep_return; e.ep_substeps = ep_substeps;
  e.counters = h->ep.counters;
  CU(hsrb_episode_launch(*p, e, (cudaStream_t)stream));
  h->launches++;
  return 0;
}

// FP32 FMA-loop peak of the device (the denominator of bench.py's FP32 roofline): 8 independent chains per thread
__global__ void __launch_bounds__(1024) fma_peak_kernel(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int k = 0; k < 8; k++) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

// ---------------------------------------------------------------------------------------------- 'openai' observation
// The 25-d Fetch-style observation of HSREnv._get_observation (/root/reference/hsr/env.py:72-110; the branch is dead code in
// the snapshot, SURVEY.md App. C #8: this is its intent, stated in hsr_env_b200/kin.py, which stays as the test-side
// oracle) from the resident state, one thread per environment, fp64: forward kinematics with 6-D body velocities down
// the tree (bodies are in tree order), then
//   grip_pos | object_pos | object_pos - grip_pos | finger qpos (2) | mat2euler(object xmat) | (object_velp - grip_velp) dt |
//   object_velr dt | grip_velp dt | finger qvel dt (2)
__device__ __forceinline__ void oq_mul(const double* a, const double* b, double* r) {
  const double r0 = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], r1 = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
  const double r2 = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], r3 = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
  r[0] = r0; r[1] = r1; r[2] = r2; r[3] = r3;
}
__device__ __forceinline__ void oq_mat(const double* q, double* R) {
  const double w = q[0], x = q[1], y = q[2], z = q[3];
  R[0] = w * w + x * x - y * y - z * z; R[1] = 2 * (x * y - w * z); R[2] = 2 * (x * z + w * y);
  R[3] = 2 * (x * y + w * z); R[4] = w * w - x * x + y * y - z * z; R[5] = 2 * (y * z - w * x);
  R[6] = 2 * (x * z - w * y); R[7] = 2 * (y * z + w * x); R[8] = w * w - x * x - y * y + z * z;
}
__device__ __forceinline__ void oq_norm(double* q) {
  double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  n = n < 1e-15 ? 1e-15 : n;
  q[0] /= n; q[1] /= n; q[2] /= n; q[3] /= n;
}
#define OMV(R, v, o) { o[0] = R[0] * v[0] + R[1] * v[1] + R[2] * v[2]; o[1] = R[3] * v[0] + R[4] * v[1] + R[5] * v[2]; o[2] = R[6] * v[0] + R[7] * v[1] + R[8] * v[2]; }
#define OCROSS(a, b, o) { o[0] = a[1] * b[2] - a[2] * b[1]; o[1] = a[2] * b[0] - a[0] * b[2]; o[2] = a[0] * b[1] - a[1] * b[0]; }
__global__ void __launch_bounds__(128) openai_obs_kernel(const ModelT<float> m, const float* __restrict__ state, int n, int S, int block_body,
                                                        int adr_l, int adr_r, int dof_l, int dof_r, float* __restrict__ obs) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const float* qpos = state + (size_t)e * S;
  const float* qvel = qpos + m.nq;
  double xpos[HSRB_MAXBODY][3], xquat[HSRB_MAXBODY][4], velp[HSRB_MAXBODY][3], velr[HSRB_MAXBODY][3];
  for (int k = 0; k < 3; k++) { xpos[0][k] = 0; velp[0][k] = 0; velr[0][k] = 0; }
  xquat[0][0] = 1; xquat[0][1] = xquat[0][2] = xquat[0][3] = 0;
  for (int b = 1; b < m.nbody; b++) {
    const int p = m.body_parent[b], j0 = m.body_jntadr[b], nj = m.body_jntnum[b];
    if (nj == 1 && m.jnt_type[j0] == JNT_FREE) {
      const int a = m.jnt_qposadr[j0], v = m.jnt_dofadr[j0];
      double q[4] = {(double)qpos[a + 3], (double)qpos[a + 4], (double)qpos[a + 5], (double)qpos[a + 6]}, R[9];
      oq_norm(q); oq_mat(q, R);
      const double w[3] = {(double)qvel[v + 3], (double)qvel[v + 4], (double)qvel[v + 5]};
      double wr[3];
      OMV(R, w, wr);
      for (int k = 0; k < 3; k++) { xpos[b][k] = (double)qpos[a + k]; velp[b][k] = (double)qvel[v + k]; velr[b][k] = wr[k]; }
      for (int k = 0; k < 4; k++) xquat[b][k] = q[k];
      continue;
    }
    double Rp[9], pos[3], quat[4], w[3], vel[3], t3[3], d3[3];
    oq_mat(xquat[p], Rp);
    const double bp[3] = {(double)m.body_pos[3 * b], (double)m.body_pos[3 * b + 1], (double)m.body_pos[3 * b + 2]};
    const double bq[4] = {(double)m.body_quat[4 * b], (double)m.body_quat[4 * b + 1], (double)m.body_quat[4 * b + 2], (double)m.body_quat[4 * b + 3]};
    OMV(Rp, bp, t3);
    for (int k = 0; k < 3; k++) { pos[k] = xpos[p][k] + t3[k]; w[k] = velr[p][k]; d3[k] = pos[k] - xpos[p][k]; }
    oq_mul(xquat[p], bq, quat);
    OCROSS(velr[p], d3, t3);
    for (int k = 0; k < 3; k++) vel[k] = velp[p][k] + t3[k];   // origin of b carried rigidly by its parent
    for (int j = j0; j < j0 + nj; j++) {
      double R[9], anchor[3], axis[3];
      oq_mat(quat, R);
      const double jp[3] = {(double)m.jnt_pos[3 * j], (double)m.jnt_pos[3 * j + 1], (double)m.jnt_pos[3 * j + 2]};
      const double ja[3] = {(double)m.jnt_axis[3 * j], (double)m.jnt_axis[3 * j + 1], (double)m.jnt_axis[3 * j + 2]};
      OMV(R, jp, t3);
      for (int k = 0; k < 3; k++) anchor[k] = pos[k] + t3[k];
      OMV(R, ja, axis);
      const int a = m.jnt_qposadr[j], v = m.jnt_dofadr[j];
      const double q = (double)qpos[a] - (double)m.qpos0[a], qd = (double)qvel[v];
      if (m.jnt_type[j] == JNT_SLIDE) {
        for (int k = 0; k < 3; k++) { pos[k] += axis[k] * q; vel[k] += axis[k] * qd; }
      } else {
        const double half = 0.5 * q, sh = sin(half);
        const double dq[4] = {cos(half), sh * ja[0], sh * ja[1], sh * ja[2]};
        oq_mul(quat, dq, quat);
        oq_mat(quat, R);
        OMV(R, jp, t3);
        for (int k = 0; k < 3; k++) { pos[k] = anchor[k] - t3[k]; w[k] += axis[k] * qd; d3[k] = pos[k] - anchor[k]; }
        const double aw[3] = {axis[0] * qd, axis[1] * qd, axis[2] * qd};
        OCROSS(aw, d3, t3);
        for (int k = 0; k < 3; k++) vel[k] += t3[k];
      }
    }
    oq_norm(quat);
    for (int k = 0; k < 3; k++) { xpos[b][k] = pos[k]; velp[b][k] = vel[k]; velr[b][k] = w[k]; }
    for (int k = 0; k < 4; k++) xquat[b][k] = quat[k];
  }
  double gp[3] = {0, 0, 0}, gv[3] = {0, 0, 0};
  for (int f = 0; f < 2; f++) {
    const int b = m.finger_body[f];
    double R[9], r[3], t3[3];
    oq_mat(xquat[b], R);
    const double fp[3] = {(double)m.finger_pos[3 * f], (double)m.finger_pos[3 * f + 1], (double)m.finger_pos[3 * f + 2]};
    OMV(R, fp, r);
    OCROSS(velr[b], r, t3);
    for (int k = 0; k < 3; k++) { gp[k] += 0.5 * (xpos[b][k] + r[k]); gv[k] += 0.5 * (velp[b][k] + t3[k]); }
  }
  const double dt = (double)m.timestep;
  double Rb[9];
  oq_mat(xquat[block_body], Rb);
  // mat2euler, /root/reference/hsr/env.py:256-272
  const double cy = sqrt(Rb[8] * Rb[8] + Rb[5] * Rb[5]);
  const bool cond = cy > 2.220446049250313e-16 * 4;
  const double e2 = cond ? -atan2(Rb[1], Rb[0]) : -atan2(-Rb[3], Rb[4]);
  const double e1 = -atan2(-Rb[2], cy);
  const double e0 = cond ? -atan2(Rb[5], Rb[8]) : 0.0;
  float* o = obs + (size_t)e * 25;
  const double* op = xpos[block_body];
  for (int k = 0; k < 3; k++) {
    o[k] = (float)gp[k]; o[3 + k] = (float)op[k]; o[6 + k] = (float)(op[k] - gp[k]);
    o[14 + k] = (float)((velp[block_body][k] - gv[k]) * dt); o[17 + k] = (float)(velr[block_body][k] * dt); o[20 + k] = (float)(gv[k] * dt);
  }
  o[9] = adr_l >= 0 ? qpos[adr_l] : 0.f; o[10] = adr_r >= 0 ? qpos[adr_r] : 0.f;
  o[11] = (float)e0; o[12] = (float)e1; o[13] = (float)e2;
  o[23] = dof_l >= 0 ? (float)((double)qvel[dof_l] * dt) : 0.f; o[24] = dof_r >= 0 ? (float)((double)qvel[dof_r] * dt) : 0.f;
}
#undef OMV
#undef OCROSS

__global__ void gather_state(const float* __restrict__ st, int n, int S, int off, int w, float* __restrict__ out) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)n * w) return;
  int e = (int)(i / w), k = (int)(i % w);
  out[i] = st[(size_t)e * S + off + k];
}
__global__ void scatter_state(float* __restrict__ st, int n, int S, int off, int w, const float* __restrict__ in) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)n * w) return;
  int e = (int)(i / w), k = (int)(i % w);
  st[(size_t)e * S + off + k] = in[i];
}

}  // namespace

extern "C" {

const char* hsrb_last_error(void) { return g_err; }

int hsrb_create(const void* model_blob, size_t bytes, int n_envs, int device, uint64_t seed, uint64_t env_id_offset,
                hsrb_t** out) {
  if (!model_blob || !out || n_envs <= 0) return fail(-1, "hsrb_create: bad arguments");
  *out = nullptr;
  hsrb* h = new (std::nothrow) hsrb();
  if (!h) return fail(-1, "out of host memory");
  std::string err;
  if (!h->hm.parse(model_blob, bytes, err)) { delete h; return fail(-1, "model blob: %s", err.c_str()); }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    delete h;
    return fail(-2, "no CUDA device (%s): this backend has no CPU fallback", cudaGetErrorString(e));
  }
  if (device < 0 || device >= ndev) { delete h; return fail(-1, "device %d out of range (%d visible)", device, ndev); }
  h->n = n_envs; h->device = device; h->seed = seed; h->env_off = env_id_offset;
  h->knobs = read_knobs();
  h->S = h->hm.m.nq + 2 * h->hm.m.nv + 3;
  memset(&h->cfg, 0, sizeof(h->cfg));
  h->cfg.qidx0 = 0; h->cfg.qidx1 = 2;
#define CUH(call)                                                                                    \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess) { int rc_ = fail(-2, "%s: %s", #call, cudaGetErrorString(e_)); hsrb_destroy(h); return rc_; } \
  } while (0)
  CUH(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUH(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    int rc = fail(-2, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    hsrb_destroy(h);
    return rc;
  }
  h->num_sm = prop.multiProcessorCount;
  CUH(cudaMalloc(&h->d_model, h->hm.buf.size()));
  CUH(cudaMemcpy(h->d_model, h->hm.buf.data(), h->hm.buf.size(), cudaMemcpyHostToDevice));
  HostModel<float> tmp = h->hm;  // copy the table, then point it at the device buffer
  tmp.rebase(h->d_model);
  h->dm = tmp.m;
  h->hm.rebase(h->hm.buf.data());
  CUH(cudaMalloc(&h->d_state, sizeof(float) * (size_t)h->n * h->S));
  CUH(cudaMalloc(&h->d_episode, sizeof(unsigned) * (size_t)h->n));
  CUH(cudaMalloc(&h->d_stats, sizeof(unsigned long long) * ST_COUNT));
  CUH(cudaMemset(h->d_episode, 0, sizeof(unsigned) * (size_t)h->n));
  CUH(cudaMemset(h->d_stats, 0, sizeof(unsigned long long) * ST_COUNT));
  // state after load = mj_resetData: qpos0, zero velocities (MjSim(model), mujoco_env.py:34)
  {
    std::vector<float> row(h->S, 0.f);
    for (int i = 0; i < h->hm.m.nq; i++) row[i] = h->hm.m.qpos0[i];
    for (int k = 0; k < 3; k++) row[h->hm.m.nq + 2 * h->hm.m.nv + k] = h->hm.m.mocap_pos0[k];
    std::vector<float> all((size_t)h->n * h->S);
    for (int e2 = 0; e2 < h->n; e2++) memcpy(all.data() + (size_t)e2 * h->S, row.data(), sizeof(float) * h->S);
    CUH(cudaMemcpy(h->d_state, all.data(), sizeof(float) * all.size(), cudaMemcpyHostToDevice));
  }
#undef CUH
  h->fast_ok = push_fill_info(h->hm.m, h->fast, h->fast_tab, h->fast_why, sizeof(h->fast_why));
  if (h->fast_ok) {
    cudaError_t e2 = cudaMalloc(&h->d_fast_tab, h->fast_tab.bytes());
    if (e2 == cudaSuccess) e2 = cudaMemcpy(h->d_fast_tab, h->fast_tab.tab.data(), h->fast_tab.bytes(), cudaMemcpyHostToDevice);
    if (e2 != cudaSuccess) { int rc_ = fail(-2, "fast-path tables: %s", cudaGetErrorString(e2)); hsrb_destroy(h); return rc_; }
    h->fast_tab.point(h->fast, h->d_fast_tab);
    int nbg = 0;
    for (int gi = 0; gi < h->hm.m.ngeom; gi++) nbg += h->hm.m.geom_body[gi] == h->fast.block_body ? 1 : 0;
    h->wpe_ok = nbg <= WPE_MAXBG && h->hm.m.npair <= WPE_MAXPAIR && h->hm.m.ngeom <= WPE_MAXGEOM;
  }
  *out = h;
  return 0;
}

int hsrb_set_path(hsrb_t* h, int path) {
  if (!h) return fail(-1, "null handle");
  if (path < 0 || path > 3) return fail(-1, "path must be 0 (auto), 1 (general kernel), 2 (lock-step fast kernel) or 3 (warp-per-environment fast kernel)");
  if (path >= 2 && !h->fast_ok) return fail(-3, "fast path not available for this model: %s", h->fast_why);
  if (path == 3 && !h->wpe_ok) return fail(-3, "warp-per-environment kernel not available for this model");
  h->path = path;
  Kernel k;
  const int rc = select(h, &k);
  return rc ? rc : kPathCode[k];
}

int hsrb_destroy(hsrb_t* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaFree(h->d_fast_tab); cudaFree(h->d_model); cudaFree(h->d_state); cudaFree(h->d_episode); cudaFree(h->d_stats);
  cudaFree(h->d_ctrl); cudaFree(h->d_obs); cudaFree(h->d_reward); cudaFree(h->d_done); cudaFree(h->d_taken);
  cudaFree(h->d_fd);
  h->sort.free();
  h->ep.free();
  h->prm.free();
  delete h;
  return 0;
}

int hsrb_dims(hsrb_t* h, int* nq, int* nv, int* nu, int* nbody, int* nblock) {
  if (!h) return fail(-1, "null handle");
  if (nq) *nq = h->hm.m.nq;
  if (nv) *nv = h->hm.m.nv;
  if (nu) *nu = h->hm.m.nu;
  if (nbody) *nbody = h->hm.m.nbody;
  if (nblock) *nblock = h->hm.m.nblock;
  return 0;
}

int hsrb_config(hsrb_t* h, int lanes_per_env, int ncon_max, int nefc_max) {
  if (!h) return fail(-1, "null handle");
  if (lanes_per_env != 0 && lanes_per_env != 4 && lanes_per_env != 8 && lanes_per_env != 16 && lanes_per_env != 32)
    return fail(-1, "lanes_per_env must be 0, 4, 8, 16 or 32");
  h->lanes_req = lanes_per_env;
  if (ncon_max > 0) h->dm.ncon_max = h->hm.m.ncon_max = ncon_max;
  if (nefc_max > 0) h->dm.nefc_max = h->hm.m.nefc_max = nefc_max;
  for (Plan& p : h->plan) p = Plan();
  CU(cudaSetDevice(h->device));
  const Plan* p = nullptr;
  return configure(h, K_GENERAL, &p);
}

int hsrb_set_goals(hsrb_t* h, const float* goal_lohi, const float* block_lohi, float geofence, float min_sep, int qidx0,
                   int qidx1) {
  if (!h) return fail(-1, "null handle");
  if (qidx0 < 0 || qidx0 > 3 || qidx1 < 0 || qidx1 > 3) return fail(-1, "quaternion indices must be in 0..3");
  EnvCfg<float>& c = h->cfg;
  c.has_goal = goal_lohi ? 1 : 0;
  c.has_block = block_lohi ? 1 : 0;
  c.ngoal = 0;
  c.qidx0 = qidx0; c.qidx1 = qidx1; c.geofence = geofence; c.min_sep = min_sep;
  for (int k = 0; k < 3; k++) { c.goal_lo[k] = goal_lohi ? goal_lohi[k] : 0.f; c.goal_hi[k] = goal_lohi ? goal_lohi[3 + k] : 0.f; }
  for (int k = 0; k < 4; k++) { c.block_lo[k] = block_lohi ? block_lohi[k] : 0.f; c.block_hi[k] = block_lohi ? block_lohi[4 + k] : 0.f; }
  return 0;
}

int hsrb_set_goal_list(hsrb_t* h, int ngoal, const int32_t* a_codes, const int32_t* b_codes, const float* distance,
                       const float* point_lohi, const float* fixed_pts, int nfixed) {
  if (!h) return fail(-1, "null handle");
  if (ngoal < 0 || ngoal > HSRB_MAXGOAL) return fail(-1, "at most %d GoalSpecs", HSRB_MAXGOAL);
  if (nfixed < 0 || nfixed > HSRB_MAXFIXED) return fail(-1, "at most %d fixed goal points", HSRB_MAXFIXED);
  if (ngoal > 0 && (!a_codes || !b_codes || !distance)) return fail(-1, "goal list arrays are NULL");
  EnvCfg<float>& c = h->cfg;
  for (int k = 0; k < ngoal; k++) {
    const int codes[2] = {a_codes[k], b_codes[k]};
    for (int e = 0; e < 2; e++) {
      if (codes[e] >= h->hm.m.nbody) return fail(-1, "goal %d: body id %d out of range", k, codes[e]);
      if (codes[e] < -1 - nfixed) return fail(-1, "goal %d: fixed point %d not given", k, -2 - codes[e]);
    }
  }
  c.ngoal = ngoal;
  c.has_goal = ngoal > 0 ? 1 : 0;
  c.has_block = 0;
  for (int k = 0; k < ngoal; k++) { c.goal_a[k] = a_codes[k]; c.goal_b[k] = b_codes[k]; c.goal_dist[k] = distance[k]; }
  for (int k = 0; k < 3; k++) {
    c.goal_lo[k] = point_lohi ? point_lohi[k] : h->hm.m.mocap_pos0[k];
    c.goal_hi[k] = point_lohi ? point_lohi[3 + k] : h->hm.m.mocap_pos0[k];
  }
  for (int k = 0; k < nfixed; k++) for (int i = 0; i < 3; i++) c.fixed_pt[k][i] = fixed_pts[3 * k + i];
  return 0;
}

int hsrb_set_starts(hsrb_t* h, int nstart, const int32_t* qpos_adr, const int32_t* width, const float* lo, const float* hi) {
  if (!h) return fail(-1, "null handle");
  if (nstart < 0 || nstart > HSRB_MAXSTART) return fail(-1, "at most %d joints with a start space", HSRB_MAXSTART);
  if (nstart > 0 && (!qpos_adr || !width || !lo || !hi)) return fail(-1, "start arrays are NULL");
  EnvCfg<float>& c = h->cfg;
  for (int s = 0; s < nstart; s++) {
    if (width[s] != 1 && width[s] != 7) return fail(-1, "start %d: width must be 1 (slide / hinge) or 7 (free joint)", s);
    if (qpos_adr[s] < 0 || qpos_adr[s] + width[s] > h->hm.m.nq) return fail(-1, "start %d: qpos slice out of range", s);
  }
  c.nstart = nstart;
  for (int s = 0; s < nstart; s++) {
    c.start_adr[s] = qpos_adr[s]; c.start_width[s] = width[s];
    for (int k = 0; k < 7; k++) { c.start_lo[s][k] = k < width[s] ? lo[7 * s + k] : 0.f; c.start_hi[s][k] = k < width[s] ? hi[7 * s + k] : 0.f; }
  }
  return 0;
}

#if defined(WPE_CHAIN_CLOCKS)
// experiment hook (not part of include/hsrb.h): the per-environment work array of the last wpe launch -> host
extern "C" int hsrb_debug_work(hsrb_t* h, int* out_host) {
  if (!h || !h->sort.work) return -1;
  cudaDeviceSynchronize();
  return cudaMemcpy(out_host, h->sort.work, sizeof(int) * (size_t)h->n, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -2;
}
#endif

int hsrb_set_env_params(hsrb_t* h, const float* params, void* stream) {
  if (!h) return fail(-1, "null handle");
  CU(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (!params) {   // nominal model, no ranges, the instances without parameters
    h->prm.on = false; h->prm.draw = false;
    return h->prm.d ? h->prm.nominal(h->n, s) : 0;
  }
  int rc = h->prm.alloc(h->n, s);
  if (rc) return rc;
  CU(cudaMemcpyAsync(h->prm.d, params, sizeof(float) * (size_t)h->n * PRM_COUNT, cudaMemcpyDeviceToDevice, s));
  h->prm.on = true;
  return 0;
}

int hsrb_get_env_params(hsrb_t* h, float* params, void* stream) {
  if (!h || !params) return fail(-1, "bad arguments");
  CU(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t cnt = (size_t)h->n * PRM_COUNT;
  if (h->prm.d) CU(cudaMemcpyAsync(params, h->prm.d, sizeof(float) * cnt, cudaMemcpyDeviceToDevice, s));
  else {
    fill_f32<<<(unsigned)((cnt + 255) / 256), 256, 0, s>>>(params, cnt, 1.f);
    CU(cudaGetLastError());
  }
  return 0;
}

int hsrb_set_env_param_ranges(hsrb_t* h, const float* lo_host, const float* hi_host) {
  if (!h) return fail(-1, "null handle");
  if (!lo_host != !hi_host) return fail(-1, "lo and hi must both be given or both be NULL");
  if (!lo_host) { h->prm.draw = false; return 0; }   // parameters persist across resets
  static const char* const names[PRM_COUNT] = {"friction", "block_mass", "actuator_gain", "damping"};
  for (int k = 0; k < PRM_COUNT; k++) {
    const float lo = lo_host[k], hi = hi_host[k];
    const bool positive = k == PRM_FRICTION || k == PRM_BLOCK_MASS;   // > 0; gain and damping >= 0
    if (!std::isfinite(lo) || !std::isfinite(hi) || !(lo <= hi) || (positive ? !(lo > 0.f) : !(lo >= 0.f)))
      return fail(-1, "%s range [%g, %g]: needs finite lo <= hi with lo %s 0", names[k], (double)lo, (double)hi, positive ? ">" : ">=");
  }
  CU(cudaSetDevice(h->device));
  if (!h->prm.d) {   // first use: filled with 1.0 before any stream of the caller's can read it
    int rc = h->prm.alloc(h->n, nullptr);
    if (rc) return rc;
    CU(cudaStreamSynchronize(nullptr));
  }
  for (int k = 0; k < PRM_COUNT; k++) { h->prm.lo[k] = lo_host[k]; h->prm.hi[k] = hi_host[k]; }
  h->prm.draw = true; h->prm.on = true;
  return 0;
}

int hsrb_reset(hsrb_t* h, const uint8_t* mask, float* obs, void* stream) {
  if (!h) return fail(-1, "null handle");
  CU(cudaSetDevice(h->device));
  KArgs a = base_args(h);
  a.mode = MODE_RESET; a.mask = mask; a.obs = obs; a.nsub = 0;
  const int rc = run(h, a, stream);
  if (rc || !h->ep.age) return rc;
  CU(hsrb_episode_clear(mask, h->n, h->ep.age, h->ep.ret, h->ep.sub, (cudaStream_t)stream));
  return 0;
}

int hsrb_step(hsrb_t* h, const float* ctrl, int nsubsteps, float* obs, float* reward, uint8_t* done, uint8_t* success,
              int32_t* substeps_taken, uint8_t* bad_state, void* stream) {
  if (!h) return fail(-1, "null handle");
  if (!ctrl && h->hm.m.nu > 0) return fail(-1, "ctrl is NULL");
  if (nsubsteps < 0) return fail(-1, "nsubsteps < 0");
  CU(cudaSetDevice(h->device));
  KArgs a = base_args(h);
  a.mode = MODE_STEP; a.ctrl = ctrl; a.nsub = nsubsteps; a.obs = obs; a.reward = reward; a.done = done;
  a.success = success; a.taken = substeps_taken; a.bad = bad_state;
  return run(h, a, stream);
}

int hsrb_rollout(hsrb_t* h, const float* ctrl, int nactions, int nsubsteps, float* obs, float* reward, uint8_t* done,
                 int32_t* substeps_taken, uint8_t* bad_state, void* stream) {
  if (!h) return fail(-1, "null handle");
  if (nactions < 0) return fail(-1, "nactions < 0");
  if (!ctrl && h->hm.m.nu > 0) return fail(-1, "ctrl is NULL");
  if (nsubsteps < 0) return fail(-1, "nsubsteps < 0");
  if (nactions == 0) return 0;
  CU(cudaSetDevice(h->device));
  KArgs a = base_args(h);
  a.mode = MODE_STEP; a.ctrl = ctrl; a.nsub = nsubsteps; a.obs = obs; a.reward = reward; a.done = done;
  a.taken = substeps_taken; a.bad = bad_state;
  Kernel k = K_GENERAL;
  const Plan* p = nullptr;
  int rc = select(h, &k);
  if (!rc) rc = configure(h, k, &p);
  if (rc) return rc;
  if (p->rollout) return run(h, a, stream, nactions);   // one launch: the phase-locked wpe and general kernels
  // every other kernel: one hsrb_step launch per action on slice k of each array
  const size_t n = (size_t)h->n, nobs = (size_t)(h->hm.m.nq + h->hm.m.nv), nu = (size_t)h->hm.m.nu;
  for (int i = 0; i < nactions; i++) {
    KArgs b = a;
    const size_t r = (size_t)i * n;
    if (ctrl) b.ctrl = ctrl + r * nu;
    if (obs) b.obs = obs + r * nobs;
    if (reward) b.reward = reward + r;
    if (done) b.done = done + r;
    if (substeps_taken) b.taken = substeps_taken + r;
    if (bad_state) b.bad = bad_state + r;
    if ((rc = run(h, b, stream))) return rc;
  }
  return 0;
}

int hsrb_step_episode(hsrb_t* h, const float* ctrl, int nsubsteps, int max_episode_steps, int autoreset, float* obs, float* reward,
                      uint8_t* terminated, uint8_t* truncated, float* final_obs, int32_t* ep_length, float* ep_return,
                      int32_t* ep_substeps, int32_t* substeps_taken, uint8_t* bad_state, void* stream) {
  if (!h) return fail(-1, "null handle");
  if (max_episode_steps < 0) return fail(-1, "max_episode_steps < 0");
  CU(cudaSetDevice(h->device));
  int rc = h->ep.alloc(h->n, (cudaStream_t)stream);
  if (rc) return rc;
  // what the episode kernel reads goes to the handle's buffers when the caller does not want it
  uint8_t* term = terminated ? terminated : h->ep.term;
  float* rew = reward ? reward : h->ep.reward;
  int32_t* taken = substeps_taken ? substeps_taken : h->ep.taken;
  uint8_t* bad = bad_state ? bad_state : h->ep.bad;
  rc = hsrb_step(h, ctrl, nsubsteps, obs, rew, term, nullptr, taken, bad, stream);
  if (rc) return rc;
  return run_episode(h, max_episode_steps, autoreset, term, rew, taken, bad, obs, truncated, final_obs, ep_length, ep_return,
                     ep_substeps, stream);
}

int hsrb_episode_update(hsrb_t* h, int max_episode_steps, int autoreset, const uint8_t* terminated, const float* reward,
                        const int32_t* substeps_taken, const uint8_t* bad_state, float* obs, uint8_t* truncated, float* final_obs,
                        int32_t* ep_length, float* ep_return, int32_t* ep_substeps, void* stream) {
  if (!h) return fail(-1, "null handle");
  if (!terminated) return fail(-1, "terminated is NULL");
  if (max_episode_steps < 0) return fail(-1, "max_episode_steps < 0");
  CU(cudaSetDevice(h->device));
  return run_episode(h, max_episode_steps, autoreset, terminated, reward, substeps_taken, bad_state, obs, truncated, final_obs,
                     ep_length, ep_return, ep_substeps, stream);
}

int hsrb_set_episode_ages(hsrb_t* h, const int32_t* age, void* stream) {
  if (!h) return fail(-1, "null handle");
  CU(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  int rc = h->ep.alloc(h->n, s);
  if (rc) return rc;
  const size_t n = (size_t)h->n;
  if (age) CU(cudaMemcpyAsync(h->ep.age, age, sizeof(int) * n, cudaMemcpyDeviceToDevice, s));
  else CU(cudaMemsetAsync(h->ep.age, 0, sizeof(int) * n, s));
  CU(cudaMemsetAsync(h->ep.ret, 0, sizeof(float) * n, s));
  CU(cudaMemsetAsync(h->ep.sub, 0, sizeof(int) * n, s));
  return 0;
}

int hsrb_get_episode_ages(hsrb_t* h, int32_t* age, void* stream) {
  if (!h || !age) return fail(-1, "bad arguments");
  CU(cudaSetDevice(h->device));
  int rc = h->ep.alloc(h->n, (cudaStream_t)stream);
  if (rc) return rc;
  CU(cudaMemcpyAsync(age, h->ep.age, sizeof(int) * (size_t)h->n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int hsrb_episode_stats(hsrb_t* h, int64_t* out8, void* stream) {
  static_assert(EP_COUNT == 8, "hsrb.h documents 8 counters");
  if (!h || !out8) return fail(-1, "bad arguments");
  CU(cudaSetDevice(h->device));
  int rc = h->ep.alloc(h->n, (cudaStream_t)stream);
  if (rc) return rc;
  unsigned long long v[EP_COUNT];
  CU(cudaMemcpyAsync(v, h->ep.counters, sizeof(v), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CU(cudaStreamSynchronize((cudaStream_t)stream));
  for (int i = 0; i < EP_COUNT; i++) out8[i] = (int64_t)v[i];
  return 0;
}

int hsrb_step_host(hsrb_t* h, const float* ctrl_host, int nsubsteps, float* obs_host, float* reward_host,
                   uint8_t* done_host, int32_t* taken_host, void* stream) {
  if (!h) return fail(-1, "null handle");
  if (!ctrl_host && h->hm.m.nu > 0) return fail(-1, "ctrl_host is NULL");
  CU(cudaSetDevice(h->device));
  const int n = h->n, nu = h->hm.m.nu, nobs = h->hm.m.nq + h->hm.m.nv;
  if (!h->d_obs) {
    CU(cudaMalloc(&h->d_ctrl, sizeof(float) * (size_t)n * (nu > 0 ? nu : 1)));
    CU(cudaMalloc(&h->d_obs, sizeof(float) * (size_t)n * nobs));
    CU(cudaMalloc(&h->d_reward, sizeof(float) * (size_t)n));
    CU(cudaMalloc(&h->d_done, (size_t)n));
    CU(cudaMalloc(&h->d_taken, sizeof(int) * (size_t)n));
  }
  // Everything is enqueued on the CALLER's stream, behind whatever the caller launched there before (hsrb_reset,
  // hsrb_set_state, a previous step), so no cross-stream ordering is left to the caller; the call returns after the
  // device->host copies have completed.
  cudaStream_t s = (cudaStream_t)stream;
  if (nu > 0) CU(cudaMemcpyAsync(h->d_ctrl, ctrl_host, sizeof(float) * (size_t)n * nu, cudaMemcpyHostToDevice, s));
  int rc = hsrb_step(h, h->d_ctrl, nsubsteps, h->d_obs, h->d_reward, h->d_done, nullptr, h->d_taken, nullptr, s);
  if (rc) return rc;
  if (obs_host) CU(cudaMemcpyAsync(obs_host, h->d_obs, sizeof(float) * (size_t)n * nobs, cudaMemcpyDeviceToHost, s));
  if (reward_host) CU(cudaMemcpyAsync(reward_host, h->d_reward, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, s));
  if (done_host) CU(cudaMemcpyAsync(done_host, h->d_done, (size_t)n, cudaMemcpyDeviceToHost, s));
  if (taken_host) CU(cudaMemcpyAsync(taken_host, h->d_taken, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

int hsrb_get_state(hsrb_t* h, float* qpos, float* qvel, float* qacc_warm, float* mocap_pos, void* stream) {
  if (!h) return fail(-1, "null handle");
  CU(cudaSetDevice(h->device));
  const int nq = h->hm.m.nq, nv = h->hm.m.nv;
  float* outs[4] = {qpos, qvel, qacc_warm, mocap_pos};
  int offs[4] = {0, nq, nq + nv, nq + 2 * nv}, ws[4] = {nq, nv, nv, 3};
  for (int k = 0; k < 4; k++) {
    if (!outs[k] || ws[k] == 0) continue;
    long long tot = (long long)h->n * ws[k];
    gather_state<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->d_state, h->n, h->S, offs[k], ws[k], outs[k]);
  }
  CU(cudaGetLastError());
  return 0;
}

int hsrb_set_state(hsrb_t* h, const float* qpos, const float* qvel, const float* qacc_warm, const float* mocap_pos,
                   void* stream) {
  if (!h) return fail(-1, "null handle");
  CU(cudaSetDevice(h->device));
  const int nq = h->hm.m.nq, nv = h->hm.m.nv;
  const float* ins[4] = {qpos, qvel, qacc_warm, mocap_pos};
  int offs[4] = {0, nq, nq + nv, nq + 2 * nv}, ws[4] = {nq, nv, nv, 3};
  for (int k = 0; k < 4; k++) {
    if (!ins[k] || ws[k] == 0) continue;
    long long tot = (long long)h->n * ws[k];
    scatter_state<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->d_state, h->n, h->S, offs[k], ws[k], ins[k]);
  }
  CU(cudaGetLastError());
  return 0;
}

int hsrb_forward(hsrb_t* h, float* body_xpos, float* gripper_pos, void* stream) {
  if (!h) return fail(-1, "null handle");
  CU(cudaSetDevice(h->device));
  KArgs a = base_args(h);
  a.mode = MODE_FORWARD; a.body_xpos = body_xpos; a.gripper = gripper_pos;
  return run(h, a, stream);
}

int hsrb_openai_obs(hsrb_t* h, int finger_qposadr_l, int finger_qposadr_r, int finger_dofadr_l, int finger_dofadr_r, float* obs25,
                    void* stream) {
  if (!h) return fail(-1, "null handle");
  if (!obs25) return fail(-1, "obs25 is NULL");
  const auto& m = h->hm.m;
  if (m.nblock < 1) return fail(-3, "the 'openai' observation needs a block (hsr/env.py:58)");
  if (m.nbody > HSRB_MAXBODY) return fail(-3, "more than %d bodies", HSRB_MAXBODY);
  if (finger_qposadr_l >= m.nq || finger_qposadr_r >= m.nq || finger_dofadr_l >= m.nv || finger_dofadr_r >= m.nv)
    return fail(-1, "finger joint address out of range");
  CU(cudaSetDevice(h->device));
  openai_obs_kernel<<<(h->n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->dm, h->d_state, h->n, h->S, m.block_body[0], finger_qposadr_l,
                                                                        finger_qposadr_r, finger_dofadr_l, finger_dofadr_r, obs25);
  CU(cudaGetLastError());
  return 0;
}

int hsrb_compute_reward(hsrb_t* h, float* reward, uint8_t* success, void* stream) {
  if (!h) return fail(-1, "null handle");
  CU(cudaSetDevice(h->device));
  KArgs a = base_args(h);
  a.mode = MODE_FORWARD; a.reward = reward; a.success = success;
  return run(h, a, stream);
}

int hsrb_debug_size(hsrb_t* h) {
  if (!h) return fail(-1, "null handle");
  return (int)debug_size(h->dm);
}

int hsrb_debug_substep(hsrb_t* h, const float* ctrl, double* dump, void* stream) {
  if (!h) return fail(-1, "null handle");
  if (!dump) return fail(-1, "dump is NULL");
  CU(cudaSetDevice(h->device));
  KArgs a = base_args(h);
  a.mode = MODE_DEBUG; a.ctrl = ctrl; a.nsub = 1; a.dump = dump; a.dump_stride = (unsigned)debug_size(h->dm);
  return run(h, a, stream);
}

int hsrb_contact_capacity(hsrb_t* h) {
  if (!h) return fail(-1, "null handle");
  return h->dm.ncon_max;   // the general plan's ncon_max (configure_general)
}

// mj_forward + data.contact / mj_contactForce / per-body contact wrenches of the current state, in the lean launch layout of
// the general path whatever kernel hsrb_step selects (hsrb_contacts.cuh)
int hsrb_contacts(hsrb_t* h, const float* ctrl, int max_contacts, int32_t* count, int32_t* pair, float* dist, float* pos,
                  float* frame, float* force, float* body_wrench, uint8_t* bad_state, void* stream) {
  if (!h) return fail(-1, "null handle");
  const bool rows = pair || dist || pos || frame || force;
  if (rows && max_contacts < 1) return fail(-1, "max_contacts < 1 with per-contact outputs");
  CU(cudaSetDevice(h->device));
  const Plan* p = nullptr;
  int rc = configure(h, K_GENERAL, &p);
  if (rc) return rc;
  if (h->con_lanes != p->lanes) {
    CU(hsrb_contacts_prepare(*p));
    h->con_lanes = p->lanes;
  }
  ConArgs c;
  memset(&c, 0, sizeof(c));
  c.k = base_args(h);
  c.k.ws_bytes = p->ws;
  c.k.m.ncon_max = p->ncon_max; c.k.m.nefc_max = p->nefc_max;
  c.k.ctrl = ctrl;
  c.C = rows ? max_contacts : 0;
  c.count = count; c.pair = pair; c.dist = dist; c.pos = pos; c.frame = frame; c.force = force; c.wrench = body_wrench;
  c.bad = bad_state;
  CU(hsrb_contacts_launch(*p, c, (cudaStream_t)stream));
  h->launches++;
  return 0;
}

// mjd_transitionFD for every environment: (environment, run) jobs in the lean launch layout of the general path whatever
// kernel hsrb_step selects, then the forming kernel (hsrb_fd.cuh)
int hsrb_transition_fd(hsrb_t* h, const float* ctrl, float eps, int centered, int nsubsteps, float* A, float* B,
                       float* next_obs, uint8_t* bad_state, void* stream) {
  if (!h) return fail(-1, "null handle");
  if (!(eps > 0.f) || !std::isfinite(eps)) return fail(-1, "eps must be finite and > 0");
  if (nsubsteps < 1) return fail(-1, "nsubsteps < 1");
  CU(cudaSetDevice(h->device));
  const Plan* p = nullptr;
  int rc = configure(h, K_GENERAL, &p);
  if (rc) return rc;
  if (h->fd_lanes != p->lanes || h->fd_smem != p->smem) {
    CU(hsrb_fd_prepare(*p, &h->fd_bps));
    if (h->fd_bps < 1) return fail(-3, "transition-derivative kernel does not fit on an SM (%zu bytes of shared memory)", p->smem);
    h->fd_lanes = p->lanes; h->fd_smem = p->smem;
  }
  FdArgs f;
  memset(&f, 0, sizeof(f));
  f.k = base_args(h);
  f.k.ws_bytes = p->ws;
  f.k.m.ncon_max = p->ncon_max; f.k.m.nefc_max = p->nefc_max;
  f.k.ctrl = ctrl;
  f.eps = eps;
  f.rot_c = cos(0.5 * (double)eps); f.rot_s = sin(0.5 * (double)eps);
  f.centered = centered ? 1 : 0;
  f.nsub = nsubsteps;
  f.nruns = fd_nruns(h->hm.m, centered != 0);
  const size_t words = (size_t)h->n * f.nruns * fd_row(h->hm.m);
  if (words > h->fd_words) {
    CU(cudaFree(h->d_fd));
    h->d_fd = nullptr; h->fd_words = 0;
    CU(cudaMalloc(&h->d_fd, words * sizeof(float)));
    h->fd_words = words;
  }
  f.scratch = h->d_fd;
  f.A = A; f.B = B; f.next_obs = next_obs; f.bad = bad_state;
  const long long blocks = ((long long)h->n * f.nruns + 32 / p->lanes - 1) / (32 / p->lanes);
  const long long cap = (long long)h->fd_bps * h->num_sm;
  CU(hsrb_fd_launch(*p, f, (int)(blocks < cap ? blocks : cap), (cudaStream_t)stream));
  h->launches += 2;
  return 0;
}

int hsrb_stats(hsrb_t* h, int64_t* out9, void* stream) {
  static_assert(ST_COUNT == 16, "hsrb.h documents 16 counters");
  if (!h || !out9) return fail(-1, "bad arguments");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize((cudaStream_t)stream));
  unsigned long long v[ST_COUNT];
  CU(cudaMemcpy(v, h->d_stats, sizeof(v), cudaMemcpyDeviceToHost));
  for (int i = 0; i < ST_COUNT; i++) out9[i] = (int64_t)v[i];
  out9[ST_LAUNCHES] = h->launches;
  return 0;
}

int hsrb_measure_fp32_peak(int device, double* tflops_out) {
  if (!tflops_out) return fail(-1, "bad arguments");
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 2, threads = 1024, iters = 4096;
  float* out = nullptr;
  CU(cudaMalloc(&out, sizeof(float) * (size_t)blocks * threads));
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  double best = 0;
  for (int rep = 0; rep < 5; rep++) {
    cudaEventRecord(e0, 0);
    fma_peak_kernel<<<blocks, threads>>>(out, iters, 0.999f, 0.001f);
    cudaEventRecord(e1, 0);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    const double tf = 2.0 * 64.0 * iters * (double)blocks * threads / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(out);
  CU(cudaGetLastError());
  *tflops_out = best;
  return 0;
}

int hsrb_launch_info(hsrb_t* h, int* out6) {
  if (!h || !out6) return fail(-1, "bad arguments");
  CU(cudaSetDevice(h->device));
  Kernel k;
  const Plan* p = nullptr;
  int rc = select(h, &k);
  if (!rc) rc = configure(h, k, &p);
  if (rc) return rc;
  out6[0] = p->lanes; out6[1] = (int)p->ws; out6[2] = p->bps * (p->threads / p->lanes); out6[3] = p->grid;
  out6[4] = kPathCode[k]; out6[5] = p->threads;
  return 0;
}

}  // extern "C"
