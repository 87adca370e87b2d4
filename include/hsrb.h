/* hsrb.h - C ABI of the B200 batched physics backend for hsr-env (libhsrb.so).
 *
 * The reference has no FFI of its own: the seam its hot path sits behind is the mujoco-py object API as used
 * by hsr/ (SURVEY.md §8b).  Each entry point below names the reference call site(s) it replaces.  All pointers
 * are plain device pointers owned by the caller unless the name says "host"; every call is asynchronous on
 * the cudaStream_t passed as `stream` (0 = legacy default stream) unless it says otherwise; nothing throws:
 * the return value is 0 on success and <0 on error, with a thread-local message from hsrb_last_error().
 * One handle per (process, GPU); a handle is not thread-safe.  There is NO CPU fallback.
 */
#ifndef HSRB_H
#define HSRB_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hsrb hsrb_t;

/* mujoco_py.load_model_from_path + MjSim(model)            /root/reference/hsr/mujoco_env.py:33-34
 * model_blob: output of hsr_env_b200.model.Model.to_blob() (MJCF -> flat arrays, hsr_env_b200/mjcf.py).
 * env_id_offset: global id of local env 0 (Philox streams are keyed on the global id, so a trajectory does
 * not depend on how environments are sharded across ranks). */
int hsrb_create(const void* model_blob, size_t bytes, int n_envs, int device, uint64_t seed, uint64_t env_id_offset,
                hsrb_t** out);
int hsrb_destroy(hsrb_t* h);

/* model.nq / nv / nu (mujoco_env.py:88, 44), number of fused bodies, number of blocks (goals) */
int hsrb_dims(hsrb_t* h, int* nq, int* nv, int* nu, int* nbody, int* nblock);

/* Tuning knobs, valid before the first reset/step: lanes of a warp per environment (0 = auto from n_envs;
 * 4, 8, 16 or 32) and the contact / constraint-row capacities (0 = model default; MuJoCo's nconmax/njmax,
 * /root/reference/hsr/models/world.xml:44).  The capacities apply to the general kernel; the fast kernel of the
 * sliding-base family has a fixed capacity of 8 contacts (48 contact rows + 2 limit rows) per environment, which the
 * one-block model cannot exceed by more than a transient (4 floor corners + hull contacts); an overflow sets bit 0 of
 * bad_state on either path. */
int hsrb_config(hsrb_t* h, int lanes_per_env, int ncon_max, int nefc_max);

/* Kernel selection: 0 = auto (for the sliding base with at most one free box - the README block-push family - the
 * warp-per-environment kernel hsrb_wpe.cuh; else the general kernel), 1 = general kernel, 2 = the 8-lane lock-step
 * kernel of the family (hsrb_push.cuh), 3 = the warp-per-environment kernel (2, 3: error if the model is outside the
 * family).  The fast kernels take the single-goal form of hsrb_set_goals only: with a goal list, 3 runs the general
 * kernel and 2 is an error.  Returns the path that will run (1, 2 or 3), or the error hsrb_step would return. */
int hsrb_set_path(hsrb_t* h, int path);

/* GoalSpec(a=block_space, b=goal_space, distance=geofence)  /root/reference/hsr/util.py:70-74, env.py:161-172
 * goal_lohi = {lo[3], hi[3]} (NULL: goals=None, the env is never done), block_lohi = {lo[4], hi[4]} over
 * (x, y, quat[qidx0], quat[qidx1]); min_sep > 0 rejection-samples block (x,y) at least that far apart. */
int hsrb_set_goals(hsrb_t* h, const float* goal_lohi_host, const float* block_lohi_host, float geofence,
                   float min_sep, int qidx0, int qidx1);

/* The general list-of-GoalSpec form of HSREnv              /root/reference/hsr/env.py:126,137-147,161-172
 * success = all_k |pos(a_k) - pos(b_k)| < distance_k, evaluated after every substep.  Endpoint codes: >= 0 a (fused)
 * body id (a body-name endpoint, data.get_body_xpos), -1 the per-environment goal point (a Space endpoint sampled at
 * reset from point_lohi = {lo[3], hi[3]}, or an ndarray endpoint with lo == hi; written to mocap_pos as env.py:169-172
 * does; NULL = the model's mocap_pos0), -2-k fixed point k of fixed_pts[nfixed][3] (further ndarray endpoints).
 * ngoal <= 4, nfixed <= 4.  Replaces any hsrb_set_goals configuration (and vice versa); ngoal = 0 means goals=None.
 * Callable endpoints (env.py:139-140) cannot run inside a kernel: the Python front-end rejects them in batched mode.
 * Models of the sliding-base family run the general kernel when this form is active. */
int hsrb_set_goal_list(hsrb_t* h, int ngoal, const int32_t* a_codes_host, const int32_t* b_codes_host,
                       const float* distance_host, const float* point_lohi_host, const float* fixed_pts_host, int nfixed);

/* HSREnv.new_state: per-joint start spaces                   /root/reference/hsr/env.py:149-156
 * qpos[qpos_adr[s] .. + width[s]) ~ U[lo[s], hi[s]] at every reset (width 1, or 7 for a free joint; lo / hi are
 * [nstart][7]), drawn inside the reset kernel from the environment's Philox stream (key = seed, GLOBAL env id; counter =
 * episode, draw block 4096 + 2 s): reproducible and independent of batch size / sharding.  nstart <= 8; 0 clears. */
int hsrb_set_starts(hsrb_t* h, int nstart, const int32_t* qpos_adr_host, const int32_t* width_host, const float* lo_host,
                    const float* hi_host);

/* MujocoEnv.reset + HSREnv.reset_model                      mujoco_env.py:83-85, env.py:158-177
 * mask[N] (NULL = all): environments to reset.  obs[N, nq+nv] (nullable) receives the new observation. */
int hsrb_reset(hsrb_t* h, const uint8_t* mask, float* obs, void* stream);

/* HSREnv.step: ctrl write, <= nsubsteps x (mj_step, goal test, early break), obs/reward/done   env.py:115-135
 * ctrl[N, nu]; obs[N, nq+nv]; reward[N] = float(success); done = success; substeps_taken[N] = executed
 * substeps (env.py:127-131 breaks early); bad_state[N] bit flags (1 contact overflow, 2 non-finite/huge
 * state, 4 Cholesky pivot clamp).  Any output pointer may be NULL. */
int hsrb_step(hsrb_t* h, const float* ctrl, int nsubsteps, float* obs, float* reward, uint8_t* done, uint8_t* success,
              int32_t* substeps_taken, uint8_t* bad_state, void* stream);

/* nactions x HSREnv.step with the actions given in advance (open-loop rollout)   env.py:115-135
 * mujoco-py has no counterpart; MuJoCo's mujoco.rollout is the analogue.  ctrl[K, N, nu] (K = nactions); obs[K, N, nq+nv],
 * reward / done / bad_state [K, N], substeps_taken[K, N] int32, all nullable: slice k holds what the k-th of K hsrb_step
 * calls would return, bit for bit, and the state afterwards is the state after the K-th.  Nothing else happens between
 * the actions: an environment that reached its goal starts the next action from that state, nothing is reset, episode
 * ages and counters are untouched (as hsrb_step leaves them), and per-environment parameters apply as in hsrb_step.  The
 * counters of hsrb_stats grow as over K steps, except launches: +1 when the selected kernel is the phase-locked wpe or
 * general kernel (one launch for all K actions), +K for every other kernel (one hsrb_step launch per action).
 * nactions < 0, nsubsteps < 0 or a NULL ctrl with nu > 0: -1; nactions == 0 does nothing.  Other errors are hsrb_step's. */
int hsrb_rollout(hsrb_t* h, const float* ctrl, int nactions, int nsubsteps, float* obs, float* reward, uint8_t* done,
                 int32_t* substeps_taken, uint8_t* bad_state, void* stream);

/* gym.wrappers.TimeLimit(max_episode_steps) + the caller's `if done: env.reset()`   hsr/__init__.py:22, control.py:73-75
 * The action kernel exactly as hsrb_step runs it, then one episode kernel.  Each environment has an episode age: the
 * actions since its last reset (hsrb_reset or auto-reset set it to 0, a step adds 1).  terminated = success (hsrb_step's
 * done); truncated = age >= max_episode_steps && !terminated (max_episode_steps 0: no limit); done = terminated |
 * truncated.  With autoreset != 0 every done environment is reset in the same call, after the step, with the Philox draw
 * hsrb_reset(mask = done) would make (key = seed, global env id; counter = its episode, which goes up by one): obs then
 * holds the new episode's first observation for those environments.  final_obs[N, nq+nv] holds, for every environment,
 * the observation the step produced, before any reset.  reward, terminated, truncated, substeps_taken and bad_state
 * describe the step taken.  Where done: ep_length[N] = the episode's length in actions, ep_return[N] = its summed reward,
 * ep_substeps[N] = its summed substeps (int32); elsewhere they are left as they were.  Without autoreset nothing is reset:
 * the caller resets (hsrb_reset) the environments it sees done, until then they report done again on every step.  Any
 * output may be NULL.  The ages, the sums of the running episodes and the counters of hsrb_episode_stats are allocated
 * (zero) on the first call of any hsrb_*episode* function; from then on hsrb_reset zeroes the ages and sums of the
 * environments it resets. */
int hsrb_step_episode(hsrb_t* h, const float* ctrl, int nsubsteps, int max_episode_steps, int autoreset, float* obs, float* reward,
                      uint8_t* terminated, uint8_t* truncated, float* final_obs, int32_t* ep_length, float* ep_return,
                      int32_t* ep_substeps, int32_t* substeps_taken, uint8_t* bad_state, void* stream);

/* The episode kernel of hsrb_step_episode alone, on the outputs of the hsrb_step before it (terminated = its done,
 * required; reward / substeps_taken / bad_state NULL = 0): lets the caller compute an observation of its own (e.g. the
 * 'openai' one, hsrb_openai_obs) of the stepped state before the reset and of the reset state after it.  obs (nullable)
 * receives the new observation of the environments it resets; the other outputs are those of hsrb_step_episode. */
int hsrb_episode_update(hsrb_t* h, int max_episode_steps, int autoreset, const uint8_t* terminated, const float* reward,
                        const int32_t* substeps_taken, const uint8_t* bad_state, float* obs, uint8_t* truncated, float* final_obs,
                        int32_t* ep_length, float* ep_return, int32_t* ep_substeps, void* stream);

/* TimeLimit._elapsed_steps of every environment (hsr/__init__.py:22): age[N] int32 device arrays.  set (NULL = zeros)
 * also restarts the summed reward / substeps of the running episodes at 0: checkpoints, or staggered episode phases. */
int hsrb_set_episode_ages(hsrb_t* h, const int32_t* age, void* stream);
int hsrb_get_episode_ages(hsrb_t* h, int32_t* age, void* stream);

/* Per-environment physics parameters (domain randomization, DESIGN 4.3b): four fp32 multipliers per environment,
 * [0] friction (all five pair_friction coefficients of every contact pair, > 0), [1] block_mass (body_mass and
 * body_inertia of every body in block_body, > 0), [2] actuator_gain (act_kp, >= 0), [3] damping (dof_damping, >= 0),
 * with the meaning of editing those model fields without recomputing the compile-time derived quantities.  Not part of
 * the state.  params[N,4] device fp32, copied into the handle on `stream`; NULL: back to nominal (1.0), ranges cleared,
 * and to the kernels without parameters.  The 8-lane lock-step kernel (path 2) has no instance with parameters: with
 * parameters set, hsrb_step, hsrb_set_path(2) and hsrb_launch_info fail there (-3).  get: the current multipliers
 * (1.0 when never set). */
int hsrb_set_env_params(hsrb_t* h, const float* params, void* stream);
int hsrb_get_env_params(hsrb_t* h, float* params, void* stream);
/* lo_host[4], hi_host[4]: every reset (hsrb_reset's masked environments, the auto-reset of hsrb_step_episode /
 * hsrb_episode_update) redraws the environment's params ~ U[lo, hi) from draw block 8192 of its Philox stream (key = seed,
 * GLOBAL env id; counter = the episode the reset starts); the reset state is the same with or without ranges.  Values
 * outside the domains above, NaN or lo > hi are rejected (-1).  NULL clears: params then persist across resets. */
int hsrb_set_env_param_ranges(hsrb_t* h, const float* lo_host, const float* hi_host);

/* Cumulative counters of the episode kernel, copied to host (synchronises `stream`): [0] episodes finished (done),
 * [1] of them terminated (success), [2] truncated, [3] summed episode length in actions, [4] summed substeps of the
 * finished episodes, [5] steps with a non-zero bad_state, [6] auto-resets, [7] environment actions stepped. */
int hsrb_episode_stats(hsrb_t* h, int64_t* out8_host, void* stream);

/* Same call with HOST buffers (the way the reference's caller holds its numpy arrays, hsr/control.py:48-63):
 * copies ctrl host->device, steps, copies obs/reward/done/substeps device->host, all enqueued on `stream` - the
 * CALLER's stream, so the step is ordered after whatever the caller launched there before (hsrb_reset,
 * hsrb_set_state, a previous step) - and returns after synchronising that stream.  ctrl_host must hold [N, nu]
 * float32, the outputs [N, nq+nv] float32, [N] float32, [N] uint8, [N] int32 (nullable). */
int hsrb_step_host(hsrb_t* h, const float* ctrl_host, int nsubsteps, float* obs_host, float* reward_host,
                   uint8_t* done_host, int32_t* substeps_taken_host, void* stream);

/* sim.get_state / sim.set_state (+ qacc_warmstart, which MuJoCo keeps outside MjSimState)   env.py:69,150,175
 * qpos[N,nq] qvel[N,nv] qacc_warm[N,nv] mocap_pos[N,3]; NULL pointers are skipped. */
int hsrb_get_state(hsrb_t* h, float* qpos, float* qvel, float* qacc_warm, float* mocap_pos, void* stream);
int hsrb_set_state(hsrb_t* h, const float* qpos, const float* qvel, const float* qacc_warm, const float* mocap_pos,
                   void* stream);

/* sim.forward + data.get_body_xpos (block_pos / gripper_pos)      env.py:176,179-186
 * body_xpos[N, nbody, 3]; gripper_pos[N,3] = mean of the two distal finger links (nullable). */
int hsrb_forward(hsrb_t* h, float* body_xpos, float* gripper_pos, void* stream);

/* HSREnv._get_observation, obs_type 'openai'                      env.py:72-110
 * The 25-d Fetch-style observation from the resident state (forward kinematics with 6-D body velocities on the
 * device): grip_pos | object_pos | object_pos - grip_pos | finger qpos (2) | mat2euler(object xmat) |
 * (object_velp - grip_velp) dt | object_velr dt | grip_velp dt | finger qvel dt (2).  The reference branch is dead
 * code in the snapshot (SURVEY.md App. C #8); this is its intent as stated in hsr_env_b200/kin.py.  The finger
 * addresses are the qpos / dof addresses of hand_l_proximal_joint and hand_r_proximal_joint, -1 when --use-dof
 * removed the joint (zeros).  obs25[N, 25]. */
int hsrb_openai_obs(hsrb_t* h, int finger_qposadr_l, int finger_qposadr_r, int finger_dofadr_l, int finger_dofadr_r,
                    float* obs25, void* stream);

/* compute_reward (named by the north star; absent from the snapshot, defined as float(all in_range) to
 * agree with env.py:126,133): reward[N] / success[N] of the CURRENT state, no stepping. */
int hsrb_compute_reward(hsrb_t* h, float* reward, uint8_t* success, void* stream);

/* Teacher-forced parity hook: one substep from the current state with per-stage outputs
 * (xpos, M, qfrc_smooth, qacc_smooth, qacc, contacts, efc_J/D/aref/force, next qpos/qvel) as
 * dump[N, hsrb_debug_size()] doubles, layout = hsr::debug_dump (csrc/hsr_core.h). */
int hsrb_debug_size(hsrb_t* h);
int hsrb_debug_substep(hsrb_t* h, const float* ctrl, double* dump, void* stream);

/* Cumulative counters since creation, copied to host (synchronises `stream`):
 * [0] substeps executed, [1] Newton iterations, [2] narrowphase calls, [3] line-search evaluations,
 * [4] contacts (summed over substeps), [5] constraint rows (summed), [6] kernel launches, [7] environments
 * flagged bad, [8] algorithmic flops (SURVEY.md §8(d) stage formulas with the actual per-substep counts),
 * [9..15] lane-0 clock64 cycles / 16 per phase (kinematics, mass matrix, smooth forces, collision, constraint
 * rows, solver, integration) - zero unless the library was built with -DHSRB_PHASE_CLOCKS. */
int hsrb_stats(hsrb_t* h, int64_t* out16_host, void* stream);

/* Introspection used by bench.py, for the kernel the next hsrb_step would launch: lanes per env, shared-memory bytes
 * per env, resident envs per SM, grid, path (1 general kernel, 2 8-lane lock-step kernel, 3 warp-per-environment
 * kernel: the codes hsrb_set_path returns), threads per block.  Fails where that hsrb_step would fail to launch. */
int hsrb_launch_info(hsrb_t* h, int* out6_host);

/* Measurement aid of bench.py (no reference counterpart): the device's FP32 FMA-loop peak in TFLOP/s (8 independent FMA
 * chains per thread, 2 x 1024 threads per SM, best of 4 timed launches on the legacy stream; synchronises), the
 * denominator of the FP32 roofline fraction SURVEY.md 8(d) defines. */
int hsrb_measure_fp32_peak(int device, double* tflops_out_host);

const char* hsrb_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
