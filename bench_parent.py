"""Benchmark of the hot path: env actions/sec (300 physics substeps each) of the slide_x/slide_y block-push
configuration (BASELINE.json configs[1]: 4096 batched environments per B200, randomized block-space /
goal-space resets), one process per GPU, weak scaling (4096 environments per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs-per-gpu 4096] [--impl reference] [--no-configs]

A "step" is one env action for every environment of the batch: a masked reset of the environments whose episode
ended on the previous action - success (the caller's ``if done: env.reset()``, /root/reference/hsr/control.py:73-75) or
the reference's ``TimeLimit(max_episode_steps=20)`` (/root/reference/hsr/__init__.py:22) - followed by ``HSREnv.step``
(/root/reference/hsr/env.py:115-135) = up to 300 substeps with the per-substep goal test and early break.  Episode ages
start staggered (env i is i mod 20 actions into its episode), so the mix of episode phases - and with it the work per
action - is the same on every step.  Executed substeps are counted (``substeps_taken``), never assumed to be 300.

Both arms run the SAME workload: same Philox reset streams (global env ids), same host-generated actions, same episode
ages, the same W warm-up actions before the K timed ones.  ``--impl reference`` times the CPU side: the reference's own
implementation (mujoco-py) cannot run here (SURVEY.md §8c), so it is the oracle's fp64 C++ port on all host cores,
labelled ``kind: "port"`` (NOT MuJoCo).

Besides the headline (``value``, configs[1]) the line carries ``configs``: configs[2] (full arm + gripper, 16384 envs,
gripper-block contact workload), configs[3] (2^20 envs of the block-push model sharded over the N ranks: strong
scaling) and configs[4] (4-block clutter), each with its own substeps/s, measured flops per substep and FP32 fraction.

Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

BLOCK_LO, BLOCK_HI = [-.25, -.2, 0., -1.], [-.05, .1, 1., 1.]   # (x, y, qw, qz)   SURVEY.md §8(d) C2
GOAL_LO, GOAL_HI = [-.15, -.2, .017], [0., .1, .017]
GEOFENCE = .05
NSUB = 300
TIME_LIMIT = 20      # gym.wrappers.TimeLimit(env, max_episode_steps=20), /root/reference/hsr/__init__.py:22
BLOB = "c2_push.hsrb"
WORKLOAD = ("c2_push: --use-dof slide_x slide_y --n-blocks 1 --steps-per-action=300 --geofence=.05, "
            "block-space (-.25,-.05)(-.2,.1)(0,1)(-1,1), goal-space (-.15,0)(-.2,.1)(.017,.017), "
            "actions ~ U(ctrlrange), envs reset on success or after 20 actions (TimeLimit), staggered episode ages")
# configs[2]: block on the pan, hand hovering at block height (start spaces of the arm joints), configs[4]: four blocks
C3_BLOCK_LO, C3_BLOCK_HI = [-.1, -.18, 0., -1.], [.1, .18, 1., 1.]
C3_GOAL_LO, C3_GOAL_HI = [-.1, -.18, .422], [.1, .18, .422]
C3_STARTS = {"slide_x": (-.05, .12), "slide_y": (-.1, .1), "arm_lift_joint": (0., .12), "arm_flex_joint": (-1.9, -1.25),
             "wrist_roll_joint": (-1.57, 1.57), "hand_l_proximal_joint": (0., .349), "hand_r_proximal_joint": (0., .349)}
C5_BLOCK_LO, C5_BLOCK_HI = [-.2, -.2, 0., -1.], [.1, .2, 1., 1.]     # 0.3 x 0.4 m patch on the floor in front of the base
C5_GOAL_LO, C5_GOAL_HI = [-.15, -.2, .017], [.1, .2, .017]


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), float(d.get("sm_max_mhz", 1965.0)), "measured (MEASURED_PEAKS.json, burst copy figure)"
    return 6650.0, 1965.0, "fallback (B200_PROFILING.md)"


def host_actions(seed: int, steps: int, n: int, lo, hi, offset: int = 0):
    """Actions ~ U(ctrlrange) for `steps` actions of environments [offset, offset + n), generated on the host so that both
    arms (and every rank count) see the same numbers: one Philox stream per step, rows indexed by the global env id."""
    lo, hi = np.asarray(lo, np.float32), np.asarray(hi, np.float32)
    nu = len(lo)
    out = np.empty((steps, n, nu), np.float32)
    for k in range(steps):
        rng = np.random.Generator(np.random.Philox(key=seed + 7919 * k))
        u = rng.random(((offset + n) * nu,), dtype=np.float32)[offset * nu:]   # rows of the global env ids
        out[k] = lo + (hi - lo) * u.reshape(n, nu)
    return out


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU every 100 ms while the timed region runs (NVML)."""

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ CPU side
def cpu_port_run(n_envs: int, warmup: int, steps: int, threads: int, seed: int = 0, budget_s: float = 1e9):
    """The headline workload on the oracle's fp64 C++ port (one environment per thread at a time), environments
    [0, n_envs) of the same Philox streams, the same actions and episode ages as the GPU arm; `warmup` untimed actions,
    then up to `steps` timed ones (stops early when `budget_s` of stepping time is spent).  Returns (env_actions,
    substeps, seconds, algorithmic flops) of the timed part.  Test infrastructure used as a reported baseline only."""
    from hsr_env_b200.model import Model
    from oracle import port

    model = Model.load(ROOT / "hsr_env_b200" / "blobs" / BLOB)
    cp = port.CpuPort(model)
    cp.set_goals(np.r_[GOAL_LO, GOAL_HI], np.r_[BLOCK_LO, BLOCK_HI], GEOFENCE)
    qpos = np.zeros((n_envs, model.nq)); mocap = np.zeros((n_envs, 3))
    episode = np.zeros(n_envs, np.int64)
    for e in range(n_envs):
        qpos[e], mocap[e] = cp.reset(seed, e, 0)
    qvel = np.zeros((n_envs, model.nv)); warm = np.zeros((n_envs, model.nv))
    age = np.arange(n_envs) % TIME_LIMIT
    done = np.zeros(n_envs, bool)
    acts = host_actions(seed, warmup + steps, n_envs, model.act_ctrlrange[:, 0], model.act_ctrlrange[:, 1])
    actions = substeps = flops = 0
    t_total = 0.0
    for a in range(warmup + steps):
        t0 = time.perf_counter()
        for e in np.nonzero(done | (age >= TIME_LIMIT))[0]:
            episode[e] += 1
            qpos[e], mocap[e] = cp.reset(seed, int(e), int(episode[e]))
            qvel[e] = 0; warm[e] = 0; age[e] = 0
        out = cp.step(qpos, qvel, warm, acts[a].astype(np.float64), mocap, nsub=NSUB, nthreads=threads)
        dt = time.perf_counter() - t0
        qpos, qvel, warm = out["qpos"], out["qvel"], out["warm"]
        done = out["success"].astype(bool)
        age += 1
        if a >= warmup:
            t_total += dt
            actions += n_envs
            substeps += int(out["taken"].sum())
            flops += int(out["counters"][:, 3].sum())
            if t_total > budget_s:
                break
    return actions, substeps, t_total, flops


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_envs = args.envs_per_gpu      # the whole configuration, not a sub-sample: ~0.4 s per action on 16 threads
    acts, subs, secs, flops = cpu_port_run(n_envs, args.warmup, args.steps, cores, seed=args.seed, budget_s=150.0)
    value = acts / secs
    done_steps = acts // n_envs
    line = {
        "impl": "reference", "metric": "env_actions_per_sec", "value": value, "unit": "env-actions/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(1, done_steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "envs_per_gpu": n_envs, "total_envs": n_envs, "substeps_per_action": NSUB,
                   "time_limit": TIME_LIMIT},
        "substeps_per_s": subs / secs, "mean_substeps_per_action": subs / max(1, acts),
        "cpu_baseline": {"value": value, "unit": "env-actions/s", "cores": cores, "kind": "port",
                         "sample": f"{done_steps} of {args.steps} timed actions of all {n_envs} environments ({subs} substeps, {secs:.1f} s) "
                                   f"after {args.warmup} warm-up actions, {cores} host threads; the reference's mujoco-py cannot be "
                                   "installed here: this is the oracle's fp64 C++ port (our own restatement), NOT MuJoCo"},
        "e2e": {"value": value, "unit": "env-actions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU side
def fp32_peak(device_index: int) -> float:
    from hsr_env_b200 import lib as L

    v = ctypes.c_double()
    L.check(L.load().hsrb_measure_fp32_peak(device_index, ctypes.byref(v)))
    return float(v.value)


class _Null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def run_workload(torch, D, dev, *, blob, goals, starts, n_local, env_offset, steps, warmup, seed, kernel="auto",
                 lanes=0, min_sep=0.0, flush=None, time_limit=TIME_LIMIT, sampler=None):
    """`warmup` untimed + `steps` timed actions of one configuration on this rank's slice [env_offset, env_offset +
    n_local) of the global environments.  Returns a dict with device-timed seconds (max over ranks), substeps, flops,
    contacts, launch info and the env (open, for follow-up legs)."""
    from hsr_env_b200.env import BatchedHSREnv

    env = BatchedHSREnv(blob, goals, starts=starts, steps_per_action=NSUB, n_envs=n_local, device=dev, seed=seed,
                        env_id_offset=env_offset, lanes_per_env=lanes, kernel=kernel, min_block_separation=min_sep)
    info = env.launch_info()
    acts_h = host_actions(seed, warmup + steps, n_local, env.model.act_ctrlrange[:, 0], env.model.act_ctrlrange[:, 1], offset=env_offset)
    actions = torch.from_numpy(acts_h).to(dev)
    env.reset()
    age = ((torch.arange(n_local, device=dev) + env_offset) % time_limit).to(torch.int32)
    done = torch.zeros(n_local, dtype=torch.bool, device=dev)
    taken_sum = torch.zeros((), dtype=torch.int64, device=dev)
    succ_sum = torch.zeros((), dtype=torch.int64, device=dev)
    reset_sum = torch.zeros((), dtype=torch.int64, device=dev)
    kstart = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    kend = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]

    one = torch.ones((), dtype=torch.int32, device=dev)

    def next_mask():
        """harness bookkeeping, outside the timed bracket: which environments start a new episode before the next action"""
        return (done | (age >= time_limit)).to(torch.uint8)

    def one_step(k, mask, timed=None):
        """the timed work of a step: masked reset + action (reset kernel, action kernel, launch-order sort)"""
        nonlocal done
        env.reset(mask=mask)
        if timed is not None:
            kstart[timed].record()   # the action kernel alone (torch's current stream = the launching stream)
        obs, reward, done, inf = env.step(actions[k])
        if timed is not None:
            kend[timed].record()
        return inf["substeps_taken"]

    def after_step(mask, timed):
        """harness bookkeeping after the bracket: episode ages (reset environments are one action old), counters"""
        nonlocal age, reset_sum
        age = torch.where(mask.bool(), one, age + 1)
        if timed:
            reset_sum += mask.sum()

    for k in range(warmup):
        m_ = next_mask()
        one_step(k, m_)
        after_step(m_, False)
    torch.cuda.synchronize(dev)
    st0 = env.stats()
    starts_ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends_ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    D.barrier()
    torch.cuda.synchronize(dev)
    snap = [t.clone() for t in env.get_state()] + [done.clone(), age.clone()]
    with (sampler if sampler is not None else _Null()):
        for k in range(steps):
            if flush is not None:
                flush.fill_(k & 0xff)           # evict L2 between timed iterations (outside the event bracket)
            m_ = next_mask()
            starts_ev[k].record()
            taken = one_step(warmup + k, m_, timed=k)
            ends_ev[k].record()
            after_step(m_, True)
            taken_sum += taken.sum()
            succ_sum += done.sum()
        torch.cuda.synchronize(dev)
    D.barrier()
    secs = sum(s.elapsed_time(e) for s, e in zip(starts_ev, ends_ev)) * 1e-3
    kernel_s = sum(s.elapsed_time(e) for s, e in zip(kstart, kend)) * 1e-3 / steps   # mean action-kernel launch
    st1 = env.stats()
    secs_max = D.max_over_ranks(secs, dev)
    d = {k: float(st1[k] - st0[k]) for k in ("substeps", "flops", "contacts", "efc_rows", "newton_iters", "bad_envs", "launches")}
    tot = D.sum_over_ranks([float(taken_sum.item()), float(succ_sum.item()), d["bad_envs"], d["flops"], d["contacts"], d["newton_iters"],
                            float(reset_sum.item())], dev)
    return dict(env=env, info=info, secs=secs_max, kernel_s=kernel_s, substeps=tot[0], successes=tot[1], bad=tot[2], flops=tot[3],
                contacts=tot[4], iters=tot[5], resets=tot[6], launches=int(d["launches"]), snap=snap, actions_host=acts_h,
                local_substeps=float(taken_sum.item()), local_successes=float(succ_sum.item()), local_bad=d["bad_envs"],
                stats0=st0, stats1=st1)


def config_entry(r, n_total, steps, peak_tf, world, extra=None):
    """Throughput / roofline entry of one configuration."""
    sub_s = r["substeps"] / r["secs"]
    f_alg = r["flops"] / max(1.0, r["substeps"])
    tf = r["flops"] / r["secs"] / 1e12 / world
    e = {"envs_total": n_total, "steps": steps, "env_actions_per_s": n_total * steps / r["secs"], "substeps_per_s": sub_s,
         "substeps_per_s_per_gpu": sub_s / world, "ms_per_step": 1e3 * r["secs"] / steps,
         "mean_substeps_per_action": r["substeps"] / (n_total * steps), "mean_flops_per_substep": f_alg,
         "mean_contacts_per_substep": r["contacts"] / max(1.0, r["substeps"]),
         "mean_newton_iters_per_substep": r["iters"] / max(1.0, r["substeps"]),
         "fp32_tflops_per_gpu": tf, "fp32_frac": tf / peak_tf, "bad_states": r["bad"],
         "success_per_action": r["successes"] / (n_total * steps), "resets_per_action": r["resets"] / (n_total * steps),
         "kernel": r["info"]["kernel"], "lanes_per_env": r["info"]["lanes_per_env"], "threads_per_block": r["info"]["threads_per_block"],
         "grid": r["info"]["grid"], "smem_per_env": r["info"]["smem_per_env"], "resident_envs_per_sm": r["info"]["envs_per_sm"]}
    ph = {k: r["stats1"]["phase_cycles"][k] - r["stats0"]["phase_cycles"][k] for k in r["stats1"]["phase_cycles"]}
    if sum(ph.values()) > 0:   # only with the -DHSRB_PHASE_CLOCKS build (HSRB_LIB=.../libhsrb_prof.so)
        tot = float(sum(ph.values()))
        e["phase_share"] = {k: round(v / tot, 4) for k, v in ph.items()}
    if extra:
        e.update(extra)
    return e


def regime_census(env, blob_name, n_sample=256):
    """What kinds of contacts the states of a run hold (oracle port on a host copy of `n_sample` states, outside every
    timed region): evidence that configs[2] really is in the gripper-block regime."""
    sys.path.insert(0, str(ROOT / "tests"))
    from hsr_env_b200.model import Model
    from oracle import port
    from scenarios import regimes

    model = Model.load(ROOT / "hsr_env_b200" / "blobs" / blob_name)
    cp = port.CpuPort(model)
    cp.set_caps(64, 64 * 6 + 8)
    qpos, qvel, warm, _ = [t[:n_sample].double().cpu().numpy() for t in env.get_state()]
    dbg = cp.step(qpos, qvel, warm, np.zeros((len(qpos), model.nu)), nsub=1, debug=True)["debug"]
    counts = {}
    for d in dbg:
        for r in regimes(model, d):
            counts[r] = counts.get(r, 0) + 1
    return {k: v / len(dbg) for k, v in sorted(counts.items())}


def run_gpu(args):
    import torch

    from hsr_env_b200 import dist as D
    from hsr_env_b200.spaces import Box
    from hsr_env_b200.util import GoalSpec

    rank, local, world = D.init_from_env()
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    n = args.envs_per_gpu
    peak_tf = fp32_peak(local)       # FMA-loop peak of THIS device, measured in this run (BASELINE.md 3.4)
    # optional pre-heat (default off): repeat the FMA loop for args.preheat seconds before the warm-up actions.  (What looked
    # like a slow first process on a fresh box - 51-54 M against 55-57 M substeps/s - was the harness's own torch elementwise
    # ops inside the timed bracket, each paying a cold instruction fetch after the L2 flush; they are outside the bracket now.)
    t_heat = time.time()
    while time.time() - t_heat < args.preheat:
        peak_tf = max(peak_tf, fp32_peak(local))
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2
    goals = [GoalSpec(a=Box(BLOCK_LO, BLOCK_HI), b=Box(GOAL_LO, GOAL_HI), distance=GEOFENCE)]

    # ---------------------------------------------------------------- headline: configs[1], weak scaling
    clk = ClockSampler(local)
    r = run_workload(torch, D, dev, blob=BLOB, goals=goals, starts=None, n_local=n, env_offset=rank * n,
                     steps=args.steps, warmup=args.warmup, seed=args.seed, kernel=args.kernel, lanes=args.lanes, flush=flush,
                     sampler=clk)
    env, info = r["env"], r["info"]
    gathered = D.gather_episode_stats(dict(episodes=r["local_successes"], successes=r["local_successes"],
                                           substeps=r["local_substeps"], bad_states=r["local_bad"]), dev)

    # ---- end to end through the host-buffer API: pinned host actions in, obs/reward/done/substeps out, every step,
    #      restarted from the snapshot taken before the timed steps: the same actions on the same states
    e2e_steps = args.steps
    act_host = [torch.from_numpy(r["actions_host"][args.warmup + k]).pin_memory() for k in range(e2e_steps)]
    out = dict(obs=torch.empty(n, env.obs_dim).pin_memory(), reward=torch.empty(n).pin_memory(),
               done=torch.zeros(n, dtype=torch.uint8).pin_memory(), taken=torch.empty(n, dtype=torch.int32).pin_memory())
    mask_host = torch.zeros(n, dtype=torch.uint8).pin_memory()
    mask_dev = torch.zeros(n, dtype=torch.uint8, device=dev)
    snap = r["snap"]
    for k in range(min(3, e2e_steps)):  # warm-up of the host path
        env.step_host(act_host[k], out=out)
    env.set_state(qpos=snap[0], qvel=snap[1], qacc_warmstart=snap[2], mocap_pos=snap[3])
    out["done"].copy_(snap[4].to(torch.uint8))
    age_h = snap[5].cpu().numpy().copy()
    D.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        m = (out["done"].numpy() != 0) | (age_h >= TIME_LIMIT)      # the caller's bookkeeping, on the host
        mask_host.numpy()[:] = m
        age_h[m] = 0
        mask_dev.copy_(mask_host, non_blocking=True)              # H2D: which environments the caller resets
        env.reset(mask=mask_dev)
        env.step_host(act_host[k], out=out)                       # H2D ctrl, kernel, D2H obs/reward/done/taken, sync
        age_h += 1
    torch.cuda.synchronize(dev)
    e2e_secs = D.max_over_ranks(time.perf_counter() - t0, dev)
    h2d = n * env.nu * 4 + n
    d2h = n * (env.obs_dim * 4 + 4 + 1 + 4)

    hbm_peak, sm_max, which = peaks()
    nq, nv, nu = env.nq, env.nv, env.nu
    # algorithmic HBM bytes per env-action (SURVEY.md §8(d)): state in/out once per action
    b_alg = 4 * ((nq + 2 * nv + nu + 3 + 2) + (nq + 2 * nv + (nq + nv) + 4))
    achieved_gbs = b_alg * n / r["kernel_s"] / 1e9
    traffic = None
    tp = ROOT / "profiles" / "r02_traffic.json"
    if tp.exists() and n == 4096 and info["kernel"] == "wpe":
        traffic = json.loads(tp.read_text())["dram_bytes_per_launch"]
    clocks = clk.summary()
    secs_max = r["secs"]
    achieved_tf = r["flops"] / secs_max / 1e12 / world
    f_alg = r["flops"] / max(1.0, r["substeps"])
    value = world * n * args.steps / secs_max
    kname = {"fast": "hsrb_push_kernel", "wpe": "hsrb_wpe_kernel_t<true>"}.get(info["kernel"], "hsrb_step_kernel")
    line = {
        "metric": "env_actions_per_sec", "value": value, "unit": "env-actions/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * secs_max / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "envs_per_gpu": n, "total_envs": n * world, "substeps_per_action": NSUB,
                   "time_limit": TIME_LIMIT, "l2": "flushed (256 MiB write) between timed steps", "timed_region": "masked reset + action kernel + launch-order sort per step; the harness's episode bookkeeping (ages, reset masks, counters: torch elementwise ops) is outside the bracket", "kernel": info["kernel"],
                   "threads_per_block": info["threads_per_block"], "lanes_per_env": info["lanes_per_env"],
                   "smem_per_env": info["smem_per_env"], "resident_envs_per_sm": info["envs_per_sm"], "grid": info["grid"]},
        "substeps_per_s": r["substeps"] / secs_max, "mean_substeps_per_action": r["substeps"] / (world * n * args.steps),
        "success_per_action": r["successes"] / (world * n * args.steps), "resets_per_action": r["resets"] / (world * n * args.steps),
        "bad_states": r["bad"], "clocks": clocks,
        "e2e": {"value": world * n * e2e_steps / e2e_secs, "unit": "env-actions/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "substeps_per_s": None},
        "gpu_launches": int(r["launches"]),
        # SURVEY.md §8(d): the binding ceiling of this path is the FP32 (CUDA-core) pipe, not HBM
        "roofline": {"bound": "fp32", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                     "traffic": traffic,
                     "traffic_source": ("static: dram__bytes_read+write of one ncu --set full capture of this kernel and batch, "
                                        "profiles/r02_traffic.json; not measured in this run") if traffic is not None else None,
                     "peak_source": "FP32 FMA-loop peak measured in this run (hsrb_measure_fp32_peak: 8 FMA chains x 1024 threads x 2 blocks per SM)",
                     "kernel": kname, "kernel_ms_per_launch": 1e3 * r["kernel_s"],
                     "algorithmic_flops_per_substep": f_alg,
                     "algorithmic_flops_per_launch": r["flops"] / world / args.steps,
                     "note": "achieved = substeps/s x mean algorithmic flops per substep (SURVEY.md 8(d) stage formulas evaluated by the "
                             "kernel with the actual per-substep contact / row / iteration counts) per GPU; the kernel is bound by "
                             "dependent-instruction latency and instruction fetch, see DESIGN.md 4.1"},
        "hbm": {"achieved_gbs": achieved_gbs, "peak_gbs": hbm_peak, "frac": achieved_gbs / hbm_peak, "peak_source": which,
                "algorithmic_bytes_per_launch": b_alg * n, "algorithmic_bytes_per_env_action": b_alg,
                "note": "state crosses HBM once per action; HBM is not the bound of this path"},
        "episode_stats_per_rank": gathered,
    }
    ph = {k: r["stats1"]["phase_cycles"][k] - r["stats0"]["phase_cycles"][k] for k in r["stats1"]["phase_cycles"]}
    if sum(ph.values()) > 0:
        tot = float(sum(ph.values()))
        line["phase_share"] = {k: round(v / tot, 4) for k, v in ph.items()}
        line["phase_cycles_per_substep_lane0"] = tot / max(1.0, r["local_substeps"])
    env.close()
    del flush

    # ---------------------------------------------------------------- the other BASELINE.json configs
    if not args.no_configs:
        cfgs = {}
        # configs[3]: 2^20 environments of the block-push model sharded over the ranks (strong scaling)
        only = set(filter(None, args.only_configs.split(",")))
        n4 = args.c4_envs // world
        if only and "c4" not in only:
            n4 = 4096
        r4 = run_workload(torch, D, dev, blob=BLOB, goals=goals, starts=None, n_local=n4, env_offset=rank * n4,
                          steps=2, warmup=3, seed=args.seed + 1, kernel=args.kernel)
        cfgs["c4_1m_envs_sharded"] = config_entry(r4, n4 * world, 2, peak_tf, world, {
            "workload": f"configs[3]: {n4 * world} environments of the block-push model, {n4} per GPU on {world} GPU(s) (contiguous slices of "
                        "the global env ids, no data-path collective); 3 warm-up + 2 timed actions (the launch order of the action kernel is the "
                        "sort of the previous action's per-environment work, so the first actions after creation are not steady state)", "scaling": "strong"})
        r4["env"].close()
        # configs[2] and configs[4]: every rank runs its own batch (weak)
        c3_starts = {k: Box([lo], [hi]) for k, (lo, hi) in C3_STARTS.items()}
        c3_goals = [GoalSpec(a=Box(C3_BLOCK_LO, C3_BLOCK_HI), b=Box(C3_GOAL_LO, C3_GOAL_HI), distance=GEOFENCE)]
        n3 = args.c3_envs
        # under U(ctrlrange) the position servos lift the arm off the pan within ~50 substeps (arm_lift's target lies above
        # its range, arm_flex's at >= -1.2 rad), so the gripper contacts live at the start of an episode: one action per
        # episode here (TimeLimit 1), every action starts with the hand on / above the block
        r3 = run_workload(torch, D, dev, blob="c3_arm.hsrb", goals=c3_goals, starts=c3_starts, n_local=n3,
                          env_offset=rank * n3, steps=2, warmup=1, seed=args.seed + 2, time_limit=1)
        census = None
        if rank == 0:
            e3 = r3["env"]
            e3.reset()
            e3.step(torch.from_numpy(r3["actions_host"][0]).to(dev), steps=15)
            census = regime_census(e3, "c3_arm.hsrb")
        cfgs["c3_arm_gripper"] = config_entry(r3, n3 * world, 2, peak_tf, world, {
            "workload": f"configs[2]: full arm + gripper (nv = 13), {n3} environments per GPU, block on the pan (block-space over the pan), "
                        "hand starting at block height above it (start spaces of the seven robot joints), actions ~ U(ctrlrange), "
                        "every environment reset before every action (episodes of one action: the servos lift the arm off the pan "
                        "within ~50 substeps); 1 warm-up + 2 timed actions of 300 substeps",
            "contact_regimes_fraction_of_states_at_substep_15": census, "scaling": "weak"})
        r3["env"].close()
        c5_goals = [GoalSpec(a=Box(C5_BLOCK_LO, C5_BLOCK_HI), b=Box(C5_GOAL_LO, C5_GOAL_HI), distance=GEOFENCE)]
        n5 = args.c5_envs
        r5 = run_workload(torch, D, dev, blob="c5_clutter.hsrb", goals=c5_goals, starts=None, n_local=n5,
                          env_offset=rank * n5, steps=1, warmup=1, seed=args.seed + 3, min_sep=.115)
        census5 = regime_census(r5["env"], "c5_clutter.hsrb") if rank == 0 else None
        cfgs["c5_clutter"] = config_entry(r5, n5 * world, 1, peak_tf, world, {
            "workload": f"configs[4]: slide_x/slide_y base + 4 blocks (nv = 26), {n5} environments per GPU, blocks ~ U over a 0.3 x 0.4 m patch in "
                        "front of the base, rejection-sampled 11.5 cm apart; 1 warm-up + 1 timed action",
            "contact_regimes_fraction_of_states": census5, "scaling": "weak"})
        r5["env"].close()
        line["configs"] = cfgs

    if rank == 0 and world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        # the same actions of the same environments after the same warm-up: the first `n_cpu` environments, bounded by time
        n_cpu = min(n, max(cores * 32, 256))
        acts, subs, csecs, _ = cpu_port_run(n_cpu, args.warmup, args.steps, cores, seed=args.seed, budget_s=args.cpu_seconds)
        line["cpu_baseline"] = {
            "value": acts / csecs, "unit": "env-actions/s", "cores": cores, "kind": "port",
            "substeps_per_s": subs / csecs,
            "sample": f"environments 0..{n_cpu - 1} of the same workload (same reset streams, actions, episode ages), {acts // n_cpu} timed actions after "
                      f"{args.warmup} warm-up actions ({subs} substeps, {csecs:.1f} s) on {cores} host threads; oracle fp64 C++ port (our own "
                      "restatement, NOT mujoco-py: it cannot be installed here)"}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--envs-per-gpu", type=int, default=4096)
    ap.add_argument("--lanes", type=int, default=0, help="lanes of a warp per environment (0 = auto)")
    ap.add_argument("--kernel", default="auto", choices=["auto", "general", "fast", "wpe"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-configs", action="store_true", help="skip configs[2], [3], [4]")
    ap.add_argument("--only-configs", default="", help="comma list of c3,c4,c5: run only these extra configs (experiments)")
    ap.add_argument("--c3-envs", type=int, default=16384)
    ap.add_argument("--c4-envs", type=int, default=1 << 20, help="total over all ranks")
    ap.add_argument("--c5-envs", type=int, default=4096)
    ap.add_argument("--preheat", type=float, default=0.0, help="seconds of untimed FMA-loop work before the warm-up actions")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
