"""Cost of per-environment physics parameters on the bench workload (c2_push, 4096 environments, block / goal spaces,
TimeLimit 20 with staggered ages and auto-reset, host Philox actions), L2 overwritten between actions as bench.py does,
CUDA events around each action.  Three arms on handles of their own, alternated `--reps` times:

  none   no parameters (the kernels without parameters);
  unit   set_env_params(ones): the instances with parameters at the nominal model (their own cost);
  ranges randomize every multiplier over [0.5, 2] (draws at every reset, per-environment physics).

Writes the JSON line it prints to profiles/env_params_rate.json (or --out), with the card name and power limit.

    python tools/env_params_rate.py [--envs 4096] [--steps 20] [--warmup 5] [--reps 3] [--out PATH]
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import bench  # noqa: E402  (the workload's constants and host actions)
from episode_loop_rate import card  # noqa: E402

ARMS = ("none", "unit", "ranges")


def make_env(torch, n, arm):
    from hsr_env_b200.env import PARAM_NAMES, BatchedHSREnv
    from hsr_env_b200.spaces import Box
    from hsr_env_b200.util import GoalSpec

    goals = [GoalSpec(a=Box(bench.BLOCK_LO, bench.BLOCK_HI), b=Box(bench.GOAL_LO, bench.GOAL_HI), distance=bench.GEOFENCE)]
    randomize = {k: (0.5, 2.0) for k in PARAM_NAMES} if arm == "ranges" else None
    env = BatchedHSREnv(bench.BLOB, goals, steps_per_action=bench.NSUB, n_envs=n, device="cuda:0", seed=0,
                        max_episode_steps=bench.TIME_LIMIT, autoreset=True, randomize=randomize)
    if arm == "unit":
        env.set_env_params(torch.ones(n, len(PARAM_NAMES)))
    env.reset()
    env.set_episode_ages((torch.arange(n, device="cuda:0") % bench.TIME_LIMIT).to(torch.int32))
    return env


def time_arm(torch, env, actions, flush, warmup, steps):
    for k in range(warmup):
        env.step(actions[k])
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for k in range(steps):
        flush.fill_(k & 0xff)        # evict L2 between actions (outside the event bracket), as bench.py
        ev[k][0].record()
        env.step(actions[warmup + k])
        ev[k][1].record()
    torch.cuda.synchronize()
    return sum(s.elapsed_time(e) for s, e in ev) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "env_params_rate.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("env_params_rate.py measures on the GPU; no CUDA device is visible")
    n = args.envs
    from hsr_env_b200.model import Model

    model = Model.load(ROOT / "hsr_env_b200" / "blobs" / bench.BLOB)
    actions = torch.from_numpy(bench.host_actions(0, args.warmup + args.steps, n, model.act_ctrlrange[:, 0],
                                                  model.act_ctrlrange[:, 1])).cuda()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda:0")
    ms = {a: [] for a in ARMS}
    substeps = {}
    for _ in range(args.reps):
        for arm in ARMS:
            env = make_env(torch, n, arm)
            ms[arm].append(time_arm(torch, env, actions, flush, args.warmup, args.steps))
            substeps[arm] = env.stats()["substeps"]
            env.close()
    med = {a: float(np.median(v)) for a, v in ms.items()}
    res = {"card": card(), "envs": n, "steps": args.steps, "warmup": args.warmup, "reps": args.reps, "ms_per_action": ms,
           "median_ms": med, "unit_over_none": med["unit"] / med["none"], "ranges_over_none": med["ranges"] / med["none"],
           "substeps_last_rep": substeps,
           "l2": "overwritten (256 MiB write) between actions, outside the event bracket"}
    line = json.dumps(res)
    print(line)
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(line + "\n")


if __name__ == "__main__":
    main()
