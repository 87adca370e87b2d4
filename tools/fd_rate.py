"""Cost of the transition derivatives on the bench workload: one transition_fd() call (centered and forward, one substep)
against one step() of 300 substeps, for c2_push at 4096 and 131072 environments and c3_arm at 4096.  CUDA events around
each call, L2 overwritten before each timed call, every call warmed up, the arms alternated over the repetitions (the step
moves the state on, so each repetition differentiates a new state), medians.

Writes the JSON line it prints to profiles/fd_rate.json (or --out), with the card name, power limit and max SM clock.

    python tools/fd_rate.py [--reps 7] [--out PATH]
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

from episode_loop_rate import card  # noqa: E402
from rollout_rate import make_env, timed  # noqa: E402  (the bench workload's handle, the L2-flushed event bracket)

CASES = [("c2_push", 4096), ("c2_push", 131072), ("c3_arm", 4096)]


def handle(name, n):
    if name == "c2_push":
        return make_env(n)
    import bench
    from hsr_env_b200.env import BatchedHSREnv

    return BatchedHSREnv(f"{name}.hsrb", None, steps_per_action=bench.NSUB, n_envs=n, device="cuda:0", seed=0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "fd_rate.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("fd_rate.py measures on the GPU; no CUDA device is visible")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda:0")
    rows = []
    for name, n in CASES:
        env = handle(name, n)
        rng = np.random.default_rng(n)
        lo, hi = env.model.act_ctrlrange[:, 0], env.model.act_ctrlrange[:, 1]
        env.reset()
        arms = {"step": lambda a: env.step(a), "fd_centered": lambda a: env.transition_fd(a, centered=True),
                "fd_forward": lambda a: env.transition_fd(a, centered=False)}
        act = torch.tensor(rng.uniform(lo, hi, (n, env.nu)), dtype=torch.float32, device="cuda:0")
        for fn in arms.values():   # warm-up: module load, the allocator, the scratch
            fn(act)
        torch.cuda.synchronize()
        ms = {k: [] for k in arms}
        for r in range(args.reps):
            act = torch.tensor(rng.uniform(lo, hi, (n, env.nu)), dtype=torch.float32, device="cuda:0")
            order = list(arms.items())
            order = order[r % 3:] + order[:r % 3]
            for k, fn in order:
                t, _ = timed(torch, lambda: fn(act), flush, r)
                ms[k].append(t)
        med = {k: float(np.median(v)) for k, v in ms.items()}
        nr_c, nr_f = 1 + 2 * (2 * env.nv + env.nu), 1 + 2 * env.nv + env.nu
        rows.append({"model": name, "envs": n, "ms": ms, "median_ms": med, "runs_per_env": {"centered": nr_c, "forward": nr_f},
                     "centered_over_step": med["fd_centered"] / med["step"], "forward_over_step": med["fd_forward"] / med["step"],
                     "spread": {k: (max(v) - min(v)) / med[k] for k, v in ms.items()}})
        print(json.dumps(rows[-1]), file=sys.stderr)
        env.close()
    import bench

    res = {"card": card(), "workload": f"{bench.NSUB} substeps per step, uniform actions; c2_push with the goal spaces of "
                                       "bench.py, c3_arm without goals; transition_fd at eps 1e-2, one substep",
           "reps": args.reps, "rows": rows, "l2": "overwritten (256 MiB write) before each timed call, outside the event bracket"}
    line = json.dumps(res)
    print(line)
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(line + "\n")


if __name__ == "__main__":
    main()
