"""Open-loop rollouts against step() loops on the bench workload (c2_push, 300 substeps, uniform actions from
act_ctrlrange): (a) K step() calls against (b) one rollout() of the same K actions, on twin handles reset alike, at
4096 and 131072 environments and K in {1, 5, 20}.  CUDA events around each call (a: around the K steps), L2 overwritten
before each timed call, every shape warmed up, three alternating runs of each arm; the outputs of (a) and (b) are
checked bit for bit on every timed run.

Writes the JSON line it prints to profiles/rollout_rate.json (or --out), with the card name, power limit and max SM clock.

    python tools/rollout_rate.py [--envs 4096 131072] [--ks 1 5 20] [--reps 3] [--out PATH]
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

import bench  # noqa: E402  (the workload's constants)
from episode_loop_rate import card  # noqa: E402


def make_env(n):
    from hsr_env_b200.env import BatchedHSREnv
    from hsr_env_b200.spaces import Box
    from hsr_env_b200.util import GoalSpec

    goals = [GoalSpec(a=Box(bench.BLOCK_LO, bench.BLOCK_HI), b=Box(bench.GOAL_LO, bench.GOAL_HI), distance=bench.GEOFENCE)]
    return BatchedHSREnv(bench.BLOB, goals, steps_per_action=bench.NSUB, n_envs=n, device="cuda:0", seed=0)


def run_steps(env, act):
    outs = [env.step(a) for a in act]
    return [outs[k][j] for k in range(len(outs)) for j in range(3)] + [o[3][key] for o in outs for key in ("substeps_taken", "bad_state")]


def run_rollout(env, act):
    obs, reward, done, info = env.rollout(act)
    return [x[k] for k in range(len(act)) for x in (obs, reward, done)] + [info[key][k] for k in range(len(act))
                                                                            for key in ("substeps_taken", "bad_state")]


def timed(torch, fn, flush, tag):
    flush.fill_(tag & 0xff)          # evict L2 before the call, outside the event bracket
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    out = fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 131072])
    ap.add_argument("--ks", type=int, nargs="+", default=[1, 5, 20])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "rollout_rate.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("rollout_rate.py measures on the GPU; no CUDA device is visible")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda:0")
    rows = []
    for n in args.envs:
        A, B = make_env(n), make_env(n)
        rng = np.random.default_rng(n)
        lo, hi = A.model.act_ctrlrange[:, 0], A.model.act_ctrlrange[:, 1]
        for K in args.ks:
            # warm-up of this shape on both handles (module load, the sort buffers, the allocator)
            act = torch.tensor(rng.uniform(lo, hi, (K, n, A.nu)), dtype=torch.float32, device="cuda:0")
            run_steps(A, act); run_rollout(B, act)
            ms = {"steps": [], "rollout": []}
            for r in range(args.reps):
                # the same start state on both handles: reset (same seed, same episode counters) then K actions
                assert torch.equal(A.reset(), B.reset())
                act = torch.tensor(rng.uniform(lo, hi, (K, n, A.nu)), dtype=torch.float32, device="cuda:0")
                order = (("steps", A, run_steps), ("rollout", B, run_rollout))
                if r % 2:
                    order = order[::-1]
                outs = {}
                for arm, env, fn in order:
                    t, outs[arm] = timed(torch, lambda: fn(env, act), flush, r)
                    ms[arm].append(t)
                assert all(torch.equal(x, y) for x, y in zip(outs["steps"], outs["rollout"])), (n, K, r)
                assert all(torch.equal(x, y) for x, y in zip(A.get_state(), B.get_state())), (n, K, r)
            med = {a: float(np.median(v)) for a, v in ms.items()}
            rows.append({"envs": n, "K": K, "ms": ms, "median_ms": med, "rollout_over_steps": med["rollout"] / med["steps"],
                         "spread_steps": (max(ms["steps"]) - min(ms["steps"])) / med["steps"],
                         "spread_rollout": (max(ms["rollout"]) - min(ms["rollout"])) / med["rollout"],
                         "env_actions_per_s_rollout": n * K / (med["rollout"] * 1e-3),
                         "env_actions_per_s_steps": n * K / (med["steps"] * 1e-3)})
            print(json.dumps(rows[-1]), file=sys.stderr)
        A.close(); B.close()
    res = {"card": card(), "workload": f"{bench.BLOB}, {bench.NSUB} substeps, uniform actions, goal spaces of bench.py",
           "reps": args.reps, "bit_equal": True, "rows": rows,
           "l2": "overwritten (256 MiB write) before each timed call, outside the event bracket"}
    line = json.dumps(res)
    print(line)
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(line + "\n")


if __name__ == "__main__":
    main()
