"""Cost of the contact query on the bench workload (c2_push, 300 substeps, uniform actions from act_ctrlrange): one
contacts() call and one contact_wrench() call against one step(), at 4096 and 131072 environments.  CUDA events around
each call, L2 overwritten before each timed call, every call warmed up, the three arms alternated over the repetitions
(the step moves the state on, so each repetition queries a new state).

Writes the JSON line it prints to profiles/contacts_rate.json (or --out), with the card name, power limit and max SM clock.

    python tools/contacts_rate.py [--envs 4096 131072] [--reps 7] [--out PATH]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 131072])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "contacts_rate.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("contacts_rate.py measures on the GPU; no CUDA device is visible")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda:0")
    rows = []
    for n in args.envs:
        env = make_env(n)
        rng = np.random.default_rng(n)
        lo, hi = env.model.act_ctrlrange[:, 0], env.model.act_ctrlrange[:, 1]
        env.reset()
        arms = {"step": lambda a: env.step(a), "contacts": lambda a: env.contacts(a), "contact_wrench": lambda a: env.contact_wrench(a)}
        act = torch.tensor(rng.uniform(lo, hi, (n, env.nu)), dtype=torch.float32, device="cuda:0")
        for fn in arms.values():   # warm-up: module load, the allocator, the pair table
            fn(act)
        torch.cuda.synchronize()
        ms = {k: [] for k in arms}
        ncon = []
        for r in range(args.reps):
            act = torch.tensor(rng.uniform(lo, hi, (n, env.nu)), dtype=torch.float32, device="cuda:0")
            order = list(arms.items())
            order = order[r % 3:] + order[:r % 3]
            for name, fn in order:
                t, out = timed(torch, lambda: fn(act), flush, r)
                ms[name].append(t)
                if name == "contacts":
                    ncon.append(float(out["count"].float().mean().item()))
        med = {k: float(np.median(v)) for k, v in ms.items()}
        rows.append({"envs": n, "ms": ms, "median_ms": med, "contacts_over_step": med["contacts"] / med["step"],
                     "wrench_over_step": med["contact_wrench"] / med["step"], "mean_contacts_per_env": float(np.mean(ncon)),
                     "spread": {k: (max(v) - min(v)) / med[k] for k, v in ms.items()}})
        print(json.dumps(rows[-1]), file=sys.stderr)
        env.close()
    import bench

    res = {"card": card(), "workload": f"{bench.BLOB}, {bench.NSUB} substeps per step, uniform actions, goal spaces of bench.py",
           "reps": args.reps, "rows": rows, "l2": "overwritten (256 MiB write) before each timed call, outside the event bracket"}
    line = json.dumps(res)
    print(line)
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(line + "\n")


if __name__ == "__main__":
    main()
