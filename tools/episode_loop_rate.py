"""Rate of the whole RL loop per action on the bench workload (c2_push, 4096 environments, block / goal spaces, TimeLimit 20
with staggered ages, host Philox actions), L2 overwritten between actions as bench.py does, CUDA events around each action:

  (a) the loop a caller writes today: torch bookkeeping (mask = done | age >= 20, ages), reset(mask), step();
  (b) step() with max_episode_steps=20, autoreset=True (the episode kernel after the action kernel).

Each loop runs `--reps` times, alternating (a), (b), (a), ...  Before timing, (a) and (b) are run side by side from the same
start and their outputs compared bit for bit.  Prints one JSON line with the card name and power limit.

    python tools/episode_loop_rate.py [--envs 4096] [--steps 20] [--warmup 5] [--reps 3]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402  (the workload's constants and host actions)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable: {e!r}"


def make_env(n, episode_loop):
    from hsr_env_b200.env import BatchedHSREnv
    from hsr_env_b200.spaces import Box
    from hsr_env_b200.util import GoalSpec

    goals = [GoalSpec(a=Box(bench.BLOCK_LO, bench.BLOCK_HI), b=Box(bench.GOAL_LO, bench.GOAL_HI), distance=bench.GEOFENCE)]
    kw = dict(max_episode_steps=bench.TIME_LIMIT, autoreset=True) if episode_loop else {}
    return BatchedHSREnv(bench.BLOB, goals, steps_per_action=bench.NSUB, n_envs=n, device="cuda:0", seed=0, **kw)


class Loop:
    """One of the two loops on its own handle; step(k) runs action k (the timed unit)."""

    def __init__(self, torch, n, episode_loop, actions):
        self.torch, self.n, self.episodic, self.actions = torch, n, episode_loop, actions
        self.env = make_env(n, episode_loop)
        self.env.reset()
        self.age = (torch.arange(n, device="cuda:0") % bench.TIME_LIMIT).to(torch.int32)
        self.done = torch.zeros(n, dtype=torch.bool, device="cuda:0")
        if episode_loop:
            self.env.set_episode_ages(self.age)

    def step(self, k):
        torch = self.torch
        if self.episodic:
            return self.env.step(self.actions[k])
        mask = self.done | (self.age >= bench.TIME_LIMIT)
        self.age = torch.where(mask, 0, self.age)
        obs_r = self.env.reset(mask=mask)
        out = self.env.step(self.actions[k])
        self.done = out[2]
        self.age = self.age + 1
        return out, obs_r, mask


def check_equal(torch, n, actions, steps):
    """(a) and (b) side by side: (b)'s final observation is (a)'s step obs; (b)'s obs after its auto-reset is what (a)'s
    masked reset before the next action returns, and (b)'s done is that reset's mask."""
    a, b = Loop(torch, n, False, actions), Loop(torch, n, True, actions)
    prev_b = None
    for k in range(steps + 1):
        (oa, ra, da, _), obs_r, mask = a.step(k)
        if prev_b is not None:
            assert torch.equal(obs_r, prev_b[0]) and torch.equal(mask, prev_b[1]), k
        if k == steps:
            break
        ob, rb, db, ib = b.step(k)
        assert torch.equal(ib["final_observation"], oa) and torch.equal(rb, ra) and torch.equal(ib["terminated"], da), k
        prev_b = (ob, db)
    a.env.close(); b.env.close()
    return steps


def time_loop(torch, loop, flush, warmup, steps):
    for k in range(warmup):
        loop.step(k)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for k in range(steps):
        flush.fill_(k & 0xff)        # evict L2 between actions (outside the event bracket), as bench.py
        ev[k][0].record()
        loop.step(warmup + k)
        ev[k][1].record()
    torch.cuda.synchronize()
    return sum(s.elapsed_time(e) for s, e in ev) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--check-steps", type=int, default=25)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("episode_loop_rate.py measures on the GPU; no CUDA device is visible")
    n = args.envs
    from hsr_env_b200.model import Model

    model = Model.load(ROOT / "hsr_env_b200" / "blobs" / bench.BLOB)
    total = max(args.check_steps + 1, args.warmup + args.steps)
    actions = torch.from_numpy(bench.host_actions(0, total, n, model.act_ctrlrange[:, 0], model.act_ctrlrange[:, 1])).cuda()
    checked = check_equal(torch, n, actions, args.check_steps)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda:0")
    ms = {"a_torch_bookkeeping_reset_step": [], "b_step_autoreset": []}
    for _ in range(args.reps):
        for key, episodic in (("a_torch_bookkeeping_reset_step", False), ("b_step_autoreset", True)):
            loop = Loop(torch, n, episodic, actions)
            ms[key].append(time_loop(torch, loop, flush, args.warmup, args.steps))
            loop.env.close()
    a, b = np.median(ms["a_torch_bookkeeping_reset_step"]), np.median(ms["b_step_autoreset"])
    print(json.dumps({"card": card(), "envs": n, "steps": args.steps, "warmup": args.warmup, "reps": args.reps,
                      "ms_per_action": ms, "median_ms": {"a": a, "b": b}, "saving_ms": a - b,
                      "env_actions_per_s": {"a": n / a * 1e3, "b": n / b * 1e3},
                      "bit_equal_outputs": f"checked over {checked} actions at {n} environments",
                      "l2": "overwritten (256 MiB write) between actions, outside the event bracket"}))


if __name__ == "__main__":
    main()
