"""The episode kernel (hsr_env_b200/csrc/hsrb_episode.cuh: TimeLimit + auto-reset on the device), compiled unchanged by g++
on the SIMT emulator, against a numpy restatement of the bookkeeping and the oracle port's Philox reset
(oracle.port.reset), with random done / age patterns.  CPU only; the GPU side is tests/test_episodes.py."""
import sys
from pathlib import Path

import numpy as np
import pytest

from scenarios import BLOCK_HI, BLOCK_LO, GOAL_HI, GOAL_LO, rollout_states

sys.path.insert(0, str(Path(__file__).resolve().parent / "simt_emu"))

T = 20
SEED, OFF = 77, 1000
CUPBOARD_STARTS = {"blockjoint": ([-.1, -.2, .418, 0, 0, -1, 0], [.1, .2, .418, 1, 0, 1, 0]), "slide_x": ([-.05], [.02])}
CUPBOARD_POINT = np.array([0, 0, .498, 0, 0, .498])


@pytest.fixture(scope="module")
def emu():
    import emu_episode

    emu_episode.build()
    return emu_episode


def _starts(model, starts):
    names = list(model.names["joint"])
    adr, width, lo, hi = [], [], [], []
    for joint, (l, h) in starts.items():
        j = names.index(joint)
        w = 7 if int(model.jnt_type[j]) == 0 else 1
        L, H = np.zeros(7), np.zeros(7)
        L[:w], H[:w] = l, h
        adr.append(int(model.jnt_qposadr[j])); width.append(w); lo.append(L); hi.append(H)
    return adr, width, np.array(lo), np.array(hi)


def _configure(name, model, port):
    """(kwargs of the emulated launch) with the port configured the same way"""
    if name == "c2_push":
        port.set_goals(np.r_[GOAL_LO, GOAL_HI], np.r_[BLOCK_LO, BLOCK_HI], .05)
        return dict(goal_lohi=np.r_[GOAL_LO, GOAL_HI], block_lohi=np.r_[BLOCK_LO, BLOCK_HI])
    # f2_cupboard, the goal-list form (GoalSpec(a="block", b=ndarray)) with start spaces, as hsr/__init__.py:13-18
    st = _starts(model, CUPBOARD_STARTS)
    port.set_goal_list([int(model.block_body[0])], [-1], [.05], CUPBOARD_POINT)
    port.set_starts(*st)
    return dict(goal_lohi=CUPBOARD_POINT, starts=st)


def _quat_slots(model):
    return sorted(int(model.jnt_qposadr[j]) + 3 + k for j in range(model.njnt) if int(model.jnt_type[j]) == 0 for k in range(4))


@pytest.mark.parametrize("name,G,grid", [("c2_push", 8, None), ("c2_push", 32, 5), ("f2_cupboard", 16, 3)])
@pytest.mark.parametrize("autoreset", [True, False])
def test_emulated_episode_kernel(name, G, grid, autoreset, models, ports, emu):
    model, port = models[name], ports[name]
    n = 40
    rng = np.random.default_rng(len(name) + G)
    qpos, qvel, warm, _ = rollout_states(port, model, n, seed=3, float32=True)
    mocap = rng.uniform(-.2, .2, (n, 3))
    state = np.concatenate([qpos, qvel, warm, mocap], 1).astype(np.float32)
    episode = rng.integers(0, 5, n).astype(np.uint32)
    age = rng.integers(0, T + 3, n).astype(np.int32)
    age[:4] = [T - 1, T - 1, T - 2, 0]
    term = (rng.random(n) < .25).astype(np.uint8)
    term[:4] = [1, 0, 0, 0]                                  # success exactly at the limit: terminated, not truncated
    reward = term.astype(np.float32)
    ret = rng.integers(0, 3, n).astype(np.float32)
    sub = rng.integers(0, 3000, n).astype(np.int32)
    taken = rng.integers(1, 301, n).astype(np.int32)
    bad = (rng.random(n) < .1).astype(np.uint8) * 2
    kw = _configure(name, model, port)
    try:
        out = emu.episode(model, state, episode, age, ret, sub, term, reward, taken, bad, max_steps=T, autoreset=autoreset,
                          seed=SEED, env_off=OFF, G=G, grid=grid, **kw)
        want_reset = {}
        # numpy restatement of the bookkeeping
        age1 = age + 1
        trunc = (age1 >= T) & (term == 0)
        done = (term != 0) | trunc
        reset = done & autoreset
        ret1, sub1 = ret + reward, sub + taken
        for e in np.nonzero(reset)[0]:
            want_reset[e] = port.reset(SEED, OFF + int(e), int(episode[e]))
    finally:
        port.set_goals(None)
        port.set_starts([], [], np.zeros((0, 7)), np.zeros((0, 7)))
    assert 0 < done.sum() < n and trunc[1] and not trunc[0] and done[0] and not done[2]
    assert np.array_equal(out["truncated"], trunc.astype(np.uint8))
    assert np.array_equal(out["ep_length"], np.where(done, age1, -1))
    assert np.array_equal(out["ep_return"][done], ret1[done]) and np.isnan(out["ep_return"][~done]).all()
    assert np.array_equal(out["ep_substeps"], np.where(done, sub1, -1))
    assert np.array_equal(out["age"], np.where(reset, 0, age1))
    assert np.array_equal(out["ret"], np.where(reset, 0, ret1).astype(np.float32))
    assert np.array_equal(out["sub"], np.where(reset, 0, sub1))
    assert np.array_equal(out["episode"], episode + reset)                     # the episode counter keys the next draw
    assert list(out["counters"]) == [done.sum(), (term != 0).sum(), trunc.sum(), age1[done].sum(), sub1[done].sum(),
                                     (bad != 0).sum(), reset.sum(), n]
    nq, nv, nobs = model.nq, model.nv, model.nq + model.nv
    assert np.array_equal(out["final_obs"], state[:, :nobs])                  # every environment, before any reset
    keep = ~reset
    assert np.array_equal(out["state"][keep].view(np.uint32), state[keep].view(np.uint32))   # untouched: bit-identical
    assert np.isnan(out["obs"][keep]).all()                                    # and their obs rows are not written
    assert sorted(want_reset) == list(np.nonzero(reset)[0])
    quat = _quat_slots(model)
    pos = [i for i in range(nq) if i not in quat]
    for e, (q, mo) in want_reset.items():
        st = out["state"][e]
        assert np.array_equal(st[pos], np.float32(q[pos])), e
        for a in range(0, len(quat), 4):
            qs = q[quat[a:a + 4]]
            np.testing.assert_allclose(st[quat[a:a + 4]], qs / np.linalg.norm(qs), atol=1e-6)
        assert not st[nq:nq + 2 * nv].any()                                    # qvel and the warm start restart at 0
        assert np.array_equal(st[nq + 2 * nv:], np.float32(mo))
        assert np.array_equal(out["obs"][e], st[:nobs])
