"""The episode loop on the device (BatchedHSREnv(max_episode_steps=..., autoreset=...) -> hsrb_step_episode): TimeLimit,
truncation, terminal observations and auto-reset against the loop a caller writes by hand in torch (step; mask = done |
age >= T; reset(mask)), bit for bit."""
import numpy as np
import pytest

from scenarios import BLOCK_HI, BLOCK_LO, GOAL_HI, GOAL_LO

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

T = 20
C3_BLOCK = ([-.1, -.18, 0., -1.], [.1, .18, 1., 1.])
C3_GOAL = ([-.1, -.18, .422], [.1, .18, .422])
CUPBOARD_STARTS = {"blockjoint": ([-.1, -.2, .418, 0, 0, -1, 0], [.1, .2, .418, 1, 0, 1, 0]), "slide_x": ([-.05], [.02])}


def _cfg(name):
    from hsr_env_b200.spaces import Box
    from hsr_env_b200.util import GoalSpec

    if name == "f2_cupboard":   # the general (goal-list) form, with start spaces (hsr/__init__.py:13-18)
        starts = {k: Box(np.array(lo), np.array(hi)) for k, (lo, hi) in CUPBOARD_STARTS.items()}
        return [GoalSpec(a="block", b=np.array([0, 0, .498]), distance=.05)], starts
    if name == "c3_arm":
        return [GoalSpec(Box(*C3_BLOCK), Box(*C3_GOAL), .05)], None
    return [GoalSpec(Box(BLOCK_LO, BLOCK_HI), Box(GOAL_LO, GOAL_HI), .05)], None


def _env(name, n, kernel="auto", goals="default", seed=3, **kw):
    from hsr_env_b200.env import BatchedHSREnv

    g, starts = _cfg(name)
    return BatchedHSREnv(f"{name}.hsrb", g if goals == "default" else goals, starts=starts, n_envs=n, device="cuda:0", seed=seed,
                         kernel=kernel, **kw)


def _actions(env, k, n=None, seed=0):
    rng = np.random.default_rng(seed + 7919 * k)
    lo, hi = env.model.act_ctrlrange[:, 0], env.model.act_ctrlrange[:, 1]
    return torch.tensor(rng.uniform(lo, hi, (n or env.n_envs, env.nu)), dtype=torch.float32, device="cuda:0")


def _state_equal(a, b):
    return all(torch.equal(x, y) for x, y in zip(a.get_state(), b.get_state()))


@pytest.mark.parametrize("name,kernel", [("c2_push", "wpe"), ("c2_push", "fast"), ("c2_push", "general"), ("c1b_readme_block", "wpe"),
                                         ("f2_cupboard", "general"), ("c3_arm", "general")])
def test_autoreset_matches_manual_loop(name, kernel):
    """Env A auto-resets on the device, env B runs the bench's hand-written loop; after every action obs, reward, done, the
    whole state, the ages and the episode statistics are bit-equal, and A's final_observation is B's step obs."""
    n, nsub, actions = 256, 100, 60
    A = _env(name, n, kernel, steps_per_action=nsub, max_episode_steps=T, autoreset=True)
    B = _env(name, n, kernel, steps_per_action=nsub)
    assert A.launch_info()["kernel"] == B.launch_info()["kernel"]
    assert torch.equal(A.reset(), B.reset())
    age = (torch.arange(n, device="cuda:0") % T).to(torch.int32)     # staggered episode phases, as bench.py
    A.set_episode_ages(age)
    assert torch.equal(A.episode_ages(), age)
    ret = torch.zeros(n, device="cuda:0"); sub = torch.zeros(n, dtype=torch.int32, device="cuda:0")
    cnt = dict(episodes=0, successes=0, truncations=0, length=0, substeps=0, bad_states=0)
    for k in range(actions):
        act = _actions(A, k)
        oa, ra, da, ia = A.step(act)
        ob, rb, db, ib = B.step(act)
        age += 1; ret += rb; sub += ib["substeps_taken"]
        mask = db | (age >= T)
        trunc = mask & ~db
        assert torch.equal(ia["final_observation"], ob)
        assert torch.equal(ra, rb) and torch.equal(da, mask)
        assert torch.equal(ia["terminated"], db) and torch.equal(ia["truncated"], trunc)
        assert torch.equal(ia["substeps_taken"], ib["substeps_taken"]) and torch.equal(ia["bad_state"], ib["bad_state"])
        ep = ia["episode"]
        assert torch.equal(ep["l"][mask], age[mask]) and torch.equal(ep["r"][mask], ret[mask])
        assert torch.equal(ep["substeps"][mask], sub[mask])
        cnt["episodes"] += int(mask.sum()); cnt["successes"] += int(db.sum()); cnt["truncations"] += int(trunc.sum())
        cnt["length"] += int(age[mask].sum()); cnt["substeps"] += int(sub[mask].sum())
        cnt["bad_states"] += int((ib["bad_state"] != 0).sum())
        obr = B.reset(mask=mask)
        age = torch.where(mask, 0, age).to(torch.int32); ret[mask] = 0; sub[mask] = 0
        assert torch.equal(oa, obr), k
        assert _state_equal(A, B), k
        assert torch.equal(A.episode_ages(), age), k
    st = A.episode_stats()
    assert cnt["truncations"] > 0
    assert {k: st[k] for k in cnt} == cnt
    assert st["resets"] == cnt["episodes"] and st["actions"] == n * actions
    A.close(); B.close()


def test_truncation_semantics():
    n = 64
    from hsr_env_b200.spaces import Box
    from hsr_env_b200.util import GoalSpec

    # success exactly at age T: terminated, not truncated (a 100 m geofence: every step succeeds)
    always = [GoalSpec(Box(BLOCK_LO, BLOCK_HI), Box(GOAL_LO, GOAL_HI), 100.)]
    A = _env("c2_push", n, goals=always, steps_per_action=10, max_episode_steps=T, autoreset=True)
    A.reset()
    A.set_episode_ages(torch.full((n,), T - 1, dtype=torch.int32))
    _, _, done, info = A.step(_actions(A, 0))
    assert done.all() and info["terminated"].all() and not info["truncated"].any()
    assert (info["episode"]["l"] == T).all()
    A.close()
    # goals=None: never terminated, truncated at ages T, 2T, ...; l and r recounted in torch
    A = _env("c2_push", n, goals=None, steps_per_action=10, max_episode_steps=T, autoreset=True)
    A.reset()
    age0 = (torch.arange(n, device="cuda:0") * 7 % T).to(torch.int32)
    A.set_episode_ages(age0)
    for k in range(2 * T + 3):
        _, rew, done, info = A.step(_actions(A, k))
        want = (age0 + k + 1) % T == 0
        assert torch.equal(info["truncated"], want) and torch.equal(done, want) and not info["terminated"].any(), k
        assert (info["episode"]["l"][want] == T).all() and (info["episode"]["r"][want] == 0).all()
        assert not rew.any()
    assert A.episode_stats()["truncations"] == int(sum((((age0 + k + 1) % T) == 0).sum() for k in range(2 * T + 3)))
    A.close()
    # without autoreset nothing is reset: the state after a truncation is a plain step's
    A = _env("c2_push", n, max_episode_steps=T, steps_per_action=50)
    B = _env("c2_push", n, steps_per_action=50)
    A.reset(); B.reset()
    A.set_episode_ages(torch.full((n,), T - 2, dtype=torch.int32))
    for k in range(3):
        oa, _, da, ia = A.step(_actions(A, k))
        ob, _, db, ib = B.step(_actions(B, k))
        assert torch.equal(oa, ob) and torch.equal(ia["final_observation"], ob) and _state_equal(A, B)
        assert torch.equal(ia["truncated"], ~db) if k >= 1 else not ia["truncated"].any()
    assert torch.equal(A.episode_ages(), torch.full((n,), T + 1, dtype=torch.int32, device="cuda:0"))
    A.close(); B.close()


def test_reset_clears_ages():
    n = 96
    A = _env("c2_push", n, max_episode_steps=T, autoreset=True)
    A.reset()
    ages = torch.randint(0, 50, (n,), dtype=torch.int32, device="cuda:0")
    A.set_episode_ages(ages)
    assert torch.equal(A.episode_ages(), ages)
    mask = torch.rand(n, device="cuda:0") < .4
    A.reset(mask=mask)
    assert torch.equal(A.episode_ages(), torch.where(mask, 0, ages))
    A.reset()
    assert not A.episode_ages().any()
    A.set_episode_ages(None)
    assert not A.episode_ages().any()
    A.close()


def test_shard_invariance():
    """Two handles with env_id_offset 0 and N/2 reproduce one handle of N environments over 40 auto-reset actions."""
    n, h = 256, 128
    full = _env("c2_push", n, steps_per_action=100, max_episode_steps=T, autoreset=True)
    shards = [_env("c2_push", h, steps_per_action=100, max_episode_steps=T, autoreset=True, env_id_offset=o) for o in (0, h)]
    age = (torch.arange(n, device="cuda:0") % T).to(torch.int32)
    full.reset(); full.set_episode_ages(age)
    for i, s in enumerate(shards):
        s.reset(); s.set_episode_ages(age[i * h:(i + 1) * h])
    for k in range(40):
        act = _actions(full, k)
        of, rf, df, inf = full.step(act)
        outs = [s.step(act[i * h:(i + 1) * h]) for i, s in enumerate(shards)]
        assert torch.equal(of, torch.cat([o[0] for o in outs])) and torch.equal(df, torch.cat([o[2] for o in outs]))
        assert torch.equal(inf["final_observation"], torch.cat([o[3]["final_observation"] for o in outs]))
    for part, i in zip(zip(*[s.get_state() for s in shards]), range(4)):
        assert torch.equal(full.get_state()[i], torch.cat(part))
    assert torch.equal(full.episode_ages(), torch.cat([s.episode_ages() for s in shards]))
    for e in [full] + shards:
        e.close()


def test_openai_final_observation():
    n = 128
    A = _env("c2_push", n, obs_type="openai", steps_per_action=100, max_episode_steps=T, autoreset=True)
    B = _env("c2_push", n, obs_type="openai", steps_per_action=100)
    assert torch.equal(A.reset(), B.reset())
    age = (torch.arange(n, device="cuda:0") % T).to(torch.int32)
    A.set_episode_ages(age)
    for k in range(25):
        act = _actions(A, k)
        oa, _, da, ia = A.step(act)
        ob, _, db, _ = B.step(act)
        age += 1
        mask = db | (age >= T)
        assert oa.shape == (n, 25) and torch.equal(ia["final_observation"], ob) and torch.equal(da, mask)
        assert torch.equal(oa, B.reset(mask=mask))
        age = torch.where(mask, 0, age).to(torch.int32)
    A.close(); B.close()


def test_facade_time_limit():
    """The facade run like hsr/control.py: done with TimeLimit.truncated on the 20th action, then the loop resets."""
    from hsr_env_b200.env import HSREnv

    env = HSREnv("c2_push.hsrb", None, steps_per_action=20, max_episode_steps=T)
    env.reset()
    ends = []
    for i in range(2 * T + 5):
        obs, reward, done, info = env.step(np.zeros(env.nu))
        assert obs.shape == (env.obs_dim,)
        if done:
            assert info["TimeLimit.truncated"] is True
            ends.append(i + 1)
            env.reset()
        else:
            assert "TimeLimit.truncated" not in info
    assert ends == [T, 2 * T]
    with pytest.raises(ValueError):
        HSREnv("c2_push.hsrb", None, max_episode_steps=T, autoreset=True)
    env.close()


def test_defaults_unchanged():
    """With the options off, step() and reset() are today's, also on a handle whose episode buffers exist."""
    n = 128
    A = _env("c2_push", n, steps_per_action=60)
    B = _env("c2_push", n, steps_per_action=60)
    A.set_episode_ages(torch.full((n,), 3, dtype=torch.int32, device="cuda:0"))
    A.episode_stats()
    assert torch.equal(A.reset(), B.reset())
    for k in range(4):
        oa, ra, da, ia = A.step(_actions(A, k))
        ob, rb, db, ib = B.step(_actions(B, k))
        assert set(ia) == set(ib) == {"log count", "substeps_taken", "bad_state"}
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
        assert torch.equal(ia["substeps_taken"], ib["substeps_taken"])
        assert torch.equal(A.reset(mask=da), B.reset(mask=db))
    assert _state_equal(A, B)
    with pytest.raises(NotImplementedError):
        _env("c2_push", 4, max_episode_steps=T).step_host(np.zeros((4, 2), np.float32))
    A.close(); B.close()
