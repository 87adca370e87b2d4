"""Open-loop rollouts on the B200 (hsrb_rollout, BatchedHSREnv.rollout): K actions in one call give, bit for bit, what K
step() calls on a twin handle (same seed, same reset) give - every slice of obs / reward / done / substeps_taken /
bad_state, the state afterwards and every work counter but `launches` - through the fused launch of the phase-locked
kernels and through the one-launch-per-action fallback of every other kernel."""
import numpy as np
import pytest

from test_episodes import _cfg

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

NSUB = 100
COUNTERS = ("substeps", "newton_iters", "narrowphase", "ls_evals", "contacts", "efc_rows", "bad_envs", "flops")


def _env(name, n, kernel="auto", goals=None, **kw):
    from hsr_env_b200.env import BatchedHSREnv

    g, starts = _cfg(name)
    return BatchedHSREnv(f"{name}.hsrb", goals or g, starts=starts, n_envs=n, device="cuda:0", seed=5, kernel=kernel,
                         steps_per_action=NSUB, **kw)


def _actions(env, K, seed=0):
    rng = np.random.default_rng(seed)
    lo, hi = env.model.act_ctrlrange[:, 0], env.model.act_ctrlrange[:, 1]
    return torch.tensor(rng.uniform(lo, hi, (K, env.n_envs, env.nu)), dtype=torch.float32, device="cuda:0")


def _twin_check(A, B, K, launches_per_call):
    """A.rollout(K actions) against K B.step() calls; A and B freshly created with the same arguments."""
    assert torch.equal(A.reset(), B.reset())
    act = _actions(A, K)
    l0 = A.stats()["launches"]
    obs, reward, done, info = A.rollout(act)
    assert A.stats()["launches"] - l0 == launches_per_call
    assert obs.shape == (K, A.n_envs, A.state_dim) and reward.shape == done.shape == (K, A.n_envs)
    assert done.dtype == torch.bool and info["substeps_taken"].dtype == torch.int32
    for k in range(K):
        o, r, d, i = B.step(act[k])
        assert torch.equal(obs[k], o) and torch.equal(reward[k], r) and torch.equal(done[k], d), k
        assert torch.equal(info["substeps_taken"][k], i["substeps_taken"]) and torch.equal(info["bad_state"][k], i["bad_state"]), k
    for x, y in zip(A.get_state(), B.get_state()):
        assert torch.equal(x, y)
    sa, sb = A.stats(), B.stats()
    for key in COUNTERS:
        assert sa[key] == sb[key], key
    assert A._time_steps == B._time_steps == K
    return done


# (model, n, kernel): the wpe kernel at 256 environments and at more than one wave, the
# phase-locked general kernel on the articulated, clutter and cupboard models
FUSED = [("c2_push", 256, "wpe"), ("c2_push", 16384, "wpe"), ("c3_arm", 64, "general"), ("c5_clutter", 32, "general"),
         ("f2_cupboard", 64, "general")]


@pytest.mark.parametrize("K", [1, 7, 20])
@pytest.mark.parametrize("name,n,kernel", FUSED)
def test_fused_rollout_bit_equal_to_steps(name, n, kernel, K):
    A, B = _env(name, n, kernel), _env(name, n, kernel)
    done = _twin_check(A, B, K, 1)
    if K == 20 and name == "c2_push":
        assert done.any()   # some environments reached the goal and carried on from there


def test_goal_list_rollout():
    """A goal list on c2_push takes the phase-locked general kernel."""
    from hsr_env_b200.spaces import Box
    from hsr_env_b200.util import GoalSpec
    from scenarios import GOAL_HI, GOAL_LO

    goals = [GoalSpec("block0", Box(GOAL_LO, GOAL_HI), .05)]
    A, B = _env("c2_push", 128, goals=goals), _env("c2_push", 128, goals=goals)
    _twin_check(A, B, 7, 1)
    assert A.launch_info()["kernel"] == "general"   # the goals are pushed at reset


@pytest.mark.parametrize("name,n,kernel", [("c2_push", 256, "wpe"), ("c2_push", 256, "general"), ("c3_arm", 64, "general")])
def test_rollout_with_params(name, n, kernel):
    prm = torch.tensor([[2, .5, 1, 2], [.5, 2, 2, .5], [1.3, .7, .9, 1.1], [1, 1, 1, 1]])[torch.arange(n) % 4]
    A, B = _env(name, n, kernel), _env(name, n, kernel)
    A.set_env_params(prm); B.set_env_params(prm)
    _twin_check(A, B, 7, 1)
    ranges = {"friction": (0.5, 2.0), "damping": (0.5, 2.0)}
    A, B = _env(name, n, kernel, randomize=ranges), _env(name, n, kernel, randomize=ranges)
    _twin_check(A, B, 7, 1)


@pytest.mark.parametrize("case", ["lockstep", "lanes8", "wpe_free", "general_free"])
def test_fallback_rollout_bit_equal(case, monkeypatch):
    """Kernels without a rollout instance run one launch per action, with the same bits."""
    name, kernel, kw = "c2_push", "auto", {}
    if case == "lockstep":
        kernel = "lockstep"
    elif case == "lanes8":
        kernel, kw = "general", {"lanes_per_env": 8}
    elif case == "wpe_free":
        monkeypatch.setenv("HSRB_WPE_LOCK", "0")
        kernel = "wpe"
    else:
        monkeypatch.setenv("HSRB_GENERAL_LOCK", "0")
        name, kernel = "c3_arm", "general"
    A, B = _env(name, 256, kernel, **kw), _env(name, 256, kernel, **kw)
    _twin_check(A, B, 5, 5)


def test_rollout_independent_of_sort(monkeypatch):
    A = _env("c2_push", 16384, "wpe")
    act = _actions(A, 7, seed=3)
    A.reset()
    ref = A.rollout(act)
    ref_state = A.get_state()
    monkeypatch.setenv("HSRB_WPE_SORT", "0")
    B = _env("c2_push", 16384, "wpe")
    B.reset()
    got = B.rollout(act)
    for x, y in zip(ref[:3], got[:3]):
        assert torch.equal(x, y)
    for key in ("substeps_taken", "bad_state"):
        assert torch.equal(ref[3][key], got[3][key])
    for x, y in zip(ref_state, B.get_state()):
        assert torch.equal(x, y)


def test_rollout_leaves_episodes_untouched():
    from hsr_env_b200 import lib

    A = _env("c2_push", 256, "wpe")
    A.reset()
    P = lib.ptr
    n = A.n_envs
    ctrl = _actions(A, 3)
    # the episode buffers exist once an episode entry point ran; set some ages, then roll out through the C ABI
    A.set_episode_ages((torch.arange(n, device="cuda:0") % 20).to(torch.int32))
    ages, stats = A.episode_ages().clone(), A.episode_stats()
    with torch.cuda.device(A.device):
        lib.check(A._lib.hsrb_rollout(A._h, P(ctrl), 3, NSUB, None, None, None, None, None, A._stream()))
    assert torch.equal(A.episode_ages(), ages) and A.episode_stats() == stats


def test_rollout_rejections():
    from hsr_env_b200 import lib

    A = _env("c2_push", 64, "wpe")
    A.reset()
    ctrl = _actions(A, 2)
    L, P, s = A._lib, lib.ptr, A._stream()
    assert L.hsrb_rollout(A._h, P(ctrl), -1, NSUB, None, None, None, None, None, s) == -1
    assert L.hsrb_rollout(A._h, P(ctrl), 2, -1, None, None, None, None, None, s) == -1
    assert L.hsrb_rollout(A._h, None, 2, NSUB, None, None, None, None, None, s) == -1
    state = A.get_state()
    launches = A.stats()["launches"]
    assert L.hsrb_rollout(A._h, P(ctrl), 0, NSUB, None, None, None, None, None, s) == 0
    assert A.stats()["launches"] == launches and all(torch.equal(x, y) for x, y in zip(state, A.get_state()))
    for bad in (ctrl[0], ctrl[:, :32], ctrl[..., :1]):
        with pytest.raises(ValueError):
            A.rollout(bad)
    with pytest.raises(NotImplementedError):
        O = _env("c3_arm", 64, "general", obs_type="openai")
        O.rollout(_actions(O, 2))
    with pytest.raises(NotImplementedError):
        _env("c2_push", 64, "wpe", max_episode_steps=20).rollout(ctrl)
    with pytest.raises(NotImplementedError):
        _env("c2_push", 64, "wpe", autoreset=True).rollout(ctrl)
