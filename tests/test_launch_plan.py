"""Kernel selection and launch plans (hsrb_api.cu: select(), one Plan per action kernel): launch_info() names the kernel a
STEP launch runs, for every model, kernel option, lanes-per-environment request and batch size; the experiment switches are
read when the handle is created."""
import numpy as np
import pytest

from scenarios import BLOCK_HI, BLOCK_LO, GOAL_HI, GOAL_LO

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

NAMES = ["c1_readme", "c1b_readme_block", "c2_push", "c3_arm", "c5_clutter", "f2_cupboard"]
FAMILY = ("c1_readme", "c1b_readme_block", "c2_push")   # sliding base + at most one free box: the fast kernels take these
FORCED = {"general": "general", "fast": "lockstep", "wpe": "wpe"}   # launch_info()["kernel"] -> the kernel= option that forces it


def _goals(name):
    from hsr_env_b200.spaces import Box
    from hsr_env_b200.util import GoalSpec

    if name == "c1_readme":
        return None
    if name == "f2_cupboard":   # the goal-list form
        return [GoalSpec(a="block", b=np.array([0, 0, .498]), distance=.05)]
    block = Box(BLOCK_LO, BLOCK_HI) if name in FAMILY else None
    return [GoalSpec(block, Box(GOAL_LO, GOAL_HI), .05)]


def _env(name, n, kernel, lanes, goals="default"):
    from hsr_env_b200.env import BatchedHSREnv

    return BatchedHSREnv(f"{name}.hsrb", _goals(name) if goals == "default" else goals, n_envs=n, device="cuda:0", seed=5,
                         kernel=kernel, lanes_per_env=lanes)


def _action(env):
    rng = np.random.default_rng(11)
    lo, hi = env.model.act_ctrlrange[:, 0], env.model.act_ctrlrange[:, 1]
    return torch.tensor(rng.uniform(lo, hi, (env.n_envs, env.nu)), dtype=torch.float32, device="cuda:0")


def _step(env, act):
    launches = env.stats()["launches"]
    obs, reward, done, info = env.step(act, steps=10)
    assert env.stats()["launches"] == launches + 1
    return [obs, reward, done, info["substeps_taken"], info["bad_state"], *env.get_state()]


@pytest.mark.parametrize("n", [1, 4100])
@pytest.mark.parametrize("lanes", [0, 8])
@pytest.mark.parametrize("name,kernel", [(m, k) for m in NAMES for k in ("auto", "general", "lockstep", "wpe")
                                         if m in FAMILY or k in ("auto", "general")])
def test_launch_info_names_the_kernel_that_runs(name, kernel, lanes, n):
    env = _env(name, n, kernel, lanes)
    env.reset()
    info = env.launch_info()
    assert info["kernel"] == {"auto": "wpe" if name in FAMILY else "general", "general": "general", "lockstep": "fast",
                              "wpe": "wpe"}[kernel]
    ref = _env(name, n, FORCED[info["kernel"]], lanes)
    assert ref.launch_info() == info
    ref.reset()
    act = _action(env)
    for got, want in zip(_step(env, act), _step(ref, act)):
        assert torch.equal(got, want)


def test_goal_list_on_the_fast_family():
    """The fast kernels take the env_wrapper goal form only: under kernel='wpe' a goal list runs the general kernel, under
    kernel='lockstep' it is an error, from launch_info() and step() alike."""
    from hsr_env_b200.lib import HsrbError
    from hsr_env_b200.spaces import Box
    from hsr_env_b200.util import GoalSpec

    goals = [GoalSpec("block0", Box(GOAL_LO, GOAL_HI), .05)]
    env = _env("c2_push", 64, "wpe", 0, goals)
    env.reset()
    assert env.launch_info()["kernel"] == "general"
    ref = _env("c2_push", 64, "general", 0, goals)
    ref.reset()
    act = _action(env)
    for got, want in zip(_step(env, act), _step(ref, act)):
        assert torch.equal(got, want)
    env = _env("c2_push", 64, "lockstep", 0, goals)
    env.reset()
    with pytest.raises(HsrbError, match="fast path not available"):
        env.launch_info()
    with pytest.raises(HsrbError, match="fast path not available"):
        env.step(act)


def test_switches_are_read_at_creation(monkeypatch):
    monkeypatch.setenv("HSRB_WPE_WPB", "14")
    env = _env("c2_push", 4096, "auto", 0)
    monkeypatch.delenv("HSRB_WPE_WPB")
    info = env.launch_info()
    assert info["kernel"] == "wpe" and info["threads_per_block"] == 448
    assert _env("c2_push", 4096, "auto", 0).launch_info()["threads_per_block"] != 448
    env.reset()
    env.step(_action(env), steps=1)
    assert env.launch_info() == info


def test_wpe_layout_at_4096_envs():
    """DESIGN 4.0: 4096 environments of the block-push model run as 148 blocks of 27-28 warps (not 147 of 28 and an idle SM)."""
    if torch.cuda.get_device_properties(0).multi_processor_count != 148:
        pytest.skip("the layout is stated for a 148-SM B200")
    info = _env("c2_push", 4096, "auto", 0).launch_info()
    assert (info["kernel"], info["grid"], info["threads_per_block"]) == ("wpe", 148, 896)
