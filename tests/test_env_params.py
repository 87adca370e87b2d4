"""Per-environment physics parameters on the B200 (BatchedHSREnv.set_env_params / randomize): unit multipliers give the
bits of a handle without parameters, power-of-two multipliers the bits of default handles built from edited models,
other multipliers match the fp64 port on the edited model, resets draw the parameters of hsr_core.h sample_env_params,
and friction changes how far a sliding block goes.

The reference of an environment with multipliers s is the model whose arrays were scaled by s and written out as a blob
(tests/test_env_params_emu.py: edited)."""
import numpy as np
import pytest

from scenarios import rel_err, rollout_states
from test_env_params_emu import edited, env_params

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

NSUB = 100
TUPLES = torch.tensor([[2, .5, 1, 2], [.5, 2, 2, .5], [2, 2, .5, 1], [.5, .5, 2, 2], [1, 1, 1, 1]])


def _env(name, n, kernel="auto", model=None, lanes=0, **kw):
    from test_episodes import _cfg
    from hsr_env_b200.env import BatchedHSREnv

    g, starts = _cfg(name)
    return BatchedHSREnv(model if model is not None else f"{name}.hsrb", g, starts=starts, n_envs=n, device="cuda:0", seed=3,
                         kernel=kernel, lanes_per_env=lanes, steps_per_action=NSUB, **kw)


def _actions(env, k):
    rng = np.random.default_rng(7919 * k + 1)
    lo, hi = env.model.act_ctrlrange[:, 0], env.model.act_ctrlrange[:, 1]
    return torch.tensor(rng.uniform(lo, hi, (env.n_envs, env.nu)), dtype=torch.float32, device="cuda:0")


def _outputs(env, act):
    obs, reward, done, info = env.step(act)
    return [obs, reward, done, info["substeps_taken"], info["bad_state"], *env.get_state()]


# (model, n, kernel, lanes_per_env): the wpe kernel at 256 environments and at more than it holds resident, the general
# path's phase-locked (lanes 0) and 8-lane kernels, and the general kernel on the articulated and goal-list models
CASES = [("c2_push", 256, "wpe", 0), ("c2_push", 16384, "wpe", 0), ("c2_push", 256, "general", 0), ("c2_push", 256, "general", 8),
         ("c3_arm", 64, "general", 0), ("c5_clutter", 32, "general", 0), ("f2_cupboard", 64, "general", 0)]


@pytest.mark.parametrize("name,n,kernel,lanes", CASES)
def test_unit_params_bit_equal(name, n, kernel, lanes):
    A = _env(name, n, kernel, lanes=lanes)
    B = _env(name, n, kernel, lanes=lanes)
    A.set_env_params(torch.ones(n, 4))
    assert torch.equal(A.env_params(), torch.ones(n, 4, device="cuda:0"))
    assert A.launch_info() == B.launch_info()
    assert torch.equal(A.reset(), B.reset())
    for k in range(20):
        act = _actions(A, k)
        for x, y in zip(_outputs(A, act), _outputs(B, act)):
            assert torch.equal(x, y), k
    sa, sb = A.stats(), B.stats()
    for key in ("substeps", "newton_iters", "narrowphase", "ls_evals", "contacts", "efc_rows", "bad_envs", "flops"):
        assert sa[key] == sb[key], key


@pytest.mark.parametrize("name,n,kernel,lanes", CASES)
def test_power_of_two_params_match_edited_models(name, n, kernel, lanes, models):
    idx = torch.arange(n) % len(TUPLES)
    A = _env(name, n, kernel, lanes=lanes)
    A.set_env_params(TUPLES[idx])
    refs = [_env(name, n, kernel, lanes=lanes, model=edited(models[name], t.numpy())) for t in TUPLES]
    obs = A.reset()
    for R in refs:
        assert torch.equal(R.reset(), obs)
    for k in range(20):
        act = _actions(A, k)
        got = _outputs(A, act)
        for t, R in enumerate(refs):
            rows = (idx == t).to("cuda:0")
            for x, y in zip(got, _outputs(R, act)):
                assert torch.equal(x[rows], y[rows]), (k, t)


@pytest.mark.parametrize("name,n,kernel,lanes", [c for c in CASES if c[1] <= 256])
def test_params_match_oracle(name, n, kernel, lanes, models, ports):
    """Multipliers ~ U[0.5, 2]: one substep against the fp64 port on each environment's edited model, at the tolerance and
    allowance of tests/test_gpu_parity.py."""
    from oracle import port

    n = min(n, 48)
    model = models[name]
    qpos, qvel, warm, ctrl = rollout_states(ports[name], model, n, seed=len(name) * 7, pan=name in ("c3_arm", "f2_cupboard"),
                                            float32=True)
    prm = np.random.default_rng(9).uniform(0.5, 2.0, (n, 4)).astype(np.float32)
    env = _env(name, n, kernel, lanes=lanes)
    env.set_env_params(torch.tensor(prm))
    env.set_state(qpos, qvel, warm)
    obs, _, _, info = env.step(torch.tensor(ctrl, dtype=torch.float32), steps=1)
    got = obs.double().cpu().numpy()
    over = 0
    for e in range(n):
        ref = port.CpuPort(edited(model, prm[e].astype(np.float64))).step(qpos[e:e + 1], qvel[e:e + 1], warm[e:e + 1], ctrl[e:e + 1], nsub=1)
        assert rel_err(got[e:e + 1, :model.nq], ref["qpos"]).max() <= 1e-4, e
        over += int(rel_err(got[e:e + 1, model.nq:], ref["qvel"]).max() > 1e-4)
    assert over <= max(1, n // 100), over


RANGES = {"friction": (.5, 2.), "block_mass": (.5, 2.), "actuator_gain": (.5, 2.), "damping": (.5, 2.)}
LO, HI = np.array([.5] * 4, np.float32), np.array([2.] * 4, np.float32)


def test_reset_draws_match_port():
    n, off = 300, 17
    from hsr_env_b200.env import BatchedHSREnv
    from test_episodes import _cfg

    g, _ = _cfg("c2_push")
    env = BatchedHSREnv("c2_push.hsrb", g, n_envs=n, device="cuda:0", seed=11, env_id_offset=off, randomize=RANGES)
    plain = BatchedHSREnv("c2_push.hsrb", g, n_envs=n, device="cuda:0", seed=11, env_id_offset=off)
    assert torch.equal(env.reset(), plain.reset())          # the reset state does not depend on the ranges
    want = np.array([env_params(LO, HI, 11, off + e, 0) for e in range(n)])
    assert np.array_equal(env.env_params().cpu().numpy(), want)
    # a masked reset redraws only the masked environments
    mask = torch.zeros(n, dtype=torch.bool, device="cuda:0"); mask[::3] = True
    before = env.env_params()
    env.reset(mask=mask); plain.reset(mask=mask)
    after = env.env_params()
    assert torch.equal(after[~mask], before[~mask])
    m = mask.cpu().numpy()
    want2 = np.array([env_params(LO, HI, 11, off + e, 1) for e in np.nonzero(m)[0]])
    assert np.array_equal(after[mask].cpu().numpy(), want2)
    assert all(torch.equal(x, y) for x, y in zip(env.get_state(), plain.get_state()))
    # a handle whose environments are rows k.. of a larger one
    big = BatchedHSREnv("c2_push.hsrb", g, n_envs=n + off, device="cuda:0", seed=11, randomize=RANGES)
    big.reset()
    small = BatchedHSREnv("c2_push.hsrb", g, n_envs=n, device="cuda:0", seed=11, env_id_offset=off, randomize=RANGES)
    small.reset()
    assert torch.equal(big.env_params()[off:], small.env_params())
    assert all(torch.equal(x[off:], y) for x, y in zip(big.get_state(), small.get_state()))


@pytest.mark.parametrize("kernel", ["wpe", "general"])
def test_autoreset_draws_match_manual_loop(kernel):
    n, T = 256, 20
    A = _env("c2_push", n, kernel, max_episode_steps=T, autoreset=True, randomize=RANGES)
    B = _env("c2_push", n, kernel, randomize=RANGES)
    assert torch.equal(A.reset(), B.reset())
    age = (torch.arange(n, device="cuda:0") % T).to(torch.int32)
    A.set_episode_ages(age)
    for k in range(45):
        act = _actions(A, k)
        oa, ra, da, _ = A.step(act)
        ob, rb, db, _ = B.step(act)
        age += 1
        mask = db | (age >= T)
        assert torch.equal(da, mask)
        ob = B.reset(mask=mask)
        age[mask] = 0
        assert torch.equal(oa, ob), k
        assert torch.equal(A.env_params(), B.env_params()), k
        assert all(torch.equal(x, y) for x, y in zip(A.get_state(), B.get_state())), k


def test_lockstep_kernel_refuses_params():
    from hsr_env_b200.lib import HsrbError

    env = _env("c2_push", 64, "lockstep")
    env.reset()
    env.set_env_params(torch.ones(64, 4))
    with pytest.raises(HsrbError, match="per-environment parameters"):
        env.step(_actions(env, 0))
    with pytest.raises(HsrbError, match="per-environment parameters"):
        env.launch_info()
    with pytest.raises(HsrbError, match="per-environment parameters"):
        from hsr_env_b200 import lib as L
        L.check(env._lib.hsrb_set_path(env._h, 2))
    env.set_env_params(None)
    assert env.launch_info()["kernel"] == "fast"
    with pytest.raises(HsrbError):
        env.set_param_ranges({"friction": (0.0, 1.0)})        # friction must stay > 0
    with pytest.raises(HsrbError):
        env.set_param_ranges({"damping": (float("nan"), 1.0)})
    with pytest.raises(ValueError):
        env.set_env_params({"block_mass": torch.zeros(64)})


@pytest.mark.parametrize("kernel", ["wpe", "general"])
def test_clearing_params_returns_to_default_kernel(kernel):
    n = 256
    A = _env("c2_push", n, kernel)
    B = _env("c2_push", n, kernel)
    A.set_env_params(TUPLES[torch.arange(n) % len(TUPLES)])
    A.reset(); B.reset()
    A.step(_actions(A, 0))
    A.set_env_params(None)
    assert torch.equal(A.env_params(), torch.ones(n, 4, device="cuda:0"))
    st = B.get_state()
    A.set_state(*st)
    for k in range(1, 6):
        act = _actions(A, k)
        for x, y in zip(_outputs(A, act), _outputs(B, act)):
            assert torch.equal(x, y), k


def _slide_distance(friction, block_mass, backend, models=None):
    """The block of the block-push model resting on the floor far from the robot, pushed to 0.5 m/s along x: the distance
    it slides (Coulomb: v^2 / (2 mu g)).  backend 'gpu': one environment per multiplier pair on the wpe kernel;
    'port': the fp64 port on the edited model."""
    from scenarios import block_adr

    model = models["c2_push"]
    a = block_adr(model)[0]
    q = model.qpos0.astype(np.float64).copy()
    q[a:a + 3] = [.6, .3, .017]          # a 3.4 cm cube on the floor, 0.6 m in front of the base
    q[a + 3:a + 7] = [1, 0, 0, 0]
    v = np.zeros(model.nv)
    dof = int(model.jnt_dofadr[model.body_jntadr[model.block_body[0]]])
    v[dof] = .5
    n = len(friction)
    qpos, qvel, warm = np.tile(q, (n, 1)), np.tile(v, (n, 1)), np.zeros((n, model.nv))
    ctrl = np.zeros((n, model.nu))
    steps = 400
    if backend == "port":
        from oracle import port
        out = []
        for f, m in zip(friction, block_mass):
            r = port.CpuPort(edited(model, (f, m, 1, 1))).step(qpos[:1], qvel[:1], warm[:1], ctrl[:1], nsub=steps)
            out.append(r["qpos"][0, a] - q[a])
        return np.array(out)
    from hsr_env_b200.env import BatchedHSREnv
    env = BatchedHSREnv("c2_push.hsrb", None, n_envs=n, device="cuda:0", kernel="wpe")
    env.set_env_params({"friction": torch.tensor(friction), "block_mass": torch.tensor(block_mass)})
    env.set_state(qpos, qvel, warm)
    obs, _, _, _ = env.step(torch.zeros(n, model.nu, device="cuda:0"), steps=steps)
    return obs[:, a].double().cpu().numpy() - q[a]


def test_friction_changes_sliding_distance(models):
    fr = [.5, 1., 2., 1., 1.]
    mb = [1., 1., 1., .5, 2.]
    got = _slide_distance(fr, mb, "gpu", models)
    ref = _slide_distance(fr, mb, "port", models)
    print("sliding distance gpu", got, "port", ref)
    assert np.all(got > 0)
    assert got[0] > got[1] > got[2]
    assert 1.6 < got[0] / got[1] < 2.4 and 1.6 < got[1] / got[2] < 2.4
    # the mass of the block does not change the Coulomb distance; tolerance: the port's own spread on the edited models
    tol = 2 * max(abs(ref[3] - ref[1]), abs(ref[4] - ref[1])) + 1e-4
    assert abs(got[3] - got[1]) <= tol and abs(got[4] - got[1]) <= tol, (got, ref, tol)
    np.testing.assert_allclose(got, ref, rtol=2e-2, atol=2e-4)   # fp32 over 400 substeps against the fp64 port
