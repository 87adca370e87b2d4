"""Transition derivatives on the B200 (hsrb_transition_fd, BatchedHSREnv.transition_fd, HSREnv.transition_fd): next_obs is
nsubsteps chained hsrb_debug_substep calls on a twin handle, bit for bit; A and B equal the columns rebuilt from twin-handle
set_state(perturbed input) + debug_substep chains (bit for bit, 2 fp32 ulp in free-joint rotation rows and columns); with and
without per-environment parameters; no effect on the state, the next step or the work counters; the same bits whatever
kernel step() runs; the c1_readme known answer; rejected inputs; and the single-environment form."""
import numpy as np
import pytest

from test_contacts import _actions, _env, _params, _warm_up
from test_transition_fd_emu import numpy_AB, nruns, perturbed, tolerant_mask, within_ulps

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

EPS = 1e-3


def chain(env, act, nsub):
    """nsub debug_substep calls from the current state; returns qpos | qvel [N, nq + nv] and leaves the state advanced"""
    for _ in range(nsub):
        env.debug_substep(act)
    q, v, _, _ = env.get_state()
    return torch.cat([q, v], 1).cpu().numpy()


def reconstruct(env, act, nsub, centered, rows_out=None):
    """A, B of every environment from set_state(perturbed input) + debug_substep chains on the handle (restores its state)"""
    m = env.model
    n, nq, nv = env.n_envs, env.nq, env.nv
    state = env.get_state()
    q0, v0, w0, mo = (t.cpu().numpy() for t in state)
    u0 = act.cpu().numpy()
    x0 = np.concatenate([q0, v0], 1)
    nr = nruns(m, centered)
    rows = np.zeros((n, nr, nq + nv), np.float32)
    hs = np.zeros((n, nr))
    for r in range(nr):
        ins = [perturbed(m, x0[e], u0[e], r, centered, EPS) for e in range(n)]
        v = np.stack([i[0] for i in ins])
        hs[:, r] = [i[1] for i in ins]
        env.set_state(v[:, :nq], v[:, nq:nq + nv], w0, mo)
        rows[:, r] = chain(env, torch.tensor(v[:, nq + nv:], device="cuda:0"), nsub)
    env.set_state(*state)
    A = np.zeros((n, 2 * nv, 2 * nv), np.float32)
    B = np.zeros((n, 2 * nv, env.nu), np.float32)
    for e in range(n):
        A[e], B[e] = numpy_AB(m, rows[e], hs[e], u0[e], centered, EPS)
    return A, B, rows


def check(env, got, A, B):
    mA, mB = tolerant_mask(env.model)
    for g, w, msk in ((got["A"].cpu().numpy(), A, mA), (got["B"].cpu().numpy(), B, mB)):
        assert np.array_equal(g[:, ~msk], w[:, ~msk])
        assert np.all(within_ulps(g[:, msk], w[:, msk]))


@pytest.mark.parametrize("nsub", [1, 3])
@pytest.mark.parametrize("with_params", [False, True], ids=["nominal", "params"])
@pytest.mark.parametrize("name,n", [("c2_push", 4096), ("c3_arm", 64), ("f2_cupboard", 64)])
def test_equals_debug_substep_reconstruction(name, n, with_params, nsub):
    env = _env(name, n)
    _warm_up(env, name)
    if with_params:
        env.set_env_params(_params(n))
    act = _actions(env, 7)
    before = env.get_state()
    s0 = env.stats()
    out = env.transition_fd(act, eps=EPS, nsubsteps=nsub)
    s1 = env.stats()
    assert all(torch.equal(x, y) for x, y in zip(env.get_state(), before))
    assert s1["launches"] == s0["launches"] + 2 and all(s0[k] == s1[k] for k in s0 if k != "launches")
    # next_obs: the chained debug substeps of the unperturbed input
    ref = chain(env, act, nsub)
    env.set_state(*before)
    assert np.array_equal(out["next_obs"].cpu().numpy(), ref)
    if n > 64:   # the full reconstruction on a slice of c2_push (37 debug chains per environment)
        sub = _env(name, 64)
        sub.reset()
        sub.set_state(*(t[:64] for t in before))
        if with_params:
            sub.set_env_params(env.env_params()[:64].contiguous())
        A, B, rows = reconstruct(sub, act[:64].contiguous(), nsub, True)
        got = {k: v[:64] for k, v in out.items()}
    else:
        A, B, rows = reconstruct(env, act, nsub, True)
        got = out
    check(env, got, A, B)
    assert np.abs(A).max() > 0 and np.all(np.isfinite(A))


def test_forward_mode_and_rebuild():
    env = _env("c3_arm", 32)
    _warm_up(env, "c3_arm")
    act = _actions(env, 9)
    act[:4, 2] = float(env.model.act_ctrlrange[2, 1])        # at the upper limit: backward columns
    act[4:8, 3] = float(env.model.act_ctrlrange[3, 0]) - 0.1   # outside the range: zero columns
    out = env.transition_fd(act, eps=EPS, centered=False)
    A, B, _ = reconstruct(env, act, 1, False)
    check(env, out, A, B)
    assert torch.all(out["B"][4:8, :, 3] == 0)


def test_query_changes_nothing():
    """After transition_fd the next step gives the bits of a twin handle that skipped it."""
    A, B = _env("c2_push", 1024), _env("c2_push", 1024)
    for env in (A, B):
        _warm_up(env, "c2_push")
    act = _actions(A, 11)
    A.transition_fd(act, nsubsteps=3)
    oa, ra, da, ia = A.step(act)
    ob, rb, db, ib = B.step(act)
    assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
    assert torch.equal(ia["bad_state"], ib["bad_state"]) and torch.equal(ia["substeps_taken"], ib["substeps_taken"])
    assert all(torch.equal(x, y) for x, y in zip(A.get_state(), B.get_state()))


def test_independent_of_kernel_choice():
    ref = None
    for kernel in ("auto", "wpe", "lockstep", "general"):
        env = _env("c2_push", 512, kernel=kernel)
        env.reset()
        act = _actions(env, 4)
        out = env.transition_fd(act, nsubsteps=2)
        if ref is None:
            ref = out
        else:
            for k in ref:
                assert torch.equal(out[k], ref[k]), (kernel, k)


def test_affine_known_answer():
    """c1_readme, contact-free with no limit active and ctrl inside its range: the closed form of implicit-damping Euler."""
    from hsr_env_b200.env import BatchedHSREnv

    env = BatchedHSREnv("c1_readme.hsrb", None, n_envs=2, device="cuda:0")
    env.reset()
    m = env.model
    q = np.array([[0.03, -0.02], [0.05, 0.08]], np.float32)
    v = np.array([[0.1, -0.2], [0.0, 0.05]], np.float32)
    env.set_state(qpos=q, qvel=v, qacc_warmstart=np.zeros((2, 2), np.float32))
    u = torch.tensor([[0.12, -0.05], [0.2, 0.3]], device="cuda:0")
    out = env.transition_fd(u, eps=EPS)
    dump = env.debug_substep(u).cpu().numpy()
    dt, kp, g, D = m.timestep, m.act_kp, m.act_gear, np.diag(m.dof_damping)
    nb, nv = env.nbody, env.nv
    for e in range(2):
        assert dump[e, 0] == 0 and dump[e, 1] == 0   # ncon, nefc
        M = dump[e, 4 + nb * 3:4 + nb * 3 + nv * nv].reshape(nv, nv)
        Hi = np.linalg.inv(M + dt * D)
        dvdq, dvdv, dvdu = -dt * Hi @ np.diag(g * kp * g), np.eye(2) - dt * Hi @ D, dt * Hi @ np.diag(g * kp)
        A = np.block([[np.eye(2) + dt * dvdq, dt * dvdv], [dvdq, dvdv]])
        B = np.vstack([dt * dvdu, dvdu])
        assert np.allclose(out["A"][e].cpu().numpy(), A, rtol=1e-3, atol=2e-4)
        assert np.allclose(out["B"][e].cpu().numpy(), B, rtol=1e-3, atol=2e-4)


def test_rejections():
    from hsr_env_b200 import lib

    env = _env("c2_push", 8)
    env.reset()
    for eps, nsub in ((0.0, 1), (-1e-3, 1), (float("inf"), 1), (float("nan"), 1), (1e-3, 0)):
        rc = env._lib.hsrb_transition_fd(env._h, None, eps, 1, nsub, None, None, None, None, env._stream())
        assert rc == -1, (eps, nsub)
    for kw in (dict(eps=0), dict(eps=-1.0), dict(nsubsteps=0)):
        with pytest.raises(ValueError):
            env.transition_fd(**kw)
    with pytest.raises(ValueError):
        env.transition_fd(torch.zeros(8, env.nu + 1, device="cuda:0"))
    # a NULL ctrl reads as zeros; every output is nullable
    a = env.transition_fd()
    b = env.transition_fd(torch.zeros(8, env.nu, device="cuda:0"))
    assert all(torch.equal(a[k], b[k]) for k in a)
    assert env._lib.hsrb_transition_fd(env._h, None, 1e-3, 1, 1, None, None, None, None, env._stream()) == 0


def test_single_env_and_openai_obs():
    from hsr_env_b200.env import BatchedHSREnv, HSREnv

    from test_episodes import _cfg

    g, starts = _cfg("c2_push")
    env = HSREnv("c2_push.hsrb", g, starts=starts, steps_per_action=40, seed=2)
    env.reset()
    a = np.array([0.5, 0.0], np.float32)
    env.step(a)
    r = env.transition_fd(a, eps=EPS)
    assert r["A"].shape == (2 * env.nv, 2 * env.nv) and r["B"].shape == (2 * env.nv, env.nu) and r["A"].dtype == np.float64
    assert r["next_obs"].shape == (env.nq + env.nv,) and isinstance(r["bad_state"], int)
    b = BatchedHSREnv.transition_fd(env, torch.tensor(a[None], device="cuda:0"), eps=EPS)
    assert np.array_equal(r["A"], b["A"][0].double().cpu().numpy())
    # any obs_type and episode handles: the call reads only the resident state
    e2 = _env("c2_push", 16, obs_type="openai", max_episode_steps=5, autoreset=True)
    e2.reset()
    e2.step(_actions(e2, 1))
    out = e2.transition_fd(_actions(e2, 2))
    assert out["A"].shape == (16, 2 * e2.nv, 2 * e2.nv) and torch.isfinite(out["A"]).all()
