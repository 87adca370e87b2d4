"""The contact query on the B200 (hsrb_contacts, BatchedHSREnv.contacts / contact_wrench, HSREnv.contacts): bit for bit the
contact part of hsrb_debug_substep's dump on the same state and action, with and without per-environment parameters; no
effect on the state, the next step or the work counters; the same bits whatever kernel step() runs; the block-at-rest
known answer; rejected inputs; and the single-environment form."""
import numpy as np
import pytest

from test_episodes import _cfg

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

NSUB = 40


def _env(name, n, kernel="auto", seed=5, **kw):
    from hsr_env_b200.env import BatchedHSREnv

    g, starts = _cfg(name)
    return BatchedHSREnv(f"{name}.hsrb", g, starts=starts, n_envs=n, device="cuda:0", seed=seed, kernel=kernel,
                         steps_per_action=NSUB, **kw)


def _actions(env, seed=0):
    rng = np.random.default_rng(seed)
    lo, hi = env.model.act_ctrlrange[:, 0], env.model.act_ctrlrange[:, 1]
    return torch.tensor(rng.uniform(lo, hi, (env.n_envs, env.nu)), dtype=torch.float32, device="cuda:0")


def _warm_up(env, name):
    """A state with contacts: reset and two actions (c3_arm: arm over the pan, block under the fingers)."""
    env.reset()
    if name == "c3_arm":
        from oracle import port
        from scenarios import initial_states

        q = initial_states(env.model, env.n_envs, seed=9, pan=True, port=port.CpuPort(env.model))
        env.set_state(qpos=q.astype(np.float32), qvel=np.zeros((env.n_envs, env.nv), np.float32))
    for k in range(2):
        env.step(_actions(env, 100 + k))


def dump_contacts(env, dump):
    """count [N], pair [N, nc], dist, pos [N, nc, 3], frame [N, nc, 3, 3], force [N, nc, 6] of a debug dump (hsr_core.h
    debug_dump layout; the efc_force rows of contact c follow the joint-limit rows and the rows of contacts < c)."""
    m = env.model
    d = dump.cpu().numpy()
    nq, nv, nb, nc = env.nq, env.nv, env.nbody, env.contact_capacity()
    ne = (d.shape[1] - (4 + nb * 3 + nv * nv + 3 * nv + nc * 14 + nq + nv)) // (nv + 3)
    off = 4 + nb * 3 + nv * nv + 3 * nv
    con = d[:, off:off + nc * 14].reshape(-1, nc, 14)
    efc = d[:, off + nc * 14:off + nc * 14 + ne * (nv + 3)].reshape(-1, ne, nv + 3)
    n = d.shape[0]
    count = d[:, 0].astype(np.int64)
    pair = con[:, :, 0].astype(np.int64)
    force = np.zeros((n, nc, 6))
    for e in range(n):
        r = int(d[e, 2])
        for c in range(count[e]):
            dim = int(m.pair_condim[pair[e, c]])
            force[e, c, :dim] = efc[e, r:r + dim, nv + 2]
            r += dim
    return dict(count=count, pair=pair, dist=con[:, :, 1], pos=con[:, :, 2:5], frame=con[:, :, 5:14].reshape(n, nc, 3, 3),
                force=force)


def check_equal_to_dump(c, ref):
    assert np.array_equal(c["count"].cpu().numpy(), ref["count"])
    assert np.array_equal(c["pair"].cpu().numpy(), ref["pair"])   # padding: -1 in both
    for k in ("dist", "pos", "frame", "force"):
        assert np.array_equal(c[k].cpu().numpy().astype(np.float64), ref[k]), k


def _params(n, seed=3):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (0.5 + 1.5 * torch.rand(n, 4, generator=g)).to("cuda:0")


@pytest.mark.parametrize("with_params", [False, True], ids=["nominal", "params"])
@pytest.mark.parametrize("name,n", [("c2_push", 4096), ("c3_arm", 64), ("f2_cupboard", 64)])
def test_contacts_equal_debug_substep(name, n, with_params):
    env = _env(name, n)
    _warm_up(env, name)
    if with_params:
        env.set_env_params(_params(n))
    act = _actions(env, 7)
    qpos, qvel, warm, mocap = env.get_state()
    c = env.contacts(act)
    assert all(torch.equal(x, y) for x, y in zip(env.get_state(), (qpos, qvel, warm, mocap)))
    dump = env.debug_substep(act)            # advances the state
    env.set_state(qpos, qvel, warm, mocap)
    ref = dump_contacts(env, dump)
    check_equal_to_dump(c, ref)
    assert ref["count"].sum() > 0
    # geom / body / dim from the model's pair tables, -1 on padding rows
    m = env.model
    pair = c["pair"].cpu().numpy()
    on = pair >= 0
    assert np.array_equal(c["geom"][..., 0].cpu().numpy()[on], m.pair_geom1[pair[on]])
    assert np.array_equal(c["body"][..., 1].cpu().numpy()[on], m.geom_body[m.pair_geom2[pair[on]]])
    assert np.array_equal(c["dim"].cpu().numpy()[on], m.pair_condim[pair[on]])
    assert np.all(c["geom"].cpu().numpy()[~on] == -1) and np.all(c["dim"].cpu().numpy()[~on] == -1)
    # the wrench call (contact rows NULL) runs the same forward pass; its rows sum to zero force
    w = env.contact_wrench(act).double()
    scale = max(1.0, w.abs().max().item())
    assert w[:, :, :3].sum(dim=1).abs().max().item() < 1e-5 * scale


def test_query_changes_nothing():
    """After contacts() and contact_wrench(), the state is unchanged, the next step gives the bits of a twin handle that
    skipped them, and the work counters are unchanged except launches (+1 per call)."""
    A, B = _env("c2_push", 1024), _env("c2_push", 1024)
    for env in (A, B):
        _warm_up(env, "c2_push")
    before, s0 = A.get_state(), A.stats()
    act = _actions(A, 11)
    A.contacts(act)
    s1 = A.stats()
    A.contact_wrench(act)
    s2 = A.stats()
    assert s1["launches"] == s0["launches"] + 1 and s2["launches"] == s1["launches"] + 1
    for k in s0:
        if k != "launches":
            assert s0[k] == s1[k] == s2[k], k
    assert all(torch.equal(x, y) for x, y in zip(A.get_state(), before))
    oa, ra, da, ia = A.step(act)
    ob, rb, db, ib = B.step(act)
    assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
    assert torch.equal(ia["bad_state"], ib["bad_state"]) and torch.equal(ia["substeps_taken"], ib["substeps_taken"])
    assert all(torch.equal(x, y) for x, y in zip(A.get_state(), B.get_state()))


def test_independent_of_kernel_choice():
    """auto / wpe / lockstep / general handles in the same state report the same bits: the query always runs the general
    path's stages."""
    ref = None
    for kernel in ("auto", "wpe", "lockstep", "general"):
        env = _env("c2_push", 512, kernel=kernel)   # same seed: the same reset state (resets run the general kernel)
        env.reset()
        act = _actions(env, 4)
        c = env.contacts(act)
        c["wrench"] = env.contact_wrench(act)
        if ref is None:
            ref = c
            assert c["count"].sum().item() > 0
        else:
            for k in ref:
                assert torch.equal(c[k], ref[k]), (kernel, k)


@pytest.mark.parametrize("mb", [1.0, 2.0])
def test_block_at_rest_known_answer(mb):
    """The block of c2_push settled on the floor (fp64 port, 600 substeps, with the block mass the multiplier gives): its
    contact wrench is (0, 0, mb m g) with no torque; the floor's row holds the reaction."""
    from oracle import port as P

    from test_contacts_emu import edited

    env = _env("c2_push", 1)
    env.reset()
    m = env.model
    q = m.qpos0.copy()
    a = int(m.jnt_qposadr[m.body_jntadr[m.block_body[0]]])
    q[a:a + 7] = [0.3, 0.4, 0.017, 1, 0, 0, 0]
    z = np.zeros(m.nv)
    r = P.CpuPort(edited(m, (1, mb, 1, 1))).step(q, z, z, np.zeros(m.nu), nsub=600)
    env.set_state(qpos=r["qpos"].astype(np.float32), qvel=r["qvel"].astype(np.float32), qacc_warmstart=r["warm"].astype(np.float32))
    if mb != 1.0:
        env.set_env_params(torch.tensor([[1, mb, 1, 1]], dtype=torch.float32, device="cuda:0"))
    w = env.contact_wrench().double().cpu().numpy()[0]
    c = env.contacts()
    b = int(m.block_body[0])
    mg = mb * float(m.body_mass[b]) * abs(float(m.opt[3]))
    assert c["count"][0].item() == 4 and c["bad_state"][0].item() == 0
    assert np.allclose(w[b, :3], [0, 0, mg], rtol=1e-4, atol=1e-4 * mg), (w[b], mg)
    assert np.abs(w[b, 3:]).max() < 1e-4 * mg
    assert np.allclose(w[0, :3], [0, 0, -mg], rtol=1e-4, atol=1e-4 * mg)


def test_rejections():
    from hsr_env_b200 import lib

    env = _env("c2_push", 8)
    env.reset()
    pair = torch.zeros(8, 4, dtype=torch.int32, device="cuda:0")
    rc = env._lib.hsrb_contacts(env._h, None, 0, None, lib.ptr(pair), None, None, None, None, None, None, env._stream())
    assert rc == -1
    with pytest.raises(lib.HsrbError):
        lib.check(rc)
    # without per-contact outputs max_contacts is not read
    assert env._lib.hsrb_contacts(env._h, None, 0, lib.ptr(pair[:, 0].contiguous()), None, None, None, None, None, None, None,
                                  env._stream()) == 0
    with pytest.raises(ValueError):
        env.contacts(max_contacts=0)
    with pytest.raises(ValueError):
        env.contacts(torch.zeros(8, env.nu + 1, device="cuda:0"))
    with pytest.raises(ValueError):
        env.contact_wrench(torch.zeros(4, env.nu, device="cuda:0"))
    c = env.contacts(max_contacts=2)
    assert c["pair"].shape == (8, 2) and c["force"].shape == (8, 2, 6) and c["frame"].shape == (8, 2, 3, 3)


def test_single_env_contacts():
    from hsr_env_b200.env import BatchedHSREnv, HSREnv

    g, starts = _cfg("c2_push")
    env = HSREnv("c2_push.hsrb", g, starts=starts, steps_per_action=NSUB, seed=2)
    env.reset()
    env.set_state(qpos=env.model.qpos0.astype(np.float32))   # the block lying flat on the floor: four corner contacts
    a = np.array([0.5, 0.0], np.float32)
    env.step(a)
    c = env.contacts(a)
    k = c["ncon"]
    assert k > 0
    assert c["pair"].shape == (k,) and c["geom"].shape == (k, 2) and c["body"].shape == (k, 2) and c["dim"].shape == (k,)
    assert c["pos"].shape == (k, 3) and c["frame"].shape == (k, 3, 3) and c["force"].shape == (k, 6) and c["dist"].shape == (k,)
    names = env.model.names
    assert c["geom_names"] == [(names["geom"][i], names["geom"][j]) for i, j in c["geom"]]
    assert c["body_names"] == [(names["body"][i], names["body"][j]) for i, j in c["body"]]
    b = BatchedHSREnv.contacts(env, torch.tensor(a[None], device="cuda:0"))
    assert int(b["count"][0]) == k
    assert np.array_equal(b["pair"][0, :k].cpu().numpy(), c["pair"])
    assert np.array_equal(b["force"][0, :k].cpu().numpy().astype(np.float64), c["force"])
    w = env.contact_wrench(a)
    assert w.shape == (env.nbody, 6)
    assert np.array_equal(w, BatchedHSREnv.contact_wrench(env, a[None])[0].double().cpu().numpy())
