"""The contact query without a GPU: hsrb_contacts_kernel on the SIMT emulator against the MODE_DEBUG launch of the general
action kernel (hsrb_debug_substep's dump) on the same inputs, bit for bit; against the fp64 port; known answers of a block
at rest; the per-body wrenches against a numpy recomputation; purity; capacities; and the ptxas budget of the instances."""
import ctypes
import re
import subprocess
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest

from scenarios import initial_states, rollout_states

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
EMU = HERE / "simt_emu"
LIB = ROOT / "oracle" / "_build" / "libcontacts_emu.so"
CSRC = ROOT / "hsr_env_b200" / "csrc"
DEPS = [EMU / "emu_contacts.cpp", EMU / "simt_emu.h"] + [CSRC / h for h in ("hsr_core.h", "hsr_model.h", "hsrb_kernels.cuh",
                                                                          "hsrb_contacts.cuh")]
ST_COUNT = 16   # hsrb_kernels.cuh: ST_PHASE0 + PH_COUNT
_vp = ctypes.c_void_p
MODELS = ("c2_push", "c1b_readme_block", "c3_arm", "f2_cupboard", "c5_clutter")
POW2 = np.array([[2, .5, 1, 2], [.5, 2, 2, .5], [1, 1, 1, 1], [2, 2, .5, 1]], np.float32)
NONPOW2 = np.array([[1.3, .7, .9, 1.1], [.6, 1.7, 1.4, .8], [1.9, 1.2, .55, 1.6]], np.float32)


def _lib():
    LIB.parent.mkdir(exist_ok=True)
    if not LIB.exists() or any(LIB.stat().st_mtime < d.stat().st_mtime for d in DEPS):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-D__CUDACC__", "-DHSRB_SIMT_EMU",
                               "-include", str(EMU / "simt_emu.h"), "-I", str(EMU), "-o", str(LIB), str(EMU / "emu_contacts.cpp"),
                               "-lpthread"])
    lib = ctypes.CDLL(str(LIB))
    lib.emu_contacts.argtypes = [ctypes.c_char_p, ctypes.c_size_t] + [ctypes.c_int] * 5 + [_vp] * 15
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(_vp)


def caps_of(port, ncon_max=0, nefc_max=0):
    """dims for oracle.port.unpack_debug at the capacities of a launch (0: the model's)"""
    return SimpleNamespace(nq=port.nq, nv=port.nv, nbody=port.nbody, ncon_max=ncon_max or port.ncon_max,
                           nefc_max=nefc_max or port.nefc_max)


def query(model, state, ctrl, G=8, params=None, C=None, caps=(0, 0), port=None, debug=True, rows=True):
    """One launch of the contact query (and, with debug, the MODE_DEBUG launch on a copy of the state)."""
    from oracle.port import unpack_debug

    n = state.shape[0]
    dims = caps_of(port, *caps)
    C = dims.ncon_max if C is None else C
    st = np.ascontiguousarray(state, np.float32).copy()
    ctrl = None if ctrl is None else np.ascontiguousarray(ctrl, np.float32)
    prm = None if params is None else np.ascontiguousarray(params, np.float32)
    o = dict(count=np.full(n, -7, np.int32), pair=np.full((n, C), -7, np.int32), dist=np.full((n, C), np.nan, np.float32),
             pos=np.full((n, C, 3), np.nan, np.float32), frame=np.full((n, C, 3, 3), np.nan, np.float32),
             force=np.full((n, C, 6), np.nan, np.float32), wrench=np.full((n, model.nbody, 6), np.nan, np.float32),
             bad=np.full(n, 0xff, np.uint8), stats=np.zeros(ST_COUNT, np.uint64), xipos=np.zeros((n, model.nbody, 3)))
    if not rows:
        for k in ("pair", "dist", "pos", "frame", "force"):
            o[k] = None
    size = 4 + dims.nbody * 3 + dims.nv * dims.nv + 3 * dims.nv + dims.ncon_max * 14 + dims.nefc_max * (dims.nv + 3) + dims.nq + dims.nv
    dump = np.zeros((n, size)) if debug else None   # hsr_core.h debug_size
    dbg_bad = np.zeros(n, np.uint8)
    blob = model.to_blob()
    rc = _lib().emu_contacts(blob, len(blob), G, n, caps[0], caps[1], C, _p(st), _p(ctrl), _p(prm), _p(o["count"]), _p(o["pair"]),
                             _p(o["dist"]), _p(o["pos"]), _p(o["frame"]), _p(o["force"]), _p(o["wrench"]), _p(o["bad"]),
                             _p(o["stats"]), _p(dump), _p(dbg_bad), _p(o["xipos"]))
    assert rc == 0, rc
    o["state"] = st
    if debug:
        o["debug"] = [unpack_debug(dims, dump[e]) for e in range(n)]
        o["dbg_bad"] = dbg_bad
    return o


def debug_rows(model, d):
    """The contact rows of a debug dump: (pair, dist, pos, frame [k, 3, 3], force [k, 6]) with the efc_force rows of each
    contact (joint-limit rows first, then condim rows per contact in contact order)."""
    k = d["ncon"]
    force = np.zeros((k, 6))
    r = d["nlimit"]
    for c in range(k):
        dim = int(model.pair_condim[d["con_pair"][c]])
        force[c, :dim] = d["efc_force"][r:r + dim]
        r += dim
    assert r == d["nefc"]
    return d["con_pair"], d["con_dist"], d["con_pos"], d["con_frame"], force


def check_against_debug(model, o, C=None):
    """Count and every contact row equal the debug dump bit for bit; padding rows are exactly -1 / 0."""
    n, Cq = o["pair"].shape
    for e in range(n):
        d = o["debug"][e]
        k = d["ncon"]
        assert o["count"][e] == k, e
        m = min(k, Cq)
        pair, dist, pos, frame, force = debug_rows(model, d)
        assert np.array_equal(o["pair"][e, :m], pair[:m]), e
        assert np.array_equal(o["dist"][e, :m].astype(np.float64), dist[:m]), e
        assert np.array_equal(o["pos"][e, :m].astype(np.float64), pos[:m]), e
        assert np.array_equal(o["frame"][e, :m].astype(np.float64), frame[:m]), e
        assert np.array_equal(o["force"][e, :m].astype(np.float64), force[:m]), e
        assert np.all(o["pair"][e, m:] == -1) and np.all(o["dist"][e, m:] == 0) and np.all(o["pos"][e, m:] == 0)
        assert np.all(o["frame"][e, m:] == 0) and np.all(o["force"][e, m:] == 0)
    # bit 0 (contact overflow) is the forward pass's; bit 2 of the query is set only where the debug launch has it too
    # (that launch adds the Cholesky of the implicit-damping Euler step); bit 1 belongs to the Euler step alone
    assert np.array_equal(o["bad"] & 1, o["dbg_bad"] & 1)
    assert np.all((o["bad"] & ~np.uint8(5)) == 0) and np.all((o["bad"] & 4) <= (o["dbg_bad"] & 4))


def numpy_wrench(model, o, e):
    """body_wrench of environment e recomputed in fp64 from the query's own rows and xipos."""
    out = np.zeros((model.nbody, 6))
    for c in range(int(o["count"][e])):
        pk = int(o["pair"][e, c])
        b1, b2 = int(model.geom_body[model.pair_geom1[pk]]), int(model.geom_body[model.pair_geom2[pk]])
        F = o["force"][e, c].astype(np.float64)
        fr = o["frame"][e, c].astype(np.float64)
        fc, tc = F[:3] @ fr, F[3:] @ fr
        for b, s in ((b2, 1.0), (b1, -1.0)):
            d = o["pos"][e, c].astype(np.float64) - o["xipos"][e, b]
            out[b, :3] += s * fc
            out[b, 3:] += s * (tc + np.cross(d, fc))
    return out


def edited(model, s):
    """The model whose arrays carry the multipliers s = (friction, block_mass, actuator_gain, damping)."""
    f, mb, g, d = (float(x) for x in s)
    mass, inertia = model.body_mass.copy(), model.body_inertia.copy()
    for b in model.block_body:
        mass[b] *= mb
        inertia[b] *= mb
    return model.replace(pair_friction=model.pair_friction * f, body_mass=mass, body_inertia=inertia,
                         act_kp=model.act_kp * g, dof_damping=model.dof_damping * d)


def make_state(qpos, qvel, warm, mocap=None):
    mocap = np.zeros((len(qpos), 3)) if mocap is None else mocap
    return np.concatenate([qpos, qvel, warm, mocap], axis=1).astype(np.float32)


@pytest.fixture(scope="module")
def cases(models, ports):
    """States [n, S] and controls per model: the ends of short fp64-port rollouts (resting, pushing, limit, gripper-pan
    contacts) and start states on the pan with a random control."""
    out = {}
    for name in MODELS:
        model, port = models[name], ports[name]
        qpos, qvel, warm, ctrl = rollout_states(port, model, 12, seed=31, pan=name == "c3_arm", float32=True)
        q0 = initial_states(model, 6, seed=32, pan=True, port=port).astype(np.float32).astype(np.float64)
        rng = np.random.default_rng(33)
        c0 = rng.uniform(model.act_ctrlrange[:, 0], model.act_ctrlrange[:, 1], (6, model.nu)).astype(np.float32)
        z = np.zeros((6, model.nv))
        out[name] = (np.concatenate([make_state(qpos, qvel, warm), make_state(q0, z, z)]),
                     np.concatenate([ctrl.astype(np.float32), c0]))
    return out


def prm_rows(kind, n):
    if kind is None:
        return None
    tab = POW2 if kind == "pow2" else NONPOW2
    return tab[np.arange(n) % len(tab)]


# ---------------------------------------------------------------------------------------------- 1. bit-equal to the dump
@pytest.mark.parametrize("kind", [None, "pow2", "nonpow2"], ids=["nominal", "pow2", "nonpow2"])
@pytest.mark.parametrize("G", [4, 8, 32])
@pytest.mark.parametrize("name", MODELS)
def test_bit_equal_to_debug_dump(name, G, kind, models, ports, cases):
    model = models[name]
    state, ctrl = cases[name]
    o = query(model, state, ctrl, G=G, params=prm_rows(kind, len(state)), port=ports[name])
    check_against_debug(model, o)
    assert o["count"].sum() > 0
    assert np.array_equal(o["state"], state)                   # purity: the resident state is not written
    assert np.all(o["stats"] == 0)                             # nor the work counters


def test_null_ctrl_is_zeros_and_ctrl_matters(models, ports, cases):
    """A NULL ctrl reads as zeros; the forces depend on the control (actuation in qacc_smooth)."""
    model = models["c3_arm"]
    state, ctrl = cases["c3_arm"]
    a = query(model, state, None, port=ports["c3_arm"], debug=False)
    b = query(model, state, np.zeros_like(ctrl), port=ports["c3_arm"], debug=False)
    c = query(model, state, ctrl, port=ports["c3_arm"], debug=False)
    for k in ("count", "pair", "force", "wrench", "bad"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    assert not np.array_equal(a["force"], c["force"])


# ---------------------------------------------------------------------------------------------- 2. against the fp64 port
# Forces within RTOL |f| + ATOL of the fp64 port.  The port's own fp32 build (use_float=True: the solver in fp32, geometry
# in fp64, as on the device) exceeds RTOL |f| by at most 7.1e-6 N on these states, the kernel by 7.4e-6 N (printed below,
# nominal; 7.7e-6 / 7.8e-6 N with multipliers): the bound leaves two orders of magnitude for other states.  An environment on a contact-activation edge (a pair whose distance is at the fp32 noise
# floor of zero, or a cone zone switch) may resolve differently in fp32: <= 1 % of environments, at least one.
RTOL, ATOL = 1e-3, 1e-3


def force_mismatch(model, got_pairs, got_force, dbg):
    pair, _, _, _, force = debug_rows(model, dbg)
    if len(got_pairs) != len(pair) or not np.array_equal(got_pairs, pair):
        return np.inf
    if len(pair) == 0:
        return 0.0
    return float(np.max(np.abs(got_force - force) - RTOL * np.abs(force)))


@pytest.mark.parametrize("kind", [None, "nonpow2"], ids=["nominal", "params"])
def test_matches_fp64_port(kind, models, ports, cases):
    from oracle import port as P

    worst_kernel, worst_f32, over, total = 0.0, 0.0, 0, 0
    for name in MODELS:
        model, port = models[name], ports[name]
        state, ctrl = cases[name]
        n = len(state)
        prm = prm_rows(kind, n)
        o = query(model, state, ctrl, params=prm, port=port, debug=False)
        nq, nv = model.nq, model.nv
        x = state.astype(np.float64)
        for e in range(n):
            pm = port if prm is None else P.CpuPort(edited(model, prm[e].astype(np.float64)))
            args = (x[e:e + 1, :nq], x[e:e + 1, nq:nq + nv], x[e:e + 1, nq + nv:nq + 2 * nv], ctrl[e:e + 1].astype(np.float64))
            ref = pm.step(*args, nsub=1, debug=True)["debug"][0]
            f32 = pm.step(*args, nsub=1, debug=True, use_float=True)["debug"][0]
            k = int(o["count"][e])
            dk = force_mismatch(model, o["pair"][e, :k], o["force"][e, :k].astype(np.float64), ref)
            pair32, _, _, _, force32 = debug_rows(model, f32)
            d32 = force_mismatch(model, pair32, force32, ref)
            total += 1
            if dk > ATOL:
                over += 1
            else:
                worst_kernel = max(worst_kernel, dk)
            if np.isfinite(d32):
                worst_f32 = max(worst_f32, d32)
    print(f"max |f - f64| - rtol |f64|: kernel {worst_kernel:.2e} N, port fp32 {worst_f32:.2e} N; {over}/{total} over")
    assert over <= max(1, total // 100), (over, total)
    assert worst_f32 <= ATOL   # the bound holds for the port's own fp32 build


# ---------------------------------------------------------------------------------------------- 3. known answers
@pytest.fixture(scope="module")
def resting(models, ports):
    """The block of c2_push settled on the floor (tests/test_oracle_kat.py kat3), with its nominal mass and with twice it:
    600 substeps of the fp64 port from x = 0.3, y = 0.4, flat."""
    from oracle import port as P

    model = models["c2_push"]
    out = {}
    for mb in (1.0, 2.0):
        pm = ports["c2_push"] if mb == 1.0 else P.CpuPort(edited(model, (1, mb, 1, 1)))
        q = model.qpos0.copy()
        a = int(model.jnt_qposadr[model.body_jntadr[model.block_body[0]]])
        q[a:a + 7] = [0.3, 0.4, 0.017, 1, 0, 0, 0]
        z = np.zeros(model.nv)
        r = pm.step(q, z, z, np.zeros(model.nu), nsub=600)
        out[mb] = make_state(r["qpos"], r["qvel"], r["warm"])
    return out


@pytest.mark.parametrize("mb", [1.0, 2.0])
def test_block_at_rest_carries_its_weight(mb, models, ports, resting):
    model = models["c2_push"]
    state = resting[mb]
    prm = None if mb == 1.0 else np.array([[1, mb, 1, 1]], np.float32)
    o = query(model, state, np.zeros((1, model.nu)), params=prm, port=ports["c2_push"])
    check_against_debug(model, o)
    b = int(model.block_body[0])
    mg = mb * float(model.body_mass[b]) * abs(float(model.opt[3]))
    w = o["wrench"][0].astype(np.float64)
    assert o["count"][0] == 4 and o["bad"][0] == 0
    assert np.allclose(w[b, :3], [0, 0, mg], rtol=1e-4, atol=1e-4 * mg), (w[b], mg)
    assert np.abs(w[b, 3:]).max() < 1e-4 * mg
    assert np.allclose(w[0, :3], [0, 0, -mg], rtol=1e-4, atol=1e-4 * mg)   # the floor's reaction
    assert np.abs(w[:, :3].sum(axis=0)).max() < 1e-5 * mg                    # row 0 holds the reactions: the forces sum to 0


@pytest.mark.parametrize("kind", [None, "nonpow2"], ids=["nominal", "params"])
def test_wrench_rows_sum_to_zero_and_forces_in_cone(kind, models, ports, cases):
    for name in MODELS:
        model = models[name]
        state, ctrl = cases[name]
        prm = prm_rows(kind, len(state))
        o = query(model, state, ctrl, params=prm, port=ports[name], debug=False)
        for e in range(len(state)):
            w = o["wrench"][e].astype(np.float64)
            scale = max(1.0, np.abs(w).max())
            # the torques sum to zero about a common point only: move every row's torque to the world origin
            t0 = w[:, 3:] + np.cross(o["xipos"][e], w[:, :3])
            assert np.abs(w[:, :3].sum(axis=0)).max() < 1e-5 * scale, (name, e)
            assert np.abs(t0.sum(axis=0)).max() < 1e-5 * scale, (name, e)
            fscale = 1.0 if prm is None else float(prm[e, 0])
            for c in range(int(o["count"][e])):
                pk = int(o["pair"][e, c])
                dim = int(model.pair_condim[pk])
                f = o["force"][e, c].astype(np.float64)
                assert f[0] >= 0, (name, e, c, f)
                if dim >= 3:
                    mu = model.pair_friction[pk].astype(np.float32) * np.float32(fscale)
                    assert np.linalg.norm(f[1:dim] / mu[:dim - 1]) <= f[0] * (1 + 1e-4) + 1e-6, (name, e, c, f)


# ---------------------------------------------------------------------------------------------- 4. wrench recomputation
@pytest.mark.parametrize("name", MODELS)
def test_wrench_matches_numpy_recomputation(name, models, ports, cases):
    model = models[name]
    state, ctrl = cases[name]
    o = query(model, state, ctrl, port=ports[name], debug=False)
    for e in range(len(state)):
        ref = numpy_wrench(model, o, e)
        scale = max(1.0, np.abs(ref).max())
        assert np.allclose(o["wrench"][e], ref, rtol=1e-6, atol=1e-6 * scale), (e, o["wrench"][e], ref)
    # the wrench alone (contact rows NULL) gives the same bits
    w = query(model, state, ctrl, port=ports[name], debug=False, rows=False, C=0)
    assert np.array_equal(w["wrench"], o["wrench"]) and np.array_equal(w["count"], o["count"])


# ---------------------------------------------------------------------------------------------- 6. capacity
def test_overflow_keeps_the_dumps_contacts(models, ports, cases):
    """At ncon_max = 4 the forward pass keeps the contacts the debug launch keeps, and flags the overflow."""
    flagged = 0
    for name in ("c2_push", "c3_arm", "c5_clutter"):
        model = models[name]
        state, ctrl = cases[name]
        o = query(model, state, ctrl, caps=(4, 0), port=ports[name])
        check_against_debug(model, o)
        assert np.all(o["count"] <= 4)
        flagged += int(np.sum(o["bad"] & 1))
    assert flagged >= 3


def test_fewer_rows_than_contacts(models, ports, cases):
    """max_contacts < count: the first max_contacts rows, count and the wrenches unchanged (all held contacts)."""
    model = models["c3_arm"]
    state, ctrl = cases["c3_arm"]
    full = query(model, state, ctrl, port=ports["c3_arm"], debug=False)
    cut = query(model, state, ctrl, C=2, port=ports["c3_arm"], debug=False)
    assert np.any(full["count"] > 2)
    assert np.array_equal(cut["count"], full["count"]) and np.array_equal(cut["wrench"], full["wrench"])
    for k in ("pair", "dist", "pos", "frame", "force"):
        assert np.array_equal(cut[k], full[k][:, :2]), k


# ---------------------------------------------------------------------------------------------- 7. ptxas budget
# registers / stack of the instances (ptxas -v, sm_100a, the flags of hsrb_step_g8.cu), measured 236-254 registers and
# 1536-1584 bytes of stack frame, no spills; the MODE_DEBUG general instance they share their stages with has 240 / 1568
STACK_CEIL = 1600


def test_contacts_kernel_resources():
    from hsr_env_b200 import build as B

    B.build()
    log = (B.CSRC / "hsrb_contacts.ptxas.log").read_text()
    names = [f"_Z20hsrb_contacts_kernelILi{G}ELb{int(P)}EEv7ConArgs" for G in (4, 8, 16, 32) for P in (False, True)]
    for name in names:
        block = log.split(f"Function properties for {name}", 1)[1]
        stack = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", block)
        regs = re.search(r"Used (\d+) registers", block)
        assert int(regs.group(1)) <= 255, (name, regs.group(1))
        assert int(stack.group(1)) <= STACK_CEIL and int(stack.group(2)) == 0 and int(stack.group(3)) == 0, (name, stack.groups())
