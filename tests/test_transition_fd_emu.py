"""Transition derivatives without a GPU: hsrb_fd_kernel and hsrb_fd_form_kernel on the SIMT emulator.  Every run's x' and
flags equal the general action kernel (MODE_DEBUG, or a goal-free STEP launch for several substeps) on that run's perturbed
input, bit for bit; the perturbed inputs equal a numpy restatement of the perturbation rule; A and B equal a numpy
recomputation from the runs; the derivatives agree with centered differences of the fp64 port as well as the port's own fp32
build does; known answers (an affine model, a block in free flight, slide kinematics); MuJoCo's ctrl-limit rule; purity;
and the ptxas budget of the instances.

Mutations that make this file fail (each checked by hand): the rotation perturbed in the world frame (dq (x) q); the columns
divided by eps instead of the realised h; the ctrl-limit rule ignored (every side used); the perturbed runs started from the
warm start the group's previous run left (qpos / qvel reloaded, qacc_warmstart not); A's row and column indices swapped."""
import ctypes
import math
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

from scenarios import initial_states, rollout_states
from test_contacts_emu import POW2, NONPOW2, edited, make_state, prm_rows

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
EMU = HERE / "simt_emu"
LIB = ROOT / "oracle" / "_build" / "libfd_emu.so"
CSRC = ROOT / "hsr_env_b200" / "csrc"
DEPS = [EMU / "emu_fd.cpp", EMU / "simt_emu.h"] + [CSRC / h for h in ("hsr_core.h", "hsr_model.h", "hsrb_kernels.cuh", "hsrb_fd.cuh")]
ST_COUNT = 16
JNT_FREE = 0
_vp = ctypes.c_void_p
MODELS = ("c2_push", "c1b_readme_block", "c3_arm", "f2_cupboard")


def _lib():
    LIB.parent.mkdir(exist_ok=True)
    if not LIB.exists() or any(LIB.stat().st_mtime < d.stat().st_mtime for d in DEPS):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-D__CUDACC__", "-DHSRB_SIMT_EMU",
                               "-include", str(EMU / "simt_emu.h"), "-I", str(EMU), "-o", str(LIB), str(EMU / "emu_fd.cpp"),
                               "-lpthread"])
    lib = ctypes.CDLL(str(LIB))
    lib.emu_fd.argtypes = [ctypes.c_char_p, ctypes.c_size_t] + [ctypes.c_int] * 4 + [ctypes.c_float, ctypes.c_double, ctypes.c_double,
                                                                                     ctypes.c_int] + [_vp] * 13
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(_vp)


def nruns(model, centered):
    return 1 + (2 if centered else 1) * (2 * model.nv + model.nu)


def rot_cs(eps):
    """cos / sin of eps / 2 in double, as hsrb_transition_fd computes them (eps as the fp32 the call receives)"""
    e = float(np.float32(eps))
    return math.cos(0.5 * e), math.sin(0.5 * e)


def fd(model, state, ctrl, G=8, nsub=1, centered=True, eps=1e-3, params=None, grid_cap=0, ref=True):
    """One call of the transition derivatives on the emulator (and the reference launch on every run's input)."""
    n = state.shape[0]
    nr, nx, nobs, nu = nruns(model, centered), 2 * model.nv, model.nq + model.nv, model.nu
    R = nobs + 3
    st = np.ascontiguousarray(state, np.float32).copy()
    ctrl = None if ctrl is None else np.ascontiguousarray(ctrl, np.float32)
    prm = None if params is None else np.ascontiguousarray(params, np.float32)
    o = dict(A=np.full((n, nx, nx), np.nan, np.float32), B=np.full((n, nx, nu), np.nan, np.float32),
             next_obs=np.full((n, nobs), np.nan, np.float32), bad=np.full(n, 0xff, np.uint8), stats=np.zeros(ST_COUNT, np.uint64),
             scratch=np.zeros(n * nr * R, np.float32), inputs=np.zeros((n, nr, nobs + nu), np.float32), h=np.zeros((n, nr)))
    if ref:
        o["ref"] = np.zeros((n * nr, nobs), np.float32)
        o["ref_bad"] = np.zeros(n * nr, np.uint8)
    c, s = rot_cs(eps)
    blob = model.to_blob()
    rc = _lib().emu_fd(blob, len(blob), G, n, nsub, int(centered), eps, c, s, grid_cap, _p(st), _p(ctrl), _p(prm), _p(o["A"]),
                       _p(o["B"]), _p(o["next_obs"]), _p(o["bad"]), _p(o["stats"]), _p(o["scratch"]), _p(o["inputs"]), _p(o["h"]),
                       _p(o.get("ref")), _p(o.get("ref_bad")))
    assert rc == 0, rc
    rows = o["scratch"].reshape(n, nr, R)
    o["rows"] = rows[:, :, :nobs]
    o["flags"] = rows[:, :, nobs].copy().view(np.int32)
    o["row_h"] = rows[:, :, nobs + 1:nobs + 3].copy().view(np.float64)[..., 0]
    o["state"] = st
    return o


# ---------------------------------------------------------------------------------------------- numpy restatement
def rot_dofs(model):
    """dof -> (qpos address of the joint's quaternion, k) for the rotation dofs of free joints"""
    out = {}
    for j in range(model.njnt):
        if model.jnt_type[j] == JNT_FREE:
            for k in range(3):
                out[int(model.jnt_dofadr[j]) + 3 + k] = (int(model.jnt_qposadr[j]) + 3, k)
    return out


def qpos_of_dof(model, d):
    j = int(model.dof_jnt[d])
    return int(model.jnt_qposadr[j]) + d - int(model.jnt_dofadr[j])


def nudge(x, eps, side):
    x, eps = np.float32(x), np.float32(eps)
    y = np.float32(x + eps) if side > 0 else np.float32(x - eps)
    return y if y != x else np.nextafter(x, np.float32(np.inf if side > 0 else -np.inf))


def ctrl_ok(model, i, u, eps, side):
    if not model.act_ctrllimited[i]:
        return True
    lo, hi = np.float32(model.act_ctrlrange[i, 0]), np.float32(model.act_ctrlrange[i, 1])
    un = nudge(u, eps, side)
    return lo <= np.float32(u) <= hi and lo <= un <= hi


def quatmul(a, b):
    return np.array([a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                     a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]])


def subquat(qa, qb):
    """MuJoCo's mju_subQuat: axis-angle of conj(qb) (x) qa"""
    d = quatmul(np.array([qb[0], -qb[1], -qb[2], -qb[3]], float), np.asarray(qa, float))
    ax = d[1:].copy()
    s = math.sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2])
    ax = np.array([1.0, 0, 0]) if s < 1e-15 else ax * (1 / s)
    speed = 2 * math.atan2(s, d[0])
    if speed > math.pi:
        speed -= 2 * math.pi
    return ax * speed


def perturbed(model, x, u, r, centered, eps):
    """(qpos | qvel | ctrl) fp32 and h of run r from the nominal x = qpos | qvel and ctrl u: the rule of include/hsrb.h"""
    nq, nv = model.nq, model.nv
    v = np.concatenate([x, u]).astype(np.float32)
    if r == 0:
        return v, 0.0
    S = 2 if centered else 1
    c = (r - 1) // S
    side = (1 if (r - 1) % S == 0 else -1) if centered else (-1 if c >= 2 * nv and not ctrl_ok(model, c - 2 * nv, u[c - 2 * nv], eps, 1) else 1)
    rot = rot_dofs(model)
    if c < nv and c in rot:
        a, k = rot[c]
        q0 = [float(t) for t in v[a:a + 4]]
        cs, sn = rot_cs(eps)
        e = [0.0, 0.0, 0.0]
        e[k] = sn if side > 0 else -sn
        p = [q0[0] * cs - q0[1] * e[0] - q0[2] * e[1] - q0[3] * e[2], q0[0] * e[0] + q0[1] * cs + q0[2] * e[2] - q0[3] * e[1],
             q0[0] * e[1] - q0[1] * e[2] + q0[2] * cs + q0[3] * e[0], q0[0] * e[2] + q0[1] * e[1] - q0[2] * e[0] + q0[3] * cs]
        nrm = math.sqrt(p[0] * p[0] + p[1] * p[1] + p[2] * p[2] + p[3] * p[3])
        v[a:a + 4] = [np.float32(t / nrm) for t in p]
        return v, float(subquat(v[a:a + 4].astype(float), q0)[k])
    i = qpos_of_dof(model, c) if c < nv else (nq + c - nv if c < 2 * nv else nq + nv + c - 2 * nv)
    x0 = v[i]
    v[i] = nudge(x0, eps, side)
    return v, float(v[i]) - float(x0)


def numpy_AB(model, rows, h, u, centered, eps):
    """A [2nv, 2nv], B [2nv, nu] of one environment from its runs' x' [nruns, nq + nv] and h [nruns] (include/hsrb.h)"""
    nq, nv, nu = model.nq, model.nv, model.nu
    nxs = 2 * nv
    x0 = rows[0].astype(np.float64)
    rot = rot_dofs(model)
    out = np.zeros((nxs, nxs + nu), np.float32)
    S = 2 if centered else 1

    def diff(x):
        x = x.astype(np.float64)
        d = np.zeros(nxs)
        done = set()
        for i in range(nv):
            if i in rot:
                a, k = rot[i]
                if a not in done:
                    done.add(a)
                    d[i - k:i - k + 3] = subquat(x[a:a + 4], x0[a:a + 4])
            else:
                d[i] = x[qpos_of_dof(model, i)] - x0[qpos_of_dof(model, i)]
        d[nv:] = x[nq:] - x0[nq:]
        return d

    for c in range(nxs + nu):
        rp = 1 + c * S
        rm = rp + 1 if centered else rp
        usep, usem = True, centered
        if c >= nxs:
            okp, okm = ctrl_ok(model, c - nxs, u[c - nxs], eps, 1), ctrl_ok(model, c - nxs, u[c - nxs], eps, -1)
            usep, usem = okp, (okm if centered else (not okp and okm))
        dp, dm = diff(rows[rp]), diff(rows[rm])
        if usep and usem:
            col = (dp - dm) / (h[rp] - h[rm])
        elif usep:
            col = dp / h[rp]
        elif usem:
            col = dm / h[rm]
        else:
            col = np.zeros(nxs)
        out[:, c] = col.astype(np.float32)
    return out[:, :nxs], out[:, nxs:]


def tolerant_mask(model):
    """entries of A | B that go through transcendental functions: rows and columns of free-joint rotations"""
    nv, nu = model.nv, model.nu
    rot = np.zeros(2 * nv + nu, bool)
    rot[list(rot_dofs(model))] = True
    m = np.zeros((2 * nv, 2 * nv + nu), bool)
    m[rot[:2 * nv], :] = True
    m[:, rot] = True
    return m[:, :2 * nv], m[:, 2 * nv:]


def within_ulps(a, b, k=2):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return np.abs(a.astype(np.float64) - b) <= k * np.spacing(np.maximum(np.abs(a), np.abs(b))).astype(np.float64)


def check_AB(model, o, ctrl, centered, eps):
    n = o["A"].shape[0]
    mA, mB = tolerant_mask(model)
    u = np.zeros((n, model.nu), np.float32) if ctrl is None else ctrl
    for e in range(n):
        A, B = numpy_AB(model, o["rows"][e], o["h"][e], u[e], centered, eps)
        for got, want, m in ((o["A"][e], A, mA), (o["B"][e], B, mB)):
            assert np.array_equal(got[~m], want[~m]), e
            assert np.all(within_ulps(got[m], want[m])), (e, np.abs(got - want)[m].max())


# ---------------------------------------------------------------------------------------------- fixtures
@pytest.fixture(scope="module")
def cases(models, ports):
    """States [n, S] and controls per model: ends of short fp64-port rollouts (resting, pushing, limit and pan contacts) and a
    start state on the pan with a random control."""
    out = {}
    for name in MODELS:
        model, port = models[name], ports[name]
        k = 3 if name == "c3_arm" else 4
        qpos, qvel, warm, ctrl = rollout_states(port, model, k, seed=41, pan=name == "c3_arm", float32=True)
        q0 = initial_states(model, 1, seed=42, pan=True, port=port).astype(np.float32).astype(np.float64)
        c0 = np.random.default_rng(43).uniform(model.act_ctrlrange[:, 0], model.act_ctrlrange[:, 1], (1, model.nu)).astype(np.float32)
        z = np.zeros((1, model.nv))
        out[name] = (np.concatenate([make_state(qpos, qvel, warm), make_state(q0, z, z)]), np.concatenate([ctrl.astype(np.float32), c0]))
    return out


# ---------------------------------------------------------------------------------------------- 1. runs bit for bit
# (G, nsub, parameter kind, centered, grid cap): every G, 1 and 3 substeps, both multiplier kinds and the grid-stride loop
COMBOS = [(4, 1, None, True, 0), (8, 3, "pow2", True, 3), (32, 1, "nonpow2", True, 0), (8, 1, None, False, 2),
          (32, 3, None, True, 0), (4, 1, "pow2", False, 0)]


@pytest.mark.parametrize("G,nsub,kind,centered,cap", COMBOS, ids=[f"G{c[0]}-n{c[1]}-{c[2] or 'nominal'}-{'c' if c[3] else 'f'}"
                                                                  f"{'-cap' if c[4] else ''}" for c in COMBOS])
@pytest.mark.parametrize("name", MODELS)
def test_runs_bit_equal_to_general_kernel(name, G, nsub, kind, centered, cap, models, cases):
    model = models[name]
    state, ctrl = cases[name]
    if name == "c3_arm" and (G, nsub) not in ((8, 3), (32, 1), (4, 1)):
        pytest.skip("c3_arm: three of the combinations (emulator time)")
    n = len(state)
    prm = prm_rows(kind, n)
    o = fd(model, state, ctrl, G=G, nsub=nsub, centered=centered, params=prm, grid_cap=cap)
    nr, nobs = nruns(model, centered), model.nq + model.nv
    # every run's x' and flags are the general kernel's on the same perturbed input
    assert np.array_equal(o["rows"].reshape(-1, nobs), o["ref"])
    assert np.array_equal(o["flags"].reshape(-1), o["ref_bad"].astype(np.int32))
    # the harness's inputs are the rule of include/hsrb.h (numpy restatement): the fp32 values bit for bit, h to rounding
    x = state[:, :nobs]
    for e in range(n):
        for r in range(nr):
            v, h = perturbed(model, x[e], ctrl[e], r, centered, 1e-3)
            assert np.array_equal(o["inputs"][e, r], v), (e, r)
            assert abs(o["h"][e, r] - h) <= 1e-12 * max(abs(h), 1e-3), (e, r, o["h"][e, r], h)
    assert np.array_equal(o["row_h"], o["h"])
    # next_obs is the unperturbed run; bad_state the OR over the runs
    assert np.array_equal(o["next_obs"], o["rows"][:, 0])
    assert np.array_equal(o["bad"], np.bitwise_or.reduce(o["flags"], axis=1).astype(np.uint8))
    check_AB(model, o, ctrl, centered, 1e-3)
    # purity: the resident state and the work counters are untouched
    assert np.array_equal(o["state"], state) and np.all(o["stats"] == 0)


def test_perturbations_touch_one_coordinate(models, cases):
    """Each perturbed input differs from the nominal one in its own coordinate only (a free joint's rotation: its four
    quaternion components), and differentiatePos(perturbed, nominal) = h e_k to the fp32 rounding of the quaternion."""
    model = models["c2_push"]
    state, ctrl = cases["c2_push"]
    o = fd(model, state[:2], ctrl[:2], ref=False)
    nq, nv, nu = model.nq, model.nv, model.nu
    rot = rot_dofs(model)
    for e in range(2):
        v0 = o["inputs"][e, 0]
        for r in range(1, nruns(model, True)):
            c = (r - 1) // 2
            v, h = o["inputs"][e, r], o["h"][e, r]
            changed = set(np.nonzero(v != v0)[0])
            if c < nv and c in rot:
                a, k = rot[c]
                assert changed <= set(range(a, a + 4)) and changed
                dp = subquat(v[a:a + 4].astype(float), v0[a:a + 4].astype(float))
                assert abs(dp[k] - h) <= 1e-15, (r, dp, h)
                # off-axis: the rotation the fp32 rounding of the quaternion adds (2^-24 per component)
                assert np.abs(np.delete(dp, k)).max() < 2 * 2.0 ** -23, (r, dp)
                assert 0.9e-3 < abs(h) < 1.1e-3
            else:
                i = qpos_of_dof(model, c) if c < nv else (nq + c - nv if c < 2 * nv else nq + nv + c - 2 * nv)
                assert changed == {i}, (r, changed, i)
                assert h == float(v[i]) - float(v0[i]) and h != 0


# ---------------------------------------------------------------------------------------------- 2. against the fp64 port
def port_fd(port, model, x, warm, u, eps, use_float=False, perturb_fp32=False):
    """Centered differences of one substep of the port: fp64 perturbations (perturb_fp32: the kernel's rule at eps)."""
    nq, nv, nu = model.nq, model.nv, model.nu
    nxs = 2 * nv
    rot = rot_dofs(model)
    ins, hs = [], []
    for c in range(nxs + nu):
        for side in (1, -1):
            if perturb_fp32:
                v, h = perturbed(model, x.astype(np.float32), u.astype(np.float32), 1 + 2 * c + (side < 0), True, eps)
                v = v.astype(np.float64)
            else:
                v = np.concatenate([x, u]).astype(np.float64)
                if c < nv and c in rot:
                    a, k = rot[c]
                    dq = np.zeros(4)
                    dq[0], dq[1 + k] = math.cos(0.5 * side * eps), math.sin(0.5 * side * eps)
                    q = quatmul(v[a:a + 4], dq)
                    v[a:a + 4] = q / np.linalg.norm(q)
                    h = side * eps
                else:
                    i = qpos_of_dof(model, c) if c < nv else (nq + c - nv if c < 2 * nv else nq + nv + c - 2 * nv)
                    v[i] += side * eps
                    h = side * eps
            ins.append(v)
            hs.append(h)
    ins = np.array([np.concatenate([x, u]).astype(np.float32 if perturb_fp32 else np.float64).astype(np.float64)] + ins)
    k = len(ins)
    r = port.step(ins[:, :nq], ins[:, nq:nq + nv], np.tile(warm, (k, 1)), ins[:, nq + nv:], nsub=1, use_float=use_float)
    xs = np.concatenate([r["qpos"], r["qvel"]], axis=1)
    return numpy_AB_f64(model, xs, np.array([0.0] + hs))


def numpy_AB_f64(model, rows, h):
    """centered columns in double (no rounding to fp32), every side used"""
    nq, nv, nu = model.nq, model.nv, model.nu
    nxs = 2 * nv
    rot = rot_dofs(model)
    x0 = rows[0]

    def diff(x):
        d = np.zeros(nxs)
        for i in range(nv):
            if i in rot:
                a, k = rot[i]
                d[i] = subquat(x[a:a + 4], x0[a:a + 4])[k]
            else:
                d[i] = x[qpos_of_dof(model, i)] - x0[qpos_of_dof(model, i)]
        d[nv:] = x[nq:] - x0[nq:]
        return d

    out = np.zeros((nxs, nxs + nu))
    for c in range(nxs + nu):
        out[:, c] = (diff(rows[1 + 2 * c]) - diff(rows[2 + 2 * c])) / (h[1 + 2 * c] - h[2 + 2 * c])
    return out[:, :nxs], out[:, nxs:]


def tight(model):
    """the model with the solver run to convergence: the fp64 reference's own noise below the comparison"""
    opt = model.opt.copy()
    opt[5], opt[6], opt[7], opt[8] = 1e-15, 1e-15, 1000, 200
    return model.replace(opt=opt)


def err(X, ref):
    return float(np.abs(X - ref).max() / max(1.0, np.abs(ref).max()))


@pytest.fixture(scope="module")
def smooth_cases(models, cases):
    """States of the fixtures whose inputs keep the ctrl inside its range by more than 1e-2 (a limit column is one-sided by
    design and is compared elsewhere)"""
    out = {}
    for name in ("c2_push", "c1b_readme_block", "f2_cupboard"):
        model = models[name]
        state, ctrl = cases[name]
        lo, hi = model.act_ctrlrange[:, 0], model.act_ctrlrange[:, 1]
        keep = np.all((ctrl > lo + 1e-2) & (ctrl < hi - 1e-2), axis=1)
        out[name] = (state[keep], ctrl[keep])
    return out


# The fp64 reference: centered differences of the port at eps 1e-6 on the model with the solver run to convergence.  A
# state where it is not smooth at that scale itself (a contact on its activation edge: eps 1e-6 against 1e-7 differ by more
# than REF_NOISE) says nothing about the kernel and is left out; the tests check that enough states remain.
REF_NOISE = 1e-3


@pytest.fixture(scope="module")
def fp64_refs(models, smooth_cases):
    """per model: (states, ctrls, [A | B] of the fp64 reference, the reference's noise) of the states where it is smooth"""
    from oracle import port as P

    out = {}
    for name, (state, ctrl) in smooth_cases.items():
        model = models[name]
        p64 = P.CpuPort(tight(model))
        nobs = model.nq + model.nv
        keep, refs, noise = [], [], []
        for e in range(len(state)):
            x, warm, u = state[e, :nobs].astype(np.float64), state[e, nobs:nobs + model.nv].astype(np.float64), ctrl[e].astype(np.float64)
            ref = np.concatenate(port_fd(p64, model, x, warm, u, 1e-6), 1)
            nz = err(np.concatenate(port_fd(p64, model, x, warm, u, 1e-7), 1), ref)
            if nz < REF_NOISE:
                keep.append(e); refs.append(ref); noise.append(nz)
        out[name] = (state[keep], ctrl[keep], refs, noise)
    assert sum(len(v[2]) for v in out.values()) >= 8
    return out


# The kernel runs hsr_core.h's stages in fp32 like the port's fp32 build (use_float=True; geometry in fp64 in both), with
# the same perturbations: measured on these fixtures (printed below), their errors against the fp64 reference agree to three
# digits on 11 of 12 states and the kernel's is the smaller on the twelfth (0.144 against 0.145).  The margin: 10 % of the
# port's own error plus 1e-5.
PORT_MARGIN_ABS, PORT_MARGIN_REL = 1e-5, 0.1


def test_matches_fp64_port(models, fp64_refs):
    from oracle import port as P

    rows = []
    for name, (state, ctrl, refs, noise) in fp64_refs.items():
        model = models[name]
        p32 = P.CpuPort(model)
        nobs = model.nq + model.nv
        o = fd(model, state, ctrl, eps=1e-3, ref=False)
        for e in range(len(state)):
            x, warm, u = state[e, :nobs].astype(np.float64), state[e, nobs:nobs + model.nv].astype(np.float64), ctrl[e].astype(np.float64)
            e32 = err(np.concatenate(port_fd(p32, model, x, warm, u, 1e-3, use_float=True, perturb_fp32=True), 1), refs[e])
            ek = err(np.concatenate([o["A"][e], o["B"][e]], 1).astype(np.float64), refs[e])
            rows.append((name, e, noise[e], ek, e32))
    print("\nname env  ref-noise(1e-6 vs 1e-7)  kernel  port-fp32   (max |X - X64| / max(1, |X64|), eps 1e-3)")
    for r in rows:
        print(f"{r[0]:>16} {r[1]:2d}  {r[2]:.2e}  {r[3]:.2e}  {r[4]:.2e}")
    for name, e, noise, ek, e32 in rows:
        assert ek <= e32 * (1 + PORT_MARGIN_REL) + PORT_MARGIN_ABS, (name, e, ek, e32)


EPS_SWEEP = (1e-2, 3e-3, 1e-3, 3e-4, 1e-4)


def test_eps_sweep(models, fp64_refs):
    """The default eps of BatchedHSREnv.transition_fd is the best power of ten of the sweep (median error over the
    fixtures); DESIGN 4.3e has the table."""
    import inspect

    from hsr_env_b200.env import BatchedHSREnv

    tab = {}
    for name, (state, ctrl, refs, _) in fp64_refs.items():
        model = models[name]
        for eps in EPS_SWEEP:
            o = fd(model, state, ctrl, eps=eps, ref=False)
            tab.setdefault(eps, []).extend(err(np.concatenate([o["A"][e], o["B"][e]], 1).astype(np.float64), refs[e])
                                           for e in range(len(state)))
    print("\neps      median    max      (max |X - X64| / max(1, |X64|) over the fixtures)")
    for eps in EPS_SWEEP:
        print(f"{eps:.0e}  {np.median(tab[eps]):.2e}  {np.max(tab[eps]):.2e}")
    best = min((1e-2, 1e-3, 1e-4), key=lambda e: np.median(tab[e]))
    assert inspect.signature(BatchedHSREnv.transition_fd).parameters["eps"].default == best


# ---------------------------------------------------------------------------------------------- 3. known answers
def test_affine_known_answer(models, ports):
    """c1_readme (two slides, position servos kp 300 with gear 3, damping 2200), contact-free, no limit active, ctrl inside
    its range: one substep is affine, v' = v + dt H^-1 (gear kp (u - gear q) - D v), q' = q + dt v', H = M + dt D."""
    model = models["c1_readme"]
    q = np.array([[0.03, -0.02], [0.05, 0.08]])
    v = np.array([[0.1, -0.2], [0.0, 0.05]])
    u = np.array([[0.12, -0.05], [0.2, 0.3]], np.float32)
    state = make_state(q, v, np.zeros_like(v))
    o = fd(model, state, u, ref=False)
    dbg = ports["c1_readme"].step(state[:, :2].astype(float), state[:, 2:4].astype(float), np.zeros((2, 2)), u.astype(float),
                                  nsub=1, debug=True, use_float=True)["debug"]
    dt, kp, g, D = model.timestep, model.act_kp, model.act_gear, np.diag(model.dof_damping)
    for e in range(2):
        assert dbg[e]["ncon"] == 0 and dbg[e]["nefc"] == 0
        Hi = np.linalg.inv(dbg[e]["M"] + dt * D)
        dvdq, dvdv, dvdu = -dt * Hi @ np.diag(g * kp * g), np.eye(2) - dt * Hi @ D, dt * Hi @ np.diag(g * kp)
        A = np.block([[np.eye(2) + dt * dvdq, dt * dvdv], [dvdq, dvdv]])
        B = np.vstack([dt * dvdu, dvdu])
        assert np.allclose(o["A"][e], A, rtol=1e-3, atol=2e-4), (o["A"][e], A)
        assert np.allclose(o["B"][e], B, rtol=1e-3, atol=2e-4), (o["B"][e], B)


def test_block_in_free_flight(models):
    """c2_push with the block 1 m above the floor: the block's rows of A are [[I, dt I], [0, I]] over its own coordinates
    and zero elsewhere, and its rows of B are zero."""
    model = models["c2_push"]
    q = model.qpos0.copy()
    a = int(model.jnt_qposadr[model.body_jntadr[model.block_body[0]]])
    q[a:a + 7] = [0.3, 0.1, 1.0, np.cos(0.3), 0, 0, np.sin(0.3)]
    v = np.zeros(model.nv)
    v[2:8] = [0.1, -0.05, 0.2, 0.0, 0.0, 0.0]
    state = make_state(q[None], v[None], np.zeros((1, model.nv)))
    o = fd(model, state, np.array([[0.3, -0.2]], np.float32), ref=False)
    nv = model.nv
    d0 = int(model.jnt_dofadr[model.body_jntadr[model.block_body[0]]])
    blk = np.r_[d0:d0 + 6, nv + d0:nv + d0 + 6]
    dt = model.timestep
    want = np.block([[np.eye(6), dt * np.eye(6)], [np.zeros((6, 6)), np.eye(6)]])
    A = o["A"][0]
    assert np.allclose(A[np.ix_(blk, blk)], want, atol=2e-4), A[np.ix_(blk, blk)]
    other = np.setdiff1d(np.arange(2 * nv), blk)
    assert np.abs(A[np.ix_(blk, other)]).max() < 1e-6
    assert np.abs(o["B"][0][blk]).max() < 1e-6


def test_slide_rows_are_kinematic(models, cases):
    """One substep of a slide joint is q' = q + dt v': its qpos row of [A | B] is e_q + dt x its qvel row, to the fp32
    resolution of q' over the perturbation."""
    for name in ("c2_push", "f2_cupboard"):
        model = models[name]
        state, ctrl = cases[name]
        o = fd(model, state, ctrl, ref=False)
        nv, dt = model.nv, model.timestep
        for d in range(nv):
            j = int(model.dof_jnt[d])
            if model.jnt_type[j] != 1:
                continue
            for e in range(len(state)):
                row = np.concatenate([o["A"][e, d], o["B"][e, d]])
                vrow = np.concatenate([o["A"][e, nv + d], o["B"][e, nv + d]])
                want = dt * vrow
                want[d] += 1
                assert np.allclose(row, want, atol=3e-4), (name, e, d, np.abs(row - want).max())


# ---------------------------------------------------------------------------------------------- 4. ctrl-limit rule
def test_ctrl_limit_rule(models, cases):
    """u = hi: the centered call gives the backward column; u outside the range: a zero column; forward mode with
    u + eps > hi falls back to the backward column."""
    # the actuators' force limits widened: at u = hi the servo force of c2_push saturates, which zeroes the column itself
    model = models["c2_push"].replace(act_forcerange=models["c2_push"].act_forcerange * 100)
    state, ctrl = cases["c2_push"]
    state = state[:2]
    hi, lo = model.act_ctrlrange[:, 1].astype(np.float32), model.act_ctrlrange[:, 0].astype(np.float32)
    u = np.array([[hi[0], hi[1] + 0.5], [hi[0] - np.float32(4e-4), lo[1] - 0.5]], np.float32)
    nxs = 2 * model.nv
    for centered in (True, False):
        o = fd(model, state, u, centered=centered)
        assert np.array_equal(o["rows"].reshape(-1, model.nq + model.nv), o["ref"])
        check_AB(model, o, u, centered, 1e-3)
        S = 2 if centered else 1
        for e in range(2):
            x0 = o["rows"][e, 0].astype(np.float64)
            assert np.all(o["B"][e, :, 1] == 0)                    # u outside its range
            rm = 1 + nxs * S + (1 if centered else 0)              # the - run of ctrl 0 (forward mode: its only run)
            assert o["inputs"][e, rm, model.nq + model.nv] < u[e, 0]
            want = ((x0 - o["rows"][e, rm].astype(np.float64)) / (float(u[e, 0]) - float(o["inputs"][e, rm, model.nq + model.nv])))
            got = o["B"][e, :, 0]
            nv = model.nv
            plain = [i for i in range(nxs) if i not in rot_dofs(model)]
            idx = [qpos_of_dof(model, i) if i < nv else model.nq + i - nv for i in plain]
            assert np.array_equal(got[plain], want[idx].astype(np.float32)), (centered, e)
            assert np.abs(got).max() > 0


# ---------------------------------------------------------------------------------------------- 5. ptxas budget
# registers / stack of the run instances (ptxas -v, sm_100a, the flags of hsrb_step_g8.cu): measured 247-254 registers and
# a 1552-1584 byte stack frame, no spills; the forming kernels: 68-70 registers, no stack
STACK_CEIL = 1600


def test_fd_kernel_resources():
    from hsr_env_b200 import build as B

    B.build()
    log = (B.CSRC / "hsrb_fd.ptxas.log").read_text()
    names = [f"_Z14hsrb_fd_kernelILi{G}ELb{int(P)}EEv6FdArgs" for G in (4, 8, 16, 32) for P in (False, True)]
    for name in names + [f"_Z19hsrb_fd_form_kernelILb{c}EEv6FdArgs" for c in (0, 1)]:
        block = log.split(f"Function properties for {name}", 1)[1]
        stack = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", block)
        regs = re.search(r"Used (\d+) registers", block)
        assert int(regs.group(1)) <= 255, (name, regs.group(1))
        assert int(stack.group(1)) <= STACK_CEIL and int(stack.group(2)) == 0 and int(stack.group(3)) == 0, (name, stack.groups())
