"""Per-environment physics parameters without a GPU: the kernels' instances with parameters on the SIMT emulator against
their instances without, the reset draw of the parameters, and the ptxas budget of the warp-per-environment instance.

The reference of an environment with multipliers s is the model whose arrays were scaled by s (pair_friction, the block
bodies' body_mass and body_inertia, act_kp, dof_damping), written out as a blob: the compile-time derived quantities stay
as they are.  A power-of-two multiplier is exact in fp32 and fp64, so those environments must match bit for bit."""
import ctypes
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from scenarios import rel_err, rollout_states

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
EMU = HERE / "simt_emu"
LIB = ROOT / "oracle" / "_build" / "libparams_emu.so"
CSRC = ROOT / "hsr_env_b200" / "csrc"
DEPS = [EMU / "emu_params.cpp", EMU / "simt_emu.h"] + [CSRC / h for h in (
    "hsr_core.h", "hsr_model.h", "hsrb_kernels.cuh", "hsrb_push.cuh", "hsrb_wpe.cuh", "hsrb_wpe_kernel.cuh")]
PARAM_NAMES = ("friction", "block_mass", "actuator_gain", "damping")
_dp = ctypes.POINTER(ctypes.c_double)
_fp = ctypes.POINTER(ctypes.c_float)


def _lib():
    LIB.parent.mkdir(exist_ok=True)
    if not LIB.exists() or any(LIB.stat().st_mtime < d.stat().st_mtime for d in DEPS):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-D__CUDACC__", "-DHSRB_SIMT_EMU",
                               "-include", str(EMU / "simt_emu.h"), "-I", str(EMU), "-o", str(LIB), str(EMU / "emu_params.cpp"),
                               "-lpthread"])
    lib = ctypes.CDLL(str(LIB))
    lib.emu_params_step.argtypes = [ctypes.c_char_p, ctypes.c_size_t] + [ctypes.c_int] * 4 + [_dp] * 4 + [_fp] + [_dp] * 3 + [
        ctypes.POINTER(ctypes.c_ubyte)]
    lib.emu_env_params.argtypes = [_fp, _fp, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, _fp]
    lib.emu_params_reset.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_ulonglong] + [_fp] * 6
    return lib


def _p(a, t=ctypes.c_double):
    return None if a is None else a.ctypes.data_as(ctypes.POINTER(t))


def edited(model, s):
    """The model whose arrays carry the multipliers s = (friction, block_mass, actuator_gain, damping)."""
    f, mb, g, d = (float(x) for x in s)
    mass, inertia = model.body_mass.copy(), model.body_inertia.copy()
    for b in model.block_body:
        mass[b] *= mb
        inertia[b] *= mb
    return model.replace(pair_friction=model.pair_friction * f, body_mass=mass, body_inertia=inertia,
                         act_kp=model.act_kp * g, dof_damping=model.dof_damping * d)


def emu_step(model, kernel, qpos, qvel, warm, ctrl, params=None, nsub=1, wpb=3):
    lib = _lib()
    n = qpos.shape[0]
    qpos, qvel, warm, ctrl = (np.ascontiguousarray(x, float) for x in (qpos, qvel, warm, ctrl))
    prm = None if params is None else np.ascontiguousarray(params, np.float32)
    qo, vo, wo = np.zeros_like(qpos), np.zeros_like(qvel), np.zeros_like(warm)
    flags = np.zeros(n, np.uint8)
    blob = model.to_blob()
    rc = lib.emu_params_step(blob, len(blob), kernel, wpb, n, nsub, _p(qpos), _p(qvel), _p(warm), _p(ctrl), _p(prm, ctypes.c_float),
                             _p(qo), _p(vo), _p(wo), _p(flags, ctypes.c_ubyte))
    assert rc == 0, rc
    return np.concatenate([qo, vo, wo], axis=1), flags


def env_params(lo, hi, seed, env_id, episode):
    out = np.zeros(4, np.float32)
    _lib().emu_env_params(_p(np.asarray(lo, np.float32), ctypes.c_float), _p(np.asarray(hi, np.float32), ctypes.c_float),
                          seed, env_id, episode, _p(out, ctypes.c_float))
    return out


# (model, kernel code of emu_params_step): the warp-per-environment kernel both ways, the general kernel at 8 lanes and
# the phase-locked general kernel
CASES = [("c2_push", -1), ("c2_push", -2), ("c2_push", 8), ("c2_push", 0), ("c3_arm", 8), ("c3_arm", 0)]
TUPLES = np.array([[1, 1, 1, 1], [2, .5, 1, 2], [.5, 2, 2, .5], [2, 2, .5, 1], [.5, .5, 2, 2], [1, 2, .5, .5]], np.float32)


@pytest.fixture(scope="module")
def states(models, ports):
    out = {}
    for name in ("c2_push", "c3_arm"):
        out[name] = rollout_states(ports[name], models[name], 12, seed=11, pan=name == "c3_arm", float32=True)
    return out


@pytest.mark.parametrize("name,kernel", CASES)
def test_unit_scales_match_default_instance(name, kernel, models, states):
    model = models[name]
    qpos, qvel, warm, ctrl = states[name]
    ref, fr = emu_step(model, kernel, qpos, qvel, warm, ctrl, nsub=3)
    got, fg = emu_step(model, kernel, qpos, qvel, warm, ctrl, params=np.ones((len(qpos), 4), np.float32), nsub=3)
    assert np.array_equal(got, ref) and np.array_equal(fg, fr)


@pytest.mark.parametrize("name,kernel", CASES)
def test_power_of_two_scales_match_edited_models(name, kernel, models, states):
    """Per-environment tuples from {0.5, 1, 2}: each environment has the bits of the instance without parameters run on
    the model edited with its tuple.  The three warps of the wpe kernel's one block run 4 environments each: the
    multipliers must be read per environment of the grid-stride loop, not once per warp."""
    model = models[name]
    qpos, qvel, warm, ctrl = states[name]
    n = len(qpos)
    idx = np.arange(n) % len(TUPLES)
    got, _ = emu_step(model, kernel, qpos, qvel, warm, ctrl, params=TUPLES[idx], nsub=3)
    for t in range(len(TUPLES)):
        rows = idx == t
        ref, _ = emu_step(edited(model, TUPLES[t]), kernel, qpos[rows], qvel[rows], warm[rows], ctrl[rows], nsub=3)
        assert np.array_equal(got[rows], ref), (t, TUPLES[t])


@pytest.mark.parametrize("name,kernel", CASES)
def test_scales_match_oracle_one_substep(name, kernel, models, states):
    """Multipliers that are not powers of two: one substep within 1e-4 of the fp64 port on the edited model."""
    from oracle import port

    model = models[name]
    qpos, qvel, warm, ctrl = states[name]
    n = len(qpos)
    rng = np.random.default_rng(5)
    prm = rng.uniform(0.5, 2.0, (n, 4)).astype(np.float32)
    got, _ = emu_step(model, kernel, qpos, qvel, warm, ctrl, params=prm, nsub=1)
    over = 0
    for e in range(n):
        ref = port.CpuPort(edited(model, prm[e].astype(np.float64))).step(qpos[e:e + 1], qvel[e:e + 1], warm[e:e + 1], ctrl[e:e + 1], nsub=1)
        assert rel_err(got[e:e + 1, :model.nq], ref["qpos"]).max() <= 1e-4
        over += int(rel_err(got[e:e + 1, model.nq:model.nq + model.nv], ref["qvel"]).max() > 1e-4)
    assert over <= 1, over   # a state on a contact-activation edge may resolve differently in fp32 (tests/test_gpu_parity.py)


def test_reset_draws():
    lo, hi = np.array([.5, .8, 0., 1.], np.float32), np.array([2., 1.25, 3., 1.], np.float32)
    vals = np.array([env_params(lo, hi, 123, e, ep) for e in range(64) for ep in range(3)])
    assert np.all(vals >= lo) and np.all(vals <= hi)
    assert np.all(vals[:, 3] == 1.0)                       # lo == hi draws exactly lo
    assert len(np.unique(vals[:, 0])) == len(vals)         # a stream per environment and episode
    assert not np.array_equal(env_params(lo, hi, 123, 0, 0), env_params(lo, hi, 124, 0, 0))


def test_reset_state_independent_of_ranges(models):
    """The lean reset instance with parameter ranges: the same state bits as without, the parameters of
    sample_env_params for every global environment id."""
    from scenarios import BLOCK_HI, BLOCK_LO, GOAL_HI, GOAL_LO

    lib = _lib()
    model = models["c2_push"]
    n, seed, off = 40, 77, 1000
    S = model.nq + 2 * model.nv + 3
    blob = model.to_blob()
    goal = np.r_[GOAL_LO, GOAL_HI].astype(np.float32)
    block = np.r_[BLOCK_LO, BLOCK_HI].astype(np.float32)
    lo, hi = np.array([.5, .5, .5, .5], np.float32), np.array([2, 2, 2, 2], np.float32)
    outs = []
    for lohi in ((None, None), (lo, hi)):
        st = np.zeros(n * S, np.float32); prm = np.zeros(n * 4, np.float32)
        assert lib.emu_params_reset(blob, len(blob), n, seed, off, _p(goal, ctypes.c_float), _p(block, ctypes.c_float),
                                    _p(lohi[0], ctypes.c_float), _p(lohi[1], ctypes.c_float), _p(st, ctypes.c_float),
                                    _p(prm, ctypes.c_float)) == 0
        outs.append((st, prm.reshape(n, 4)))
    assert np.array_equal(outs[0][0], outs[1][0])
    assert np.all(outs[0][1] == 1.0)
    want = np.array([env_params(lo, hi, seed, off + e, 0) for e in range(n)])
    assert np.array_equal(outs[1][1], want)


# ceilings of the instances with parameters (ptxas -v, sm_100a, the flags of hsrb_wpe.cu); the instances without have
# 234 / 288 (locked) and 178 / 232 (free) bytes, held by tests/test_wpe_resources.py
PARAMS_KERNELS = {"_Z24hsrb_wpe_params_kernel_tILb1EEv5KArgs8PushInfo": (250, 300),
                  "_Z24hsrb_wpe_params_kernel_tILb0EEv5KArgs8PushInfo": (194, 264)}


def test_wpe_params_resources(tmp_path):
    from hsr_env_b200 import build as B

    if not Path(B.NVCC).exists() and shutil.which(B.NVCC) is None:
        pytest.skip(f"nvcc not found at {B.NVCC}")
    src = B.CSRC / "hsrb_wpe_params.cu"
    r = subprocess.run([B.NVCC, *B.FLAGS, *B.TU_FLAGS[src.name], "-c", str(src), "-o", str(tmp_path / "p.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    for name, (st_ceil, ld_ceil) in PARAMS_KERNELS.items():
        block = r.stderr.split(f"Function properties for {name}", 1)[1]
        spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", block)
        regs = re.search(r"Used (\d+) registers", block)
        assert int(regs.group(1)) <= 72, (name, regs.group(1))   # 28 warps per SM
        assert int(spill.group(1)) <= st_ceil and int(spill.group(2)) <= ld_ceil, (name, spill.groups())
