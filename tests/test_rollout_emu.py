"""Open-loop rollouts without a GPU: the rollout instances of the phase-locked action kernels (K actions per environment
in one launch, hsrb_rollout) against K launches of the step instances on the SIMT emulator, bit for bit: every slice of
every output, the state afterwards and the work counters.  Plus the ptxas budget of the wpe rollout instances."""
import ctypes
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from scenarios import rollout_states

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
EMU = HERE / "simt_emu"
LIB = ROOT / "oracle" / "_build" / "librollout_emu.so"
CSRC = ROOT / "hsr_env_b200" / "csrc"
DEPS = [EMU / "emu_rollout.cpp", EMU / "simt_emu.h"] + [CSRC / h for h in (
    "hsr_core.h", "hsr_model.h", "hsrb_kernels.cuh", "hsrb_step_lock_kernel.cuh", "hsrb_push.cuh", "hsrb_wpe.cuh",
    "hsrb_wpe_kernel.cuh")]
ST_COUNT = 16   # hsrb_kernels.cuh: ST_PHASE0 + PH_COUNT
GEOFENCE = 0.05
_vp = ctypes.c_void_p


def _lib():
    LIB.parent.mkdir(exist_ok=True)
    if not LIB.exists() or any(LIB.stat().st_mtime < d.stat().st_mtime for d in DEPS):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-D__CUDACC__", "-DHSRB_SIMT_EMU",
                               "-include", str(EMU / "simt_emu.h"), "-I", str(EMU), "-o", str(LIB), str(EMU / "emu_rollout.cpp"),
                               "-lpthread"])
    lib = ctypes.CDLL(str(LIB))
    lib.emu_rollout.argtypes = [ctypes.c_char_p, ctypes.c_size_t] + [ctypes.c_int] * 6 + [ctypes.c_float] + [_vp] * 10
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(_vp)


def emu_rollout(model, kernel, state, ctrl, rollout, params=None, nsub=40, geofence=GEOFENCE, wpb=3):
    """(state after, obs, reward, done, taken, bad, stats, sep) of K = len(ctrl) actions; sep: the wpe kernel's
    separating-direction cache of each warp at the end (the outputs cannot show it: the cache only saves work)."""
    K, n = ctrl.shape[0], state.shape[0]
    st = np.ascontiguousarray(state, np.float32).copy()
    ctrl = np.ascontiguousarray(ctrl, np.float32)
    prm = None if params is None else np.ascontiguousarray(params, np.float32)
    obs = np.full((K, n, model.nq + model.nv), np.nan, np.float32)
    reward = np.full((K, n), np.nan, np.float32)
    done, bad = np.full((K, n), 7, np.uint8), np.full((K, n), 7, np.uint8)
    taken = np.full((K, n), -1, np.int32)
    stats = np.zeros(ST_COUNT, np.uint64)
    sep = np.zeros((wpb, 4 * 24), np.float32)   # WPE_MAXPAIR
    blob = model.to_blob()
    rc = _lib().emu_rollout(blob, len(blob), kernel, wpb, int(rollout), n, K, nsub, geofence, _p(st), _p(ctrl), _p(prm), _p(obs),
                            _p(reward), _p(done), _p(taken), _p(bad), _p(stats), _p(sep))
    assert rc == 0, rc
    return st, obs, reward, done, taken, bad, stats, sep


def block_qadr(model):
    """qpos address of the block's free joint (its position = the block body's position)."""
    b = int(model.block_body[0])
    j = [j for j in range(model.njnt) if model.jnt_type[j] == 0 and model.jnt_body[j] == b][0]
    return int(model.jnt_qposadr[j])


@pytest.fixture(scope="module")
def starts(models, ports):
    """Start state rows [n, S] per model: the goal point (mocap) sits on the block for every third environment (reached
    in the first action), far away for the others (never reached)."""
    out = {}
    for name in ("c2_push", "c1b_readme_block", "c3_arm", "f2_cupboard"):
        model = models[name]
        qpos, qvel, warm, _ = rollout_states(ports[name], model, 12, seed=23, pan=name == "c3_arm", float32=True)
        qa = block_qadr(model)
        mocap = np.where((np.arange(len(qpos)) % 3 == 0)[:, None], qpos[:, qa:qa + 3], 10.0)
        out[name] = np.concatenate([qpos, qvel, warm, mocap], axis=1).astype(np.float32)
    return out


def actions(model, K, n, seed=1):
    rng = np.random.default_rng(seed)
    lo, hi = model.act_ctrlrange[:, 0], model.act_ctrlrange[:, 1]
    return rng.uniform(lo, hi, (K, n, model.nu)).astype(np.float32)


def check_equal(got, ref):
    names = ("state", "obs", "reward", "done", "taken", "bad", "stats", "sep")
    for nm, x, y in zip(names, got, ref):
        assert x.shape == y.shape and np.array_equal(x, y, equal_nan=False), nm


# (model, kernel code of emu_rollout): the phase-locked wpe kernel on the two block-push models, the phase-locked general
# kernel on the articulated arm and the cupboard
CASES = [("c2_push", -2), ("c1b_readme_block", -2), ("c3_arm", 0), ("f2_cupboard", 0)]
PARAMS = np.array([[2, .5, 1, 2], [.5, 2, 2, .5], [1.3, .7, .9, 1.1], [1, 1, 1, 1]], np.float32)


@pytest.mark.parametrize("with_params", [False, True], ids=["nominal", "params"])
@pytest.mark.parametrize("name,kernel", CASES)
def test_rollout_bit_equal_to_sequential_steps(name, kernel, with_params, models, starts):
    model = models[name]
    state = starts[name]
    n, K = len(state), 4
    ctrl = actions(model, K, n)
    prm = PARAMS[np.arange(n) % len(PARAMS)] if with_params else None
    ref = emu_rollout(model, kernel, state, ctrl, rollout=False, params=prm)
    got = emu_rollout(model, kernel, state, ctrl, rollout=True, params=prm)
    check_equal(got, ref)
    done = ref[3].astype(bool)
    assert done[0].any() and not done.all()         # some environments reach the goal in the first action, others never
    assert not np.array_equal(ref[1][0], ref[1][-1])   # the actions move the state
    assert np.all(ref[4][:, ~done[0]] == 40)


@pytest.mark.parametrize("name,kernel", CASES[:1] + CASES[2:3])
@pytest.mark.parametrize("K,nsub", [(1, 40), (3, 0)])
def test_rollout_single_action_and_zero_substeps(name, kernel, K, nsub, models, starts):
    model = models[name]
    state = starts[name]
    ctrl = actions(model, K, len(state), seed=K)
    ref = emu_rollout(model, kernel, state, ctrl, rollout=False, nsub=nsub)
    got = emu_rollout(model, kernel, state, ctrl, rollout=True, nsub=nsub)
    check_equal(got, ref)
    if nsub == 0:
        assert np.array_equal(got[0], state) and np.all(got[4] == 0)


# ceilings of the wpe rollout instances (ptxas -v, sm_100a, the flags of hsrb_wpe.cu); the step instances they are built
# from have 234 / 288 (tests/test_wpe_resources.py) and 250 / 300 bytes (tests/test_env_params_emu.py): the action loop
# keeps its counter and row offset live across the substep loop
ROLLOUT_KERNELS = {"_Z25hsrb_wpe_rollout_kernel_tILb1EEv5KArgs8PushInfoi": (242, 304),
                   "_Z32hsrb_wpe_rollout_params_kernel_tILb1EEv5KArgs8PushInfoi": (298, 372)}


def test_wpe_rollout_resources(tmp_path):
    from hsr_env_b200 import build as B

    if not Path(B.NVCC).exists() and shutil.which(B.NVCC) is None:
        pytest.skip(f"nvcc not found at {B.NVCC}")
    src = B.CSRC / "hsrb_wpe_rollout.cu"
    r = subprocess.run([B.NVCC, *B.FLAGS, *B.TU_FLAGS[src.name], "-c", str(src), "-o", str(tmp_path / "r.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    for name, (st_ceil, ld_ceil) in ROLLOUT_KERNELS.items():
        block = r.stderr.split(f"Function properties for {name}", 1)[1]
        spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", block)
        regs = re.search(r"Used (\d+) registers", block)
        assert int(regs.group(1)) <= 72, (name, regs.group(1))   # 28 warps per SM
        assert int(spill.group(1)) <= st_ceil and int(spill.group(2)) <= ld_ceil, (name, spill.groups())
