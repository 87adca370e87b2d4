"""TEST INFRASTRUCTURE: g++ build of the CUDA action kernel on top of the SIMT emulator (no GPU needed)."""
from __future__ import annotations

import ctypes
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
LIB = ROOT / "oracle" / "_build" / "libpush_emu.so"
DEPS = [HERE / "emu_push.cpp", HERE / "simt_emu.h", ROOT / "hsr_env_b200/csrc/hsrb_push.cuh", ROOT / "hsr_env_b200/csrc/hsrb_wpe.cuh", ROOT / "hsr_env_b200/csrc/hsr_core.h",
        ROOT / "hsr_env_b200/csrc/hsrb_kernels.cuh", ROOT / "hsr_env_b200/csrc/hsr_model.h"]


def lib_path(base, defines):
    """Library of one set of extra -D flags: the default build keeps `base`, every other set gets its own file, so that a
    reduced-capacity build never stands in for the default one (or the other way round) on the mtime check."""
    if not defines:
        return base
    tag = "_".join(d.replace("=", "") for d in defines)
    return base.with_name(f"{base.stem}_{tag}{base.suffix}")


def build(force=False, defines=()):
    """The fast-path kernels on the emulator; `defines` (and EMU_DEFINES in the environment) are extra -D flags, e.g.
    ("PUSH_MAXCON=4", "WPE_MAXCON=4") for a build with a contact capacity of 4."""
    import os
    extra = [*defines, *os.environ.get("EMU_DEFINES", "").split()]
    lib = lib_path(LIB, extra)
    lib.parent.mkdir(exist_ok=True)
    if not force and lib.exists() and all(lib.stat().st_mtime >= d.stat().st_mtime for d in DEPS):
        return lib
    cmd = ["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-D__CUDACC__", "-DHSRB_SIMT_EMU", "-DHSR_COMPACT", *[f"-D{d}" for d in extra],
           "-include", str(HERE / "simt_emu.h"), "-I", str(HERE), "-o", str(lib), str(HERE / "emu_push.cpp"), "-lpthread"]
    subprocess.check_call(cmd)
    return lib


_dp = ctypes.POINTER(ctypes.c_double)


def _p(a, t=ctypes.c_double):
    return a.ctypes.data_as(ctypes.POINTER(t))


def step(model, qpos, qvel, warm, ctrl, mocap=None, nsub=1, G=8, threads=32, geofence=None, defines=()):
    lib = ctypes.CDLL(str(build(defines=defines)))
    qpos = np.ascontiguousarray(np.atleast_2d(qpos), float); n = qpos.shape[0]
    qvel = np.ascontiguousarray(np.atleast_2d(qvel), float); warm = np.ascontiguousarray(np.atleast_2d(warm), float)
    ctrl = np.ascontiguousarray(np.atleast_2d(ctrl), float)
    mocap = np.zeros((n, 3)) if mocap is None else np.ascontiguousarray(np.atleast_2d(mocap), float)
    qo, vo, wo = np.zeros_like(qpos), np.zeros_like(qvel), np.zeros_like(warm)
    taken = np.zeros(n, np.int32); succ = np.zeros(n, np.uint8); flags = np.zeros(n, np.uint8); stats = np.zeros(16, np.int64)
    blob = model.to_blob()
    lib.emu_push_step.argtypes = [ctypes.c_char_p, ctypes.c_size_t] + [ctypes.c_int] * 4 + [_dp] * 5 + [ctypes.c_int, ctypes.c_double] + [_dp] * 3 + [
        ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_ubyte), ctypes.POINTER(ctypes.c_ubyte), ctypes.POINTER(ctypes.c_longlong)]
    rc = lib.emu_push_step(blob, len(blob), G, threads, n, nsub, _p(qpos), _p(qvel), _p(warm), _p(ctrl), _p(mocap),
                           int(geofence is not None), float(geofence or 0.0), _p(qo), _p(vo), _p(wo), _p(taken, ctypes.c_int),
                           _p(succ, ctypes.c_ubyte), _p(flags, ctypes.c_ubyte), _p(stats, ctypes.c_longlong))
    if rc:
        raise RuntimeError(f"emu_push_step failed: {rc}")
    return dict(qpos=qo, qvel=vo, warm=wo, taken=taken, success=succ, flags=flags, stats=stats)


# ---------------------------------------------------------------------------------------------- general kernel
LIB_G = ROOT / "oracle" / "_build" / "libstep_emu.so"
DEPS_G = [HERE / "emu_step.cpp", HERE / "simt_emu.h", ROOT / "hsr_env_b200/csrc/hsr_core.h", ROOT / "hsr_env_b200/csrc/hsrb_kernels.cuh",
          ROOT / "hsr_env_b200/csrc/hsr_model.h"]


def build_general(force=False):
    LIB_G.parent.mkdir(exist_ok=True)
    if not force and LIB_G.exists() and all(LIB_G.stat().st_mtime >= d.stat().st_mtime for d in DEPS_G):
        return LIB_G
    cmd = ["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-D__CUDACC__", "-DHSRB_SIMT_EMU",
           "-include", str(HERE / "simt_emu.h"), "-I", str(HERE), "-o", str(LIB_G), str(HERE / "emu_step.cpp"), "-lpthread"]
    subprocess.check_call(cmd)
    return LIB_G


def step_general(model, qpos, qvel, warm, ctrl, nsub=1, G=8, ncon_max=0, nefc_max=0):
    """The general action kernel (hsrb_kernels.cuh) on the emulator: G lanes per environment, one warp per block (G = 0:
    the phase-locked kernel).  ncon_max / nefc_max > 0 replace the model's contact / constraint-row capacities, as
    hsrb_config does on the device."""
    lib = ctypes.CDLL(str(build_general()))
    qpos = np.ascontiguousarray(np.atleast_2d(qpos), float); n = qpos.shape[0]
    qvel = np.ascontiguousarray(np.atleast_2d(qvel), float); warm = np.ascontiguousarray(np.atleast_2d(warm), float)
    ctrl = np.ascontiguousarray(np.atleast_2d(ctrl), float)
    qo, vo, wo = np.zeros_like(qpos), np.zeros_like(qvel), np.zeros_like(warm)
    taken = np.zeros(n, np.int32); flags = np.zeros(n, np.uint8); stats = np.zeros(16, np.int64)
    blob = model.to_blob()
    lib.emu_general_step.argtypes = [ctypes.c_char_p, ctypes.c_size_t] + [ctypes.c_int] * 5 + [_dp] * 7 + [
        ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_ubyte), ctypes.POINTER(ctypes.c_longlong)]
    rc = lib.emu_general_step(blob, len(blob), G, n, nsub, int(ncon_max), int(nefc_max), _p(qpos), _p(qvel), _p(warm), _p(ctrl), _p(qo), _p(vo), _p(wo),
                              _p(taken, ctypes.c_int), _p(flags, ctypes.c_ubyte), _p(stats, ctypes.c_longlong))
    if rc:
        raise RuntimeError(f"emu_general_step failed: {rc}")
    return dict(qpos=qo, qvel=vo, warm=wo, taken=taken, flags=flags, stats=stats)
