"""TEST INFRASTRUCTURE: g++ build of the episode kernel (hsr_env_b200/csrc/hsrb_episode.cuh) on the SIMT emulator."""
from __future__ import annotations

import ctypes
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
LIB = ROOT / "oracle" / "_build" / "libepisode_emu.so"
DEPS = [HERE / "emu_episode.cpp", HERE / "simt_emu.h", ROOT / "hsr_env_b200/csrc/hsrb_episode.cuh", ROOT / "hsr_env_b200/csrc/hsr_core.h",
        ROOT / "hsr_env_b200/csrc/hsrb_kernels.cuh", ROOT / "hsr_env_b200/csrc/hsr_model.h"]


def build(force=False):
    """EMU_EPISODE_LIB in the environment names a prebuilt library instead (tools/emu_sanitize.sh: a sanitizer build)."""
    if os.environ.get("EMU_EPISODE_LIB"):
        return Path(os.environ["EMU_EPISODE_LIB"])
    LIB.parent.mkdir(exist_ok=True)
    if not force and LIB.exists() and all(LIB.stat().st_mtime >= d.stat().st_mtime for d in DEPS):
        return LIB
    cmd = ["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-D__CUDACC__", "-DHSRB_SIMT_EMU",
           "-include", str(HERE / "simt_emu.h"), "-I", str(HERE), "-o", str(LIB), str(HERE / "emu_episode.cpp"), "-lpthread"]
    subprocess.check_call(cmd)
    return LIB


def _p(a, t):
    return a.ctypes.data_as(ctypes.POINTER(t))


def episode(model, state, episode_ctr, age, ret, sub, term, reward, taken, bad, *, max_steps, autoreset, seed=0, env_off=0,
            goal_lohi=None, block_lohi=None, min_sep=0.0, qidx=(0, 2), starts=None, G=8, grid=None):
    """One launch of the episode kernel.  state [n, nq + 2 nv + 3] float32, episode_ctr uint32, age / sub int32, ret float32
    are updated in place (copies are returned); starts = (adr, width, lo [k, 7], hi [k, 7]).  grid None: one block per
    32 / G environments (smaller: the grid-stride loop)."""
    lib = ctypes.CDLL(str(build()))
    n = len(state)
    state = np.ascontiguousarray(state, np.float32).copy()
    episode_ctr = np.ascontiguousarray(episode_ctr, np.uint32).copy()
    age = np.ascontiguousarray(age, np.int32).copy(); ret = np.ascontiguousarray(ret, np.float32).copy()
    sub = np.ascontiguousarray(sub, np.int32).copy()
    term = np.ascontiguousarray(term, np.uint8); reward = np.ascontiguousarray(reward, np.float32)
    taken = np.ascontiguousarray(taken, np.int32); bad = np.ascontiguousarray(bad, np.uint8)
    nobs = model.nq + model.nv
    trunc = np.full(n, 7, np.uint8)
    final = np.full((n, nobs), np.nan, np.float32)
    obs = np.full((n, nobs), np.nan, np.float32)
    ep_len = np.full(n, -1, np.int32); ep_ret = np.full(n, np.nan, np.float32); ep_sub = np.full(n, -1, np.int32)
    counters = np.zeros(8, np.uint64)
    gl = np.zeros(6) if goal_lohi is None else np.asarray(goal_lohi, float)
    bl = np.zeros(8) if block_lohi is None else np.asarray(block_lohi, float)
    adr, width, lo, hi = starts if starts is not None else ([], [], np.zeros((0, 7)), np.zeros((0, 7)))
    adr = np.ascontiguousarray(adr, np.int32); width = np.ascontiguousarray(width, np.int32)
    lo = np.ascontiguousarray(lo, float).reshape(-1, 7); hi = np.ascontiguousarray(hi, float).reshape(-1, 7)
    if grid is None:
        grid = (n + 32 // G - 1) // (32 // G)
    c_int, c_u8, c_f, c_d = ctypes.c_int, ctypes.c_ubyte, ctypes.c_float, ctypes.c_double
    P = ctypes.POINTER
    lib.emu_episode.argtypes = ([ctypes.c_char_p, ctypes.c_size_t, c_int, c_int, c_int, ctypes.c_ulonglong, ctypes.c_ulonglong,
                                 c_int, P(c_d), c_int, P(c_d), c_d, c_int, c_int, c_int, P(c_int), P(c_int), P(c_d), P(c_d),
                                 c_int, c_int, P(c_f), P(ctypes.c_uint), P(c_int), P(c_f), P(c_int),
                                 P(c_u8), P(c_f), P(c_int), P(c_u8), P(c_u8), P(c_f), P(c_f), P(c_int), P(c_f), P(c_int),
                                 P(ctypes.c_ulonglong)])
    blob = model.to_blob()
    rc = lib.emu_episode(blob, len(blob), G, grid, n, seed, env_off, int(goal_lohi is not None), _p(gl, c_d), int(block_lohi is not None),
                         _p(bl, c_d), float(min_sep), qidx[0], qidx[1], len(adr), _p(adr, c_int), _p(width, c_int), _p(lo, c_d), _p(hi, c_d),
                         int(max_steps), int(autoreset), _p(state, c_f), _p(episode_ctr, ctypes.c_uint), _p(age, c_int), _p(ret, c_f),
                         _p(sub, c_int), _p(term, c_u8), _p(reward, c_f), _p(taken, c_int), _p(bad, c_u8), _p(trunc, c_u8), _p(final, c_f),
                         _p(obs, c_f), _p(ep_len, c_int), _p(ep_ret, c_f), _p(ep_sub, c_int), _p(counters, ctypes.c_ulonglong))
    if rc:
        raise RuntimeError(f"emu_episode failed: {rc}")
    return dict(state=state, episode=episode_ctr, age=age, ret=ret, sub=sub, truncated=trunc, final_obs=final, obs=obs,
                ep_length=ep_len, ep_return=ep_ret, ep_substeps=ep_sub, counters=counters)
