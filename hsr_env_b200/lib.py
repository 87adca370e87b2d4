"""ctypes binding of libhsrb.so (include/hsrb.h).  No CPU fallback: a missing library or GPU raises.

The binding exchanges PyTorch CUDA tensors by raw device pointer (``tensor.data_ptr()``) and launches on
torch's current stream, so calls order naturally with the caller's torch work.
"""
from __future__ import annotations

import ctypes
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint8, c_uint64, c_void_p
from pathlib import Path

CSRC = Path(__file__).resolve().parent / "csrc"
import os

LIB_PATH = Path(os.environ.get("HSRB_LIB", CSRC / "libhsrb.so"))  # HSRB_LIB: e.g. the phase-clock build

# every symbol include/hsrb.h declares: (restype, argtypes)
SIGNATURES = {
    "hsrb_create": (c_int, [c_void_p, c_size_t, c_int, c_int, c_uint64, c_uint64, POINTER(c_void_p)]),
    "hsrb_destroy": (c_int, [c_void_p]),
    "hsrb_dims": (c_int, [c_void_p] + [POINTER(c_int)] * 5),
    "hsrb_config": (c_int, [c_void_p, c_int, c_int, c_int]),
    "hsrb_set_path": (c_int, [c_void_p, c_int]),
    "hsrb_set_goals": (c_int, [c_void_p, POINTER(c_float), POINTER(c_float), c_float, c_float, c_int, c_int]),
    "hsrb_set_goal_list": (c_int, [c_void_p, c_int, POINTER(c_int32), POINTER(c_int32), POINTER(c_float), POINTER(c_float),
                                   POINTER(c_float), c_int]),
    "hsrb_set_starts": (c_int, [c_void_p, c_int, POINTER(c_int32), POINTER(c_int32), POINTER(c_float), POINTER(c_float)]),
    "hsrb_reset": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "hsrb_step": (c_int, [c_void_p, c_void_p, c_int] + [c_void_p] * 7),
    "hsrb_rollout": (c_int, [c_void_p, c_void_p, c_int, c_int] + [c_void_p] * 6),
    "hsrb_step_episode": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int] + [c_void_p] * 11),
    "hsrb_episode_update": (c_int, [c_void_p, c_int, c_int] + [c_void_p] * 11),
    "hsrb_set_episode_ages": (c_int, [c_void_p, c_void_p, c_void_p]),
    "hsrb_get_episode_ages": (c_int, [c_void_p, c_void_p, c_void_p]),
    "hsrb_episode_stats": (c_int, [c_void_p, POINTER(c_int64), c_void_p]),
    "hsrb_set_env_params": (c_int, [c_void_p, c_void_p, c_void_p]),
    "hsrb_get_env_params": (c_int, [c_void_p, c_void_p, c_void_p]),
    "hsrb_set_env_param_ranges": (c_int, [c_void_p, POINTER(c_float), POINTER(c_float)]),
    "hsrb_step_host":(c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hsrb_get_state": (c_int, [c_void_p] + [c_void_p] * 5),
    "hsrb_set_state": (c_int, [c_void_p] + [c_void_p] * 5),
    "hsrb_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "hsrb_openai_obs": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hsrb_compute_reward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "hsrb_contact_capacity": (c_int, [c_void_p]),
    "hsrb_contacts": (c_int, [c_void_p, c_void_p, c_int] + [c_void_p] * 9),
    "hsrb_transition_fd": (c_int, [c_void_p, c_void_p, c_float, c_int, c_int] + [c_void_p] * 5),
    "hsrb_debug_size": (c_int, [c_void_p]),
    "hsrb_debug_substep": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "hsrb_stats": (c_int, [c_void_p, POINTER(c_int64), c_void_p]),
    "hsrb_launch_info": (c_int, [c_void_p, POINTER(c_int)]),
    "hsrb_measure_fp32_peak": (c_int, [c_int, POINTER(c_double)]),
    "hsrb_last_error": (c_char_p, []),
}

_lib = None


class HsrbError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """Load libhsrb.so (built in-tree by ``python -m hsr_env_b200.build``).  Fails loudly when absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise HsrbError(f"{LIB_PATH} is missing: build it with `python -m hsr_env_b200.build` "
                        "(there is no CPU fallback for the physics path)")
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int):
    if rc < 0:
        raise HsrbError(load().hsrb_last_error().decode())
    return rc


def ptr(t):
    """Device (or host) pointer of a contiguous tensor / numpy array, or NULL."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        assert t.is_contiguous(), "tensor must be contiguous"
        return c_void_p(t.data_ptr())
    assert t.flags["C_CONTIGUOUS"]
    return c_void_p(t.ctypes.data)
