"""The C-ABI library loads without a GPU and exports every symbol include/hsrb.h declares."""
import ctypes
import os
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def declared_symbols():
    text = (ROOT / "include" / "hsrb.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hsrb_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound():
    from hsr_env_b200 import build, lib

    build.build()
    cdll = lib.load()
    syms = declared_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(cdll, s), s
        assert s in lib.SIGNATURES, f"{s} declared in hsrb.h but not bound in lib.py"
    assert set(lib.SIGNATURES) == set(syms)


NO_GPU_CHECK = """
import ctypes
import torch
from hsr_env_b200 import lib
from hsr_env_b200.env import BatchedHSREnv
from hsr_env_b200.model import Model

assert not torch.cuda.is_available()
cdll = lib.load()
blob = Model.load("hsr_env_b200/blobs/c2_push.hsrb").to_blob()
h = ctypes.c_void_p()
rc = cdll.hsrb_create(blob, len(blob), 4, 0, 0, 0, ctypes.byref(h))
assert rc < 0 and not h.value
assert b"no CPU fallback" in cdll.hsrb_last_error()
try:
    BatchedHSREnv("c2_push.hsrb", None, n_envs=4, device="cuda:0")
except lib.HsrbError:
    pass
else:
    raise AssertionError("BatchedHSREnv was created without a GPU")
"""


def test_create_fails_loudly_without_gpu():
    """In a process that sees no GPU (CUDA_VISIBLE_DEVICES empty), so that a machine with one checks the path too."""
    env = {**os.environ, "CUDA_VISIBLE_DEVICES": ""}
    r = subprocess.run([sys.executable, "-c", NO_GPU_CHECK], cwd=ROOT, env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_bad_blob_rejected():
    from hsr_env_b200 import lib

    cdll = lib.load()
    h = ctypes.c_void_p()
    assert cdll.hsrb_create(b"\0" * 128, 128, 1, 0, 0, 0, ctypes.byref(h)) < 0
    assert b"blob" in cdll.hsrb_last_error()
