"""In-tree build of libhsrb.so (nvcc, sm_100a only).  ``python -m hsr_env_b200.build [--force]``.

The shared library is built next to the sources (``hsr_env_b200/csrc/libhsrb.so``) so that it travels to the
GPU box with the repository snapshot; it is git-ignored.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

CSRC = Path(__file__).resolve().parent / "csrc"
LIB = CSRC / "libhsrb.so"
TUS = ["hsrb_api.cu", "hsrb_push.cu", "hsrb_wpe.cu", "hsrb_wpe_params.cu", "hsrb_step_g4.cu", "hsrb_step_g8.cu", "hsrb_step_g16.cu", "hsrb_step_g32.cu", "hsrb_step_lock.cu", "hsrb_episode.cu",
       "hsrb_step_g4_params.cu", "hsrb_step_g8_params.cu", "hsrb_step_g16_params.cu", "hsrb_step_g32_params.cu",
       "hsrb_step_lock_params.cu", "hsrb_wpe_rollout.cu", "hsrb_step_lock_rollout.cu"]
HEADERS = ["hsr_core.h", "hsr_model.h", "hsrb_kernels.cuh", "hsrb_push.cuh", "hsrb_wpe.cuh", "hsrb_wpe_kernel.cuh", "hsrb_step_lock_kernel.cuh", "hsrb_episode.cuh", "../../include/hsrb.h"]
# per-TU flags: the fast-path kernel uses the 2-ulp fp32 division / square root (MUFU.RCP / MUFU.RSQ sequences without
# the IEEE fix-up path; measured +6 % substeps/s, one-step error vs the fp64 oracle unchanged at the 1e-7 level); the
# general kernel and the reset / forward paths keep IEEE division.
TU_FLAGS = {"hsrb_push.cu": ([] if os.environ.get("HSRB_PRECISE_DIV") else ["--prec-div=false", "--prec-sqrt=false"])
            + os.environ.get("NVCC_PUSH_EXTRA", "").split()}
TU_FLAGS["hsrb_wpe.cu"] = ([] if os.environ.get("HSRB_PRECISE_DIV") else ["--prec-div=false", "--prec-sqrt=false"]) \
    + os.environ.get("NVCC_WPE_EXTRA", "").split()
# the instance with per-environment parameters: same flags as the instances without
TU_FLAGS["hsrb_wpe_params.cu"] = TU_FLAGS["hsrb_wpe.cu"]
for _g in (4, 8, 16, 32):
    TU_FLAGS[f"hsrb_step_g{_g}.cu"] = os.environ.get("NVCC_STEP_EXTRA", "").split()
# the episode kernel resets environments with the stages of the lean reset instance above: same (IEEE) flags, same bits
TU_FLAGS["hsrb_episode.cu"] = TU_FLAGS["hsrb_step_g8.cu"]
# the phase-locked general kernel takes the same 2-ulp fp32 division / square root as the block-push kernels
TU_FLAGS["hsrb_step_lock.cu"] = ([] if os.environ.get("HSRB_PRECISE_DIV") else ["--prec-div=false", "--prec-sqrt=false"]) \
    + os.environ.get("NVCC_STEP_EXTRA", "").split()
# the instances with per-environment parameters: the flags of the instances without
for _tu in ("hsrb_step_g4.cu", "hsrb_step_g8.cu", "hsrb_step_g16.cu", "hsrb_step_g32.cu", "hsrb_step_lock.cu"):
    TU_FLAGS[_tu.replace(".cu", "_params.cu")] = TU_FLAGS[_tu]
# the instances with the action loop of hsrb_rollout: the flags of the instances hsrb_step launches
TU_FLAGS["hsrb_wpe_rollout.cu"] = TU_FLAGS["hsrb_wpe.cu"]
TU_FLAGS["hsrb_step_lock_rollout.cu"] = TU_FLAGS["hsrb_step_lock.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
         "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False, phase_clocks: bool = False, defines=(), tag: str = "") -> Path:
    """phase_clocks=True builds the instrumented variant libhsrb_prof.so (-DHSRB_PHASE_CLOCKS); ``defines`` + ``tag``
    build an experiment variant libhsrb_<tag>.so with extra -D flags (selected at run time with HSRB_LIB)."""
    hdrs = [CSRC / h for h in HEADERS]
    objs = []
    jobs = []
    name = tag
    tag = ".prof" if phase_clocks else (f".{tag}" if tag else "")
    flags = FLAGS + (["-DHSRB_PHASE_CLOCKS"] if phase_clocks else []) + [f"-D{d}" for d in defines] + os.environ.get("NVCC_EXTRA", "").split()
    lib = CSRC / "libhsrb_prof.so" if phase_clocks else (CSRC / f"libhsrb_{name}.so" if name else LIB)
    for tu in TUS:
        src = CSRC / tu
        obj = CSRC / (src.stem + tag + ".o")
        objs.append(obj)
        if force or _stale(obj, [src] + hdrs):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [NVCC, *flags, *TU_FLAGS.get(src.name, []), "-c", str(src), "-o", str(obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        (CSRC / (src.stem + tag + ".ptxas.log")).write_text(r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src.name}:\n{r.stderr}")
        return src.name, r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            for name, log in ex.map(compile_one, jobs):
                if verbose:
                    print(f"--- {name}\n{log}")
    if force or jobs or _stale(lib, objs):
        cmd = [NVCC, "-shared", "-o", str(lib), *map(str, objs), "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
        subprocess.check_call(cmd)
    return lib


if __name__ == "__main__":
    defs = [a.split("=", 1)[1] if a.startswith("--define=") else None for a in sys.argv]
    defs = [d for d in defs if d]
    tags = [a.split("=", 1)[1] for a in sys.argv if a.startswith("--tag=")]
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, phase_clocks="--prof" in sys.argv, defines=defs,
                tag=tags[0] if tags else ""))
