"""Register and local-memory budget of the warp-per-environment action kernels (hsrb_wpe.cu), from ptxas, without a GPU.

The kernels run 28 warps per SM at a cap of 72 registers.  Local memory under that cap is the kernel's stack: spill slots
and address-taken objects.  Its reloads sit on the dependent chain of an environment, and 28 warps' slots compete for the
~24 KB of L1 that the 227 KB shared-memory carve-out leaves.  The test compiles the
translation unit with the build's own flags and holds the figures of this layout as ceilings, so that a change that
brings spills back fails here rather than as a slower benchmark.
"""
import re
import shutil
import subprocess
from pathlib import Path

import pytest

from hsr_env_b200 import build as B

KERNELS = {"_Z17hsrb_wpe_kernel_tILb1EEv5KArgs8PushInfo": "locked", "_Z17hsrb_wpe_kernel_tILb0EEv5KArgs8PushInfo": "free"}
MPR = "_ZN3wpe3mprEiiiifii"
# ceilings (bytes) of the kernel bodies; before the fixed shared-memory layout and the narrow mpr() call the locked kernel
# had 406 B of spill stores and 392 B of spill loads, the free-running one 254 B and 264 B
SPILL_CEIL = {"locked": (234, 288), "free": (178, 232)}
# the stack of a kernel includes its callees' frames: hsr::box_box's clip polygons (2 x 16 points, 768 B) and spill slots
STACK_CEIL = 1920


def ptxas_report(tmp: Path) -> str:
    if not Path(B.NVCC).exists() and shutil.which(B.NVCC) is None:
        pytest.skip(f"nvcc not found at {B.NVCC}")
    src = B.CSRC / "hsrb_wpe.cu"
    cmd = [B.NVCC, *B.FLAGS, *B.TU_FLAGS.get(src.name, []), "-c", str(src), "-o", str(tmp / "hsrb_wpe.o")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    return r.stderr


def parse(log: str):
    """{entry: {"regs": n, "stack": b, "functions": {name: (stack, spill_st, spill_ld)}}} from ptxas -v."""
    out, entry, fn = {}, None, None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            entry = m.group(1)
            out[entry] = {"regs": None, "stack": None, "functions": {}}
            continue
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            fn = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and entry and fn:
            out[entry]["functions"][fn] = tuple(int(x) for x in m.groups())
            continue
        m = re.search(r"Used (\d+) registers.*?(\d+) bytes cumulative stack size", line)
        if m and entry:
            out[entry]["regs"], out[entry]["stack"] = int(m.group(1)), int(m.group(2))
    return out


@pytest.fixture(scope="module")
def report(tmp_path_factory):
    return parse(ptxas_report(tmp_path_factory.mktemp("wpe_ptxas")))


@pytest.mark.parametrize("entry", sorted(KERNELS))
def test_wpe_registers_and_spills(report, entry):
    r = report[entry]
    kind = KERNELS[entry]
    assert r["regs"] is not None and r["regs"] <= 72, r            # 28 warps x 32 lanes x 72 = the register file
    _, st, ld = r["functions"][entry]
    assert st <= SPILL_CEIL[kind][0] and ld <= SPILL_CEIL[kind][1], (kind, st, ld)
    assert r["stack"] <= STACK_CEIL, (kind, r["stack"])


@pytest.mark.parametrize("entry", sorted(KERNELS))
def test_wpe_mpr_call_is_narrow(report, entry):
    """The portal refinement is called with 32-bit arguments only (its mangled signature is (int, int, int, int, float,
    int, int)): no 64-bit pointers to the tables, the slices or the hull vertices cross the call."""
    fns = report[entry]["functions"]
    assert MPR in fns, sorted(fns)
    _, st, ld = fns[MPR]
    assert st <= 8 and ld <= 20, (st, ld)   # 136 B of loads before
