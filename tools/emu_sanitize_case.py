"""Driver of tools/emu_sanitize.sh: a few substeps of every fast-family kernel layout on the SIMT emulator (library given by
EMU_LIB, built with a sanitizer), on states with floor, hull and limit contacts.  With EMU_CAP=4 (libraries built with
PUSH_MAXCON=4 WPE_MAXCON=4, general kernel library EMU_LIB_G) the states are ones that overflow a capacity of 4 contacts,
and the general kernels run at (4 contacts, 26 rows) and (4, 12)."""
import ctypes
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests")); sys.path.insert(0, str(ROOT / "tests" / "simt_emu"))
import build as emu  # noqa: E402
from hsr_env_b200.model import Model  # noqa: E402

emu.LIB = Path(os.environ["EMU_LIB"])
emu.build = lambda force=False, defines=(): emu.LIB
g = np.load(ROOT / "tests" / "golden" / "c2_push.npz")
g1 = np.load(ROOT / "tests" / "golden" / "c1_readme.npz")
m2 = Model.load(ROOT / "hsr_env_b200" / "blobs" / "c2_push.hsrb")
m1 = Model.load(ROOT / "hsr_env_b200" / "blobs" / "c1_readme.hsrb")
if os.environ.get("EMU_CAP"):
    from oracle import port as P
    emu.LIB_G = Path(os.environ["EMU_LIB_G"])
    emu.build_general = lambda force=False: emu.LIB_G
    port = P.CpuPort(m2)
    port.set_caps(4, 26)
    x = [g[k] for k in ("qpos", "qvel", "warm", "ctrl")]
    ov = np.nonzero(port.step(*x, nsub=1)["flags"] & 1)[0]
    idx = np.r_[ov, 0, 1]
    xs = [a[idx] for a in x]
    for G, threads in ((1, 64), (8, 32), (16, 32), (32, 32)):
        out = emu.step(m2, *xs, nsub=3, G=G, threads=threads)
        print("c2_push cap 4 G", G, "envs", len(idx), "overflow", int((out["flags"] & 1).sum()), "stats", out["stats"][:6], flush=True)
    for caps in ((4, 26), (4, 12)):
        for G in (8, 0):
            out = emu.step_general(m2, *xs, nsub=3, G=G, ncon_max=caps[0], nefc_max=caps[1])
            print("c2_push general G", G, "caps", caps, "overflow", int((out["flags"] & 1).sum()), "stats", out["stats"][:6], flush=True)
    print("done")
    sys.exit(0)
sel = np.r_[np.nonzero(g["regime"] & 4)[0][:6], np.nonzero(g["regime"] & 1)[0][:4], 0, 1][:12]   # hull contacts, limits, plain
for name, model, fx, idx in (("c2_push", m2, g, sel), ("c1_readme", m1, g1, np.nonzero(g1["regime"])[0][:8])):
    for G, threads in ((1, 64), (8, 32), (16, 32), (32, 32)):
        out = emu.step(model, fx["qpos"][idx], fx["qvel"][idx], fx["warm"][idx], fx["ctrl"][idx], nsub=3, G=G, threads=threads)
        print(name, "G", G, "threads", threads, "envs", len(idx), "flags", np.unique(out["flags"]), "stats", out["stats"][:6], flush=True)
print("done")
