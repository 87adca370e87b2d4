"""Golden fixture of the reference's own ReplayBuffer (rl_utils/replay_buffer.py, imported from a checkout of the
reference under a stubbed gym): a scripted sequence of extend / append / indexed reads, with everything the reference
returned.  The tests replay the script on the buffer, on the host and on the device, without the reference.

    HSR_REFERENCE=<checkout of the reference> python tests/golden/make_replay_golden.py   ->  tests/golden/replay.npz
"""
import importlib
import os
import sys
import types
from pathlib import Path

import numpy as np

if not os.environ.get("HSR_REFERENCE"):
    sys.exit("set HSR_REFERENCE to a checkout of the reference's repository")
REF = Path(os.environ["HSR_REFERENCE"])
gym = types.ModuleType("gym"); gym.spaces = types.ModuleType("gym.spaces")
gym.Env = object; gym.Space = object; gym.Wrapper = object
for n in ("Box", "Discrete", "Dict", "Tuple", "Space"):
    setattr(gym.spaces, n, type(n, (), {}))
sys.modules.setdefault("gym", gym); sys.modules.setdefault("gym.spaces", gym.spaces)
sys.path.insert(0, str(REF))
Ref = importlib.import_module("rl_utils.replay_buffer").ReplayBuffer

rng = np.random.default_rng(7)
ref = Ref(maxlen=64)
out = {}
sizes = [9, 25, 17, 40, 3, 31]          # wraps around the 64-slot ring several times
out["sizes"] = np.array(sizes)
for s, k in enumerate(sizes):
    b = [rng.normal(size=(k, 17)).astype(np.float32), rng.normal(size=(k, 2)).astype(np.float32), rng.normal(size=(k,)).astype(np.float32)]
    ref.extend(b)
    for j, a in enumerate(b):
        out[f"in{s}_{j}"] = a
    out[f"pos{s}"] = np.array([ref.pos, int(ref.full), len(ref)])
    for j, a in enumerate(ref.array()):
        out[f"all{s}_{j}"] = np.asarray(a)
    idx = rng.integers(-len(ref), 0, size=11)
    out[f"idx{s}"] = idx
    for j, a in enumerate(ref[idx].values):
        out[f"get{s}_{j}"] = np.asarray(a)
    win = np.array([np.arange(i, i + 5) for i in idx])
    for j, a in enumerate(ref[win].values):
        out[f"win{s}_{j}"] = np.asarray(a)
np.savez_compressed(Path(__file__).with_name("replay.npz"), **out)
print("wrote", Path(__file__).with_name("replay.npz"), len(out), "arrays")
