"""Runs the REFERENCE's own ``mutate_xml`` (hsr/util.py:87-182) under stubbed ``gym`` / ``mujoco_py``
and writes a digest of the mutated MJCF trees (sha256 of their canonical form + the joints / actuators / block bodies
that survive the mutation) to tests/golden/mutate.json, the fixture tests/test_mutate_xml.py compares
hsr_env_b200.mjcf.mutate_tree with.  (The trees themselves are the reference's model files and are not copied here.)

    HSR_REFERENCE=<checkout of the reference> python tests/golden/make_mutate_golden.py
"""
import contextlib
import hashlib
import json
import importlib.util
import io
import os
import sys
import types
import xml.etree.ElementTree as ET
from pathlib import Path

import numpy as np

REF = Path(os.environ["HSR_REFERENCE"]) if os.environ.get("HSR_REFERENCE") else None   # the reference's repository
OUT = Path(__file__).resolve().parent / "mutate.json"

ALL_DOFS = ["slide_x", "slide_y", "arm_lift_joint", "arm_flex_joint", "wrist_roll_joint", "hand_l_proximal_joint", "hand_r_proximal_joint"]
# case -> (xml file, dofs, n_blocks, goal-space point(s) used for the block positions, --set-xml changes)
CASES = {
    "c1_readme": ("models/world.xml", ["slide_x", "slide_y"], 0, [(0, 0, 0)], []),
    "c1b_readme_block": ("models/world.xml", ["slide_x", "slide_y"], 1, [(0, 0, 0)], []),
    "c3_arm": ("models/world.xml", ALL_DOFS, 1, [(0.02, -0.05, 0.422)], []),
    "c5_clutter": ("models/world.xml", ["slide_x", "slide_y"], 4, [(-.1, -.1, .017), (-.1, .05, .017), (.05, -.1, .017), (.05, .05, .017)], []),
    "set_xml": ("models/world.xml", ["slide_x", "slide_y"], 1, [(0, 0, 0)],
                [('./worldbody/body[@name="goal"]/site[@name="goal"]/size', ".05 .05 .05"), ("./option/timestep", "0.004"),
                 ('./worldbody/body[@name="pan"]/geom/rgba', "1 0 0 1")]),
    "cupboard": ("models/cupboard-world.xml", ["slide_x", "slide_y"], 0, [(0, 0, 0)], []),
}


class SeqBox:
    """gym.spaces.Box stand-in whose sample() replays a given sequence (the reference draws block positions from it)."""

    def __init__(self, points):
        self.points, self.k = [np.asarray(p, float) for p in points], 0

    def sample(self):
        p = self.points[self.k % len(self.points)]
        self.k += 1
        return p


def load_reference_util():
    """hsr/util.py of the reference with its imports satisfied by stubs (gym, hsr.env, rl_utils are absent / unusable here)."""
    gym = types.ModuleType("gym")
    spaces = types.ModuleType("gym.spaces")

    class Box:   # noqa: D401
        def __init__(self, low, high, dtype=None):
            self.low, self.high = np.asarray(low), np.asarray(high)

    spaces.Box = Box
    gym.spaces = spaces
    env = types.ModuleType("hsr.env")
    env.get_xml_filepath = lambda p=Path("models/world.xml"): Path(REF / "hsr", p).absolute()
    from collections import namedtuple
    env.GoalSpec = namedtuple("GoalSpec", "a b distance")
    hsr = types.ModuleType("hsr")
    hsr.env = env
    rl = types.ModuleType("rl_utils")
    rl.parse_space = lambda dim: (lambda s: s)
    rl.parse_vector = lambda length, delim: (lambda s: s)
    saved = {k: sys.modules.get(k) for k in ("gym", "gym.spaces", "hsr", "hsr.env", "rl_utils")}
    sys.modules.update({"gym": gym, "gym.spaces": spaces, "hsr": hsr, "hsr.env": env, "rl_utils": rl})
    try:
        spec = importlib.util.spec_from_file_location("ref_hsr_util", REF / "hsr" / "util.py")
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod


def canonical(elem, drop=()):
    """Order-preserving, whitespace-free dump of an element tree; attributes sorted; `drop` = (tag, attribute) pairs the
    reference rewrites to machine-specific paths."""
    attrs = " ".join(f'{k}="{v}"' for k, v in sorted(elem.attrib.items()) if (elem.tag, k) not in drop)
    kids = "".join(canonical(c, drop) for c in elem)
    return f"<{elem.tag}{' ' + attrs if attrs else ''}>{kids}</{elem.tag}>\n"


DROP = (("include", "file"), ("compiler", "meshdir"))


def reference_mutation(mod, case):
    xml, dofs, n_blocks, points, changes = CASES[case]
    path = Path(REF / "hsr", xml).absolute()
    setters = [mod.XMLSetter(p, v) for p, v in changes]
    with contextlib.redirect_stdout(io.StringIO()):
        with mod.mutate_xml(changes=setters, dofs=dofs, goal_space=SeqBox(points), n_blocks=n_blocks, xml_filepath=path) as tmp:
            main = ET.parse(tmp)
            out = {"main": canonical(main.getroot(), DROP)}
            for k, inc in enumerate(main.findall("*/include")):
                out[f"include{k}"] = canonical(ET.parse(Path(tmp.parent, inc.get("file"))).getroot(), DROP)
    return out


def digest(trees):
    """sha256 of each canonical tree + what the mutation is about: surviving joints / actuators, added block bodies."""
    out = {k: hashlib.sha256(v.encode()).hexdigest() for k, v in trees.items()}
    roots = [ET.fromstring(v) for v in trees.values()]
    out["joints"] = [j.get("name") for r in roots for j in r.iter("joint")]
    out["actuators"] = [a.get("name") for r in roots for acts in r.iter("actuator") for a in acts]
    out["blocks"] = [(b.get("name"), b.get("pos")) for r in roots for b in r.iter("body") if (b.get("name") or "").startswith("block")]
    return out


def main():
    if REF is None:
        sys.exit("set HSR_REFERENCE to a checkout of the reference's repository")
    mod = load_reference_util()
    res = {case: digest(reference_mutation(mod, case)) for case in CASES}
    OUT.write_text(json.dumps(res, indent=1))
    for case, d in res.items():
        print(case, d["main"][:12], "joints", len(d["joints"]), "actuators", len(d["actuators"]), "blocks", len(d["blocks"]))


if __name__ == "__main__":
    main()
