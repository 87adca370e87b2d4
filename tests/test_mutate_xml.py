"""hsr_env_b200.mjcf.mutate_tree == the reference's mutate_xml (hsr/util.py:87-182): same surviving joints
and actuators, same block bodies, same --set-xml edits, for the README model (C1), +1 block (C1b), the full arm (C3),
four blocks (C5), a --set-xml run and the cupboard scene.

The committed fixture tests/golden/mutate.json holds sha256 digests of the trees the REFERENCE'S OWN function produced
(tests/golden/make_mutate_golden.py runs it under a stubbed gym); where HSR_REFERENCE names a checkout of the reference,
it is also run live and the full canonical trees are compared.  The CLI line of the README then goes through
add_env_args / add_wrapper_args / hierarchical_parse_args / env_wrapper exactly as the reference's hsr/control.py:78-86
does.  The reference's model files are not carried here: the full-tree digests and the README model's blob need
HSR_ASSETS (its hsr/ directory).  The same cases always run on a small stand-in scene written for these tests
(tests/golden/mutate_scene: the reference's joint / actuator names and nesting, including joints every case drops), whose
surviving joints, actuators and block bodies must equal the reference's recorded ones in mutate.json."""
import hashlib
import json
import sys
import xml.etree.ElementTree as ET
from pathlib import Path

import numpy as np
import pytest

from conftest import GOLDEN

sys.path.insert(0, str(GOLDEN))
import make_mutate_golden as ref_side  # noqa: E402  (case table, canonical form, the stubbed import of the reference)

from hsr_env_b200 import mjcf  # noqa: E402

ASSETS = mjcf.default_assets_root()
STAND_IN = GOLDEN / "mutate_scene"
FIXTURE = json.loads((GOLDEN / "mutate.json").read_text())


def our_mutation(case, assets=ASSETS):
    """The same mutation with hsr_env_b200.mjcf: main file + its includes, each mutated as the reference does (util.py:171-175)."""
    xml, dofs, n_blocks, points, changes = ref_side.CASES[case]
    main, included = mjcf.load_trees(Path(assets, xml))
    setters = [mjcf.XMLSetter(p, v) for p, v in changes]
    block_pos = [points[i % len(points)] for i in range(n_blocks)]
    out = {}
    # the reference mutates the included files first, then the main file, drawing goal_space.sample() for every tree that
    # has a non-empty worldbody; only the main file has one
    for k, (name, tree) in enumerate(included.items()):
        mjcf.mutate_tree(tree, dofs, n_blocks, [np.asarray(p, float) for p in block_pos], setters)
        out[f"include{k}"] = ref_side.canonical(tree.getroot(), ref_side.DROP)
    mjcf.mutate_tree(main, dofs, n_blocks, [np.asarray(p, float) for p in block_pos], setters)
    out = {"main": ref_side.canonical(main.getroot(), ref_side.DROP), **out}
    return out


needs_assets = pytest.mark.skipif(ASSETS is None, reason="HSR assets (hsr/models) not found: set HSR_ASSETS")


@pytest.mark.parametrize("case", list(ref_side.CASES))
def test_mutate_tree_matches_reference_lists_on_stand_in(case):
    ours = our_mutation(case, STAND_IN)
    want = FIXTURE[case]
    got = ref_side.digest(ours)
    assert got["joints"] == want["joints"]
    assert got["actuators"] == want["actuators"]
    assert [list(b) for b in got["blocks"]] == [list(b) for b in want["blocks"]]
    main = ET.fromstring(ours["main"])
    for path, value in ref_side.CASES[case][4]:                  # --set-xml edits
        elt, attr = path.rsplit("/", 1)
        assert main.find(elt).get(attr) == value


@needs_assets
@pytest.mark.parametrize("case", list(ref_side.CASES))
def test_mutate_tree_matches_reference_digest(case):
    ours = our_mutation(case)
    want = FIXTURE[case]
    got = ref_side.digest(ours)
    assert got["joints"] == want["joints"]
    assert got["actuators"] == want["actuators"]
    assert [list(b) for b in got["blocks"]] == [list(b) for b in want["blocks"]]
    for k in ours:
        assert got[k] == want[k], f"{case}/{k}: mutated tree differs from the reference's"


@pytest.mark.skipif(ref_side.REF is None, reason="the reference's repository is not part of this one: set HSR_REFERENCE")
@pytest.mark.parametrize("case", list(ref_side.CASES))
def test_mutate_tree_matches_reference_live(case):
    mod = ref_side.load_reference_util()
    want = ref_side.reference_mutation(mod, case)
    ours = our_mutation(case)
    assert set(ours) == set(want)
    for k in want:
        assert ours[k] == want[k]
    for k in want:
        assert hashlib.sha256(want[k].encode()).hexdigest() == FIXTURE[case][k], "tests/golden/mutate.json is stale"


def readme_through_env_wrapper():
    """README.md:5 of the reference, parsed and wrapped as hsr/control.py:78-86 does: (parsed args, env_args the wrapped
    main received, the model it loaded)."""
    import argparse

    from hsr_env_b200 import util
    from hsr_env_b200.model import Model

    argv = ("--block-space (0,0)(0,0)(0,0)(0,0) --goal-space (0,0)(0,0)(0,0) --use-dof slide_x --use-dof slide_y "
            "--steps-per-action=300 --geofence=.5 --n-blocks 1").split()
    parser = argparse.ArgumentParser()
    wrapper_parser = parser.add_argument_group("wrapper_args")
    env_parser = parser.add_argument_group("env_args")
    util.add_env_args(env_parser)
    util.add_wrapper_args(wrapper_parser)
    args = util.hierarchical_parse_args(parser, argv=argv)
    seen = {}

    def main(env_args):
        seen.update(env_args)
        return Model.load(env_args["xml_file"]) if str(env_args["xml_file"]).endswith(".hsrb") else env_args["xml_file"]

    return args, seen, util.env_wrapper(main)(**args)


def test_readme_command_line_through_env_wrapper(monkeypatch):
    """The wrapped main receives env_args with the compiled model, goals=[GoalSpec(block_space, goal_space, geofence)] and
    starts={} (hsr/util.py:69-74); on the stand-in scene where the reference's model files are absent."""
    from hsr_env_b200.model import Model

    if ASSETS is None:
        monkeypatch.setenv("HSR_ASSETS", str(STAND_IN))
    args, seen, model = readme_through_env_wrapper()
    assert set(args) == {"wrapper_args", "env_args"}
    assert args["wrapper_args"]["use_dof"] == ["slide_x", "slide_y"] and args["wrapper_args"]["geofence"] == .5
    assert args["env_args"]["steps_per_action"] == 300
    assert seen["starts"] == {} and len(seen["goals"]) == 1
    g = seen["goals"][0]
    assert g.distance == .5 and g.a.shape == (4,) and g.b.shape == (3,)
    assert isinstance(model, Model) and (model.nq, model.nv, model.nu) == (9, 8, 2)      # SURVEY App. A.2: C1b
    assert model.names["joint"] == ["slide_x", "slide_y", "block0joint"]
    assert model.names["actuator"] == ["slide_x_motor", "slide_y_motor"]


@needs_assets
def test_readme_model_is_the_committed_blob():
    """The README model compiled from the reference's files is the model the committed blob holds: the GPU test of the
    single-environment facade (tests/test_gpu_parity.py::test_control_loop_through_the_single_env_facade) starts from
    that blob, because the reference's model files are not part of this repository."""
    from conftest import BLOBS
    from hsr_env_b200.model import Model

    model = readme_through_env_wrapper()[2]
    assert model.to_blob() == Model.load(BLOBS / "c1b_readme_block.hsrb").to_blob()
