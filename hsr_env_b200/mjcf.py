"""MJCF loader + model compiler for the HSR scenes.

Replaces, for the element/attribute subset the HSR models use, what the reference gets from
``mujoco_py.load_model_from_path`` (/root/reference/hsr/mujoco_env.py:33) after the temp-file
mutation done by ``mutate_xml`` (/root/reference/hsr/util.py:87-182):

* ``mutate_tree``   – the mutation semantics (append ``n_blocks`` free boxes, apply ``--set-xml`` edits,
                      drop every actuator / ``<joint>`` whose name is not in ``--use-dof``), applied to the
                      parsed trees in memory instead of temp files.
* ``compile_model`` – MuJoCo's compile rules for that subset (local coordinates, ``angle=degree``,
                      ``inertiafromgeom=true``, meshes -> convex hulls, contact filtering, parameter mixing,
                      ``qpos0``, ``invweight0``) -> ``model.Model``.

MuJoCo itself is not available (SURVEY.md §8c), so every version-dependent choice is a named option
(``CompileOptions``) and the result is a plain blob that a dump from a real MuJoCo could replace.
The asset directory (``hsr/models``, ``hsr/hsr_meshes``) is *read* from the reference checkout at compile
time only; runtime code consumes the pre-compiled blobs in ``hsr_env_b200/blobs``.
"""
from __future__ import annotations

import copy
import os
import re
import struct
import xml.etree.ElementTree as ET
from dataclasses import dataclass, field
from pathlib import Path
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import model as M

MJMINVAL = 1e-15


# ----------------------------------------------------------------------------- small math helpers
def quat_mul(a, b):
    aw, ax, ay, az = a
    bw, bx, by, bz = b
    return np.array([
        aw * bw - ax * bx - ay * by - az * bz,
        aw * bx + ax * bw + ay * bz - az * by,
        aw * by - ax * bz + ay * bw + az * bx,
        aw * bz + ax * by - ay * bx + az * bw,
    ])


def quat_to_mat(q):
    w, x, y, z = q
    return np.array([
        [w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y)],
        [2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x)],
        [2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z],
    ])


def quat_normalize(q):
    q = np.asarray(q, float)
    n = np.linalg.norm(q)
    if n < MJMINVAL:
        return np.array([1.0, 0, 0, 0])
    return q / n


def _floats(s: Optional[str], n: Optional[int] = None, default=None):
    """Tolerant float-vector parser (hsr.mjcf:13 has ``pos="0 0hsr"`` -> treated as zeros, SURVEY A.1)."""
    if s is None:
        return None if default is None else np.array(default, float)
    out = []
    for tok in s.split():
        try:
            out.append(float(tok))
        except ValueError:
            m = re.match(r"[-+]?(\d+\.?\d*|\.\d+)([eE][-+]?\d+)?", tok)
            out.append(float(m.group(0)) if m else 0.0)
    if n is not None:
        out = (out + [0.0] * n)[:n]
    return np.array(out, float)


# ----------------------------------------------------------------------------- options
@dataclass
class CompileOptions:
    """Version-dependent compile choices (SURVEY.md App. B.9)."""
    mesh_inertia: str = "legacy"  # legacy | exact | convex   (App. A.5)
    solimp_params: int = 5  # 5-parameter impedance (MuJoCo >= 2.0); 3 pads to a linear ramp
    prune_static_pairs: bool = True  # drop candidate pairs that joint ranges make unreachable (same contacts, less work)
    block_quat_index: Tuple[int, int] = (0, 2)  # which free-joint quaternion comps block-space drives
    # (hsr/__init__.py:15-17 varies q1 and q3 of [x y z q1 q2 q3 q4]  ->  indices 0 and 2)


@dataclass
class XMLSetter:
    path: str
    value: str


# ----------------------------------------------------------------------------- XML loading + mutation
def load_trees(xml_path: Path):
    """Parse the main file and every ``<include>`` it references (one level, as the reference does)."""
    xml_path = Path(xml_path)
    main = ET.parse(xml_path)
    included = {}
    for inc in main.findall("*/include"):
        p = Path(xml_path.parent, inc.get("file"))
        included[inc.get("file")] = ET.parse(p)
    return main, included


def mutate_tree(tree: ET.ElementTree, dofs: Sequence[str], n_blocks: int, block_pos: Sequence[Sequence[float]],
                changes: Sequence[XMLSetter]):
    """In-memory restatement of ``mutate_tree`` in /root/reference/hsr/util.py:91-159.

    ``block_pos[i]`` plays the role of ``goal_space.sample()`` at util.py:108 (the caller draws it).
    """
    worldbody = tree.getroot().find("./worldbody")
    rgba = ["0 1 0 1", "0 0 1 1", "0 1 1 1", "1 0 0 1", "1 0 1 1", "1 1 0 1", "1 1 1 1"]
    if worldbody is not None and len(worldbody):  # reference relies on Element truthiness (util.py:106)
        for i in range(n_blocks):
            pos = " ".join(map(str, block_pos[i]))
            name = f"block{i}"
            body = ET.SubElement(worldbody, "body", attrib=dict(name=name, pos=pos))
            ET.SubElement(body, "geom", attrib=dict(
                name=name, type="box", mass="1", size=".05 .025 .017", rgba=rgba[i % len(rgba)], condim="6",
                solimp="0.99 0.99 0.01", solref="0.01 1"))
            ET.SubElement(body, "freejoint", attrib=dict(name=f"block{i}joint"))
    for change in changes:
        parent = re.sub("/[^/]*$", "", change.path)
        elt = tree.find(parent)
        if isinstance(elt, ET.Element):
            name = re.search("[^/]*$", change.path)[0]
            elt.set(name, change.value)
    for actuators in tree.iter("actuator"):
        for actuator in list(actuators):
            if actuator.get("joint") not in dofs:
                actuators.remove(actuator)
    for body in tree.iter("body"):
        for joint in body.findall("joint"):
            if joint.get("name") not in dofs:
                body.remove(joint)
    return tree


def expand_includes(main: ET.ElementTree, included: Dict[str, ET.ElementTree]) -> ET.Element:
    root = copy.deepcopy(main.getroot())
    for parent in root.iter():
        for idx, child in enumerate(list(parent)):
            if child.tag == "include":
                inc_root = included[child.get("file")].getroot()
                pos = list(parent).index(child)
                parent.remove(child)
                for k, sub in enumerate(list(inc_root)):
                    parent.insert(pos + k, copy.deepcopy(sub))
    return root


# ----------------------------------------------------------------------------- meshes
def read_stl(path: Path):
    data = Path(path).read_bytes()
    if data[:5] == b"solid" and b"facet" in data[:512]:
        raise ValueError(f"{path}: ASCII STL not supported (all HSR meshes are binary)")
    (ntri,) = struct.unpack_from("<I", data, 80)
    rec = np.frombuffer(data, dtype=np.dtype([("n", "<f4", 3), ("v", "<f4", (3, 3)), ("a", "<u2")]), count=ntri,
                        offset=84)
    tri = rec["v"].astype(np.float64)  # (ntri,3,3)
    verts, inv = np.unique(tri.reshape(-1, 3), axis=0, return_inverse=True)
    faces = inv.reshape(-1, 3)
    return verts, faces


def _tet_props(a, b, c, d):
    """volume (signed), centroid and second-moment (covariance integral about origin) of tetra (a,b,c,d)."""
    vol = np.dot(np.cross(b - a, c - a), d - a) / 6.0
    cen = (a + b + c + d) / 4.0
    # integral of x x^T over the tetra = vol/20 * (sum_i v_i v_i^T + (sum v)(sum v)^T)
    s = a + b + c + d
    P = (np.outer(a, a) + np.outer(b, b) + np.outer(c, c) + np.outer(d, d) + np.outer(s, s)) * (vol / 20.0)
    return vol, cen, P


def mesh_mass_props(verts, faces, mode: str):
    """(volume, com, inertia-per-unit-density about com) of a triangle mesh.

    ``legacy``: pyramids from the surface centroid with |volume| (MuJoCo <= 2.1 behaviour, exact only for
    convex meshes); ``exact``: signed tetrahedra; ``convex``: exact on the convex hull.  SURVEY.md A.5.
    """
    if mode == "convex":
        from scipy.spatial import ConvexHull
        hull = ConvexHull(verts)
        faces = hull.simplices.copy()
        cen = verts[hull.vertices].mean(0)
        for k, f in enumerate(faces):  # orient outward
            n = np.cross(verts[f[1]] - verts[f[0]], verts[f[2]] - verts[f[0]])
            if np.dot(n, verts[f[0]] - cen) < 0:
                faces[k] = f[::-1]
        mode = "exact"
    tri = verts[faces]
    area = 0.5 * np.linalg.norm(np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]), axis=1)
    fcen = tri.mean(1)
    apex = (fcen * area[:, None]).sum(0) / max(area.sum(), MJMINVAL)
    vol = 0.0
    com = np.zeros(3)
    P = np.zeros((3, 3))
    for t in tri:
        v, c, p = _tet_props(apex, t[0], t[1], t[2])
        if mode == "legacy" and v < 0:
            v, p = -v, -p
        vol += v
        com += v * c
        P += p
    com = com / vol
    # P is the second moment about the origin; shift to com, convert to inertia tensor
    Pc = P - vol * np.outer(com, com)
    I = np.trace(Pc) * np.eye(3) - Pc
    return vol, com, I


def convex_hull_vertices(verts):
    from scipy.spatial import ConvexHull
    hull = ConvexHull(verts)
    return verts[np.sort(hull.vertices)]


# ----------------------------------------------------------------------------- parsed (un-fused) tree
@dataclass
class _Geom:
    name: str
    type: int
    pos: np.ndarray
    quat: np.ndarray
    size: np.ndarray
    mesh: Optional[str]
    contype: int
    conaffinity: int
    condim: int
    friction: np.ndarray
    solref: np.ndarray
    solimp: np.ndarray
    solmix: float
    mass: Optional[float]
    density: float
    group: int


@dataclass
class _Joint:
    name: str
    type: int
    pos: np.ndarray
    axis: np.ndarray
    limited: bool
    range: np.ndarray
    damping: float
    solref: np.ndarray
    solimp: np.ndarray


@dataclass
class _Body:
    name: str
    parent: int
    pos: np.ndarray
    quat: np.ndarray
    mocap: bool
    joints: List[_Joint] = field(default_factory=list)
    geoms: List[_Geom] = field(default_factory=list)
    inertial: Optional[dict] = None
    # compile products
    mass: float = 0.0
    ipos: np.ndarray = field(default_factory=lambda: np.zeros(3))
    inertia: np.ndarray = field(default_factory=lambda: np.zeros((3, 3)))
    weld: int = 0


_GEOM_TYPES = {"plane": M.GEOM_PLANE, "cylinder": M.GEOM_CYLINDER, "box": M.GEOM_BOX, "mesh": M.GEOM_MESH,
               "sphere": 2}
_DEF_SOLREF = np.array([0.02, 1.0])
_DEF_SOLIMP = np.array([0.9, 0.95, 0.001, 0.5, 2.0])


def _solimp(s, opts: CompileOptions):
    v = _floats(s)
    if v is None:
        return _DEF_SOLIMP.copy()
    out = _DEF_SOLIMP.copy()
    out[:min(len(v), 5)] = v[:5]
    if opts.solimp_params == 3:
        out[3:] = (0.5, 1.0)
    return out


def _collect_defaults(root):
    """class name -> {tag -> attrib}.  Nested classes inherit from their parent class."""
    table: Dict[str, Dict[str, dict]] = {}

    def visit(elt, inherited):
        cur = {k: dict(v) for k, v in inherited.items()}
        for child in elt:
            if child.tag != "default":
                cur.setdefault(child.tag, {}).update(child.attrib)
        table[elt.get("class", "main")] = cur
        for child in elt:
            if child.tag == "default":
                visit(child, cur)

    for d in root.findall("default"):
        # a second top-level <default class="all"> (world.xml:35-37) is accepted; nothing references it
        visit(d, {} if d.get("class") else table.get("main", {}))
    return table


def _parse_tree(root, opts: CompileOptions):
    compiler = {}
    for c in root.findall("compiler"):
        compiler.update(c.attrib)
    degree = compiler.get("angle", "degree") == "degree"
    option = {}
    for o in root.findall("option"):
        option.update(o.attrib)
    defaults = _collect_defaults(root)

    def with_defaults(elt):
        cls = elt.get("class")
        base = dict(defaults.get("main", {}).get(elt.tag, {}))
        if cls and cls in defaults:
            base.update(defaults[cls].get(elt.tag, {}))
        base.update(elt.attrib)
        return base

    bodies: List[_Body] = [_Body("world", -1, np.zeros(3), np.array([1.0, 0, 0, 0]), False)]

    def parse_geom(e, body_name, k):
        a = with_defaults(e)
        gtype = _GEOM_TYPES[a.get("type", "sphere")]
        fr = _floats(a.get("friction"), default=[1.0, 0.005, 0.0001])
        fr = np.concatenate([fr, [1.0, 0.005, 0.0001][len(fr):]])
        return _Geom(
            name=a.get("name", f"{body_name}_geom{k}"), type=gtype,
            pos=_floats(a.get("pos"), 3, [0, 0, 0]), quat=quat_normalize(_floats(a.get("quat"), 4, [1, 0, 0, 0])),
            size=_floats(a.get("size"), 3, [0, 0, 0]), mesh=a.get("mesh"),
            contype=int(a.get("contype", 1)), conaffinity=int(a.get("conaffinity", 1)),
            condim=int(a.get("condim", 3)), friction=fr,
            solref=_floats(a.get("solref"), 2, _DEF_SOLREF), solimp=_solimp(a.get("solimp"), opts),
            solmix=float(a.get("solmix", 1.0)), mass=float(a["mass"]) if "mass" in a else None,
            density=float(a.get("density", 1000.0)), group=int(a.get("group", 0)))

    def parse_joint(e):
        if e.tag == "freejoint":
            return _Joint(e.get("name", ""), M.JNT_FREE, np.zeros(3), np.array([0, 0, 1.0]), False, np.zeros(2), 0.0,
                          _DEF_SOLREF.copy(), _DEF_SOLIMP.copy())
        a = with_defaults(e)
        jt = {"slide": M.JNT_SLIDE, "hinge": M.JNT_HINGE, "free": M.JNT_FREE}[a.get("type", "hinge")]
        rng = _floats(a.get("range"), 2, [0, 0])
        if jt == M.JNT_HINGE and degree:
            rng = np.deg2rad(rng)
        axis = _floats(a.get("axis"), 3, [0, 0, 1])
        axis = axis / np.linalg.norm(axis)
        return _Joint(a.get("name", ""), jt, _floats(a.get("pos"), 3, [0, 0, 0]), axis,
                      a.get("limited", "false") == "true", rng, float(a.get("damping", 0.0)),
                      _floats(a.get("solreflimit"), 2, _DEF_SOLREF), _solimp(a.get("solimplimit"), opts))

    def visit(elt, parent_id):
        for child in elt:
            if child.tag == "body":
                b = _Body(child.get("name", f"body{len(bodies)}"), parent_id, _floats(child.get("pos"), 3, [0, 0, 0]),
                          quat_normalize(_floats(child.get("quat"), 4, [1, 0, 0, 0])),
                          child.get("mocap", "false") == "true")
                bid = len(bodies)
                bodies.append(b)
                for k, sub in enumerate(child):
                    if sub.tag in ("joint", "freejoint"):
                        b.joints.append(parse_joint(sub))
                    elif sub.tag == "geom":
                        b.geoms.append(parse_geom(sub, b.name, k))
                    elif sub.tag == "inertial":
                        b.inertial = dict(pos=_floats(sub.get("pos"), 3, [0, 0, 0]),
                                          quat=quat_normalize(_floats(sub.get("quat"), 4, [1, 0, 0, 0])),
                                          mass=float(sub.get("mass")),
                                          diag=_floats(sub.get("diaginertia"), 3, [0, 0, 0]))
                visit(child, bid)
            elif child.tag == "geom" and parent_id == 0 and elt.tag == "worldbody":
                bodies[0].geoms.append(parse_geom(child, "world", len(bodies[0].geoms)))

    wb = root.find("worldbody")
    visit(wb, 0)
    meshes = {m.get("name"): m.get("file") for m in root.findall("asset/mesh")}
    actuators = []
    for act in root.findall("actuator/position"):
        a = dict(act.attrib)
        actuators.append(dict(
            name=a.get("name"), joint=a["joint"], gear=_floats(a.get("gear"), 1, [1.0])[0], kp=float(a.get("kp", 1)),
            ctrllimited=a.get("ctrllimited", "false") == "true", ctrlrange=_floats(a.get("ctrlrange"), 2, [0, 0]),
            forcelimited=a.get("forcelimited", "false") == "true", forcerange=_floats(a.get("forcerange"), 2, [0, 0])))
    excludes = [(e.get("body1"), e.get("body2")) for e in root.findall("contact/exclude")]
    return bodies, meshes, actuators, excludes, compiler, option


# ----------------------------------------------------------------------------- inertia of primitives
def _geom_mass_props(g: _Geom, mesh_cache, opts):
    """mass, com (geom frame offset in body frame), inertia about com in body frame."""
    R = quat_to_mat(g.quat)
    if g.type == M.GEOM_BOX:
        a, b, c = g.size
        vol = 8 * a * b * c
        I = np.diag([b * b + c * c, a * a + c * c, a * a + b * b]) * vol / 3.0
        com = np.zeros(3)
    elif g.type == M.GEOM_CYLINDER:
        r, h = g.size[0], g.size[1]
        vol = np.pi * r * r * 2 * h
        I = np.diag([(3 * r * r + 4 * h * h) / 12.0] * 2 + [r * r / 2.0]) * vol
        com = np.zeros(3)
    elif g.type == 2:  # sphere
        r = g.size[0]
        vol = 4.0 / 3.0 * np.pi * r ** 3
        I = np.eye(3) * 0.4 * r * r * vol
        com = np.zeros(3)
    elif g.type == M.GEOM_MESH:
        vol, com, I = mesh_cache[g.mesh]["props"]
    else:
        return 0.0, np.zeros(3), np.zeros((3, 3))
    mass = g.mass if g.mass is not None else g.density * vol
    I = I * (mass / vol)
    return mass, g.pos + R @ com, R @ I @ R.T


def _combine(parts):
    """parts: list of (mass, com, I_about_com) in one frame -> combined (mass, com, I)."""
    mass = sum(p[0] for p in parts)
    if mass <= 0:
        return 0.0, np.zeros(3), np.zeros((3, 3))
    com = sum(p[0] * p[1] for p in parts) / mass
    I = np.zeros((3, 3))
    for m_, c, Ic in parts:
        d = c - com
        I += Ic + m_ * (np.dot(d, d) * np.eye(3) - np.outer(d, d))
    return mass, com, I


# ----------------------------------------------------------------------------- compile
def compile_model(xml_path: Path, use_dof: Sequence[str], n_blocks: int = 0,
                  block_pos: Optional[Sequence[Sequence[float]]] = None, set_xml: Sequence[XMLSetter] = (),
                  opts: Optional[CompileOptions] = None, block_name: str = "block") -> M.Model:
    opts = opts or CompileOptions()
    xml_path = Path(xml_path)
    if block_pos is None:
        block_pos = [(0.0, 0.0, 0.0)] * n_blocks
    main, included = load_trees(xml_path)
    for t in [main] + list(included.values()):
        mutate_tree(t, use_dof, n_blocks, block_pos, list(set_xml))
    root = expand_includes(main, included)
    bodies, meshes, actuators, excludes, compiler, option = _parse_tree(root, opts)
    meshdir = Path(xml_path.parent, compiler.get("meshdir", "."))

    # ---- meshes: hulls + mass properties (only those referenced by geoms)
    mesh_cache = {}
    for b in bodies:
        for g in b.geoms:
            if g.type == M.GEOM_MESH and g.mesh not in mesh_cache:
                verts, faces = read_stl(meshdir / meshes[g.mesh])
                mesh_cache[g.mesh] = dict(verts=verts, faces=faces,
                                          props=mesh_mass_props(verts, faces, opts.mesh_inertia), hull=None)

    # ---- per original body inertia (inertiafromgeom=true: geoms override <inertial> where geoms exist)
    from_geom = compiler.get("inertiafromgeom", "auto")
    for b in bodies[1:]:
        parts = [_geom_mass_props(g, mesh_cache, opts) for g in b.geoms]
        parts = [p for p in parts if p[0] > 0]
        use_geoms = bool(parts) and (from_geom == "true" or (from_geom == "auto" and b.inertial is None))
        if use_geoms:
            b.mass, b.ipos, b.inertia = _combine(parts)
        elif b.inertial is not None:
            R = quat_to_mat(b.inertial["quat"])
            b.mass, b.ipos, b.inertia = b.inertial["mass"], b.inertial["pos"], R @ np.diag(b.inertial["diag"]) @ R.T

    # ---- weld groups and fused bodies
    fused_of = {0: 0}
    fused_ids = [0]
    for i, b in enumerate(bodies):
        if i == 0:
            continue
        if b.joints:
            b.weld = i
            fused_of[i] = len(fused_ids)
            fused_ids.append(i)
        else:
            b.weld = bodies[b.parent].weld
    nbody = len(fused_ids)
    # transform of every original body relative to its weld root
    rel_pos = [np.zeros(3) for _ in bodies]
    rel_quat = [np.array([1.0, 0, 0, 0]) for _ in bodies]
    for i, b in enumerate(bodies):
        if i == 0 or b.weld == i:
            continue
        p = b.parent
        rel_pos[i] = rel_pos[p] + quat_to_mat(rel_quat[p]) @ b.pos
        rel_quat[i] = quat_mul(rel_quat[p], b.quat)

    arr: Dict[str, np.ndarray] = {}
    body_parent = np.zeros(nbody, np.int32)
    body_pos = np.zeros((nbody, 3))
    body_quat = np.tile(np.array([1.0, 0, 0, 0]), (nbody, 1))
    body_mass = np.zeros(nbody)
    body_ipos = np.zeros((nbody, 3))
    body_inertia = np.zeros((nbody, 6))
    for f, i in enumerate(fused_ids):
        if f == 0:
            body_parent[f] = -1
            continue
        b = bodies[i]
        p = b.parent
        body_parent[f] = fused_of[bodies[p].weld]
        body_pos[f] = rel_pos[p] + quat_to_mat(rel_quat[p]) @ b.pos
        body_quat[f] = quat_mul(rel_quat[p], b.quat)
        parts = []
        for j, ob in enumerate(bodies):
            if j and ob.weld == i and ob.mass > 0:
                R = quat_to_mat(rel_quat[j])
                parts.append((ob.mass, rel_pos[j] + R @ ob.ipos, R @ ob.inertia @ R.T))
        m_, c_, I_ = _combine(parts)
        body_mass[f], body_ipos[f] = m_, c_
        body_inertia[f] = [I_[0, 0], I_[1, 1], I_[2, 2], I_[0, 1], I_[0, 2], I_[1, 2]]

    # ---- joints / dofs / qpos0
    jt, jb, jq, jd, jax, jpos, jlim, jrng, jsr, jsi = [], [], [], [], [], [], [], [], [], []
    dof_body, dof_parent, dof_jnt, dof_damp = [], [], [], []
    qpos0: List[float] = []
    body_jntadr = np.zeros(nbody, np.int32)
    body_jntnum = np.zeros(nbody, np.int32)
    body_dofadr = np.zeros(nbody, np.int32)
    body_dofnum = np.zeros(nbody, np.int32)
    jnt_names = []
    last_dof_of_body = {0: -1}
    for f, i in enumerate(fused_ids):
        if f == 0:
            continue
        b = bodies[i]
        body_jntadr[f] = len(jt)
        body_jntnum[f] = len(b.joints)
        body_dofadr[f] = len(dof_body)
        prev = last_dof_of_body[int(body_parent[f])]
        for j in b.joints:
            jnt_names.append(j.name)
            jt.append(j.type); jb.append(f); jq.append(len(qpos0)); jd.append(len(dof_body))
            jax.append(j.axis); jpos.append(j.pos); jlim.append(int(j.limited)); jrng.append(j.range)
            jsr.append(j.solref); jsi.append(j.solimp)
            nd = 6 if j.type == M.JNT_FREE else 1
            for k in range(nd):
                dof_body.append(f); dof_parent.append(prev); dof_jnt.append(len(jt) - 1); dof_damp.append(j.damping)
                prev = len(dof_body) - 1
            if j.type == M.JNT_FREE:
                qpos0 += list(body_pos[f]) + list(body_quat[f])
            else:
                qpos0.append(0.0)
        body_dofnum[f] = len(dof_body) - body_dofadr[f]
        last_dof_of_body[f] = prev
    nq, nv, njnt = len(qpos0), len(dof_body), len(jt)

    def A(x, dt, shape):
        return np.asarray(x, dt).reshape(shape)

    arr.update(
        qpos0=A(qpos0, float, (nq,)), body_parent=body_parent, body_pos=body_pos, body_quat=body_quat,
        body_mass=body_mass, body_ipos=body_ipos, body_inertia=body_inertia, body_jntadr=body_jntadr,
        body_jntnum=body_jntnum, body_dofadr=body_dofadr, body_dofnum=body_dofnum,
        jnt_type=A(jt, np.int32, (njnt,)), jnt_body=A(jb, np.int32, (njnt,)), jnt_qposadr=A(jq, np.int32, (njnt,)),
        jnt_dofadr=A(jd, np.int32, (njnt,)), jnt_axis=A(jax, float, (njnt, 3)), jnt_pos=A(jpos, float, (njnt, 3)),
        jnt_limited=A(jlim, np.int32, (njnt,)), jnt_range=A(jrng, float, (njnt, 2)),
        jnt_solref=A(jsr, float, (njnt, 2)), jnt_solimp=A(jsi, float, (njnt, 5)),
        dof_body=A(dof_body, np.int32, (nv,)), dof_parent=A(dof_parent, np.int32, (nv,)),
        dof_jnt=A(dof_jnt, np.int32, (nv,)), dof_damping=A(dof_damp, float, (nv,)))

    # ---- actuators
    nu = len(actuators)
    act_dof = np.zeros(nu, np.int32); act_q = np.zeros(nu, np.int32)
    for k, a in enumerate(actuators):
        jid = jnt_names.index(a["joint"])
        act_dof[k], act_q[k] = jd[jid], jq[jid]
    arr.update(
        act_dof=act_dof, act_qposadr=act_q, act_gear=A([a["gear"] for a in actuators], float, (nu,)),
        act_kp=A([a["kp"] for a in actuators], float, (nu,)),
        act_ctrllimited=A([a["ctrllimited"] for a in actuators], np.int32, (nu,)),
        act_ctrlrange=A([a["ctrlrange"] for a in actuators], float, (nu, 2)),
        act_forcelimited=A([a["forcelimited"] for a in actuators], np.int32, (nu,)),
        act_forcerange=A([a["forcerange"] for a in actuators], float, (nu, 2)))

    # ---- colliding geoms, in fused-body frames
    geoms = []  # (orig body id, _Geom, pos, mat, verts-or-None)
    for i, b in enumerate(bodies):
        for g in b.geoms:
            if g.contype == 0 and g.conaffinity == 0:
                continue
            Rb = quat_to_mat(rel_quat[i])
            Rg = Rb @ quat_to_mat(g.quat)
            pg = rel_pos[i] + Rb @ g.pos
            verts = None
            if g.type == M.GEOM_MESH:
                mc = mesh_cache[g.mesh]
                if mc["hull"] is None:
                    mc["hull"] = convex_hull_vertices(mc["verts"])
                com = mc["props"][1]
                verts = mc["hull"] - com  # geom frame is centred at the mesh CoM (MuJoCo recentres meshes)
                pg = pg + Rg @ com
            geoms.append((i, g, pg, Rg, verts))
    ngeom = len(geoms)
    geom_type = np.array([g.type for _, g, *_ in geoms], np.int32)
    geom_body = np.array([fused_of[bodies[i].weld] for i, *_ in geoms], np.int32)
    geom_pos = np.array([p for *_, p, _, _ in geoms]).reshape(ngeom, 3)
    geom_mat = np.array([Rg.reshape(9) for *_, Rg, _ in geoms]).reshape(ngeom, 9)
    geom_size = np.array([g.size for _, g, *_ in geoms]).reshape(ngeom, 3)
    geom_rbound = np.zeros(ngeom); geom_aabb = np.zeros((ngeom, 3))
    vertadr = np.zeros(ngeom, np.int32); vertnum = np.zeros(ngeom, np.int32)
    hull_chunks = []
    nvert = 0
    for k, (_, g, _, _, verts) in enumerate(geoms):
        if g.type == M.GEOM_MESH:
            vertadr[k], vertnum[k] = nvert, len(verts)
            hull_chunks.append(verts); nvert += len(verts)
            geom_rbound[k] = np.linalg.norm(verts, axis=1).max()
            geom_aabb[k] = np.abs(verts).max(0)
        elif g.type == M.GEOM_BOX:
            geom_rbound[k] = np.linalg.norm(g.size); geom_aabb[k] = g.size
        elif g.type == M.GEOM_CYLINDER:
            geom_rbound[k] = np.hypot(g.size[0], g.size[1]); geom_aabb[k] = [g.size[0], g.size[0], g.size[1]]
        elif g.type == M.GEOM_PLANE:
            geom_rbound[k] = 0.0
        else:
            raise NotImplementedError(f"colliding geom type {g.type} ({g.name}) is outside the HSR subset")
    hull_vert = np.concatenate(hull_chunks).reshape(-1, 3) if hull_chunks else np.zeros((0, 3))

    # ---- options
    opt = np.zeros(16)
    opt[0] = float(option.get("timestep", 0.002))
    opt[1:4] = _floats(option.get("gravity"), 3, [0, 0, -9.81])
    opt[4] = float(option.get("impratio", 1.0))
    opt[5] = float(option.get("tolerance", 1e-8))
    opt[6] = float(option.get("ls_tolerance", 0.01))
    opt[7] = float(option.get("iterations", 100))
    opt[8] = float(option.get("ls_iterations", 50))
    opt[9] = float(option.get("mpr_tolerance", 1e-6))
    opt[10] = float(option.get("mpr_iterations", 50))
    if option.get("cone", "pyramidal") != "elliptic":
        raise NotImplementedError("only cone=elliptic (world.xml:38) is implemented")
    arr.update(opt=opt, geom_type=geom_type, geom_body=geom_body, geom_pos=geom_pos, geom_mat=geom_mat,
               geom_size=geom_size, geom_rbound=geom_rbound, geom_aabb=geom_aabb, geom_vertadr=vertadr,
               geom_vertnum=vertnum, hull_vert=hull_vert)

    # ---- mass matrix at qpos0 on the fused tree -> invweights, meaninertia
    kin = kinematics(arr, nbody, np.asarray(qpos0, float))
    Mq = np.zeros((nv, nv))
    for f in range(1, nbody):
        Jp, Jr = jacobian(arr, kin, f, kin["xipos"][f])
        Iw = kin["xmat"][f] @ _sym6(body_inertia[f]) @ kin["xmat"][f].T
        Mq += body_mass[f] * Jp.T @ Jp + Jr.T @ Iw @ Jr
    Minv = np.linalg.inv(Mq) if nv else np.zeros((0, 0))
    dof_invweight0 = np.zeros(nv)
    for j in range(njnt):
        d0 = jd[j]
        if jt[j] == M.JNT_FREE:
            dof_invweight0[d0:d0 + 3] = np.mean(np.diag(Minv)[d0:d0 + 3])
            dof_invweight0[d0 + 3:d0 + 6] = np.mean(np.diag(Minv)[d0 + 3:d0 + 6])
        else:
            dof_invweight0[d0] = Minv[d0, d0]
    opt[11] = float(np.mean(np.diag(Mq))) if nv else 1.0
    # body_invweight0 (translational part) of every ORIGINAL body, evaluated at its own CoM
    orig_invweight = np.zeros(len(bodies))
    for i, b in enumerate(bodies):
        f = fused_of[b.weld]
        if f == 0:
            continue
        p_local = rel_pos[i] + quat_to_mat(rel_quat[i]) @ b.ipos
        pw = kin["xpos"][f] + kin["xmat"][f] @ p_local
        Jp, Jr = jacobian(arr, kin, f, pw)
        Aj = Jp @ Minv @ Jp.T
        orig_invweight[i] = np.trace(Aj) / 3.0
    geom_invweight = np.array([orig_invweight[i] for i, *_ in geoms]).reshape(ngeom)
    arr.update(dof_invweight0=dof_invweight0, geom_invweight=geom_invweight)

    # ---- static candidate pair list (collision filtering on the original tree)
    name_to_id = {b.name: i for i, b in enumerate(bodies)}
    excl = set()
    for b1, b2 in excludes:
        if b1 in name_to_id and b2 in name_to_id:
            i1, i2 = name_to_id[b1], name_to_id[b2]
            excl.add((min(i1, i2), max(i1, i2)))
    weldparent = {i: (bodies[bodies[b.weld].parent].weld if b.weld else 0) for i, b in enumerate(bodies)}
    mdl_info_prune = {}
    pairs = []
    for a in range(ngeom):
        for c in range(a + 1, ngeom):
            (i1, g1, *_), (i2, g2, *_) = geoms[a], geoms[c]
            if i1 == i2:
                continue
            w1, w2 = bodies[i1].weld, bodies[i2].weld
            if w1 == w2:
                continue
            if w1 != 0 and w2 != 0 and (w1 == weldparent[i2] or w2 == weldparent[i1]):
                continue
            if not ((g1.contype & g2.conaffinity) or (g2.contype & g1.conaffinity)):
                continue
            if (min(i1, i2), max(i1, i2)) in excl:
                continue
            ga, gb = (a, c) if g1.type <= g2.type else (c, a)
            ta, tb = geoms[ga][1].type, geoms[gb][1].type
            if ta == M.GEOM_PLANE and tb == M.GEOM_PLANE:
                continue
            if ta == M.GEOM_PLANE:
                func = M.NP_PLANE_BOX if tb == M.GEOM_BOX else M.NP_PLANE_CONVEX
            elif ta == M.GEOM_BOX and tb == M.GEOM_BOX:
                func = M.NP_BOX_BOX
            else:
                func = M.NP_CONVEX_CONVEX
            x, y = geoms[ga][1], geoms[gb][1]
            mix = x.solmix / (x.solmix + y.solmix)
            fr = np.maximum(x.friction, y.friction)
            pairs.append(dict(g1=ga, g2=gb, func=func, condim=max(x.condim, y.condim),
                              friction=[fr[0], fr[0], fr[1], fr[2], fr[2]],
                              solref=mix * x.solref + (1 - mix) * y.solref,
                              solimp=mix * x.solimp + (1 - mix) * y.solimp))
    if opts.prune_static_pairs:
        pairs = _prune_unreachable_pairs(pairs, arr, kin, nbody, geom_body, geom_type, geom_pos, geom_mat, geom_size,
                                         vertadr, vertnum, hull_vert, mesh_info=mdl_info_prune)
    npair = len(pairs)
    arr.update(
        pair_geom1=A([p["g1"] for p in pairs], np.int32, (npair,)),
        pair_geom2=A([p["g2"] for p in pairs], np.int32, (npair,)),
        pair_func=A([p["func"] for p in pairs], np.int32, (npair,)),
        pair_condim=A([p["condim"] for p in pairs], np.int32, (npair,)),
        pair_friction=A([p["friction"] for p in pairs], float, (npair, 5)),
        pair_solref=A([p["solref"] for p in pairs], float, (npair, 2)),
        pair_solimp=A([p["solimp"] for p in pairs], float, (npair, 5)))

    # ---- env bookkeeping
    block_body = [fused_of[i] for i, b in enumerate(bodies)
                  if re.fullmatch(block_name + r"\d*", b.name) and b.joints and b.joints[0].type == M.JNT_FREE]
    finger_body = np.zeros(2, np.int32); finger_pos = np.zeros((2, 3))
    for k, nm in enumerate(["hand_l_distal_link", "hand_r_distal_link"]):  # hsr/env.py:59
        if nm in name_to_id:
            i = name_to_id[nm]
            finger_body[k] = fused_of[bodies[i].weld]; finger_pos[k] = rel_pos[i]
    mocap = [b.pos for b in bodies if b.mocap]
    arr.update(block_body=A(block_body, np.int32, (len(block_body),)), finger_body=finger_body,
               finger_pos=finger_pos, mocap_pos0=A(mocap[0] if mocap else [0, 0, 0], float, (3,)))

    # Every float constant of the blob is rounded to an fp32-representable value (MuJoCo itself stores mesh
    # vertices as float): the CUDA path (fp32 model, double geometry stage) and the fp64 oracle then see identical
    # constants, so that one-step parity measures arithmetic, not a 1e-8 difference in the geometry.
    for k_, v_ in list(arr.items()):
        if v_.dtype == np.float64:
            arr[k_] = v_.astype(np.float32).astype(np.float64)
    mdl = M.Model(nq=nq, nv=nv, nu=nu, nbody=nbody, njnt=njnt, ngeom=ngeom, nvert=len(hull_vert), npair=npair,
                  nblock=len(block_body), arrays=arr)
    mdl.names = dict(body=[bodies[i].name for i in fused_ids], joint=jnt_names,
                     actuator=[a["name"] for a in actuators], geom=[g.name for _, g, *_ in geoms],
                     orig_body=[b.name for b in bodies])
    mdl.info = dict(orig_nbody=len(bodies), orig_mass={b.name: b.mass for b in bodies}, M0=Mq,
                    total_geoms=sum(len(b.geoms) for b in bodies), mesh_inertia=opts.mesh_inertia)
    mdl.validate()
    return mdl


# ----------------------------------------------------------------------------- static pair pruning
def _prune_unreachable_pairs(pairs, arr, kin, nbody, geom_body, geom_type, geom_pos, geom_mat, geom_size, vertadr,
                             vertnum, hull_vert, mesh_info, slack=0.05):
    """Drop candidate pairs between a static (world) geom and a geom whose body can only translate along limited
    slide joints, when the volume swept over the joint ranges (+ ``slack`` metres beyond each soft limit) cannot
    reach the static geom.  Purely a work reduction: a pruned pair could never produce a contact."""
    njnt = len(arr["jnt_type"])

    def slide_only_chain(f):
        """list of (axis_world, lo - q0, hi - q0) of the joints between body f and the world, or None."""
        out = []
        b = f
        while b > 0:
            for j in range(arr["body_jntadr"][b], arr["body_jntadr"][b] + arr["body_jntnum"][b]):
                if arr["jnt_type"][j] != M.JNT_SLIDE or not arr["jnt_limited"][j]:
                    return None
                q0 = arr["qpos0"][arr["jnt_qposadr"][j]]
                out.append((kin["axis"][j], arr["jnt_range"][j, 0] - q0 - slack, arr["jnt_range"][j, 1] - q0 + slack))
            b = arr["body_parent"][b]
        return out

    def local_points(g):
        t = geom_type[g]
        if t == M.GEOM_MESH:
            return hull_vert[vertadr[g]:vertadr[g] + vertnum[g]]
        s = geom_size[g]
        if t == M.GEOM_BOX:
            return np.array([[sx * s[0], sy * s[1], sz * s[2]] for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)])
        if t == M.GEOM_CYLINDER:  # conservative: bounding box of the cylinder
            return np.array([[sx * s[0], sy * s[0], sz * s[1]] for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)])
        return None

    def world_points(g):
        f = geom_body[g]
        R = kin["xmat"][f] @ geom_mat[g].reshape(3, 3)
        c = kin["xpos"][f] + kin["xmat"][f] @ geom_pos[g]
        pts = local_points(g)
        return None if pts is None else c + pts @ R.T

    kept = []
    for p in pairs:
        a, b = p["g1"], p["g2"]
        fa, fb = geom_body[a], geom_body[b]
        if (fa == 0) == (fb == 0):
            kept.append(p); continue
        st, mv = (a, b) if fa == 0 else (b, a)
        chain = slide_only_chain(geom_body[mv])
        pts = world_points(mv)
        if chain is None or pts is None:
            kept.append(p); continue
        lo, hi = pts.min(0).copy(), pts.max(0).copy()
        for ax, dlo, dhi in chain:
            lo += np.minimum(ax * dlo, ax * dhi); hi += np.maximum(ax * dlo, ax * dhi)
        if geom_type[st] == M.GEOM_PLANE:
            Rs = kin["xmat"][0] @ geom_mat[st].reshape(3, 3)
            n = Rs[:, 2]; p0 = geom_pos[st]
            corners = np.array([[x, y, z] for x in (lo[0], hi[0]) for y in (lo[1], hi[1]) for z in (lo[2], hi[2])])
            reachable = ((corners - p0) @ n).min() <= 1e-6
        else:
            spts = world_points(st)
            if spts is None:
                kept.append(p); continue
            slo, shi = spts.min(0), spts.max(0)
            reachable = bool(np.all(lo <= shi + 1e-6) and np.all(slo <= hi + 1e-6))
        if reachable:
            kept.append(p)
    return kept


# ----------------------------------------------------------------------------- compile-time kinematics
def _sym6(v):
    return np.array([[v[0], v[3], v[4]], [v[3], v[1], v[5]], [v[4], v[5], v[2]]])


def kinematics(arr, nbody, qpos):
    """Forward kinematics on the fused tree (used at compile time for invweight0 / meaninertia only)."""
    xpos = np.zeros((nbody, 3)); xquat = np.tile(np.array([1.0, 0, 0, 0]), (nbody, 1))
    xmat = np.tile(np.eye(3), (nbody, 1, 1)); xipos = np.zeros((nbody, 3))
    njnt = len(arr["jnt_type"])
    anchor = np.zeros((njnt, 3)); axis = np.zeros((njnt, 3))
    for b in range(1, nbody):
        p = arr["body_parent"][b]
        j0, nj = arr["body_jntadr"][b], arr["body_jntnum"][b]
        if nj == 1 and arr["jnt_type"][j0] == M.JNT_FREE:
            a = arr["jnt_qposadr"][j0]
            xpos[b] = qpos[a:a + 3]; xquat[b] = quat_normalize(qpos[a + 3:a + 7])
        else:
            xpos[b] = xpos[p] + xmat[p] @ arr["body_pos"][b]
            xquat[b] = quat_mul(xquat[p], arr["body_quat"][b])
            for j in range(j0, j0 + nj):
                R = quat_to_mat(xquat[b])
                anchor[j] = xpos[b] + R @ arr["jnt_pos"][j]; axis[j] = R @ arr["jnt_axis"][j]
                q = qpos[arr["jnt_qposadr"][j]] - arr["qpos0"][arr["jnt_qposadr"][j]]
                if arr["jnt_type"][j] == M.JNT_SLIDE:
                    xpos[b] = xpos[b] + axis[j] * q
                else:
                    ax = arr["jnt_axis"][j]
                    dq = np.concatenate([[np.cos(q / 2)], np.sin(q / 2) * ax])
                    xquat[b] = quat_mul(xquat[b], dq)
                    xpos[b] = anchor[j] - quat_to_mat(xquat[b]) @ arr["jnt_pos"][j]
        xmat[b] = quat_to_mat(xquat[b])
        xipos[b] = xpos[b] + xmat[b] @ arr["body_ipos"][b]
    return dict(xpos=xpos, xquat=xquat, xmat=xmat, xipos=xipos, anchor=anchor, axis=axis)


def jacobian(arr, kin, body, point):
    """Translational / rotational Jacobian (3 x nv each) of a world point attached to a fused body."""
    nv = len(arr["dof_body"])
    Jp = np.zeros((3, nv)); Jr = np.zeros((3, nv))
    b = body
    while b > 0:
        for j in range(arr["body_jntadr"][b], arr["body_jntadr"][b] + arr["body_jntnum"][b]):
            d = arr["jnt_dofadr"][j]
            t = arr["jnt_type"][j]
            if t == M.JNT_FREE:
                Jp[:, d:d + 3] = np.eye(3)
                R = kin["xmat"][b]
                for k in range(3):
                    Jr[:, d + 3 + k] = R[:, k]
                    Jp[:, d + 3 + k] = np.cross(R[:, k], point - kin["xpos"][b])
            elif t == M.JNT_SLIDE:
                Jp[:, d] = kin["axis"][j]
            else:
                Jr[:, d] = kin["axis"][j]
                Jp[:, d] = np.cross(kin["axis"][j], point - kin["anchor"][j])
        b = arr["body_parent"][b]
    return Jp, Jr


def default_assets_root() -> Optional[Path]:
    """Where the reference's ``hsr/`` package directory (models + meshes) lives: ``$HSR_ASSETS``, if it holds the models."""
    cand = os.environ.get("HSR_ASSETS")
    if cand and Path(cand, "models", "world.xml").exists():
        return Path(cand)
    return None
