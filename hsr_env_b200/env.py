"""Batched HSR environment on the B200 backend, with the reference's env API.

``BatchedHSREnv`` re-expresses ``HSREnv`` (/root/reference/hsr/env.py:23-209) and its ``MujocoEnv`` base
(/root/reference/hsr/mujoco_env.py:20-103) for N independent environments: same constructor kwargs
(+ ``n_envs``, ``device``, ``seed``, ``env_id_offset``), same ``reset`` / ``step`` contract, with torch tensors
``[N, ...]`` in and out.  ``HSREnv`` is the single-environment facade with numpy in/out, so a loop written
against the reference (/root/reference/hsr/control.py:66-76, /root/reference/hsr/__init__.py:9-28) runs unchanged.

The physics (``sim.step()`` x ``steps_per_action`` with the per-substep goal test and early break,
env.py:118-131) runs in one CUDA kernel launch per action behind the C ABI in include/hsrb.h.
There is no CPU fallback.
"""
from __future__ import annotations

import ctypes
from pathlib import Path
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import lib as _lib
from .model import Model
from .spaces import Box, Space
from .util import GoalSpec  # noqa: F401  (re-exported, as hsr.env does)

_BLOBS = Path(__file__).resolve().parent / "blobs"

# Columns of the per-environment physics parameters (include/hsrb.h hsrb_set_env_params): multipliers of pair_friction,
# of the block bodies' mass and inertia, of act_kp and of dof_damping.  1.0 is the model as compiled.
PARAM_NAMES = ("friction", "block_mass", "actuator_gain", "damping")
_PARAM_POSITIVE = (True, True, False, False)   # > 0, or >= 0


def get_xml_filepath(xml_filename=Path("models/world.xml")) -> Path:
    """hsr/env.py:16-17: relative model paths resolve inside the package's asset directory."""
    xml_filename = Path(xml_filename)
    if xml_filename.is_absolute():
        return xml_filename
    from .mjcf import default_assets_root

    root = default_assets_root()
    if root is None:
        raise FileNotFoundError(
            "HSR assets (hsr/models, hsr/hsr_meshes) not found: set HSR_ASSETS, or pass a pre-compiled "
            f"model blob from {_BLOBS} as xml_file")
    return Path(root, xml_filename).absolute()


def load_model(xml_file) -> Model:
    """``mujoco_py.load_model_from_path`` (mujoco_env.py:33): a compiled ``.hsrb`` blob, a ``Model``, or an MJCF
    file (compiled un-mutated, i.e. with every joint, as MuJoCo would load it)."""
    if isinstance(xml_file, Model):
        return xml_file
    p = Path(xml_file)
    if p.suffix == ".hsrb":
        if not p.is_absolute() and not p.exists():
            p = _BLOBS / p
        return Model.load(p)
    from . import mjcf

    p = get_xml_filepath(p)
    main, inc = mjcf.load_trees(p)
    full = mjcf.expand_includes(main, inc)
    dofs = [j.get("name") for j in full.iter("joint")]
    return mjcf.compile_model(p, dofs)


def _is_space(x):
    return isinstance(x, Space) or (hasattr(x, "low") and hasattr(x, "high") and hasattr(x, "sample"))


class BatchedHSREnv:
    def __init__(
            self,
            xml_file,
            goals: Optional[List[GoalSpec]],
            starts: Optional[Dict[str, Box]] = None,
            steps_per_action: int = 300,
            obs_type: str = None,
            render: bool = False,
            record: bool = False,
            record_freq: int = None,
            render_freq: int = None,
            record_path: Path = None,
            n_envs: int = 1,
            device="cuda:0",
            seed: int = 0,
            env_id_offset: int = 0,
            min_block_separation: float = 0.0,
            block_quat_index: Sequence[int] = (0, 2),
            lanes_per_env: int = 0,
            kernel: str = "auto",
            max_episode_steps: Optional[int] = None,
            autoreset: bool = False,
            randomize: Optional[dict] = None,
    ):
        """``randomize``: domain randomization, ``{name: (lo, hi)}`` over ``PARAM_NAMES`` (a missing name: (1, 1)); every
        reset, the auto-reset included, redraws the reset environments' parameters ~ U[lo, hi)."""
        if any([render, record, render_freq, record_freq, record_path]):
            raise NotImplementedError("render/record need an OpenGL viewer and are outside the batched backend "
                                      "(SURVEY.md §8f row f4)")
        if obs_type not in (None, "qpos-qvel", "openai"):
            raise NotImplementedError(f"obs_type={obs_type!r}: the default qpos|qvel observation (hsr/env.py:111-113) and "
                                      "'openai' (hsr/env.py:72-110) are implemented")
        self._obs_type = obs_type
        self._finger_adr = None   # qpos / dof addresses of the two proximal finger joints (openai observation)
        self.model = load_model(xml_file)
        self.starts = dict(starts or {})
        self.goals_specs = list(goals) if goals else []
        self.goals = None  # until the first reset (hsr/env.py:39,125): never done
        self.steps_per_action = int(steps_per_action)
        self.n_envs = int(n_envs)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.HsrbError("BatchedHSREnv needs a CUDA device: the physics path has no CPU fallback")
        if not torch.cuda.is_available():
            raise _lib.HsrbError("no CUDA device visible: the physics path has no CPU fallback")
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        blob = self.model.to_blob()
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        _lib.check(self._lib.hsrb_create(blob, len(blob), self.n_envs, dev_index, int(seed), int(env_id_offset),
                                         ctypes.byref(self._h)))
        if lanes_per_env:
            _lib.check(self._lib.hsrb_config(self._h, int(lanes_per_env), 0, 0))
        # "auto": fast kernel (hsrb_push.cuh) for the sliding-base + <=1 block family, else the general kernel
        self.kernel_path = _lib.check(self._lib.hsrb_set_path(self._h, {"auto": 0, "general": 1, "fast": 2, "lockstep": 2, "wpe": 3}[kernel]))
        m = self.model
        self.nq, self.nv, self.nu, self.nbody = m.nq, m.nv, m.nu, m.nbody
        self.state_dim = self.nq + self.nv   # what the kernel writes: qpos | qvel
        self.obs_dim = 25 if obs_type == "openai" else self.state_dim
        # spaces (mujoco_env.py:44-56)
        self.action_space = Box(m.act_ctrlrange[:, 0], m.act_ctrlrange[:, 1], dtype=np.float32)
        high = np.inf * np.ones(self.obs_dim)
        self.observation_space = Box(-high, high, dtype=np.float32)
        self.metadata = {"render.modes": "rgb_array"}
        self.reward_range = (-np.inf, np.inf)
        self.spec = None
        self._min_sep = float(min_block_separation)
        self._qidx = tuple(int(i) for i in block_quat_index)
        self._time_steps = 0
        self._geofence = 0.0
        # episode loop on the device (hsrb_step_episode): TimeLimit(max_episode_steps), hsr/__init__.py:22, and the
        # caller's `if done: env.reset()`, hsr/control.py:73-75
        if max_episode_steps is not None and int(max_episode_steps) < 0:
            raise ValueError("max_episode_steps must be >= 0 (0 or None: no time limit)")
        self.max_episode_steps = int(max_episode_steps or 0)
        self.autoreset = bool(autoreset)
        self._episodes = self.max_episode_steps > 0 or self.autoreset
        self._parse_goal_specs()
        self._push_starts()
        if randomize is not None:
            self.set_param_ranges(randomize)

    # ------------------------------------------------------------------ goals
    def _body_id(self, name: str) -> int:
        """Fused-body id of a body name (a body without joints is fused into its parent by the loader: its position is
        the parent's frame plus a constant offset, which only the renderer needs)."""
        names = list(self.model.names.get("body", []))
        if name in names:
            return names.index(name)
        if name == "block" and len(self.model.block_body):     # hsr/__init__.py:12 vs env.py:58 (SURVEY App. C #9)
            return int(self.model.block_body[0])
        raise KeyError(f"no moving body named {name!r} in the model (bodies: {names})")

    def _parse_goal_specs(self):
        """``goals`` -> kernel configuration.  Two forms:

        * the env_wrapper form (hsr/util.py:70-74): ONE GoalSpec(a=4-d block-space Box, b=3-d goal-space Box, distance)
          with the meaning SURVEY.md App. C #2 fixes: block-space (x, y, quat[i0], quat[i1]) is written into every
          block's free joint at reset, goal-space is the goal point (mocap_pos), success = all blocks within
          ``distance`` of it;
        * the general form of HSREnv (hsr/env.py:126,137-147,161-172): a list of up to four GoalSpec(a, b, distance)
          whose endpoints are body names (``data.get_body_xpos``), ndarrays or 3-d Spaces (sampled at reset);
          success = all(in_range(*g)).  As in the reference, at most one endpoint can be a Space (``mocap_pos[:] =
          concatenate(...)`` holds one point, hsr/env.py:169-172); further ndarray endpoints are fixed points.
          Callable endpoints (hsr/env.py:139-140) would have to run after every substep inside the kernel: they are
          accepted by the single-environment ``HSREnv.in_range`` only."""
        self._goal_lohi = None
        self._block_lohi = None
        self._goal_list = None
        if not self.goals_specs:
            return
        specs = [GoalSpec(*g) for g in self.goals_specs]
        a, b, dist = specs[0]
        wrapper_form = len(specs) == 1 and (a is None or (_is_space(a) and np.asarray(a.low).size == 4))
        if wrapper_form:
            self._geofence = float(dist)
            if _is_space(b):
                self._goal_lohi = np.concatenate([np.asarray(b.low, np.float32), np.asarray(b.high, np.float32)])
            else:
                b = np.asarray(b, np.float32).reshape(3)
                self._goal_lohi = np.concatenate([b, b])
            assert self._goal_lohi.shape == (6,), "goal space must be 3-d"
            if a is not None:
                self._block_lohi = np.concatenate([np.asarray(a.low, np.float32), np.asarray(a.high, np.float32)])
                assert self._block_lohi.shape == (8,), "block space must be 4-d"
            return
        if len(specs) > 4:
            raise NotImplementedError("at most four GoalSpecs")
        codes, dists, fixed, point = [], [], [], None
        for g in specs:
            pair = []
            for x in (g.a, g.b):
                if isinstance(x, str):
                    pair.append(self._body_id(x))
                elif _is_space(x):
                    if point is not None:
                        raise ValueError("only one GoalSpec endpoint can be a Space: mocap_pos holds one point (hsr/env.py:169-172)")
                    lo, hi = np.asarray(x.low, np.float32).reshape(3), np.asarray(x.high, np.float32).reshape(3)
                    point = np.concatenate([lo, hi])
                    pair.append(-1)
                elif callable(x):
                    raise NotImplementedError("callable GoalSpec endpoints cannot run inside the action kernel; "
                                              "use body names / arrays / Spaces, or HSREnv.in_range on the single-env facade")
                else:
                    v = np.asarray(x, np.float32).reshape(3)
                    if point is None and not any(_is_space(y) for h in specs for y in (h.a, h.b)):
                        point = np.concatenate([v, v])        # the ndarray endpoint that goes to mocap_pos
                        pair.append(-1)
                    else:
                        if len(fixed) >= 4:
                            raise NotImplementedError("at most four fixed goal points beside the sampled one")
                        fixed.append(v)
                        pair.append(-2 - (len(fixed) - 1))
            codes.append(pair)
            dists.append(float(g.distance))
        self._geofence = dists[0]
        self._goal_list = dict(a=np.asarray([c[0] for c in codes], np.int32), b=np.asarray([c[1] for c in codes], np.int32),
                               dist=np.asarray(dists, np.float32), point=point,
                               fixed=np.asarray(fixed, np.float32).reshape(-1, 3))

    def _push_goals(self, active: bool):
        fp = ctypes.POINTER(ctypes.c_float)
        ip = ctypes.POINTER(ctypes.c_int32)
        if self._goal_list is not None:
            g = self._goal_list
            _lib.check(self._lib.hsrb_set_goal_list(
                self._h, len(g["a"]) if active else 0, g["a"].ctypes.data_as(ip), g["b"].ctypes.data_as(ip),
                g["dist"].ctypes.data_as(fp), g["point"].ctypes.data_as(fp) if g["point"] is not None else None,
                g["fixed"].ctypes.data_as(fp) if len(g["fixed"]) else None, len(g["fixed"])))
            return
        g = self._goal_lohi if active else None
        blk = self._block_lohi
        _lib.check(self._lib.hsrb_set_goals(
            self._h, g.ctypes.data_as(fp) if g is not None else None,
            blk.ctypes.data_as(fp) if blk is not None else None, self._geofence, self._min_sep,
            self._qidx[0], self._qidx[1]))

    def _push_starts(self):
        """``starts`` (hsr/env.py:149-156) -> per-joint lo / hi table of the reset kernel (Philox draws keyed on the
        global environment id: reproducible, independent of batch size and sharding)."""
        names = list(self.model.names.get("joint", []))
        adr, width, lo, hi = [], [], [], []
        for joint, space in self.starts.items():
            assert _is_space(space), f"starts[{joint!r}] must be a Space (hsr/env.py:152)"
            j = names.index(joint)
            w = 7 if int(self.model.jnt_type[j]) == 0 else 1
            l, h = np.zeros(7, np.float32), np.zeros(7, np.float32)
            l[:w] = np.asarray(space.low, np.float32).reshape(w); h[:w] = np.asarray(space.high, np.float32).reshape(w)
            adr.append(int(self.model.jnt_qposadr[j])); width.append(w); lo.append(l); hi.append(h)
        fp = ctypes.POINTER(ctypes.c_float)
        ip = ctypes.POINTER(ctypes.c_int32)
        adr, width = np.asarray(adr, np.int32), np.asarray(width, np.int32)
        lo, hi = np.ascontiguousarray(lo, np.float32).reshape(-1, 7), np.ascontiguousarray(hi, np.float32).reshape(-1, 7)
        n = len(adr)
        _lib.check(self._lib.hsrb_set_starts(self._h, n, adr.ctypes.data_as(ip) if n else None, width.ctypes.data_as(ip) if n else None,
                                             lo.ctypes.data_as(fp) if n else None, hi.ctypes.data_as(fp) if n else None))

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _empty(self, *shape, dtype=torch.float32):
        return torch.empty(*shape, dtype=dtype, device=self.device)

    @property
    def dt(self):
        return self.model.timestep * 20  # frame_skip = record_freq default (hsr/env.py:68, mujoco_env.py:96-98)

    # ------------------------------------------------------------------ gym API
    def seed(self, seed=None):
        return [seed]

    def reset(self, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """MujocoEnv.reset + HSREnv.reset_model for all (or the masked) environments; returns obs [N, nq+nv]."""
        self._time_steps = 0
        if self.goals_specs:
            self.goals = self.goals_specs
            self._push_goals(True)
        else:
            self._push_goals(False)
        obs = self._empty(self.n_envs, self.state_dim)
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_reset(self._h, _lib.ptr(mask), _lib.ptr(obs), self._stream()))
        return self._observation(obs)

    def step(self, action: torch.Tensor, steps: Optional[int] = None):
        """HSREnv.step (hsr/env.py:115-135) for every environment: one kernel launch.  With ``max_episode_steps`` or
        ``autoreset`` (the episode loop on the device, hsrb_step_episode): done = terminated | truncated, and info adds
        ``terminated``, ``truncated``, ``final_observation`` (the step's observation before any auto-reset) and
        ``episode`` = {"l", "r", "substeps"} (length in actions, summed reward and substeps; valid where done)."""
        steps = steps or self.steps_per_action
        action = torch.as_tensor(action, dtype=torch.float32, device=self.device).reshape(self.n_envs, self.nu).contiguous()
        if self._episodes:
            return self._step_episode(action, steps)
        obs = self._empty(self.n_envs, self.state_dim)
        reward = self._empty(self.n_envs)
        done = self._empty(self.n_envs, dtype=torch.uint8)
        taken = self._empty(self.n_envs, dtype=torch.int32)
        bad = self._empty(self.n_envs, dtype=torch.uint8)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_step(self._h, _lib.ptr(action), int(steps), _lib.ptr(obs), _lib.ptr(reward),
                                           _lib.ptr(done), None, _lib.ptr(taken), _lib.ptr(bad), self._stream()))
        self._time_steps += 1
        done_b = done.bool()
        info = {"log count": {"success": done_b}, "substeps_taken": taken, "bad_state": bad}
        return self._observation(obs), reward, done_b, info

    def rollout(self, actions, steps: Optional[int] = None):
        """Open-loop rollout (MuJoCo's ``mujoco.rollout``): K step() calls with the K actions given in advance, bit for bit.
        ``actions`` [K, N, nu].  Returns obs [K, N, nq+nv], reward [K, N], done [K, N] (bool) and
        info = {"substeps_taken", "bad_state"} [K, N]: slice k is what the k-th step() would return.  Nothing happens
        between the actions: an environment that reached its goal starts the next action from that state, nothing is reset
        and the episode ages and counters are untouched.  The phase-locked kernels (the defaults) run all K actions in one
        launch, every other kernel one launch per action.  The fused launch keeps the wpe kernel's work-sorted order
        fixed for its K actions.  On the bench workload (B200) it is 2-7 % faster than K step() calls at 4096
        environments and 15-16 % slower at 131072 (K = 5, 20): there, re-sorting before every action is worth more
        than the launch boundary (DESIGN.md 4.3c).

        Raises NotImplementedError for obs_type='openai' (that observation is built from the resident state, which holds
        only the last action's) and on a handle with max_episode_steps / autoreset (the rollout has no episode loop, and
        running without the TimeLimit would silently change what the episodes mean)."""
        if self._obs_type == "openai":
            raise NotImplementedError("rollout returns the kernel's qpos|qvel observation per action; obs_type='openai' "
                                      "is built from the resident state after the last action only")
        if self._episodes:
            raise NotImplementedError("rollout has no episode loop; use step() with max_episode_steps / autoreset")
        steps = steps or self.steps_per_action
        actions = torch.as_tensor(actions, dtype=torch.float32, device=self.device)
        if actions.dim() != 3 or actions.shape[1] != self.n_envs or actions.shape[2] != self.nu:
            raise ValueError(f"rollout: actions must be [K, {self.n_envs}, {self.nu}], got {list(actions.shape)}")
        actions = actions.contiguous()
        K, n = actions.shape[0], self.n_envs
        obs = self._empty(K, n, self.state_dim)
        reward = self._empty(K, n)
        done = self._empty(K, n, dtype=torch.uint8)
        taken = self._empty(K, n, dtype=torch.int32)
        bad = self._empty(K, n, dtype=torch.uint8)
        P = _lib.ptr
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_rollout(self._h, P(actions), K, int(steps), P(obs), P(reward), P(done), P(taken), P(bad),
                                              self._stream()))
        self._time_steps += K
        return obs, reward, done.bool(), {"substeps_taken": taken, "bad_state": bad}

    def _step_episode(self, action: torch.Tensor, steps: int):
        """step() with max_episode_steps / autoreset: the action kernel, then the episode kernel (hsrb_step_episode)."""
        n = self.n_envs
        reward = self._empty(n)
        term = self._empty(n, dtype=torch.uint8)
        trunc = self._empty(n, dtype=torch.uint8)
        taken = self._empty(n, dtype=torch.int32)
        bad = self._empty(n, dtype=torch.uint8)
        # where not done the episode outputs are left as they are: zero, not garbage
        ep_l = torch.zeros(n, dtype=torch.int32, device=self.device)
        ep_r = torch.zeros(n, device=self.device)
        ep_s = torch.zeros(n, dtype=torch.int32, device=self.device)
        P = _lib.ptr
        with torch.cuda.device(self.device):
            if self._obs_type == "openai":
                # the 25-d observation of the stepped state before the reset, and of the reset state after it
                _lib.check(self._lib.hsrb_step(self._h, P(action), int(steps), None, P(reward), P(term), None, P(taken), P(bad),
                                               self._stream()))
                final = self._observation(None)
                _lib.check(self._lib.hsrb_episode_update(self._h, self.max_episode_steps, int(self.autoreset), P(term), P(reward),
                                                         P(taken), P(bad), None, P(trunc), None, P(ep_l), P(ep_r), P(ep_s),
                                                         self._stream()))
                obs = self._observation(None)
            else:
                obs = self._empty(n, self.state_dim)
                final = self._empty(n, self.state_dim)
                _lib.check(self._lib.hsrb_step_episode(self._h, P(action), int(steps), self.max_episode_steps, int(self.autoreset),
                                                       P(obs), P(reward), P(term), P(trunc), P(final), P(ep_l), P(ep_r), P(ep_s),
                                                       P(taken), P(bad), self._stream()))
        self._time_steps += 1
        term_b, trunc_b = term.bool(), trunc.bool()
        info = {"log count": {"success": term_b}, "substeps_taken": taken, "bad_state": bad, "terminated": term_b,
                "truncated": trunc_b, "final_observation": final, "episode": {"l": ep_l, "r": ep_r, "substeps": ep_s}}
        return obs, reward, term_b | trunc_b, info

    # ------------------------------------------------------------------ episode ages and counters
    def set_episode_ages(self, ages=None):
        """TimeLimit._elapsed_steps of every environment (None: zeros); the sums of the running episodes restart at 0."""
        a = None if ages is None else torch.as_tensor(ages, dtype=torch.int32, device=self.device).reshape(self.n_envs).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_set_episode_ages(self._h, _lib.ptr(a), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()  # the input may be a temporary

    def episode_ages(self) -> torch.Tensor:
        """Actions since each environment's last reset: int32 [N]."""
        out = self._empty(self.n_envs, dtype=torch.int32)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_get_episode_ages(self._h, _lib.ptr(out), self._stream()))
        return out

    def episode_stats(self) -> dict:
        """Cumulative counters of the episode kernel: the keys of dist.EPISODE_STAT_KEYS (``substeps``: summed substeps of
        the finished episodes, ``bad_states``: steps with a non-zero bad_state) plus ``truncations``, ``length`` (summed
        episode length in actions), ``resets`` (auto-resets) and ``actions`` (environment actions stepped)."""
        v = (ctypes.c_int64 * 8)()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_episode_stats(self._h, v, self._stream()))
        keys = ["episodes", "successes", "truncations", "length", "substeps", "bad_states", "resets", "actions"]
        return dict(zip(keys, [int(x) for x in v]))

    def step_host(self, action, steps: Optional[int] = None, out=None):
        """Same call with HOST buffers (numpy / pinned torch CPU tensors), copies inside: the end-to-end path.  Runs on
        torch's current stream, i.e. after any reset / set_state / step issued before it."""
        if self._obs_type == "openai":
            raise NotImplementedError("step_host returns the kernel's qpos|qvel observation; use step() for obs_type='openai'")
        if self._episodes:
            raise NotImplementedError("step_host has no episode loop; use step() with max_episode_steps / autoreset")
        steps = steps or self.steps_per_action
        if isinstance(action, torch.Tensor):
            if action.dtype != torch.float32 or not action.is_contiguous() or action.numel() != self.n_envs * self.nu or action.is_cuda:
                action = action.detach().to("cpu", torch.float32).reshape(self.n_envs, self.nu).contiguous()
        else:
            action = np.ascontiguousarray(action, np.float32).reshape(self.n_envs, self.nu)
        if out is None:
            out = dict(obs=np.empty((self.n_envs, self.state_dim), np.float32), reward=np.empty(self.n_envs, np.float32),
                       done=np.empty(self.n_envs, np.uint8), taken=np.empty(self.n_envs, np.int32))
        want = dict(obs=((self.n_envs, self.state_dim), "float32"), reward=((self.n_envs,), "float32"),
                    done=((self.n_envs,), "uint8"), taken=((self.n_envs,), "int32"))
        for k, (shape, dt) in want.items():
            buf = out[k]
            got_dt = str(buf.dtype).replace("torch.", "")
            if tuple(buf.shape) != shape or got_dt != dt:
                raise ValueError(f"step_host: out[{k!r}] must be {dt}{list(shape)}, got {got_dt}{list(buf.shape)}")
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_step_host(self._h, _lib.ptr(action), int(steps), _lib.ptr(out["obs"]),
                                                _lib.ptr(out["reward"]), _lib.ptr(out["done"]), _lib.ptr(out["taken"]),
                                                self._stream()))
        self._time_steps += 1
        return out

    def _observation(self, state: Optional[torch.Tensor]) -> torch.Tensor:
        """HSREnv._get_observation (hsr/env.py:71-113): the kernel's qpos|qvel, or the 25-d 'openai' observation built
        from it on the device (hsr_env_b200/kin.py states the intent of the reference's dead branch)."""
        if self._obs_type != "openai":
            return state
        if not len(self.model.block_body):
            raise NotImplementedError("the 'openai' observation needs a block (hsr/env.py:58 `_block_name`)")
        if self._finger_adr is None:
            names = list(self.model.names.get("joint", []))
            adr = []
            for jn in ("hand_l_proximal_joint", "hand_r_proximal_joint"):
                j = names.index(jn) if jn in names else -1
                adr.append((int(self.model.jnt_qposadr[j]), int(self.model.jnt_dofadr[j])) if j >= 0 else (-1, -1))
            self._finger_adr = adr
        (ql, dl), (qr, dr) = self._finger_adr
        obs = self._empty(self.n_envs, 25)
        with torch.cuda.device(self.device):   # one kernel on the resident state (hsrb_api.cu openai_obs_kernel); kin.py is the test oracle
            _lib.check(self._lib.hsrb_openai_obs(self._h, ql, qr, dl, dr, _lib.ptr(obs), self._stream()))
        return obs

    def compute_reward(self) -> torch.Tensor:
        """float(all in_range) of the current state (north star name; hsr/env.py:126,133)."""
        reward = self._empty(self.n_envs)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_compute_reward(self._h, _lib.ptr(reward), None, self._stream()))
        return reward

    # ------------------------------------------------------------------ per-environment physics parameters
    def set_param_ranges(self, ranges: Optional[dict]):
        """``{name: (lo, hi)}`` over ``PARAM_NAMES`` (missing: (1, 1)): every reset redraws the reset environments'
        parameters ~ U[lo, hi).  None: parameters persist across resets."""
        if ranges is None:
            _lib.check(self._lib.hsrb_set_env_param_ranges(self._h, None, None))
            return
        unknown = set(ranges) - set(PARAM_NAMES)
        if unknown:
            raise KeyError(f"unknown parameter(s) {sorted(unknown)}; names: {PARAM_NAMES}")
        lo = (ctypes.c_float * 4)(*[float(ranges.get(k, (1.0, 1.0))[0]) for k in PARAM_NAMES])
        hi = (ctypes.c_float * 4)(*[float(ranges.get(k, (1.0, 1.0))[1]) for k in PARAM_NAMES])
        _lib.check(self._lib.hsrb_set_env_param_ranges(self._h, lo, hi))

    def set_env_params(self, params):
        """Per-environment multipliers: a [N, 4] tensor (columns ``PARAM_NAMES``), a dict of [N] tensors (missing names:
        1.0), or None (nominal model, ranges cleared, the kernels without parameters).  friction and block_mass must be
        > 0, actuator_gain and damping >= 0."""
        if params is None:
            with torch.cuda.device(self.device):
                _lib.check(self._lib.hsrb_set_env_params(self._h, None, self._stream()))
            return
        if isinstance(params, dict):
            unknown = set(params) - set(PARAM_NAMES)
            if unknown:
                raise KeyError(f"unknown parameter(s) {sorted(unknown)}; names: {PARAM_NAMES}")
            cols = [torch.as_tensor(params[k], dtype=torch.float32, device=self.device).reshape(self.n_envs)
                    if k in params else torch.ones(self.n_envs, device=self.device) for k in PARAM_NAMES]
            p = torch.stack(cols, dim=1)
        else:
            p = torch.as_tensor(params, dtype=torch.float32, device=self.device).reshape(self.n_envs, len(PARAM_NAMES))
        p = p.contiguous()
        if not bool(torch.isfinite(p).all()):
            raise ValueError("environment parameters must be finite")
        for k, (name, positive) in enumerate(zip(PARAM_NAMES, _PARAM_POSITIVE)):
            col = p[:, k]
            if not bool((col > 0).all() if positive else (col >= 0).all()):
                raise ValueError(f"{name} multipliers must be {'> 0' if positive else '>= 0'}")
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_set_env_params(self._h, _lib.ptr(p), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()  # the input may be a temporary

    def env_params(self) -> torch.Tensor:
        """The current multipliers: float32 [N, 4], columns ``PARAM_NAMES``."""
        out = self._empty(self.n_envs, len(PARAM_NAMES))
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_get_env_params(self._h, _lib.ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------ state access (sim.get_state / set_state)
    def get_state(self):
        qpos = self._empty(self.n_envs, self.nq); qvel = self._empty(self.n_envs, self.nv)
        warm = self._empty(self.n_envs, self.nv); mocap = self._empty(self.n_envs, 3)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_get_state(self._h, _lib.ptr(qpos), _lib.ptr(qvel), _lib.ptr(warm), _lib.ptr(mocap),
                                                self._stream()))
        return qpos, qvel, warm, mocap

    def set_state(self, qpos=None, qvel=None, qacc_warmstart=None, mocap_pos=None):
        def prep(t, w):
            if t is None:
                return None
            return torch.as_tensor(t, dtype=torch.float32, device=self.device).reshape(self.n_envs, w).contiguous()

        ts = [prep(qpos, self.nq), prep(qvel, self.nv), prep(qacc_warmstart, self.nv), prep(mocap_pos, 3)]
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_set_state(self._h, *[_lib.ptr(t) for t in ts], self._stream()))
            torch.cuda.current_stream(self.device).synchronize()  # inputs may be temporaries

    def body_xpos(self) -> torch.Tensor:
        """data.get_body_xpos for every (fused) body: [N, nbody, 3] (sim.forward on the current state)."""
        out = self._empty(self.n_envs, self.nbody, 3)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_forward(self._h, _lib.ptr(out), None, self._stream()))
        return out

    def block_pos(self) -> torch.Tensor:
        """hsr/env.py:179-180 for every block: [N, nblock, 3]."""
        idx = torch.as_tensor(self.model.block_body, dtype=torch.long, device=self.device)
        return self.body_xpos()[:, idx]

    def gripper_pos(self) -> torch.Tensor:
        """hsr/env.py:182-186: mean of the two distal finger link positions, [N, 3]."""
        out = self._empty(self.n_envs, 3)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_forward(self._h, None, _lib.ptr(out), self._stream()))
        return out

    def goal_pos(self) -> torch.Tensor:
        return self.get_state()[3]

    def in_range(self) -> torch.Tensor:
        return self.compute_reward() > 0

    # ------------------------------------------------------------------ diagnostics
    def debug_substep(self, action):
        """One teacher-forced substep with per-stage outputs (parity tests); returns a float64 [N, D] tensor."""
        action = torch.as_tensor(action, dtype=torch.float32, device=self.device).reshape(self.n_envs, self.nu).contiguous()
        size = self._lib.hsrb_debug_size(self._h)
        dump = torch.zeros(self.n_envs, size, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_debug_substep(self._h, _lib.ptr(action), _lib.ptr(dump), self._stream()))
        return dump

    def stats(self) -> dict:
        v = (ctypes.c_int64 * 16)()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_stats(self._h, v, self._stream()))
        keys = ["substeps", "newton_iters", "narrowphase", "ls_evals", "contacts", "efc_rows", "launches", "bad_envs", "flops"]
        out = dict(zip(keys, [int(x) for x in v]))
        phases = ["kinematics", "mass_matrix", "smooth", "collision", "rows", "solver", "euler"]
        out["phase_cycles"] = {k: int(v[9 + i]) * 16 for i, k in enumerate(phases)}
        return out

    def launch_info(self) -> dict:
        v = (ctypes.c_int * 6)()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.hsrb_launch_info(self._h, v))
        return dict(lanes_per_env=v[0], smem_per_env=v[1], envs_per_sm=v[2], grid=v[3],
                    kernel={1: "general", 2: "fast", 3: "wpe"}.get(v[4], "?"), threads_per_block=v[5])

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.hsrb_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *args):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HSREnv(BatchedHSREnv):
    """Single-environment facade: numpy in / numpy out, scalars for reward and done, like the reference."""

    def __init__(self, xml_file, goals, starts=None, steps_per_action: int = 300, max_episode_steps: Optional[int] = None, **kw):
        """``max_episode_steps``: gym.wrappers.TimeLimit (hsr/__init__.py:22): done at the limit, with
        ``info["TimeLimit.truncated"]``.  No auto-reset: the caller's loop resets, as hsr/control.py:73-75 does."""
        kw.setdefault("n_envs", 1)
        assert kw["n_envs"] == 1
        if kw.get("autoreset"):
            raise ValueError("HSREnv does not auto-reset: reset() when done, as hsr/control.py:73-75 does")
        kw["max_episode_steps"] = max_episode_steps
        super().__init__(xml_file, goals, starts, steps_per_action, **kw)
        self.init_qpos = self.model.qpos0.copy()
        self.init_qvel = np.zeros(self.nv)

    def reset(self):
        return super().reset()[0].double().cpu().numpy()

    def step(self, action, steps=None):
        obs, reward, done, info = super().step(np.asarray(action, np.float32), steps)
        success = bool(info["terminated"][0].item()) if self._episodes else bool(done[0].item())
        out = {"log count": {"success": success and self._time_steps > 0}, "substeps_taken": int(info["substeps_taken"][0]),
               "bad_state": int(info["bad_state"][0])}
        if self.max_episode_steps and bool(done[0].item()) and int(info["episode"]["l"][0].item()) >= self.max_episode_steps:
            out["TimeLimit.truncated"] = not success   # what gym.wrappers.TimeLimit.step sets at the limit
        return obs[0].double().cpu().numpy(), float(reward[0].item()), bool(done[0].item()), out

    def block_pos(self):
        return super().block_pos()[0, 0].double().cpu().numpy()

    def gripper_pos(self):
        return super().gripper_pos()[0].double().cpu().numpy()

    def compute_reward(self):
        return float(super().compute_reward()[0].item())

    def in_range(self, a=None, b=None, distance=None):
        if a is None:
            return bool(super().in_range()[0].item())

        def parse(x):  # hsr/env.py:138-145
            if callable(x):
                return x()
            if isinstance(x, np.ndarray):
                return x
            if isinstance(x, str):
                xp = BatchedHSREnv.body_xpos(self)[0].double().cpu().numpy()
                return xp[self.model.names["body"].index(x)]
            raise RuntimeError(f"{x} must be function, np.ndarray, or string")

        return distance_between(parse(a), parse(b)) < distance


def distance_between(pos1, pos2):
    """hsr/env.py:231-232"""
    return np.sqrt(np.sum(np.square(pos1 - pos2), axis=-1))
