"""Batched, GPU-resident drop-in for the reference's env classes.

``Walker3DCustomVecEnv`` runs ``num_envs`` independent copies of ``Walker3DCustomEnv-v0``
(reference mocca_envs/env_locomotion.py:37-282, registered at mocca_envs/__init__.py:52-56 with
``max_episode_steps=1000``) inside one CUDA kernel launch per ``step``.  Observations, rewards and dones are
torch CUDA tensors (zero-copy; ``torch.utils.dlpack.to_dlpack`` works on them).  Auto-reset follows the baselines
VecEnv convention the reference's downstream trainers use (SURVEY.md section 3.4).

``Walker3DCustomEnv`` is the N=1 gym-protocol facade: ``reset() -> obs``, ``step(a) -> (obs, reward, done, info)``
with NumPy float64 observations, like the reference.

PyTorch is plumbing here (device memory, streams); all arithmetic is in libmocca_b200.so.
"""
from __future__ import annotations

import ctypes as C
import json
import os

import numpy as np
import torch

from . import _lib
from .seeding import create_seed, mt_state_rows

ENV_ID = "Walker3DCustomEnv-v0"
STEPPER_ID = "Walker3DStepperEnv-v0"
MONKEY_ID = "Monkey3DCustomEnv-v0"
CASSIE_ID = "CassieEnv-v0"
CHILD_ID = "Child3DCustomEnv-v0"
MIKE_ID = "MikeStepperEnv-v0"
WALKER2D_ID = "Walker2DCustomEnv-v0"
CRAB2D_ID = "Crab2DCustomEnv-v0"
_MODELS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "models")


class Box:
    """Minimal stand-in for gym.spaces.Box (gym is not a dependency of the batched path)."""

    def __init__(self, low, high, dtype=np.float32):
        self.low = np.asarray(low, dtype=dtype)
        self.high = np.asarray(high, dtype=dtype)
        self.shape = self.low.shape
        self.dtype = np.dtype(dtype)

    def sample(self, rng=np.random):
        lo = np.where(np.isfinite(self.low), self.low, -1.0)
        hi = np.where(np.isfinite(self.high), self.high, 1.0)
        return rng.uniform(lo, hi).astype(self.dtype)


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


# The tracking camera of VecEnv.render / render(mode="rgb_array") when no camera is given: PyBullet's yaw / pitch /
# distance convention about the env's base position (yaw 0 = looking along +y, i.e. at the x-z plane of the walkers)
TRACKING_CAMERA = dict(distance=3.0, yaw=0.0, pitch=-20.0, fov=60.0, near=0.01, far=100.0)
RENDER_OUTPUTS = ("rgb", "depth", "seg")


def camera_matrices(target, distance, yaw, pitch, fov=60.0, aspect=1.0, near=0.01, far=100.0):
    """(view, proj), float32 torch tensors [m, 16]: column-major OpenGL matrices in the layout of
    ``pybullet.computeViewMatrixFromYawPitchRoll(target, distance, yaw, pitch, 0, upAxisIndex=2)`` and
    ``pybullet.computeProjectionMatrixFOV(fov, aspect, near, far)``, for ``mb200_render`` / ``VecEnv.render``.

    ``target`` is [3] or [m, 3] (a tensor keeps its device).  Angles are in degrees, z is up: the eye sits at
    ``target + distance * (cos(pitch) sin(yaw), -cos(pitch) cos(yaw), -sin(pitch))`` (so a negative pitch looks down),
    looks at the target, and its up vector is ``(sin(pitch) sin(yaw), -sin(pitch) cos(yaw), cos(pitch))``.  PyBullet is
    not a dependency here, so only these geometric properties are checked, not the matrices against PyBullet's."""
    t = torch.as_tensor(target, dtype=torch.float64)
    t = t.reshape(-1, 3)
    m, dev = t.shape[0], t.device
    y, p = np.deg2rad(float(yaw)), np.deg2rad(float(pitch))
    off = torch.tensor([np.cos(p) * np.sin(y), -np.cos(p) * np.cos(y), -np.sin(p)], dtype=torch.float64, device=dev)
    up = torch.tensor([np.sin(p) * np.sin(y), -np.sin(p) * np.cos(y), np.cos(p)], dtype=torch.float64, device=dev)
    eye = t + float(distance) * off
    f = torch.nn.functional.normalize(t - eye, dim=1)
    sv = torch.nn.functional.normalize(torch.cross(f, up.expand(m, 3), dim=1), dim=1)
    u = torch.cross(sv, f, dim=1)
    view = torch.zeros(m, 16, dtype=torch.float64, device=dev)
    view[:, [0, 4, 8]] = sv
    view[:, [1, 5, 9]] = u
    view[:, [2, 6, 10]] = -f
    view[:, 12] = -(sv * eye).sum(1)
    view[:, 13] = -(u * eye).sum(1)
    view[:, 14] = (f * eye).sum(1)
    view[:, 15] = 1.0
    ys = 1.0 / np.tan(np.deg2rad(float(fov)) / 2)
    proj = torch.zeros(m, 16, dtype=torch.float64, device=dev)
    proj[:, 0], proj[:, 5] = ys / float(aspect), ys
    proj[:, 10] = (far + near) / (near - far)
    proj[:, 11] = -1.0
    proj[:, 14] = 2.0 * far * near / (near - far)
    return view.float(), proj.float()


def _unsupported(message=None):
    """A trainer-facing method the reference env does not have: it raises AttributeError(message), or does nothing
    when there is no message."""
    def method(self, *args):
        if message is not None:
            raise AttributeError(message)
    return method


class Walker3DCustomVecEnv:
    """Batched Walker3DCustomEnv-v0; also the base class of the other batched envs (env_id selects the kernels)."""

    env_id = ENV_ID
    model = "walker3d"
    control_step = 1 / 60  # env_locomotion.py:39
    llc_frame_skip = 1  # env_locomotion.py:40
    sim_frame_skip = 4  # env_locomotion.py:41
    max_episode_steps = 1000  # __init__.py:55

    def __init__(self, num_envs: int, device="cuda:0", seed: int | None = None, physics: dict | None = None,
                 return_final_obs: bool = False):
        self.num_envs = int(num_envs)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("mocca_envs_b200 has no CPU path; device must be a CUDA device")
        L = _lib.lib()
        phys = _lib.Physics()
        L.mb200_default_physics_for(self.env_id.encode(), C.byref(phys))
        for k, v in (physics or {}).items():
            if not hasattr(phys, k):
                raise KeyError(k)
            setattr(phys, k, v)
        self.physics = phys
        h = C.c_void_p()
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        _lib.check(L.mb200_create(self.env_id.encode(), self.num_envs, idx, C.byref(phys), C.byref(h)))
        self._h = h
        self._L = L
        dims = [C.c_int() for _ in range(5)]
        _lib.check(L.mb200_dims(h, *[C.byref(d) for d in dims]))
        _, self.obs_dim, self.act_dim, self.state_dim, self.nu = [d.value for d in dims]
        self.rec_stride = int(L.mb200_record_stride(h))
        with open(os.path.join(_MODELS, self.model + ".json")) as f:
            self.table = json.load(f)
        # spaces as the reference builds them (robots.py:22-29, env_locomotion.py:58-60)
        self.observation_space = Box(-np.inf * np.ones(self.obs_dim), np.inf * np.ones(self.obs_dim))
        self.action_space = self._action_space()
        kw = dict(device=self.device)
        n = self.num_envs
        self.obs = torch.zeros(n, self.obs_dim, dtype=torch.float32, **kw)
        self.rew = torch.zeros(n, dtype=torch.float32, **kw)
        self.done = torch.zeros(n, dtype=torch.uint8, **kw)
        self.trunc = torch.zeros(n, dtype=torch.uint8, **kw)
        self.final_obs = torch.zeros(n, self.obs_dim, dtype=torch.float32, **kw) if return_final_obs else None
        self._seeded = False
        self.seed(seed, _at_construction=True)

    def _action_space(self):
        return Box(-np.ones(self.act_dim), np.ones(self.act_dim))

    # ---- lifecycle
    def close(self):
        if getattr(self, "_h", None) is not None:
            self._L.mb200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- EnvBase.seed (env_base.py:164-166): env i is seeded with seed + i
    def seed(self, seed=None, _at_construction=False):
        base = create_seed(seed)
        seeds = [(base + i) % 2 ** 64 for i in range(self.num_envs)]
        rows = np.ascontiguousarray(mt_state_rows(seeds))
        _lib.check(self._L.mb200_seed(self._h, rows.ctypes.data_as(C.c_void_p), int(_at_construction)))
        self._seeded = True
        return seeds

    # ---- gym / VecEnv protocol
    def reset(self, mask: torch.Tensor | None = None) -> torch.Tensor:
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self._L.mb200_reset(self._h, _ptr(mask), _ptr(self.obs), self._stream()))
        return self.obs

    def reset_host(self, mask: np.ndarray | None = None, out: np.ndarray | None = None) -> np.ndarray:
        """Env.reset with host buffers (mb200_reset_host): no device memory on the caller's side."""
        if out is None:
            out = np.zeros((self.num_envs, self.obs_dim), np.float32)
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        _lib.check(self._L.mb200_reset_host(self._h, None if m is None else m.ctypes.data_as(C.c_void_p),
                                            out.ctypes.data_as(C.c_void_p), self._stream()))
        return out

    def step_info(self) -> torch.Tensor:
        """Integer info of the last step, one per env (mb200_info): Stepper ``steps_reached`` or -1."""
        t = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        _lib.check(self._L.mb200_info(self._h, _ptr(t), self._stream()))
        return t

    def step(self, actions: torch.Tensor):
        if actions.device != self.device or actions.dtype != torch.float32 or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.float32).contiguous()
        assert actions.shape == (self.num_envs, self.act_dim)
        _lib.check(self._L.mb200_step(self._h, _ptr(actions), _ptr(self.obs), _ptr(self.rew), _ptr(self.done),
                                      _ptr(self.trunc), _ptr(self.final_obs), self._stream()))
        info = {"TimeLimit.truncated": self.trunc}
        if self.final_obs is not None:
            info["terminal_observation"] = self.final_obs
        return self.obs, self.rew, self.done, info

    def step_host(self, actions: np.ndarray, out=None):
        """Host-buffer entry point (what a SubprocVecEnv user holds): H2D, kernel, D2H, sync in one C call."""
        n = self.num_envs
        if out is None:
            out = (np.empty((n, self.obs_dim), np.float32), np.empty(n, np.float32), np.empty(n, np.uint8),
                   np.empty(n, np.uint8))
        a = np.ascontiguousarray(actions, dtype=np.float32)
        vp = lambda x: x.ctypes.data_as(C.c_void_p)
        _lib.check(self._L.mb200_step_host(self._h, vp(a), vp(out[0]), vp(out[1]), vp(out[2]), vp(out[3]),
                                           self._stream()))
        return out

    # ---- state access (parity tests, checkpoint/resume)
    def get_state(self) -> torch.Tensor:
        s = torch.empty(self.num_envs, self.state_dim, dtype=torch.float32, device=self.device)
        _lib.check(self._L.mb200_get_state(self._h, _ptr(s), self._stream()))
        return s

    def set_state(self, s: torch.Tensor):
        s = s.to(device=self.device, dtype=torch.float32).contiguous()
        assert s.shape == (self.num_envs, self.state_dim)
        _lib.check(self._L.mb200_set_state(self._h, _ptr(s), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    def get_record(self) -> torch.Tensor:
        r = torch.empty(self.num_envs, self.rec_stride, dtype=torch.float32, device=self.device)
        _lib.check(self._L.mb200_get_record(self._h, _ptr(r), self._stream()))
        return r

    def set_record(self, r: torch.Tensor):
        r = r.to(device=self.device, dtype=torch.float32).contiguous()
        assert r.shape == (self.num_envs, self.rec_stride)
        _lib.check(self._L.mb200_set_record(self._h, _ptr(r), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    def get_rng(self) -> np.ndarray:
        """The env / robot MT19937 streams, [num_envs, 2, 640] uint32 (624 key words, position, padding)."""
        out = np.empty((self.num_envs, int(self._L.mb200_rng_words(self._h))), dtype=np.uint32)
        _lib.check(self._L.mb200_get_rng(self._h, out.ctypes.data_as(C.c_void_p)))
        return out.reshape(self.num_envs, 2, -1)

    def set_rng(self, mt: np.ndarray):
        mt = np.ascontiguousarray(mt, dtype=np.uint32)
        assert mt.size == self.num_envs * int(self._L.mb200_rng_words(self._h))
        _lib.check(self._L.mb200_set_rng(self._h, mt.ctypes.data_as(C.c_void_p)))

    def state_dict(self):
        """Complete checkpoint of the batch (physics state, bookkeeping record, RNG streams, current observation):
        a batch restored with load_state_dict continues bit-exactly."""
        d = {"state": self.get_state().cpu(), "record": self.get_record().cpu(), "rng": self.get_rng(),
             "obs": self.obs.clone().cpu(), "env_id": self.env_id, "params": self._host_params()}
        w = int(self._L.mb200_warm_width(self._h))
        if w:  # physics["warmstart"] > 0: the cached contact impulses are state too
            t = torch.empty(self.num_envs, w, dtype=torch.float32, device=self.device)
            _lib.check(self._L.mb200_get_warm(self._h, _ptr(t), self._stream()))
            d["warm"] = t.cpu()
        return d

    def _host_params(self) -> dict:
        """Host-side mirrors of what lives in the record (re-applied through mb200_set_param on load, because the
        library keeps its own copies: e.g. which stepper kernel instantiation to launch)."""
        return {"eval_mode": bool(self.eval_mode)}

    def _apply_host_params(self, params: dict):
        if params.get("eval_mode"):
            self.evaluation_mode()

    def load_state_dict(self, d):
        if d.get("env_id", self.env_id) != self.env_id:
            raise ValueError("checkpoint of %s loaded into %s" % (d["env_id"], self.env_id))
        # parameters first (they write whole record columns), then the record itself
        self._apply_host_params(d.get("params", {}))
        self.set_state(d["state"])
        self.set_record(d["record"])
        if "rng" in d:
            self.set_rng(d["rng"])
        if "warm" in d and int(self._L.mb200_warm_width(self._h)):
            t = d["warm"].to(device=self.device, dtype=torch.float32).contiguous()
            _lib.check(self._L.mb200_set_warm(self._h, _ptr(t), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()
        if "obs" in d:
            self.obs.copy_(d["obs"].to(self.device))

    def step_physics(self, tau: torch.Tensor):
        """stepSimulation only (bullet_utils.py:352-353): hold tau over the substeps; returns (rows, contacts)."""
        tau = tau.to(device=self.device, dtype=torch.float32).contiguous()
        rows = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
        nc = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
        _lib.check(self._L.mb200_step_physics(self._h, _ptr(tau), _ptr(rows), _ptr(nc), self._stream()))
        return rows, nc

    def step_physics_points(self, tau: torch.Tensor):
        """stepSimulation + pybullet.getContactPoints: returns (rows, contacts, points[n, max_points, width]); per point
        {world position (3), normal (3), distance, normal impulse, link index (-2 = unused), partner code}."""
        tau = tau.to(device=self.device, dtype=torch.float32).contiguous()
        rows = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
        nc = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
        pts = torch.zeros(self.num_envs, int(self._L.mb200_max_contact_points()),
                          int(self._L.mb200_contact_point_width()), dtype=torch.float32, device=self.device)
        _lib.check(self._L.mb200_step_physics_points(self._h, _ptr(tau), _ptr(rows), _ptr(nc), _ptr(pts), self._stream()))
        return rows, nc, pts

    def mass_matrix(self) -> torch.Tensor:
        M = torch.empty(self.num_envs, self.nu, self.nu, dtype=torch.float32, device=self.device)
        _lib.check(self._L.mb200_mass_matrix(self._h, _ptr(M), self._stream()))
        return M

    def inverse_dynamics(self, acc: torch.Tensor) -> torch.Tensor:
        acc = acc.to(device=self.device, dtype=torch.float32).contiguous()
        tau = torch.empty(self.num_envs, self.nu, dtype=torch.float32, device=self.device)
        _lib.check(self._L.mb200_inverse_dynamics(self._h, _ptr(acc), _ptr(tau), self._stream()))
        return tau

    # ---- pushes (mb200_apply_impulse)
    def link_index(self, name: str) -> int:
        """The link index ``apply_impulse`` takes for the model link ``name``: -1 for the base, else the dof of the
        link's movable frame, a fixed link folded into its nearest movable ancestor.  KeyError for unknown names."""
        t = self.table
        if name == t["base"]["name"]:
            return -1
        if name not in t["link_names"]:
            raise KeyError("%s has no link %r" % (self.model, name))
        k = t["link_names"].index(name)
        while k >= 0 and t["dof_of_link"][k] < 0:
            k = t["parent"][k]
        return -1 if k < 0 else int(t["dof_of_link"][k])

    def apply_impulse(self, impulse, link=-1, point=None):
        """Push every env between two steps: the linear impulse ``impulse`` (N s, world frame, [N, 3] or [3]) at the
        world point ``point`` ([N, 3] or [3]) rigidly attached to ``link`` (an int or an int tensor [N]; -1 = the base,
        else see ``link_index``).  The generalised velocity changes by M(q)^-1 J^T impulse (clamped to max_coord_vel);
        positions, the record and the RNG streams are untouched, and so is every env whose link is outside [-1, NJ)
        (e.g. -2 masks an env out) or whose impulse is zero or non-finite.  ``point=None`` means the base COM and needs
        ``link=-1``.  The observation already returned is the pre-push one; the next ``step`` sees the pushed state.
        CassieEnv keeps its loop closures closed; the planar walkers ignore the y components of impulse and point."""
        n, dev, nj = self.num_envs, self.device, self.nu - 6
        scalar_link = isinstance(link, (int, np.integer))
        if scalar_link:
            link = int(link)
            if not -1 <= link < nj:
                raise ValueError("link %d outside [-1, %d)" % (link, nj))
            links = torch.full((n,), link, dtype=torch.int32, device=dev)
        else:
            links = torch.as_tensor(link).to(device=dev, dtype=torch.int32).expand(n).contiguous()
        if point is None:
            if not (scalar_link and link == -1):
                raise ValueError("point=None (the base COM) needs link=-1")
            pts = self.get_state()[:, 0:3].contiguous()
        else:
            pts = torch.as_tensor(point).to(device=dev, dtype=torch.float32).expand(n, 3).contiguous()
        imp = torch.as_tensor(impulse).to(device=dev, dtype=torch.float32).expand(n, 3).contiguous()
        _lib.check(self._L.mb200_apply_impulse(self._h, _ptr(links), _ptr(pts), _ptr(imp), self._stream()))

    # ---- camera images (mb200_render)
    def render(self, env_ids=None, width=64, height=64, view=None, proj=None, outputs=RENDER_OUTPUTS):
        """Camera images of envs ``env_ids`` (None = every env, else an int tensor / sequence, any order, repeats
        allowed, an id outside the batch gives a blank frame) in their current state, by ray casting the collision
        geometry on the device: a dict with the requested ``outputs`` of "rgb" ([m, H, W, 3] uint8), "depth"
        ([m, H, W] float32, eye-space distance along the view axis, ``far`` where nothing is hit) and "seg" ([m, H, W]
        int32: -1 sky, 0 ground, 10 + k plank box, 20 + k bar, 30 walk target, 100 + link for a robot link).
        ``view`` / ``proj`` are [16] or [m, 16] column-major OpenGL matrices as ``camera_matrices`` and PyBullet build
        them; without them a tracking camera (``TRACKING_CAMERA``) looks at each env's base position.  The envs'
        state, record and RNG streams are untouched.  See include/mocca_b200.h: mb200_render."""
        unknown = set(outputs) - set(RENDER_OUTPUTS)
        if unknown:
            raise ValueError("unknown render outputs %s: choose from %s" % (sorted(unknown), RENDER_OUTPUTS))
        dev = self.device
        ids = None if env_ids is None else torch.as_tensor(env_ids).to(device=dev, dtype=torch.int32).reshape(-1)
        m = self.num_envs if ids is None else int(ids.numel())
        W, H = int(width), int(height)
        if view is None or proj is None:
            st = self.get_state()[:, 0:3]
            if ids is not None:
                ok = (ids >= 0) & (ids < self.num_envs)
                st = torch.where(ok[:, None], st[ids.clamp(0, self.num_envs - 1).long()], torch.zeros_like(st[:1]))
            v, p = camera_matrices(st, aspect=W / H if W > 0 and H > 0 else 1.0, **TRACKING_CAMERA)
            view = v if view is None else view
            proj = p if proj is None else proj
        view = torch.as_tensor(view).to(device=dev, dtype=torch.float32).expand(m, 16).contiguous()
        proj = torch.as_tensor(proj).to(device=dev, dtype=torch.float32).expand(m, 16).contiguous()
        kw = dict(device=dev)
        out = {}
        if "rgb" in outputs:
            out["rgb"] = torch.empty(m, max(H, 0), max(W, 0), 3, dtype=torch.uint8, **kw)
        if "depth" in outputs:
            out["depth"] = torch.empty(m, max(H, 0), max(W, 0), dtype=torch.float32, **kw)
        if "seg" in outputs:
            out["seg"] = torch.empty(m, max(H, 0), max(W, 0), dtype=torch.int32, **kw)
        _lib.check(self._L.mb200_render(self._h, _ptr(ids), m, _ptr(view), _ptr(proj), W, H, _ptr(out.get("rgb")),
                                        _ptr(out.get("depth")), _ptr(out.get("seg")), self._stream()))
        return out

    # ---- trainer-facing extras (env_base.py:103-118, env_locomotion.py:76-77,224-282)
    eval_mode = False  # env_locomotion.py:52

    def evaluation_mode(self):
        _lib.check(self._L.mb200_set_param(self._h, b"eval_mode", 1.0))
        self.eval_mode = True

    def set_env_params(self, params: dict):
        for k, v in params.items():
            if k == "eval_mode":
                _lib.check(self._L.mb200_set_param(self._h, b"eval_mode", float(bool(v))))
                self.eval_mode = bool(v)

    def get_env_param(self, param_name, default):
        """EnvBase.get_env_param (env_base.py:116-117): the host-side mirror of the env attribute, else ``default``."""
        return getattr(self, param_name, default)

    def set_robot_params(self, params: dict):
        """EnvBase.set_robot_params (env_base.py:108-114) ends in ``self.robot.calc_torque_limits()``, a method no
        robot class of the reference defines (quirk Q4): the reference raises AttributeError, and so does this."""
        raise AttributeError("set_robot_params: the reference calls the undefined robot.calc_torque_limits() "
                             "(env_base.py:114); no robot parameter can be changed after construction")

    # the env credits info["steps_reached"] to the statistics at every episode end (the kernel's CREDIT_STEPS_REACHED)
    reports_steps_reached = False

    def stats(self, reset=False) -> dict:
        out = (C.c_double * 8)()
        _lib.check(self._L.mb200_stats(self._h, out, int(reset)))
        d = {"episodes": out[0], "return_sum": out[1], "length_sum": out[2], "nonfinite": out[3], "overflow": out[4]}
        if self.reports_steps_reached:
            d["steps_reached_sum"] = out[5]
        return d

    def launch_count(self) -> int:
        return int(self._L.mb200_launch_count(self._h))

    # observation entries past the robot state that mirroring negates: the target's lateral offset
    mirror_neg_targets = (0,)

    def get_mirror_indices(self):
        """Walker3DCustomEnv / Walker3DStepperEnv.get_mirror_indices (env_locomotion.py:224-282,761-840) -- static
        index tables."""
        A = self.act_dim
        right_j = np.array(self.table["right_joint_indices"], dtype=np.int64)
        left_j = np.array(self.table["left_joint_indices"], dtype=np.int64)
        neg_j = np.array(self.table["negation_joint_indices"], dtype=np.int64)
        nfeet = len(self.table["foot_links"])
        robot_obs = 6 + 2 * A + nfeet
        right = np.concatenate((right_j + 6, right_j + 6 + A, [6 + 2 * A + 2 * i for i in range(nfeet // 2)]))
        left = np.concatenate((left_j + 6, left_j + 6 + A, [6 + 2 * A + 2 * i + 1 for i in range(nfeet // 2)]))
        neg_obs = np.concatenate(([2, 4], 6 + neg_j, 6 + neg_j + A, robot_obs + np.array(self.mirror_neg_targets)))
        return neg_obs, right, left, neg_j, right_j, left_j


class Walker3DStepperVecEnv(Walker3DCustomVecEnv):
    """Batched Walker3DStepperEnv-v0 (reference env_locomotion.py:330-840): seeded stepping-stone terrain, three
    recycled LargePlanks with soft contacts, fixed-order curriculum 0..9 (per env)."""

    env_id = STEPPER_ID
    ES_NEXT, ES_CURRIC, ES_STEPS_REACHED, ES_TERRAIN = 22, 27, 31, 68
    max_curriculum = 9
    curriculum = 0  # env_locomotion.py:363
    reports_steps_reached = True
    # the lateral offset and the x tilt of each of the three step targets (env_locomotion.py:761-840)
    mirror_neg_targets = (0, 3, 5, 8, 10, 13)
    evaluation_mode = _unsupported("Walker3DStepperEnv has no evaluation_mode (reference: only Walker3DCustomEnv)")

    def __init__(self, num_envs: int, device="cuda:0", seed: int | None = None, physics: dict | None = None,
                 return_final_obs: bool = False, random_reward: bool = False, plank_class: str | None = None):
        """``random_reward`` and ``plank_class`` are the reference's constructor kwargs (env_locomotion.py:355-357):
        every reward term scaled by its own np_random.uniform(0.8, 1.2) draw each step (:532-547); "LargePlank"
        (default, 0.5 x 10 m), "Plank" (0.5 x 0.75 m) or "Pillar" (capped cylinders of radius 0.25, bullet_objects.py:86-90)
        stepping stones."""
        super().__init__(num_envs, device=device, seed=seed, physics=physics, return_final_obs=return_final_obs)
        self.random_reward = bool(random_reward)
        if self.random_reward:
            _lib.check(self._L.mb200_set_param(self._h, b"random_reward", 1.0))
        classes = {"LargePlank": 0.0, "Plank": 1.0, "Pillar": 2.0}
        if plank_class is not None and plank_class not in classes:
            # the reference does globals().get(plank_class, LargePlank) (env_locomotion.py:356-357); a misspelt
            # class silently becoming LargePlank is not reproduced
            raise ValueError("plank_class %r: one of %s" % (plank_class, sorted(classes)))
        self.plank_class = plank_class or "LargePlank"
        if classes[self.plank_class]:
            _lib.check(self._L.mb200_set_param(self._h, b"plank_class", classes[self.plank_class]))

    def set_env_params(self, params: dict):
        """``{"curriculum": c}`` with an int or one value per env (env_base.py:103-106); used at the next reset
        for the terrain and immediately for gain / terminal height, like the reference's attribute."""
        for k, v in params.items():
            if k != "curriculum":
                continue
            if np.isscalar(v) or isinstance(v, int):
                _lib.check(self._L.mb200_set_param(self._h, b"curriculum", float(min(int(v), self.max_curriculum))))
                self.curriculum = min(int(v), self.max_curriculum)
            else:
                arr = np.ascontiguousarray(np.minimum(np.asarray(v), self.max_curriculum), dtype=np.float32)
                _lib.check(self._L.mb200_set_param_array(self._h, b"curriculum", arr.ctypes.data_as(C.c_void_p),
                                                         len(arr)))
                self.curriculum = arr.astype(np.int64)

    def _host_params(self) -> dict:
        cur = self.curriculum
        return {"curriculum": cur.tolist() if isinstance(cur, np.ndarray) else int(cur),
                "random_reward": self.random_reward, "plank_class": self.plank_class}

    def _apply_host_params(self, params: dict):
        classes = {"LargePlank": 0.0, "Plank": 1.0, "Pillar": 2.0}
        if "plank_class" in params:
            self.plank_class = params["plank_class"]
            _lib.check(self._L.mb200_set_param(self._h, b"plank_class", classes[self.plank_class]))
        if "random_reward" in params:
            self.random_reward = bool(params["random_reward"])
            _lib.check(self._L.mb200_set_param(self._h, b"random_reward", float(self.random_reward)))
        if "curriculum" in params:
            self.set_env_params({"curriculum": params["curriculum"]})

    def steps_reached(self) -> torch.Tensor:
        """info["steps_reached"] per env of the last step (env_locomotion.py:562-566), -1 where not reported
        (mb200_info: written by the step kernel, no record read-back)."""
        return self.step_info()

    def terrain_info(self) -> torch.Tensor:
        return self.get_record()[:, self.ES_TERRAIN:self.ES_TERRAIN + 120].reshape(self.num_envs, 20, 6)



class Child3DCustomVecEnv(Walker3DCustomVecEnv):
    """Batched Child3DCustomEnv-v0 (reference env_locomotion.py:317-327, robots.py:326-335): Walker3DCustomEnv's
    logic on the child3d model (power 0.4), started in the "crawl" pose at z = 0.38 with the base pitched by 90
    degrees, episode over below a relative height of 0.1."""

    env_id = CHILD_ID
    model = "child3d"


class Walker2DCustomVecEnv(Walker3DCustomVecEnv):
    """Batched Walker2DCustomEnv-v0 (reference env_locomotion.py:285-310, robots.py:338-370): Walker3DCustomEnv's
    logic on the planar walker2d model (7 hinges about y; the root's "ignore*" slide / hinge joints are a free base
    that stays exactly in the x-z plane).  The reference forces done to False (:303), so only the 1000-step
    TimeLimit ends an episode, and reset() returns zeros in the two target slots (:298)."""

    env_id = WALKER2D_ID
    model = "walker2d"


class Crab2DCustomVecEnv(Walker2DCustomVecEnv):
    """Batched Crab2DCustomEnv-v0 (reference env_locomotion.py:312-314, robots.py:373-404): the same env on crab2d.xml
    (6 hinges, self-collision flags on)."""

    env_id = CRAB2D_ID
    model = "crab2d"


class MikeStepperVecEnv(Walker3DStepperVecEnv):
    """Batched MikeStepperEnv-v0 (reference env_locomotion.py:843-851, robots.py:474-513): Walker3DStepperEnv's
    logic on the mike model (own power table, waist mass 8), started at (0.3, 0, 1.0)."""

    env_id = MIKE_ID
    model = "mike"


class Monkey3DCustomVecEnv(Walker3DCustomVecEnv):
    """Batched Monkey3DCustomEnv-v0 (reference env_locomotion.py:1136-1516): 23-DoF brachiator released at 20 m
    with both hands on the first two of 32 seeded monkey bars (4 physical bars, recycled); the finger joints are
    scripted by the env (swing hand opens, pivot hand closes)."""

    env_id = MONKEY_ID
    model = "monkey3d"
    EM_NEXT, EM_FREEFALL, EM_TIMESTEP, EM_SWING, EM_PIVOT, EM_BAR, EM_TERRAIN = 22, 23, 24, 25, 26, 32, 64
    reports_steps_reached = True
    evaluation_mode = _unsupported("Monkey3DCustomEnv has no evaluation_mode (reference: only Walker3DCustomEnv)")
    set_env_params = _unsupported()
    get_mirror_indices = _unsupported("Monkey3DCustomEnv defines no get_mirror_indices in the reference")

    def _action_space(self):  # env_locomotion.py:1179-1181: unbounded torque space
        return Box(-np.inf * np.ones(self.act_dim), np.inf * np.ones(self.act_dim))

    def terrain_info(self) -> torch.Tensor:
        return self.get_record()[:, self.EM_TERRAIN:self.EM_TERRAIN + 128].reshape(self.num_envs, 32, 4)

    def next_step_index(self) -> torch.Tensor:
        return self.get_record()[:, self.EM_NEXT].contiguous().view(torch.int32)


class CassieVecEnv(Walker3DCustomVecEnv):
    """Batched CassieEnv-v0 (reference env_cassie.py:285-479, registered at __init__.py:18-22): 10 residual PD targets
    per env step, 50 PD-controlled 0.6 ms physics steps inside the kernel, two point-to-point loop closures
    (achilles rods).  The reference file does not import as shipped (SURVEY App. D Q7-Q9); this is its intended
    behaviour.  The env draws no random numbers: reset restores the saved initial state."""

    env_id = CASSIE_ID
    model = "cassie"
    control_step = 0.03  # env_cassie.py:287
    llc_frame_skip = 50  # env_cassie.py:288
    sim_frame_skip = 1  # env_cassie.py:289
    EC_POTENTIAL, EC_JVEL = 22, 32
    evaluation_mode = _unsupported("CassieEnv has no evaluation_mode")
    set_env_params = _unsupported()
    get_mirror_indices = _unsupported("CassieEnv-v0 defines no get_mirror_indices in the reference")

    def rewards_info(self, obs_rew: torch.Tensor | None = None) -> dict:
        """The reference returns the reward terms as ``info`` (env_cassie.py:479): AliveRew = +2 / -1,
        ProgressRew = reward - AliveRew."""
        rew = self.rew if obs_rew is None else obs_rew
        alive = torch.where(self.done.bool() & ~self.trunc.bool(), -1.0, 2.0)
        return {"AliveRew": alive, "ProgressRew": rew - alive}


class Walker3DCustomEnv:
    """gym-protocol facade over a 1-env batch; NumPy float64 observations like the reference."""

    metadata = {"render.modes": ["rgb_array"]}
    vec_class = Walker3DCustomVecEnv
    vec_kwargs = ()  # reference constructor kwargs this env's VecEnv understands

    def __init__(self, device="cuda:0", seed=None, render=False, **kwargs):
        if render:
            raise NotImplementedError("rendering is out of scope for the GPU path (SURVEY.md section 2, row 2)")
        extra = {k: kwargs[k] for k in self.vec_kwargs if k in kwargs}
        self.vec = self.vec_class(1, device=device, seed=seed, return_final_obs=True, **extra)
        self.observation_space = self.vec.observation_space
        self.action_space = self.vec.action_space
        self._pending_reset_obs = None

    def seed(self, seed=None):
        # the kernel's auto-reset drew from the old stream: a reset() after seed() must draw from the new one
        self._pending_reset_obs = None
        return [self.vec.seed(seed)[0]]

    def reset(self):
        if self._pending_reset_obs is not None:
            # the kernel already reset this env (same RNG draws reset() would make) when the episode ended
            obs, self._pending_reset_obs = self._pending_reset_obs, None
            return obs
        return self.vec.reset()[0].double().cpu().numpy()

    def step(self, action):
        a = np.asarray(action, dtype=np.float64)
        assert np.isfinite(a).all()  # robots.py:32
        self._pending_reset_obs = None
        act = torch.as_tensor(a, dtype=torch.float32).reshape(1, -1)
        obs, rew, done, info = self.vec.step(act)
        d = bool(done[0].item())
        out_info = {}
        if d:
            self._pending_reset_obs = obs[0].double().cpu().numpy()
            o = info["terminal_observation"][0].double().cpu().numpy()
            if bool(info["TimeLimit.truncated"][0].item()):
                out_info["TimeLimit.truncated"] = True
        else:
            o = obs[0].double().cpu().numpy()
        self._extra_info(out_info)
        return o, float(rew[0].item()), d, out_info

    def _extra_info(self, info):
        pass

    def set_env_params(self, params):
        # the usual trainer pattern is set_env_params({"curriculum": c}) between done and reset(): the cached
        # auto-reset observation belongs to the OLD parameters, so reset() must run a real reset (the reference's
        # reset() reads the new attribute; the auto-reset's RNG draws are spent, documented in INTEGRATION.md)
        self._pending_reset_obs = None
        self.vec.set_env_params(params)

    def get_env_param(self, param_name, default):
        return self.vec.get_env_param(param_name, default)

    def set_robot_params(self, params):
        self.vec.set_robot_params(params)

    def evaluation_mode(self):
        self._pending_reset_obs = None
        self.vec.evaluation_mode()

    def get_mirror_indices(self):
        return self.vec.get_mirror_indices()

    def apply_impulse(self, impulse, link=-1, point=None):
        """Push the robot before the next ``step``: ``impulse`` (N s, world frame, 3 values) at the world ``point``
        on ``link`` (see ``Walker3DCustomVecEnv.apply_impulse``; ``link_index`` maps link names)."""
        pt = None if point is None else np.asarray(point, dtype=np.float32).reshape(3)
        self.vec.apply_impulse(np.asarray(impulse, dtype=np.float32).reshape(3), link=link, point=pt)

    def link_index(self, name):
        return self.vec.link_index(name)

    def render(self, mode="rgb_array", width=320, height=240):
        """An [height, width, 3] uint8 frame of the env from the tracking camera (``VecEnv.render``).  There is no
        GUI: mode="human" raises NotImplementedError."""
        if mode == "human":
            raise NotImplementedError("render(mode='human') needs a GUI; the GPU path renders mode='rgb_array' only")
        if mode != "rgb_array":
            raise ValueError("render mode %r: one of %s" % (mode, self.metadata["render.modes"]))
        return self.vec.render(width=width, height=height, outputs=("rgb",))["rgb"][0].cpu().numpy()

    def close(self):
        self.vec.close()


class Walker3DStepperEnv(Walker3DCustomEnv):
    """gym-protocol facade of Walker3DStepperEnv-v0; info carries "steps_reached" like the reference."""

    vec_class = Walker3DStepperVecEnv
    vec_kwargs = ("random_reward", "plank_class")  # env_locomotion.py:355-357
    evaluation_mode = _unsupported("Walker3DStepperEnv has no evaluation_mode")

    def _extra_info(self, info):
        sr = int(self.vec.steps_reached()[0].item())
        if sr >= 0:
            info["steps_reached"] = sr


class Child3DCustomEnv(Walker3DCustomEnv):
    """gym-protocol facade of Child3DCustomEnv-v0."""

    vec_class = Child3DCustomVecEnv


class Walker2DCustomEnv(Walker3DCustomEnv):
    """gym-protocol facade of Walker2DCustomEnv-v0."""

    vec_class = Walker2DCustomVecEnv


class Crab2DCustomEnv(Walker3DCustomEnv):
    """gym-protocol facade of Crab2DCustomEnv-v0."""

    vec_class = Crab2DCustomVecEnv


class MikeStepperEnv(Walker3DStepperEnv):
    """gym-protocol facade of MikeStepperEnv-v0."""

    vec_class = MikeStepperVecEnv


class Monkey3DCustomEnv(Walker3DCustomEnv):
    """gym-protocol facade of Monkey3DCustomEnv-v0.  The reference overwrites the two finger entries of the caller's
    action array in place (env_locomotion.py:1322-1323, quirk Q11); the kernel applies the same override internally
    and this facade mirrors the visible side effect."""

    vec_class = Monkey3DCustomVecEnv
    evaluation_mode = _unsupported("Monkey3DCustomEnv has no evaluation_mode")

    def step(self, action):
        rec = self.vec.get_record()[0]
        swing = int(rec[self.vec.EM_SWING].view(torch.int32).item())
        pivot = int(rec[self.vec.EM_PIVOT].view(torch.int32).item())
        out = super().step(action)
        if isinstance(action, np.ndarray):
            action[17 if swing == 0 else 22] = 1
            action[17 if pivot == 0 else 22] = -1
        return out


class CassieEnv(Walker3DCustomEnv):
    """gym-protocol facade of CassieEnv-v0; ``info`` carries the reward terms like the reference."""

    vec_class = CassieVecEnv
    evaluation_mode = _unsupported("CassieEnv has no evaluation_mode")

    def _extra_info(self, info):
        r = self.vec.rewards_info()
        info["AliveRew"] = float(r["AliveRew"][0].item())
        info["ProgressRew"] = float(r["ProgressRew"][0].item())


_REGISTRY = {ENV_ID: (Walker3DCustomEnv, Walker3DCustomVecEnv), STEPPER_ID: (Walker3DStepperEnv, Walker3DStepperVecEnv),
             MONKEY_ID: (Monkey3DCustomEnv, Monkey3DCustomVecEnv), CASSIE_ID: (CassieEnv, CassieVecEnv),
             CHILD_ID: (Child3DCustomEnv, Child3DCustomVecEnv), MIKE_ID: (MikeStepperEnv, MikeStepperVecEnv),
             WALKER2D_ID: (Walker2DCustomEnv, Walker2DCustomVecEnv), CRAB2D_ID: (Crab2DCustomEnv, Crab2DCustomVecEnv)}


def make(env_id: str, num_envs: int | None = None, **kwargs):
    """gym.make analogue: ``make("Walker3DCustomEnv-v0")`` -> gym-style env, ``make(id, num_envs=N)`` -> VecEnv."""
    eid = env_id.split(":")[-1]
    if eid not in _REGISTRY:
        raise KeyError("env id %r is not built yet (available: %s)" % (env_id, ", ".join(_REGISTRY)))
    single, vec = _REGISTRY[eid]
    if num_envs is None:
        return single(**kwargs)
    return vec(num_envs, **kwargs)
