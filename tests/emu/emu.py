"""ctypes binding of the lane-loop emulation of the kernel source (tests only; see emu.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libmb_emu.so")
_SRC = [os.path.join(_HERE, "emu.cpp")] + [
    os.path.join(_HERE, "..", "..", "mocca_envs_b200", "csrc", f)
    for f in ("mb_core.cuh", "mb_env.cuh", "mb_tables.h", "generated/walker3d_model.h", "generated/monkey3d_model.h",
              "generated/cassie_model.h", "generated/child3d_model.h", "generated/mike_model.h",
              "generated/walker2d_model.h", "generated/crab2d_model.h")]


class Phys(C.Structure):
    _fields_ = [("dt", C.c_float), ("substeps", C.c_int), ("iterations", C.c_int), ("gravity", C.c_float),
                ("erp_contact", C.c_float), ("erp_joint", C.c_float), ("linear_slop", C.c_float),
                ("lin_damping", C.c_float), ("ang_damping", C.c_float), ("max_coord_vel", C.c_float),
                ("limit_max_impulse", C.c_float), ("split_threshold", C.c_float), ("residual_threshold", C.c_float),
                ("ground_friction", C.c_float), ("has_ground", C.c_int), ("box_friction", C.c_float),
                ("box_erp", C.c_float), ("box_cfm", C.c_float), ("bar_friction", C.c_float), ("self_collision", C.c_int),
                ("warmstart", C.c_float)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        stale = (not os.path.exists(_LIB)) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in _SRC)
        if stale:
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                                   "-Wno-unused-variable", "-o", _LIB, _SRC[0]])
        _lib = C.CDLL(_LIB)
        assert _lib.emu_sizeof_phys() == C.sizeof(Phys)
    return _lib


def default_phys():
    """The plain reference physics (Walker3DCustomEnv has no physics of its own)."""
    return EmuW3D.phys()


def _fp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class EmuEnv:
    """One env through the emulated kernel source: emu_<prefix>_* in emu.cpp (record layout: ER_* and the kind's
    additions in mb_env.cuh).  A subclass per env kind names its prefix and dimensions."""

    prefix = None
    obs_dim = act_dim = n_dof = None
    aliased = 1  # ER_ALIASED: the robot draws from the env stream until the env is re-seeded

    @classmethod
    def phys(cls):
        """The kind's physics as mb200_create sets them when the caller passes none."""
        p = Phys()
        getattr(lib(), "emu_%s_phys" % cls.prefix)(C.byref(p))
        return p

    def __init__(self, mt_state=None, phys=None):
        self.p = phys or self.phys()
        self.state = np.zeros(64, dtype=np.float32)
        self.rec = np.zeros(self._call("rec_stride"), dtype=np.float32)
        self.rec.view(np.int32)[11] = self.aliased
        self.mt = np.zeros((2, 640), dtype=np.uint32)
        if mt_state is not None:
            self.mt[0, :625] = mt_state
        self.mt[1, 624] = 624
        self.stats = np.zeros(6)  # accumulated MbStats, in the order of mb200_stats

    def _call(self, what, *args):
        return getattr(lib(), "emu_%s_%s" % (self.prefix, what))(*args)

    def reset(self):
        obs = np.zeros(self.obs_dim, dtype=np.float32)
        self._call("reset", C.byref(self.p), _fp(self.state), _fp(self.rec), _fp(self.mt[0]), _fp(self.mt[1]), _fp(obs))
        return obs

    def step(self, act):
        act = np.ascontiguousarray(act, dtype=np.float32)
        obs = np.zeros(self.obs_dim, dtype=np.float32)
        fin = np.zeros(self.obs_dim, dtype=np.float32)
        rew = np.zeros(1, dtype=np.float32)
        done = np.zeros(1, dtype=np.uint8)
        trunc = np.zeros(1, dtype=np.uint8)
        st = np.zeros(6)
        self._call("step", C.byref(self.p), _fp(self.state), _fp(self.rec), _fp(self.mt[0]), _fp(self.mt[1]),
                   _fp(act), _fp(obs), _fp(rew), _fp(done), _fp(trunc), _fp(fin), _fp(st))
        self.stats += st
        return obs, float(rew[0]), bool(done[0]), bool(trunc[0]), fin

    def step_physics(self, tau, warm=None, points=None):
        """One stepSimulation of self.state (in place) with the obstacles of self.rec, joint torques `tau` held.
        `warm` (float32[384], updated in place) switches warm starting on; `points` (float32[16, 10]) receives the
        contact points of the last collision pass.  Returns (rows, contacts)."""
        tau = np.ascontiguousarray(tau, dtype=np.float32)
        rows, nc = C.c_int(0), C.c_int(0)
        self._call("step_physics", C.byref(self.p), _fp(self.state), _fp(self.rec), _fp(tau), _fp(warm), _fp(points),
                   C.byref(rows), C.byref(nc))
        return rows.value, nc.value

    def mass_matrix(self):
        """(mass matrix, bias forces) at self.state."""
        nu = 6 + self.n_dof
        M = np.zeros((nu, nu), dtype=np.float32)
        b = np.zeros(nu, dtype=np.float32)
        self._call("mass_matrix", C.byref(self.p), _fp(self.state), _fp(M), _fp(b))
        return M, b


class EmuW3D(EmuEnv):
    """Walker3DCustomEnv."""
    prefix = "w3d"
    obs_dim, act_dim, n_dof = 52, 21, 21


class EmuChild(EmuW3D):
    """Child3DCustomEnv-v0: the Walker3DCustomEnv template on the child3d table."""
    prefix = "child"


class EmuWalker2D(EmuW3D):
    """Walker2DCustomEnv-v0: the Walker3DCustomEnv template on the planar walker2d table."""
    prefix = "walker2d"
    obs_dim, act_dim, n_dof = 24, 7, 7


class EmuCrab2D(EmuW3D):
    """Crab2DCustomEnv-v0."""
    prefix = "crab2d"
    obs_dim, act_dim, n_dof = 22, 6, 6


class EmuStepper(EmuEnv):
    """Walker3DStepperEnv (record additions ES_*)."""

    prefix = "stepper"
    obs_dim, act_dim, n_dof = 65, 21, 21

    ES_NEXT, ES_COUNT, ES_STOP, ES_SETSTOP, ES_TIMESTEP, ES_CURRIC, ES_PLANKIDX, ES_STEPS = 22, 23, 24, 25, 26, 27, 28, 31
    ES_BOX, ES_TERRAIN = 32, 68

    def __init__(self, mt_state=None, curriculum=0, phys=None):
        super().__init__(mt_state, phys)
        self.rec.view(np.int32)[self.ES_CURRIC] = curriculum

    def terrain(self):
        return self.rec[self.ES_TERRAIN:self.ES_TERRAIN + 120].reshape(20, 6)


class EmuPillar(EmuStepper):
    """Walker3DStepperEnv with plank_class = "Pillar"."""
    prefix = "pillar"


class EmuMike(EmuStepper):
    """MikeStepperEnv-v0: the Walker3DStepperEnv template on the mike table."""
    prefix = "mike"


class EmuMonkey(EmuEnv):
    """Monkey3DCustomEnv (record additions EM_*)."""

    prefix = "monkey"
    obs_dim, act_dim, n_dof = 69, 23, 23

    EM_NEXT, EM_FREEFALL, EM_TIMESTEP, EM_SWING, EM_PIVOT, EM_SWINGPOT, EM_BARIDX, EM_BAR, EM_TERRAIN = \
        22, 23, 24, 25, 26, 27, 28, 32, 64

    def terrain(self):
        return self.rec[self.EM_TERRAIN:self.EM_TERRAIN + 128].reshape(32, 4)


class EmuCassie(EmuEnv):
    """CassieEnv-v0 (record additions EC_*).  Deterministic: its MT streams are never drawn from."""

    prefix = "cassie"
    obs_dim, act_dim, n_dof = 36, 10, 18
    aliased = 0

    EC_POTENTIAL, EC_JVEL = 22, 32
