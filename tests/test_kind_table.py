"""The env kinds' configuration (csrc/mb_env.cuh, exported through MbKindOps) is what both the library and the CPU
emulation run: the physics defaults per env id, the stepper's fix-ups, and the ids mb200_create knows."""
import ctypes as C
import re

import numpy as np
import pytest

from mocca_envs_b200 import _lib
from tests.emu import emu as E

EMU = {
    "Walker3DCustomEnv-v0": E.EmuW3D, "Walker3DStepperEnv-v0": E.EmuStepper, "Monkey3DCustomEnv-v0": E.EmuMonkey,
    "CassieEnv-v0": E.EmuCassie, "Child3DCustomEnv-v0": E.EmuChild, "MikeStepperEnv-v0": E.EmuMike,
    "Walker2DCustomEnv-v0": E.EmuWalker2D, "Crab2DCustomEnv-v0": E.EmuCrab2D,
}
STEPPER_FAMILY = (E.EmuStepper, E.EmuPillar, E.EmuMike)


@pytest.mark.parametrize("env_id", sorted(EMU))
def test_library_defaults_match_emulation(env_id):
    p = _lib.Physics()
    _lib.lib().mb200_default_physics_for(env_id.encode(), C.byref(p))
    q = EMU[env_id].phys()
    for name, _ in _lib.Physics._fields_:
        if name != "has_ground":  # the stepper's fix-up removes the ground after the public defaults
            assert getattr(p, name) == getattr(q, name), name
    assert p.has_ground == 1


@pytest.mark.parametrize("cls", [E.EmuW3D, E.EmuStepper, E.EmuPillar, E.EmuMonkey, E.EmuCassie, E.EmuChild,
                                 E.EmuMike, E.EmuWalker2D, E.EmuCrab2D])
def test_emulated_ground_and_planks(cls):
    q = cls.phys()
    assert q.has_ground == (0 if cls in STEPPER_FAMILY else 1)
    if cls in STEPPER_FAMILY:
        # contactStiffness 30000, contactDamping 1000 + a link's default 0.1, at the default dt
        f = np.float32
        dt, kp, kd = f(1.0 / 240.0), f(30000.0), f(1000.0) + f(0.1)
        denom = dt * kp + kd
        assert q.box_erp == pytest.approx(float(dt * kp / denom), rel=1e-6)
        assert q.box_cfm == pytest.approx(float(f(1.0) / denom), rel=1e-6)


def test_unsupported_id_names_every_built_id():
    L = _lib.lib()
    h = C.c_void_p()
    assert L.mb200_create(b"NoSuchEnv-v0", 4, 0, None, C.byref(h)) != 0 and h.value is None
    msg = L.mb200_last_error().decode()
    assert "unsupported env id" in msg
    built = re.search(r"\(built: (.*)\)$", msg).group(1).split(", ")
    assert sorted(built) == sorted(EMU)
