"""CPU checks of the CUDA kernel SOURCE: mb_core.cuh / mb_env.cuh compiled by g++ as a 32-lane loop
(tests/emu) and diffed against the float64 oracle.  The GPU tests (-m gpu) repeat these through the C ABI on the
real device; this file exists so that kernel-logic regressions are caught on a box without a GPU."""
import ctypes as C

import numpy as np
import pytest

from tests.emu import emu as E
from tests.helpers import contact_states, oracle_state, random_states, self_contact_states, state_error


def test_mass_matrix_and_bias(walker_table, oracle_mod):
    O, t = oracle_mod, walker_table
    A = t["n_dof"]
    m = O.model_from_table(t)
    p = O.default_params()
    emu = E.EmuW3D()
    rng = np.random.RandomState(0)
    for row in random_states(t, rng, 6):
        s = oracle_state(O, A, row)
        M = O.mass_matrix(m, s)
        emu.state[:len(row)] = row
        Me, be = emu.mass_matrix()
        assert np.abs(Me - M).max() / np.abs(M).max() < 1e-6
        acc = O.forward_dynamics(m, p, s, np.zeros(A), with_damping=True)
        bias = -M @ acc
        assert np.abs(be - bias).max() / np.abs(bias).max() < 1e-5


def test_contact_free_step(walker_table, oracle_mod):
    """north_star: contact-free single-step state within 1e-4."""
    O, t = oracle_mod, walker_table
    A = t["n_dof"]
    m = O.model_from_table(t)
    p = O.default_params()
    emu = E.EmuW3D()
    rng = np.random.RandomState(1)
    gain = np.array(t["gain"])
    for row in random_states(t, rng, 8, spin=0.5, margin=0.35):
        tau = gain * rng.uniform(-1, 1, A)
        s = oracle_state(O, A, row)
        _, rows = O.step_physics(m, p, s, tau)
        emu.state[:len(row)] = row
        erows, _ = emu.step_physics(tau)
        assert rows == erows == 0
        assert state_error(emu.state[:len(row)], O.state_vector(s, A)) < 1e-4


def test_contact_step(walker_table, oracle_mod):
    """north_star: per-step contact rollouts within a stated tolerance over 1 frame: 2e-3 (state-scaled)."""
    O, t = oracle_mod, walker_table
    A = t["n_dof"]
    m = O.model_from_table(t)
    p = O.default_params()
    emu = E.EmuW3D()
    rng = np.random.RandomState(2)
    gain = np.array(t["gain"])
    worst = 0.0
    for row in contact_states(O, t, rng, 12):
        row = row.astype(np.float32).astype(np.float64)
        tau = 0.3 * gain * rng.uniform(-1, 1, A)
        s = oracle_state(O, A, row)
        c, rows = O.step_physics(m, p, s, tau)
        emu.state[:len(row)] = row
        erows, enc = emu.step_physics(tau)
        assert enc == c.n
        assert abs(rows - erows) <= 2  # a limit row can flip at an exact boundary
        worst = max(worst, state_error(emu.state[:len(row)], O.state_vector(s, A)))
    assert worst < 2e-3, worst


def test_self_contact_step(walker_table, oracle_mod):
    """SURVEY 8 f1: self-collision (robots.py:259-264).  Limb-vs-limb contacts couple two links of the multibody;
    same 2e-3 one-frame tolerance and identical contact / row counts as the ground-contact test.  Switching the
    kernel's self-collision off must break the agreement (the test is sensitive to the feature)."""
    O, t = oracle_mod, walker_table
    A = t["n_dof"]
    m = O.model_from_table(t)
    p = O.default_params()
    emu = E.EmuW3D()
    off = E.default_phys()
    off.self_collision = 0
    emu_off = E.EmuW3D(phys=off)
    rng = np.random.RandomState(3)
    gain = np.array(t["gain"])
    worst, worst_off = 0.0, 0.0
    for row in self_contact_states(O, t, rng, 16):
        tau = gain * rng.uniform(-1, 1, A)
        s = oracle_state(O, A, row)
        c, rows = O.step_physics(m, p, s, tau)
        emu.state[:len(row)] = row
        erows, enc = emu.step_physics(tau)
        assert enc == c.n
        assert abs(rows - erows) <= 2
        worst = max(worst, state_error(emu.state[:len(row)], O.state_vector(s, A)))
        emu_off.state[:len(row)] = row
        emu_off.step_physics(tau)
        worst_off = max(worst_off, state_error(emu_off.state[:len(row)], O.state_vector(s, A)))
    assert worst < 2e-3, worst
    assert worst_off > 0.1, worst_off


def _mt_row(O, seed):
    st = np.random.RandomState(O.gym_seed_words(seed)).get_state()
    return np.concatenate([st[1], [st[2]]]).astype(np.uint32)


@pytest.mark.parametrize("eval_mode", [0, 1])
def test_reset_bit_exact(eval_mode, walker_table, oracle_mod):
    """north_star: bit-exact reset-state generation from the same seed (after rounding to the f32 state).  In
    evaluation mode randomize_target draws ONE word of the env stream (np_random.choice; dist / angle are constants,
    env_locomotion.py:67-74), so stop_frames comes from the first word and the robot's pose noise follows it."""
    O, t = oracle_mod, walker_table
    for seed in range(3):
        env = O.Walker3DCustomOracle(t, seed=seed)
        emu = E.EmuW3D(_mt_row(O, seed))
        env.e.eval_mode = eval_mode
        emu.rec.view(np.int32)[18] = eval_mode  # ER_EVAL
        for _ in range(3):
            o_ref = env.reset()
            o_emu = emu.reset()
            q_ref = np.array(env.e.s.q[:21]).astype(np.float32)
            assert np.array_equal(emu.state[13:34], q_ref)
            assert np.array_equal(emu.rec[:3], np.array(env.e.walk_target[:], dtype=np.float32))
            assert emu.rec[5] == env.e.stop_frames
            assert np.abs(o_ref - o_emu).max() < 1e-6


def test_env_step_teacher_forced(oracle_mod):
    """obs / reward / done of Walker3DCustomEnv.step from f32-identical states and bookkeeping (oracle state and record
    injected every step), random actions of amplitude 1.2, 6 envs x 40 steps.  Steps outside 1e-3 (obs) / 1e-2 (reward) must be explained by a verified
    discontinuity and bounded (tests/teacher.py), else the test fails; integer bookkeeping read back and compared
    exactly after every structurally identical step."""
    from tests import teacher as T

    js = T.run_vs_oracle(oracle_mod, "walker3d", "emu", range(5, 11), 40, lambda rng, k: rng.uniform(-1.2, 1.2, 21))
    assert np.median(np.concatenate([j.errs for j in js])) < 2e-4


# ------------------------------------------------------------------------------------------------ Stepper
def test_stepper_reset_terrain_bit_exact(walker_table, oracle_mod):
    """north_star: bit-exact terrain, stepping-stone layout and reset-state generation from the same seed
    (float64 generator on the device path, compared after rounding to the f32 record)."""
    O, t = oracle_mod, walker_table
    for seed, cur in ((0, 0), (1, 5), (2, 9)):
        env = O.Walker3DStepperOracle(t, seed=seed, curriculum=cur)
        emu = E.EmuStepper(_mt_row(O, seed), curriculum=cur)
        for _ in range(2):
            o1, o2 = env.reset(), emu.reset()
            assert np.array_equal(emu.terrain(), np.array(env.e.terrain[:]).astype(np.float32))
            assert np.array_equal(emu.state[13:34], np.array(env.e.base.s.q[:21]).astype(np.float32))
            assert np.array_equal(emu.state[0:3], np.array([0.3, 0.0, 1.32], dtype=np.float32))
            assert np.abs(o1 - o2).max() < 1e-6


def test_stepper_env_step_teacher_forced(oracle_mod):
    """Walker3DStepperEnv.step from f32-identical states and bookkeeping at curriculum 0 / 5 / 9: box contacts on soft
    planks, target advance, plank recycling, step bonus, look-ahead targets.  Steps outside 1e-3 (obs) / 1e-2 (reward) must be explained by a verified
    discontinuity and bounded (tests/teacher.py), else the test fails; integer bookkeeping read back and compared
    exactly after every structurally identical step."""
    from tests import teacher as T

    errs = []
    for seed, cur in ((300, 0), (301, 5), (302, 9), (303, 0)):
        js = T.run_vs_oracle(oracle_mod, "stepper", "emu", [seed], 50, lambda rng, k: 0.3 * rng.uniform(-1, 1, 21),
                             curriculum=cur)
        errs += js[0].errs
    assert np.median(errs) < 2e-4


def test_stepper_random_reward(walker_table, oracle_mod):
    """SURVEY 8 f2, random_reward kwarg (env_locomotion.py:355,528-547): every reward term is scaled by its own
    np_random.uniform(0.8, 1.2) draw.  Free-running from the same seed with zero actions (the first steps are
    contact-free and the stones are far away, so f32 and f64 stay together): rewards agree, differ from the plain
    reward, and the env stream stays in lockstep -- the terrain drawn at the next reset is bit-exact."""
    O, t = oracle_mod, walker_table
    seed, cur = 6, 5
    env = O.Walker3DStepperOracle(t, seed=seed, curriculum=cur, random_reward=True)
    plain = O.Walker3DStepperOracle(t, seed=seed, curriculum=cur)
    emu = E.EmuStepper(_mt_row(O, seed), curriculum=cur)
    emu.rec.view(np.int32)[3] = 1  # ES_RANDOM_REWARD
    env.reset(), plain.reset(), emu.reset()
    differs = 0
    for i in range(6):
        a = np.zeros(21)
        _, r1, d1, _ = env.step(a)
        _, r0, _, _ = plain.step(a)
        _, r2, d2, _, _ = emu.step(a)
        assert not d1 and not d2
        assert abs(r1 - r2) < 2e-3 + 1e-3 * abs(r1), (i, r1, r2)
        differs += abs(r1 - r0) > 1e-3 * abs(r0)
    assert differs >= 5
    env.reset(), emu.reset()
    assert np.array_equal(emu.terrain(), np.array(env.e.terrain[:]).astype(np.float32))


def test_stepper_plank_class(walker_table, oracle_mod):
    """plank_class kwarg (env_locomotion.py:342,356-357; bullet_objects.py:92-103): "Plank" stones are 0.75 m wide
    instead of 10 m.  A walker dropped 0.45 m to the side of the path lands with one foot off a Plank but with both
    feet on a LargePlank: kernel source and oracle agree for each class, and the two classes differ."""
    from tests.helpers import oracle_state, state_error

    O, t = oracle_mod, walker_table
    outs = {}
    for cls, flag in (("LargePlank", 0), ("Plank", 1)):
        env = O.Walker3DStepperOracle(t, seed=2, curriculum=0, plank_class=cls)
        emu = E.EmuStepper(_mt_row(O, 2), curriculum=0)
        emu.rec.view(np.int32)[4] = flag  # ES_PLANK_CLASS
        env.reset()
        emu.reset()
        m, p = env.m, O.default_params()
        p.has_ground = 0  # remove_ground=True (env_locomotion.py:359)
        sv = env.state_vector()
        sv[1] += 0.45
        sv = sv.astype(np.float32)
        emu.state[:55] = sv
        s = oracle_state(O, 21, sv.astype(np.float64))
        boxes = (O.Box * 6)(*env.e.boxes)
        worst = 0.0
        for frame in range(30):
            c, rows = O.step_physics(m, p, s, np.zeros(21), boxes=boxes)
            erows, enc = emu.step_physics(np.zeros(21, dtype=np.float32))
            ref = O.state_vector(s, 21)
            worst = max(worst, state_error(emu.state[:55], ref))
            emu.state[:55] = ref.astype(np.float32)  # teacher-forced frame by frame
            s = oracle_state(O, 21, emu.state[:55].astype(np.float64))
        assert worst < 2e-3, (cls, worst)
        outs[cls] = O.state_vector(s, 21)
    assert np.abs(outs["Plank"] - outs["LargePlank"]).max() > 1e-2


def test_stepper_pillar_class(walker_table, oracle_mod):
    """plank_class = "Pillar" (bullet_objects.py:86-90, pillar.urdf): capped cylinders of radius 0.25.  A walker
    dropped 0.3 m to the side keeps one foot on a pillar and none... on the rim: kernel source (PILLAR instantiation)
    and oracle agree frame by frame, and the result differs from the LargePlank run."""
    from tests.helpers import oracle_state, state_error

    O, t = oracle_mod, walker_table
    outs = {}
    for cls, emu_cls in (("LargePlank", E.EmuStepper), ("Pillar", E.EmuPillar)):
        env = O.Walker3DStepperOracle(t, seed=2, curriculum=0, plank_class=cls)
        emu = emu_cls(_mt_row(O, 2), curriculum=0)
        env.reset()
        emu.reset()
        m, p = env.m, O.default_params()
        p.has_ground = 0
        sv = env.state_vector()
        sv[1] += 0.3
        sv = sv.astype(np.float32)
        emu.state[:55] = sv
        s = oracle_state(O, 21, sv.astype(np.float64))
        boxes = (O.Box * 6)(*env.e.boxes)
        assert all(bool(b.cylinder) == (cls == "Pillar") for b in boxes)
        worst, contacts = 0.0, 0
        for frame in range(30):
            c, rows = O.step_physics(m, p, s, np.zeros(21), boxes=boxes)
            erows, enc = emu.step_physics(np.zeros(21, dtype=np.float32))
            assert enc == c.n
            contacts += c.n
            ref = O.state_vector(s, 21)
            worst = max(worst, state_error(emu.state[:55], ref))
            emu.state[:55] = ref.astype(np.float32)
            s = oracle_state(O, 21, emu.state[:55].astype(np.float64))
        assert contacts > 0
        assert worst < 2e-3, (cls, worst)
        outs[cls] = O.state_vector(s, 21)
    assert np.abs(outs["Pillar"] - outs["LargePlank"]).max() > 1e-2


def test_warm_start_switch(walker_table, oracle_mod):
    """Bullet-version switch MbPhysics.warmstart (SURVEY App. B.3, OQ11): contact normal rows start from f x the impulse
    of the same candidate point in the previous substep.  Flipping it changes the oracle and the kernel source TOGETHER:
    three consecutive stepSimulations from in-contact states agree within the contact-frame tolerance (2e-3) with the
    switch on, and the switched-on result differs from the switched-off one by far more than that."""
    from tests.helpers import contact_states, oracle_state, state_error

    O, t = oracle_mod, walker_table
    A = 21
    m = O.model_from_table(t)
    rng = np.random.RandomState(5)
    states = contact_states(O, t, rng, 12).astype(np.float32)
    worst_on, moved = 0.0, 0.0
    for st in states:
        tau = (0.3 * np.array(t["gain"]) * rng.uniform(-1, 1, A)).astype(np.float32)
        outs = {}
        for f in (0.0, 0.85):
            p = O.default_params()
            p.warmstart = f
            pe = E.default_phys()
            pe.warmstart = f
            s = oracle_state(O, A, st.astype(np.float64))
            warm_o = (C.c_double * 384)()
            warm_e = np.zeros(384, dtype=np.float32)
            emu = E.EmuW3D(phys=pe)
            emu.state[:len(st)] = st
            for k in range(3):
                O.step_physics(m, p, s, tau.astype(np.float64), warm=warm_o)
                emu.step_physics(tau, warm=warm_e if f > 0 else None)
            se = emu.state[:len(st)].copy()
            outs[f] = (O.state_vector(s, A), se)
            if f > 0:
                worst_on = max(worst_on, state_error(se, O.state_vector(s, A)))
                assert np.abs(warm_e - np.array(warm_o[:], dtype=np.float32)).max() < 2e-3 * max(1.0, np.abs(warm_e).max())
        moved = max(moved, state_error(outs[0.85][1], outs[0.0][1]))
    assert worst_on < 2e-3, worst_on
    assert moved > 2e-2, moved
