"""Monkey3DCustomEnv-v0: the CUDA kernel SOURCE (compiled by g++ as a 32-lane loop, tests/emu) diffed against the
float64 oracle -- model dynamics, bar contacts (sphere / capsule / box vs thin cylinder), terrain generation,
env step.  The GPU tests repeat these through the C ABI."""
import numpy as np

from tests.emu import emu as E
from tests.helpers import oracle_state, random_states, state_error


def _mt_row(O, seed):
    st = np.random.RandomState(O.gym_seed_words(seed)).get_state()
    return np.concatenate([st[1], [st[2]]]).astype(np.uint32)


def test_monkey_mass_matrix_and_bias(monkey_table, oracle_mod):
    O, t = oracle_mod, monkey_table
    A = t["n_dof"]
    m = O.model_from_table(t)
    p = O.default_params()
    emu = E.EmuMonkey()
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


def test_monkey_reset_terrain(monkey_table, oracle_mod):
    """Reset state bit-exact; bar layout from the same seed equal after f32 rounding, except that rows derived from
    the hand positions inherit the f32 forward kinematics at 20 m altitude (ulp 1.9e-6)."""
    O, t = oracle_mod, monkey_table
    for seed in range(4):
        env = O.Monkey3DOracle(t, seed=seed)
        emu = E.EmuMonkey(_mt_row(O, seed))
        for _ in range(2):
            o1, o2 = env.reset(), emu.reset()
            ref = np.array([list(r) for r in env.e.terrain]).astype(np.float32)
            assert np.abs(emu.terrain() - ref).max() < 2e-5
            # increments between bars (the seeded part) are exact to f32 rounding of the cumulative sums
            assert np.abs(np.diff(emu.terrain()[1:, 0]) - np.diff(ref[1:, 0])).max() < 4e-6
            assert np.array_equal(emu.state[13:36], np.array(env.e.base.s.q[:23]).astype(np.float32))
            assert np.array_equal(emu.state[0:3], np.array([0.0, 0.0, 20.0], dtype=np.float32))
            assert np.array_equal(emu.state[10:13], np.array([3.0, 0.0, -1.0], dtype=np.float32))
            ri = emu.rec.view(np.int32)
            assert (ri[E.EmuMonkey.EM_SWING], ri[E.EmuMonkey.EM_PIVOT]) == (env.e.swing_leg, env.e.pivot_leg)
            assert np.abs(o1 - o2).max() < 2e-5


def _force(env, emu):
    """Teacher-force the oracle's state (rounded to f32) and bookkeeping into the emulated kernel."""
    A = 23
    sv = env.state_vector().astype(np.float32)
    emu.state[:13 + 2 * A] = sv
    b = env.e.base
    for k in range(3):
        b.s.pos[k] = float(sv[k]); b.s.omega[k] = float(sv[7 + k]); b.s.vel[k] = float(sv[10 + k])
    for k in range(4):
        b.s.quat[k] = float(sv[3 + k])
    for k in range(A):
        b.s.q[k] = float(sv[13 + k]); b.s.qd[k] = float(sv[13 + A + k])
    ri = emu.rec.view(np.int32)
    emu.rec[0:3] = np.array(b.walk_target[:], dtype=np.float32)
    emu.rec[9], emu.rec[10] = b.feet_contact[0], b.feet_contact[1]
    ri[8] = b.elapsed
    M = E.EmuMonkey
    ri[M.EM_NEXT], ri[M.EM_FREEFALL], ri[M.EM_TIMESTEP] = env.e.next_step_index, env.e.free_fall_count, env.e.timestep
    ri[M.EM_SWING], ri[M.EM_PIVOT] = env.e.swing_leg, env.e.pivot_leg
    emu.rec[M.EM_SWINGPOT] = env.e.swing_potential
    emu.rec[M.EM_TERRAIN:M.EM_TERRAIN + 128] = np.array([list(r) for r in env.e.terrain], dtype=np.float32).ravel()
    for k in range(4):
        bar = env.e.bars[k]
        emu.rec[M.EM_BAR + 8 * k:M.EM_BAR + 8 * k + 8] = np.array(
            list(bar.center) + list(bar.axis) + [bar.halflen, bar.radius], dtype=np.float32)


def test_monkey_env_step_teacher_forced(oracle_mod):
    """Monkey3DCustomEnv.step (hand / palm contacts with the bars, scripted finger joints, swing progress, free-fall
    termination) from f32-identical states, 4 envs x 60 steps.  Steps outside 1e-3 (obs) / 1e-2 (reward) must be explained by a verified
    discontinuity and bounded (tests/teacher.py), else the test fails; integer bookkeeping read back and compared
    exactly after every structurally identical step."""
    from tests import teacher as T

    js = T.run_vs_oracle(oracle_mod, "monkey", "emu", (3, 4, 5, 6), 60, lambda rng, k: 0.5 * rng.uniform(-1, 1, 23))
    assert np.median(np.concatenate([j.errs for j in js])) < 3e-4
