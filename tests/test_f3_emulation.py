"""SURVEY 8 f3 -- more model tables through the same kernels: Child3DCustomEnv-v0 (env_locomotion.py:317-327,
robots.py:326-335, crawl start pose) and MikeStepperEnv-v0 (env_locomotion.py:843-851, robots.py:474-513).
CPU checks of the kernel source (tests/emu) against the float64 oracle; the GPU twins are in test_gpu_f3.py."""
import numpy as np
import pytest

from tests.emu import emu as E
from tests.helpers import force_oracle_state, oracle_record, oracle_state, random_states, state_error


def _mt_row(O, seed):
    st = np.random.RandomState(O.gym_seed_words(seed)).get_state()
    return np.concatenate([st[1], [st[2]]]).astype(np.uint32)


@pytest.mark.parametrize("name", ["child", "mike"])
def test_mass_matrix_and_bias(name, child_table, mike_table, oracle_mod):
    O, t = oracle_mod, {"child": child_table, "mike": mike_table}[name]
    A = t["n_dof"]
    m = O.model_from_table(t)
    p = O.default_params()
    emu = {"child": E.EmuChild, "mike": E.EmuMike}[name](phys=E.default_phys())
    rng = np.random.RandomState(0)
    for row in random_states(t, rng, 4):
        s = oracle_state(O, A, row)
        M = O.mass_matrix(m, s)
        emu.state[:len(row)] = row
        Me, be = emu.mass_matrix()
        assert np.abs(Me - M).max() / np.abs(M).max() < 1e-6
        acc = O.forward_dynamics(m, p, s, np.zeros(A), with_damping=True)
        bias = -M @ acc
        assert np.abs(be - bias).max() / np.abs(bias).max() < 1e-5


def test_child_reset_bit_exact(child_table, oracle_mod):
    """Crawl start pose: base pitched by 90 degrees at z = 0.38 (robots.py:314-323,335), joints bit-exact."""
    O, t = oracle_mod, child_table
    for seed in range(3):
        env = O.Walker3DCustomOracle(t, seed=seed)
        emu = E.EmuChild(_mt_row(O, seed))
        for _ in range(2):
            o_ref, o_emu = env.reset(), emu.reset()
            assert np.array_equal(emu.state[13:34], np.array(env.e.s.q[:21]).astype(np.float32))
            assert np.array_equal(emu.state[0:3], np.array([0, 0, 0.38], dtype=np.float32))
            assert np.allclose(emu.state[3:7], [0, np.sin(np.pi / 4), 0, np.cos(np.pi / 4)], atol=1e-7)
            assert np.abs(o_ref - o_emu).max() < 1e-6


def test_child_contact_step(child_table, oracle_mod):
    """One frame from the crawl pose resting on hands / knees / feet: 2e-3 like the Walker3D contact frame."""
    O, t = oracle_mod, child_table
    A = t["n_dof"]
    m = O.model_from_table(t)
    p = O.default_params()
    emu = E.EmuChild()
    rng = np.random.RandomState(2)
    gain = np.array(t["gain"])
    worst, with_contacts = 0.0, 0
    for seed in range(8):
        env = O.Walker3DCustomOracle(t, seed=seed)
        env.reset()
        for _ in range(rng.randint(8, 30)):
            env.step(0.3 * rng.uniform(-1, 1, A))
        row = env.state_vector().astype(np.float32).astype(np.float64)
        tau = 0.3 * gain * rng.uniform(-1, 1, A)
        s = oracle_state(O, A, row)
        c, rows = O.step_physics(m, p, s, tau)
        emu.state[:len(row)] = row
        erows, enc = emu.step_physics(tau)
        assert enc == c.n
        assert abs(rows - erows) <= 2
        with_contacts += c.n > 0
        worst = max(worst, state_error(emu.state[:len(row)], O.state_vector(s, A)))
    assert with_contacts >= 6
    assert worst < 2e-3, worst


def test_child_env_step_teacher_forced(oracle_mod):
    """Child3DCustomEnv.step (termination height 0.1, power 0.4) from f32-identical states and bookkeeping.  The child's
    links are small (30 kg in total, waist inertias ~1e-3 kg m^2, no armature in Bullet): its mass matrix is
    ill-conditioned more often than Walker3D's, which the judge verifies step by step (cond(M) >= 1e6).  Steps outside 1e-3 (obs) / 1e-2 (reward) must be explained by a verified
    discontinuity and bounded (tests/teacher.py), else the test fails; integer bookkeeping read back and compared
    exactly after every structurally identical step."""
    from tests import teacher as T

    js = T.run_vs_oracle(oracle_mod, "child3d", "emu", range(5, 9), 40, lambda rng, k: rng.uniform(-1.2, 1.2, 21))
    assert np.median(np.concatenate([j.errs for j in js])) < 2e-4


def test_mike_reset_and_terrain(mike_table, oracle_mod):
    """MikeStepperEnv starts at (0.3, 0, 1.0) (env_locomotion.py:845); terrain from the same stream, bit-exact."""
    O, t = oracle_mod, mike_table
    for seed, cur in ((0, 0), (1, 9)):
        env = O.Walker3DStepperOracle(t, seed=seed, curriculum=cur)
        emu = E.EmuMike(_mt_row(O, seed), curriculum=cur)
        o1, o2 = env.reset(), emu.reset()
        assert np.array_equal(emu.terrain(), np.array(env.e.terrain[:]).astype(np.float32))
        assert np.array_equal(emu.state[13:34], np.array(env.e.base.s.q[:21]).astype(np.float32))
        assert np.array_equal(emu.state[0:3], np.array([0.3, 0.0, 1.0], dtype=np.float32))
        assert np.abs(o1 - o2).max() < 1e-6


def test_mike_env_step_teacher_forced(oracle_mod):
    """MikeStepperEnv.step (Mike's power table, waist mass 8) from f32-identical states and bookkeeping.  Steps outside 1e-3 (obs) / 1e-2 (reward) must be explained by a verified
    discontinuity and bounded (tests/teacher.py), else the test fails; integer bookkeeping read back and compared
    exactly after every structurally identical step."""
    from tests import teacher as T

    for seed, cur in ((3, 5), (4, 0)):
        T.run_vs_oracle(oracle_mod, "mike", "emu", [seed], 50, lambda rng, k: 0.3 * rng.uniform(-1, 1, 21), curriculum=cur)
