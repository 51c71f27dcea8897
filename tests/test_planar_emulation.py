"""SURVEY 8 f3 -- the planar walkers: Walker2DCustomEnv-v0 / Crab2DCustomEnv-v0 (env_locomotion.py:285-314,
robots.py:338-404, data/robots/{walker2d,crab2d}.xml).  Bullet imports the root's "ignore*" slide-x / slide-z / hinge-y
joints as a fixed base with two massless dummy links; that is a free base confined to the x-z plane, and because every
joint axis is +-y and every COM has y = 0 the free-base kernels keep the out-of-plane coordinates EXACTLY zero.
CPU checks of the kernel source (tests/emu) against the float64 oracle; the GPU twins are in test_gpu_f3.py."""
import numpy as np
import pytest

from tests.emu import emu as E
from tests.helpers import force_oracle_state, oracle_record, oracle_state, state_error

ENVS = {"walker2d": E.EmuWalker2D, "crab2d": E.EmuCrab2D}


def _mt_row(O, seed):
    st = np.random.RandomState(O.gym_seed_words(seed)).get_state()
    return np.concatenate([st[1], [st[2]]]).astype(np.uint32)


def _table(name, walker2d_table, crab2d_table):
    return {"walker2d": walker2d_table, "crab2d": crab2d_table}[name]


def _planar_states(t, rng, n):
    """In-plane states: rotation about y, no out-of-plane velocity, joints inside their limits."""
    A = t["n_dof"]
    lo, hi = np.array(t["lower"]), np.array(t["upper"])
    out = np.zeros((n, 13 + 2 * A))
    for i in range(n):
        th = rng.uniform(-1, 1)
        out[i, 0:3] = [rng.uniform(-1, 1), 0.0, 2.0]
        out[i, 3:7] = [0, np.sin(th / 2), 0, np.cos(th / 2)]
        out[i, 8] = rng.randn()
        out[i, 10], out[i, 12] = rng.randn(), rng.randn()
        out[i, 13:13 + A] = lo + (hi - lo) * rng.uniform(0.15, 0.85, A)
        out[i, 13 + A:] = rng.uniform(-3, 3, A)
    return out


def test_tables(walker2d_table, crab2d_table):
    w, c = walker2d_table, crab2d_table
    assert w["planar"] and c["planar"]
    assert w["joint_names"] == ["torso_joint", "thigh_joint", "leg_joint", "foot_joint", "thigh_left_joint",
                                "leg_left_joint", "foot_left_joint"]  # joint-index order, "ignore*" skipped
    assert w["gain"] == [100, 100, 100, 50, 100, 100, 50] and c["gain"] == [100, 100, 50, 100, 100, 50]
    assert w["right_joint_indices"] == [1, 2, 3] and w["left_joint_indices"] == [4, 5, 6]  # robots.py:365-366
    assert c["right_joint_indices"] == [0, 1, 2] and c["left_joint_indices"] == [3, 4, 5]  # robots.py:399-400
    assert len(w["self_pairs"]) == 0  # contype 1 / conaffinity 0: Bullet's two-way filter rejects every pair
    assert len(c["self_pairs"]) > 0   # crab2d.xml: conaffinity 1 + the self-collision load flags
    for t in (w, c):
        assert all(abs(a[0]) < 1e-12 and abs(a[2]) < 1e-12 for a in t["axis"])


@pytest.mark.parametrize("name", ["walker2d", "crab2d"])
def test_mass_matrix_and_bias(name, walker2d_table, crab2d_table, oracle_mod):
    O, t = oracle_mod, _table(name, walker2d_table, crab2d_table)
    A = t["n_dof"]
    m, p, emu = O.model_from_table(t), O.default_params(), {"walker2d": E.EmuWalker2D, "crab2d": E.EmuCrab2D}[name]()
    rng = np.random.RandomState(0)
    for row in _planar_states(t, rng, 4):
        s = oracle_state(O, A, row)
        M = O.mass_matrix(m, s)
        emu.state[:len(row)] = row
        Me, be = emu.mass_matrix()
        assert np.abs(Me - M).max() / np.abs(M).max() < 1e-6
        # the in-plane block {omega_y, v_x, v_z, joints} decouples exactly from {omega_x, omega_z, v_y}
        inp, outp = [1, 3, 5] + list(range(6, 6 + A)), [0, 2, 4]
        assert np.all(Me[np.ix_(inp, outp)] == 0.0)
        acc = O.forward_dynamics(m, p, s, np.zeros(A), with_damping=True)
        bias = -M @ acc
        assert np.abs(be - bias).max() / np.abs(bias).max() < 1e-5
        assert np.all(be[outp] == 0.0)


@pytest.mark.parametrize("name", ["walker2d", "crab2d"])
def test_reset_bit_exact(name, walker2d_table, crab2d_table, oracle_mod):
    """Zero base pose +- 0.1 rad noise from the robot stream, pelvis origin at the world origin, zeros in the two
    target slots of the reset observation (env_locomotion.py:298)."""
    O, t = oracle_mod, _table(name, walker2d_table, crab2d_table)
    A = t["n_dof"]
    for seed in range(3):
        env = O.Walker3DCustomOracle(t, seed=seed)
        emu = ENVS[name](_mt_row(O, seed))
        for _ in range(2):
            o_ref, o_emu = env.reset(), emu.reset()
            assert np.array_equal(emu.state[13:13 + A], np.array(env.e.s.q[:A]).astype(np.float32))
            assert np.array_equal(emu.state[0:7], np.array([0, 0, 0, 0, 0, 0, 1], dtype=np.float32))
            assert o_emu[-1] == 0.0 and o_emu[-2] == 0.0 and o_ref[-1] == 0.0 and o_ref[-2] == 0.0
            assert np.abs(o_ref - o_emu).max() < 1e-6


@pytest.mark.parametrize("name", ["walker2d", "crab2d"])
def test_rollout_stays_planar_and_matches_oracle(name, walker2d_table, crab2d_table, oracle_mod):
    """120 env steps under random actions (the walker falls over and lies on the ground: many contacts, for the crab
    also self-contacts): y, v_y, omega_x, omega_z and the quaternion's x / z stay exactly zero in the f32 kernel
    source; done stays False (env_locomotion.py:303); teacher-forced obs / reward agree with the oracle."""
    O, t = oracle_mod, _table(name, walker2d_table, crab2d_table)
    A = t["n_dof"]
    from tests import teacher as T

    seen = {"contacts": 0}

    def planar(tt, backend, o, done, d1):
        st = backend.e.state
        assert not done and not d1
        assert st[1] == 0.0 and st[3] == 0.0 and st[5] == 0.0 and st[7] == 0.0 and st[9] == 0.0 and st[11] == 0.0
        seen["contacts"] += int(o.e.feet_contact[0] + o.e.feet_contact[1])

    js = T.run_vs_oracle(O, name, "emu", [3], 120, lambda rng, k: rng.uniform(-1.2, 1.2, A), on_step=planar)
    assert seen["contacts"] > 0
    assert np.median(js[0].errs) < 5e-4


def test_time_limit_is_the_only_end(walker2d_table, oracle_mod):
    O, t = oracle_mod, walker2d_table
    e = E.EmuWalker2D(_mt_row(O, 0))
    e.reset()
    e.rec.view(np.int32)[8] = 998  # ER_ELAPSED
    _, _, d, tr, _ = e.step(np.zeros(7))
    assert not d and not tr
    _, _, d, tr, _ = e.step(np.zeros(7))
    assert d and tr
    assert e.rec.view(np.int32)[8] == 0  # auto-reset
