"""CassieEnv-v0: URDF compiler checks, oracle sanity (loop closures), and the CUDA kernel SOURCE (g++ lane-loop
emulation, tests/emu) diffed against the float64 oracle."""
import numpy as np

from tests.emu import emu as E
from tests.helpers import oracle_state, random_states, state_error


def _rand_table(t):
    """random_states() draws q inside [lower, upper]; the achilles-rod joints are continuous (lower > upper)."""
    t2 = dict(t)
    lo, hi = np.array(t["lower"]), np.array(t["upper"])
    un = lo > hi
    t2["lower"], t2["upper"] = np.where(un, -1.0, lo).tolist(), np.where(un, 1.0, hi).tolist()
    return t2


def test_cassie_table_matches_urdf(cassie_table):
    """Joint order, ordered joints, masses and loop-closure consistency of the compiled table (env_cassie.py:17-62,
    114-137; SURVEY App. A.5 / E.3)."""
    t = cassie_table
    assert t["n_links"] == 21 and t["n_dof"] == 18
    assert t["link_names"][:2] == ["vectorNav", "left_pelvis_abduction"]
    names = [t["joint_names"][d] for d in t["ordered_dofs"]]
    assert names[:7] == ["hip_abduction_left", "hip_rotation_left", "hip_flexion_left", "knee_joint_left",
                         "knee_to_shin_left", "ankle_joint_left", "toe_joint_left"]
    assert abs(t["total_mass"] - (10.33 + 2 * (1.82 + 1.17 + 5.52 + 0.758 + 0.577 + 0.782 + 0.15 + 0.1567))) < 1e-9
    assert [t["gain"][d] for d in t["ordered_dofs"]][:7] == [112.5, 112.5, 195.2, 195.2, 200, 200, 45.0]


def test_cassie_loop_closure_holds_at_base_pose(cassie_table, oracle_mod):
    """The achilles-rod pivots of the saved initial state coincide to a few millimetres: pins the URDF frame
    conventions (inertial frames, joint origins, pivot frames) independently of the dynamics."""
    O, t = oracle_mod, cassie_table
    m = O.model_from_table(t)
    A = t["n_dof"]
    s = O.make_state(A, [0, 0, 1.085], [0, 0, 0, 1], [0] * 3, [0] * 3, t["base_joint_angles"], np.zeros(A))
    pos, rot = O.fk(m, s)
    for c in t["p2p"]:
        la, lb = c["link_a"] + 1, c["link_b"] + 1
        pa = pos[la] + rot[la] @ np.array(c["pivot_a"])
        pb = pos[lb] + rot[lb] @ np.array(c["pivot_b"])
        assert np.linalg.norm(pa - pb) < 6e-3
    pts = [pos[g["link"] + 1] + rot[g["link"] + 1] @ np.array(g["pos"]) for g in t["geoms"]]
    assert -0.01 < min(p[2] for p in pts) < 0.01  # the toes rest on the ground plane at the reset height


def test_cassie_oracle_loop_closure_stays_closed(cassie_table, oracle_mod):
    O, t = oracle_mod, cassie_table
    env = O.CassieOracle(t)
    env.reset()
    rng = np.random.RandomState(0)
    for _ in range(10):
        env.step(0.2 * rng.uniform(-1, 1, 10))
        pos, rot = O.fk(env.m, env.e.base.s)
        for c in t["p2p"]:
            la, lb = c["link_a"] + 1, c["link_b"] + 1
            gap = np.linalg.norm(pos[la] + rot[la] @ np.array(c["pivot_a"]) - pos[lb] - rot[lb] @ np.array(c["pivot_b"]))
            assert gap < 5e-3, gap


def test_cassie_mass_matrix_and_bias(cassie_table, oracle_mod):
    O, t = oracle_mod, cassie_table
    A = t["n_dof"]
    m = O.model_from_table(t)
    p = O.cassie_params()
    emu = E.EmuCassie()
    rng = np.random.RandomState(0)
    for row in random_states(_rand_table(t), rng, 6):
        s = oracle_state(O, A, row)
        M = O.mass_matrix(m, s)
        emu.state[:len(row)] = row
        Me, be = emu.mass_matrix()
        assert np.abs(Me - M).max() / np.abs(M).max() < 1e-6
        acc = O.forward_dynamics(m, p, s, np.zeros(A), with_damping=True)
        bias = -M @ acc
        assert np.abs(be - bias).max() / np.abs(bias).max() < 1e-5


def test_cassie_airborne_step_with_loop_closures(cassie_table, oracle_mod):
    """One 0.6 ms Bullet step away from the ground: forward dynamics + the six loop-closure rows (two compact rows
    per multiplier in the kernel) against the oracle's velocity-space PGS; state within 3e-4 (the ERP term
    divides the f32 pivot gap by dt = 0.6 ms: 1e-7 m of rounding is 1.7e-4 m/s)."""
    O, t = oracle_mod, cassie_table
    A = t["n_dof"]
    m = O.model_from_table(t)
    p = O.cassie_params()
    rng = np.random.RandomState(1)
    base = np.array(t["base_joint_angles"])
    for k in range(8):
        q = base + 0.01 * rng.randn(A)
        row = np.concatenate([[0, 0, 3.0], [0, 0, 0, 1], 0.3 * rng.randn(3), 0.3 * rng.randn(3), q, 0.2 * rng.randn(A)])
        row = row.astype(np.float32).astype(np.float64)
        tau = 20 * rng.uniform(-1, 1, A)
        s = oracle_state(O, A, row)
        _, rows = O.step_physics(m, p, s, tau)
        emu = E.EmuCassie()
        emu.state[:13 + 2 * A] = row.astype(np.float32)
        erows, enc = emu.step_physics(tau - np.array(t["damping"]) * row[13 + A:])
        assert enc == 0 and abs(rows - erows) <= 1
        assert state_error(emu.state[:13 + 2 * A], O.state_vector(s, A)) < 3e-4


def test_cassie_env_free_running(cassie_table, oracle_mod):
    """CassieEnv.step free-running from reset (deterministic env): 50 PD substeps per step, toe contacts, loop
    closures.  obs within 1e-2 (raw joint speeds in rad/s dominate), reward within 1e-3 over the first 12 steps."""
    O, t = oracle_mod, cassie_table
    env, emu = O.CassieOracle(t), E.EmuCassie()
    o1, o2 = env.reset(), emu.reset()
    assert np.abs(o1 - o2).max() < 1e-5
    rng = np.random.RandomState(0)
    for i in range(12):
        a = 0.1 * rng.uniform(-1, 1, 10)
        o1, r1, d1, _ = env.step(a)
        o2, r2, d2, tr, fin = emu.step(a)
        assert d1 == d2
        assert np.abs(o1 - (fin if d2 else o2)).max() < 1e-2
        assert abs(r1 - r2) < 1e-3
        # row counts of the 50 substeps agree up to a contact appearing one substep earlier / later
        assert abs(env.e.base.rows_sum - (emu.rec[15] - (0 if i == 0 else prev))) <= 9
        prev = emu.rec[15]
        if d1:
            break


def test_cassie_hull_self_collision(cassie_table, oracle_mod):
    """Mesh-hull self-collision (env_cassie.py:81-85: URDF_USE_SELF_COLLISION | ..._EXCLUDE_ALL_PARENTS; the non-ancestor
    pairs are left-leg vs right-leg links): warp-cooperative GJK on the 32-vertex link hulls in the kernel source against
    the oracle's float64 GJK on the same hulls.  Contact geometry (distance 2e-6, point 1e-3 (barycentric weights of a float32 Gram solve; the witness point of two nearly parallel faces slides along them with the rounding of the vertex coordinates), normal 2e-3: the normal
    is a millimetre-long difference of metre-sized float32 coordinates), contact and row counts, the state after one
    0.6 ms stepSimulation (5e-3, median 5e-4) -- and with self_collision = 0 the same states come out differently, so
    the feature is live."""
    from tests.helpers import cassie_hull_contact_states, oracle_state, state_error

    O, t = oracle_mod, cassie_table
    A = t["n_dof"]
    m = O.model_from_table(t)
    p = O.cassie_params()
    p_off = O.cassie_params()
    p_off.self_collision = 0
    emu = E.EmuCassie()
    rng = np.random.RandomState(3)
    states = cassie_hull_contact_states(O, t, rng, 24)
    errs, effect = [], []
    for st in states:
        s = oracle_state(O, A, st.astype(np.float64))
        c0 = O.collide(m, p, s)
        c, rows_ref = O.step_physics(m, p, s, np.zeros(A))
        emu.state[:len(st)] = st
        pts = np.zeros((16, 10), dtype=np.float32)
        rows, nc = emu.step_physics(np.zeros(A, dtype=np.float32), points=pts)
        out = emu.state[:len(st)].copy()
        assert nc == c.n and rows == rows_ref
        for k in range(c0.n):
            if c0.partner[k] >= 1000:
                assert int(pts[k, 9]) >= 1000
                assert abs(pts[k, 6] - c0.dist[k]) < 2e-6
                assert np.abs(pts[k, 0:3] - np.array(c0.pos_a[k][:])).max() < 1e-3
                assert np.abs(pts[k, 3:6] - np.array(c0.normal[k][:])).max() < 2e-3
        ref = O.state_vector(s, A)
        errs.append(state_error(out, ref))
        s_off = oracle_state(O, A, st.astype(np.float64))
        O.step_physics(m, p_off, s_off, np.zeros(A))
        effect.append(state_error(O.state_vector(s_off, A), ref))
    assert max(errs) < 5e-3 and np.median(errs) < 5e-4, sorted(errs)[-5:]
    assert np.median(effect) > 0.1, np.median(effect)


def test_cassie_hull_pairs_of_the_table(cassie_table):
    """The compiled hull tables: 16 link hulls of exactly 32 vertices, only left-leg vs right-leg candidate pairs (every
    other pair is an ancestor pair under EXCLUDE_ALL_PARENTS; the achilles rods carry no collision hull)."""
    t = cassie_table
    assert len(t["hulls"]) == 16 and all(len(h["verts"]) == 32 for h in t["hulls"])
    names = t["link_names"]
    assert 10 <= len(t["hull_pairs"]) <= 32
    for a, b in t["hull_pairs"]:
        na, nb = names[t["hulls"][a]["link"]], names[t["hulls"][b]["link"]]
        assert {na.split("_")[0], nb.split("_")[0]} == {"left", "right"}, (na, nb)
