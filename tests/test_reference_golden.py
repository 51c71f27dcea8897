"""The oracle's env layer against the reference's OWN Python code (tests/golden/ref_*.npz).

The fixtures were recorded by tools/gen_reference_golden.py in the build container: the reference's unmodified
env_base.py / env_locomotion.py / robots.py / bullet_utils.py, imported with stand-ins for gym and pybullet whose Bullet
client is served by the oracle's float64 physics.  So observation, reward, done, target logic, reset draws and the
quirk-Q1 seeding in these traces were computed by the reference itself; replaying the recorded actions through the
oracle's C restatement of that layer must reproduce them (same physics underneath: agreement to rounding of the
f32 casts, 1e-9).  Bullet's own arithmetic is not pinned by this (DESIGN.md section 5)."""
import glob
import os

import numpy as np
import pytest

_G = os.path.join(os.path.dirname(__file__), "golden")
GOLDEN = sorted(glob.glob(os.path.join(_G, "ref_walker3d_custom_*.npz")) + glob.glob(os.path.join(_G, "ref_child3d_custom_*.npz"))
                + glob.glob(os.path.join(_G, "ref_walker2d_custom_*.npz")) + glob.glob(os.path.join(_G, "ref_crab2d_custom_*.npz")))


def _teleport(env, table, pos):
    """The recorded state override of the teleport traces (tools/gen_reference_golden.py: reset_joint_states(base pose),
    reset_pose(pos, identity), reset_velocity(0, 0) through the reference's own robot object)."""
    s = env.e.base.s if hasattr(env.e, "base") else env.e.s
    for k in range(3):
        s.pos[k], s.omega[k], s.vel[k] = float(pos[k]), 0.0, 0.0
    s.quat[0], s.quat[1], s.quat[2], s.quat[3] = 0.0, 0.0, 0.0, 1.0
    for k, q in enumerate(table["base_joint_angles"]):
        s.q[k], s.qd[k] = float(q), 0.0


def test_fixtures_present():
    assert len(GOLDEN) >= 6


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_walker3d_custom_env_layer_matches_reference(path, walker_table, child_table, walker2d_table, crab2d_table,
                                                     oracle_mod):
    """Walker3DCustomEnv; Child3DCustomEnv (crawl start pose, power 0.4, termination height 0.1) on its table; the
    planar Walker2DCustomEnv / Crab2DCustomEnv (done forced to False, zeros in the target slots at reset, pelvis link
    accessors, restoreState at every reset: env_locomotion.py:285-314)."""
    O, g = oracle_mod, np.load(path)
    b = os.path.basename(path)
    planar = "2d_" in b
    table = (child_table if "child3d" in b else walker2d_table if "walker2d" in b else crab2d_table if "crab2d" in b
             else walker_table)
    env = O.Walker3DCustomOracle(table, seed=int(g["construction_seed"]))  # EnvBase.__init__: self.seed()
    env.seed(int(g["seed"]))  # env_base.py:164-166: the robot keeps the construction stream (quirk Q1)
    if int(g["eval_mode"]):
        env.e.eval_mode = 1
    obs = [env.reset()]
    worst_r = 0.0
    tele = {int(r[0]): r[1:4] for r in g["teleports"]} if "teleports" in g.files else {}
    for t, a in enumerate(g["actions"]):
        if t in tele:
            _teleport(env, table, tele[t])
        o, r, d, info = env.step(a)
        assert d == bool(g["dones"][t]), t
        worst_r = max(worst_r, abs(r - g["rewards"][t]))
        assert np.abs(np.array(env.e.walk_target[:]) - g["walk_target"][t]).max() < 1e-9, t
        if d:
            obs.append(o)
            o = env.reset()
        obs.append(o)
    obs = np.array(obs)
    assert obs.shape == g["obs"].shape
    assert np.abs(obs - g["obs"]).max() < 1e-12
    assert worst_r < 1e-12
    if "_target" in b:  # held at the target: the mid-episode re-randomisation ran several times
        assert len(np.unique(g["walk_target"][:, 0])) >= 4
    else:
        assert g["dones"].sum() >= (0 if planar else 2)  # the traces run through episode ends and resets


def test_mirror_indices_match_reference(walker_table):
    """get_mirror_indices (env_locomotion.py:224-282) as the reference computes it, against the table-driven mirror."""
    g = np.load(GOLDEN[0])
    t = walker_table
    A, nfeet = t["n_dof"], len(t["foot_links"])
    right_j, left_j = np.array(t["right_joint_indices"]), np.array(t["left_joint_indices"])
    neg_j = np.array(t["negation_joint_indices"])
    right = np.concatenate((right_j + 6, right_j + 6 + A, [6 + 2 * A + 2 * i for i in range(nfeet // 2)]))
    left = np.concatenate((left_j + 6, left_j + 6 + A, [6 + 2 * A + 2 * i + 1 for i in range(nfeet // 2)]))
    neg_obs = np.concatenate(([2, 4], 6 + neg_j, 6 + neg_j + A, [6 + 2 * A + nfeet]))
    ours = np.concatenate([neg_obs, right, left, neg_j, right_j, left_j])
    assert np.array_equal(ours, g["mirror"])


STEPPER = sorted(glob.glob(os.path.join(_G, "ref_walker3d_stepper_*.npz")) + glob.glob(os.path.join(_G, "ref_mike_stepper_*.npz")))


def test_stepper_fixtures_present():
    assert len(STEPPER) >= 6


@pytest.mark.parametrize("path", STEPPER, ids=[os.path.basename(p) for p in STEPPER])
def test_walker3d_stepper_env_layer_matches_reference(path, walker_table, mike_table, oracle_mod):
    """Walker3DStepperEnv (env_locomotion.py:330-840) as the reference's own code computes it -- terrain generator,
    plank placement (bullet_objects.py:47-103: geometry read from the URDFs by the stand-in, not from the oracle), foot /
    target contact logic, step bonus, curriculum gains and terminal heights, `random_reward`, `plank_class`,
    `steps_reached` -- against the oracle's restatement, on identical physics."""
    O, g = oracle_mod, np.load(path)
    pc = str(g["plank_class"])
    table = mike_table if "mike" in os.path.basename(path) else walker_table  # MikeStepperEnv: start (0.3, 0, 1.0)
    env = O.Walker3DStepperOracle(table, seed=int(g["construction_seed"]), curriculum=0,
                                  random_reward=bool(int(g["random_reward"])),
                                  plank_class=None if pc == "LargePlank" else pc)
    env.seed(int(g["seed"]))
    env.set_env_params({"curriculum": int(g["curriculum"])})
    obs = [env.reset()]
    terrain = [np.array(env.e.terrain[:])]
    worst_r = 0.0
    tele = {int(r[0]): r[1:4] for r in g["teleports"]} if "teleports" in g.files else {}
    for t, a in enumerate(g["actions"]):
        if t in tele:
            _teleport(env, table, tele[t])
        o, r, d, info = env.step(a)
        assert d == bool(g["dones"][t]), t
        assert env.e.next_step_index == int(g["next_step_index"][t]) or d, t
        assert info.get("steps_reached", -1) == int(g["steps_reached"][t]), t
        worst_r = max(worst_r, abs(r - g["rewards"][t]))
        if d:
            obs.append(o)
            o = env.reset()
            terrain.append(np.array(env.e.terrain[:]))
        obs.append(o)
    obs = np.array(obs)
    assert np.array_equal(np.array(terrain), g["terrain"])  # bit-exact: same MT19937 draws, same float64 formulas
    assert obs.shape == g["obs"].shape
    assert np.abs(obs - g["obs"]).max() < 1e-12
    assert worst_r < 1e-12
    walk = os.path.basename(path).endswith("_walk.npz")
    assert (g["next_step_index"].max() >= 14) if walk else (g["dones"].sum() >= 2 and g["next_step_index"].max() >= 2)


def _monkey_grab(env, pos):
    """tools/gen_reference_golden.py trace_monkey(grab_every): base moved to `pos`, every velocity zeroed, pose kept."""
    s = env.e.base.s
    for k in range(3):
        s.pos[k], s.omega[k], s.vel[k] = float(pos[k]), 0.0, 0.0
    for k in range(env.A):
        s.qd[k] = 0.0


MONKEY = sorted(glob.glob(os.path.join(_G, "ref_monkey3d_custom_*.npz")))


@pytest.mark.parametrize("path", MONKEY, ids=[os.path.basename(p) for p in MONKEY])
def test_monkey3d_env_layer_matches_reference(path, monkey_table, oracle_mod):
    """Monkey3DCustomEnv (env_locomotion.py:1136-1516) as the reference computes it -- bar layout generator from the
    hand positions, bar placement (bullet_objects.py:148-187), scripted finger actions, palm / hand contact logic, swing
    potential, free-fall and 180-step terminations -- against the oracle's restatement, on identical physics."""
    O, g = oracle_mod, np.load(path)
    env = O.Monkey3DOracle(monkey_table, seed=int(g["construction_seed"]))
    env.seed(int(g["seed"]))
    obs = [env.reset()]
    terrain = [np.array(env.e.terrain[:])]
    worst_r = 0.0
    tele = {int(r[0]): r[1:4] for r in g["teleports"]} if "teleports" in g.files else {}
    for t, a in enumerate(g["actions"]):
        if t in tele:  # the recorded "grab": the monkey translated so that its swing palm sits on the target bar
            _monkey_grab(env, tele[t])
        o, r, d, info = env.step(a)
        assert d == bool(g["dones"][t]), t
        assert env.e.next_step_index == int(g["next_step_index"][t]) or d, t
        worst_r = max(worst_r, abs(r - g["rewards"][t]))
        if d:
            obs.append(o)
            o = env.reset()
            terrain.append(np.array(env.e.terrain[:]))
        obs.append(o)
    obs = np.array(obs)
    assert np.abs(np.array(terrain) - g["terrain"]).max() < 1e-9
    assert obs.shape == g["obs"].shape
    assert np.abs(obs[:, :65] - g["obs"][:, :65]).max() < 1e-12
    # the swing palm's quaternion (last four entries): its overall sign comes from below the env layer (the stand-in
    # client converts the oracle's rotation matrix, Bullet multiplies quaternions down the chain) -- compare as rotations
    qa, qb = obs[:, 65:], g["obs"][:, 65:]
    assert np.minimum(np.abs(qa - qb).max(axis=1), np.abs(qa + qb).max(axis=1)).max() < 1e-9
    assert worst_r < 1e-12
    if os.path.basename(path).endswith("_grab.npz"):
        assert g["next_step_index"].max() >= 10  # eight bars grabbed: swing / pivot swaps, all four bars recycled
    else:
        assert g["dones"].sum() >= 1


CASSIE = sorted(glob.glob(os.path.join(_G, "ref_cassie_*.npz")))


@pytest.mark.parametrize("path", CASSIE, ids=[os.path.basename(p) for p in CASSIE])
def test_cassie_env_layer_matches_reference(path, cassie_table, oracle_mod):
    """CassieEnv-v0 (env_cassie.py:285-479) as the reference computes it -- residual PD targets, the filtered joint
    velocity, 50 PD + stepSimulation + calc_state rounds per env step, obs36, alive / progress rewards, termination --
    against the oracle's restatement, on identical physics (loop closures and joint damping checked by the stand-in
    against the compiled table)."""
    O, g = oracle_mod, np.load(path)
    env = O.CassieOracle(cassie_table)
    obs = [env.reset()]
    worst_r = worst_a = worst_p = 0.0
    for t, a in enumerate(g["actions"]):
        o, r, d, info = env.step(a)
        assert d == bool(g["dones"][t]), t
        worst_r = max(worst_r, abs(r - g["rewards"][t]))
        worst_a = max(worst_a, abs(info["AliveRew"] - g["alive"][t]))
        worst_p = max(worst_p, abs(info["ProgressRew"] - g["progress"][t]))
        if d:
            obs.append(o)
            o = env.reset()
        obs.append(o)
    obs = np.array(obs)
    assert obs.shape == g["obs"].shape
    assert np.array_equal(obs, g["obs"])
    assert worst_r == 0.0 and worst_a == 0.0 and worst_p == 0.0
    assert g["dones"].sum() >= 2


ALL_TRACES = sorted(glob.glob(os.path.join(_G, "ref_*.npz")))


@pytest.mark.parametrize("path", ALL_TRACES, ids=[os.path.basename(p) for p in ALL_TRACES])
def test_kernel_source_vs_reference_trace(path, oracle_mod):
    """The CUDA kernel source of every env (compiled by g++ as a lane loop, tests/emu) teacher-forced along every
    reference trace: observation / reward / done per step against the values the REFERENCE's own code recorded, within
    1e-3 / 1e-2 (Cassie: 1e-2 / 2e-3 over its 50 PD substeps) -- and every step outside that is either explained by a
    verified discontinuity (different constraint-row / contact counts, a numerically singular mass matrix, an unstable
    step map: tests/teacher.py) and bounded accordingly, or the test fails.  Oracle and kernel are seeded alike
    (construction seed + EnvBase.seed, quirk Q1), so the reset draws, mid-episode target re-draws and random_reward
    scalings come from streams in lockstep; after every structurally identical step the kernel's integer bookkeeping
    (next_step_index, target_reached_count, stop flags, swing / pivot legs, free_fall_count, plank / bar slots, feet
    contacts, elapsed) is read back and compared exactly -- Monkey3D's grab steps included, whose float comparison is
    waived (the palm starts centred ON the bar).  GPU twin: test_gpu_reference_golden.py."""
    from tests import teacher as T

    j = T.run_golden_trace(oracle_mod, path, "emu")
    assert j.book_checked >= 0.6 * j.n


CONFIG1 = os.path.join(_G, "restatement_walker3d_custom_config1.npz")


def test_config1_trace_regenerates_and_kernel_source_follows_it(oracle_mod):
    """BASELINE configs[0] (SURVEY 8d config 1): the 1000-step single-env random-action trace.  Recorded from the ORACLE
    and labelled "restatement" (PyBullet is not installable; tools/gen_pybullet_golden.py records the PyBullet twin
    where it is): the oracle regenerates it bit for bit, and the kernel source (g++ lane loop) follows it teacher-forced
    under the explained-or-fatal rules of tests/teacher.py.  GPU twin: test_gpu_reference_golden.py."""
    import importlib.util

    from tests import teacher as T

    g = np.load(CONFIG1)
    assert "restatement" in str(g["source"])
    spec = importlib.util.spec_from_file_location("gen_config1", os.path.join(os.path.dirname(_G), "..", "tools", "gen_config1_trace.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    d = mod.record()
    for k in ("actions", "obs", "states", "rewards", "dones"):
        assert np.array_equal(d[k], g[k]), k
    assert len(g["actions"]) == 1000 and g["dones"].sum() > 20
    j = T.run_golden_trace(oracle_mod, CONFIG1, "emu")
    assert j.n == 1000 and j.book_checked >= 900
