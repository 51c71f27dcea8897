"""PyBullet golden vectors (tests/golden/pybullet_<env>_<apiversion>.npz, written by tools/gen_pybullet_golden.py on a host
that has PyBullet).  None is committed: PyBullet cannot be installed in the build container (no wheel, no network), so
parity with Bullet's arithmetic is UNPINNED and the real-file checks skip.  They run by themselves once a file is
dropped in: the oracle legs on the CPU, the device legs under `-m gpu`."""
import glob
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REAL = sorted(p for p in glob.glob(os.path.join(ROOT, "tests", "golden", "pybullet_*.npz")) if "standin" not in p)
needs_golden = pytest.mark.skipif(not REAL, reason="no PyBullet golden file: parity with Bullet's arithmetic is unpinned "
                                                   "(DESIGN.md section 5); run tools/gen_pybullet_golden.py where pybullet exists")


def _env_name(g):
    from tests.teacher import env_name_of_fixture

    return env_name_of_fixture(str(g["env"]))


def _state(O, A, st):
    return O.make_state(A, st[0:3], st[3:7], st[7:10], st[10:13], st[13:13 + A], st[13 + A:13 + 2 * A])


def check_oracle_dynamics(O, path):
    """G1 / G2: mass matrix, inverse dynamics and the contact-free step of the oracle against the recorded values."""
    from tests import teacher as T

    g = np.load(path, allow_pickle=False)
    name = _env_name(g)
    kind, tname = T.SPECS[name][0], T.SPECS[name][1]
    t = T.table_of(tname)
    A = t["n_dof"]
    m = O.model_from_table(t)
    p = O.cassie_params() if kind == "cassie" else O.default_params()
    n_checked = 0
    if g["g1_mass_matrix"].dtype.kind == "f":
        for st, Mpb in zip(g["g1_states"], g["g1_mass_matrix"]):
            M = O.mass_matrix(m, _state(O, A, st))
            if Mpb.shape == M.shape:
                assert np.abs(M - Mpb).max() / np.abs(Mpb).max() < 1e-4
            else:  # a client that reports the joint block only
                assert np.abs(M[6:, 6:] - Mpb[-A:, -A:]).max() / np.abs(Mpb).max() < 1e-4
            n_checked += 1
    if kind != "stepper" and kind != "monkey":  # (their reset poses start in contact with planks / bars)
        for st, ta, ref in zip(g["g1_states"], g["g2_tau_acc"], g["g2_after_step"]):
            s = _state(O, A, st)
            O.step_physics(m, p, s, ta[:A])
            out = O.state_vector(s, A)
            assert np.max(np.abs(out - ref) / np.maximum(1.0, np.abs(ref))) < 1e-4
            n_checked += 1
    return n_checked


def check_trace(O, path, backend):
    """G4: the 1000-step random-action trace, oracle and backend restarted from the RECORDED state before every step."""
    from tests import teacher as T

    return T.run_golden_trace(O, path, backend, force_states=True)


@needs_golden
@pytest.mark.parametrize("path", REAL, ids=[os.path.basename(p) for p in REAL])
def test_oracle_vs_pybullet(path, oracle_mod):
    assert check_oracle_dynamics(oracle_mod, path) > 0
    check_trace(oracle_mod, path, "emu")


@needs_golden
@pytest.mark.gpu
@pytest.mark.parametrize("path", REAL, ids=[os.path.basename(p) for p in REAL])
def test_device_vs_pybullet(path, oracle_mod):
    """The CUDA path against PyBullet's recorded values: M(q) and inverse dynamics 1e-4, contact-free step 1e-4
    (north_star), and the G4 trace teacher-forced from the recorded states."""
    import torch

    from mocca_envs_b200 import vec_env as V
    from tests import teacher as T

    g = np.load(path)
    name = _env_name(g)
    t = T.table_of(T.SPECS[name][1])
    A = t["n_dof"]
    st = g["g1_states"].astype(np.float32)
    env = getattr(V, T.SPECS[name][4])(len(st), device="cuda:0", seed=0)
    env.reset()
    env.set_state(torch.tensor(st))
    if g["g1_mass_matrix"].dtype.kind == "f" and g["g1_mass_matrix"].shape[1:] == (6 + A, 6 + A):
        M = env.mass_matrix().cpu().numpy()
        assert np.abs(M - g["g1_mass_matrix"]).max() / np.abs(g["g1_mass_matrix"]).max() < 1e-4
    if T.SPECS[name][0] in ("custom", "cassie"):
        env.step_physics(torch.tensor(g["g2_tau_acc"][:, :A].astype(np.float32)))
        out = env.get_state().cpu().numpy()
        ref = g["g2_after_step"]
        assert np.max(np.abs(out - ref) / np.maximum(1.0, np.abs(ref))) < 1e-4
    env.close()
    check_trace(oracle_mod, path, "gpu")
