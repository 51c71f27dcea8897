"""Pushes: mb200_apply_impulse / VecEnv.apply_impulse for every env kind, against a float64 reference and against the
laws of an impulsive push.

A linear impulse i at a world point p on link l changes the generalised velocity u = [omega_w, v_w, qd] by
du = M(q)^-1 J_l(p)^T i (Cassie: projected onto its two loop closures, G du = 0), clamped to max_coord_vel.  The CPU
legs run the kernel source (mb_apply_impulse) through the lane-loop emulation (tests/emu/emu_impulse.cpp); the GPU
legs (-m gpu) push the same states through VecEnv.apply_impulse and also require the device to equal the emulation.

The float64 reference is composed here from the oracle's forward kinematics and mass matrix: the point Jacobian is
the oracle's own point_jacobian (mocca_oracle.c) restated over orc_fk's link frames, and Cassie's response is the
dense KKT solve [[M, G^T], [G, 0]] [du, lambda] = [J^T i, 0] with G = the six btMultiBodyPoint2Point rows.  States come
from seeded resets and a few random-action steps; states with cond(M) >= 1e5 are skipped (DESIGN section 5).

Worst errors measured in the emulation (du vs the reference, relative to max |du_ref| of the push): walker3d 2.6e-5,
stepper 2.3e-5, pillar 2.0e-5, monkey 2.1e-5, cassie 7.9e-5, child 2.3e-5, mike 3.2e-5, walker2d 3.2e-6, crab2d 1.8e-6
(tolerance 2e-4).  Momentum residuals <= 2.6e-6 |i| (tolerance 1e-4), Cassie's |G du| <= 1.4e-6 |J du| (1e-4), linearity
<= 3.9e-6 (1e-5)."""
import ctypes as C
import functools
import json
import os
import subprocess

import numpy as np
import pytest

from tests.emu import emu as E
from tests.helpers import oracle_state

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL_REF = 2e-4   # du vs the float64 reference, relative to max |du_ref|
TOL_MOM = 1e-4   # base rows of M du vs the impulse's momentum, relative to |i|
TOL_LOOP = 1e-4  # |G du| relative to |J du| (Cassie)
# device vs emulation, relative to max |du|: max(1e-5, 0.1 cond(M) eps_f32).  du is a linear solve with the f32 mass
# matrix and factor the step kernels share; how the device rounds them (FMA contraction, the pivots' approximate rsqrt)
# moves du by up to ~0.04 cond(M) eps_f32 -- as much as compiling the emulation itself with FMA contraction does, and as
# much as either differs from the float64 reference.  A flat 1e-5 would fail on rounding alone from cond(M) ~ 2e3 up.
TOL_DEV, TOL_DEV_COND = 1e-5, 0.1
TOL_LIN = 1e-5   # du(i1 + i2) vs du(i1) + du(i2), relative to max |du|
COND_MAX = 1e5

# env kind -> emulation class, VecEnv class (+ kwargs), model, the links pushed besides the base (URDF link names: a foot,
# a hand or arm link, and a fixed link where the model has one)
KINDS = {
    "w3d": dict(emu=E.EmuW3D, vec="Walker3DCustomVecEnv", model="walker3d",
                links=("right_foot", "right_hand", "head")),
    "stepper": dict(emu=E.EmuStepper, vec="Walker3DStepperVecEnv", model="walker3d",
                    links=("left_foot", "left_lower_arm", "head")),
    "pillar": dict(emu=E.EmuPillar, vec="Walker3DStepperVecEnv", kw=dict(plank_class="Pillar"), model="walker3d",
                   links=("right_foot", "left_hand", "head")),
    "monkey": dict(emu=E.EmuMonkey, vec="Monkey3DCustomVecEnv", model="monkey3d",
                   links=("left_foot", "right_hand", "head")),
    "cassie": dict(emu=E.EmuCassie, vec="CassieVecEnv", model="cassie",
                   links=("left_toe", "right_tarsus", "vectorNav")),
    "child": dict(emu=E.EmuChild, vec="Child3DCustomVecEnv", model="child3d",
                  links=("right_foot", "left_hand", "head")),
    "mike": dict(emu=E.EmuMike, vec="MikeStepperVecEnv", model="mike",
                 links=("right_foot", "right_hand", "left_upper_arm")),
    "walker2d": dict(emu=E.EmuWalker2D, vec="Walker2DCustomVecEnv", model="walker2d",
                     links=("foot", "thigh_left", "torso")),
    "crab2d": dict(emu=E.EmuCrab2D, vec="Crab2DCustomVecEnv", model="crab2d",
                   links=("foot_left", "leg", "thigh")),
}
PLANAR = ("walker2d", "crab2d")
BACKENDS = ["emu", pytest.param("gpu", marks=pytest.mark.gpu)]


# ------------------------------------------------------------------------------------------------ emulation
_EMU_DIR = os.path.join(ROOT, "tests", "emu")
_EMU_SRC = os.path.join(_EMU_DIR, "emu_impulse.cpp")
_EMU_LIB = os.path.join(_EMU_DIR, "libmb_emu_impulse.so")


@functools.lru_cache(maxsize=None)
def _emu_lib():
    deps = [_EMU_SRC] + E._SRC[1:]
    if not os.path.exists(_EMU_LIB) or any(os.path.getmtime(s) > os.path.getmtime(_EMU_LIB) for s in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                               "-Wno-unused-variable", "-o", _EMU_LIB, _EMU_SRC])
    L = C.CDLL(_EMU_LIB)
    assert L.emu_impulse_sizeof_phys() == C.sizeof(E.Phys)
    return L


def _fp(a):
    return a.ctypes.data_as(C.c_void_p)


def emu_push(kind, state, link, point, impulse):
    """The state after mb_apply_impulse, through the emulated kernel source."""
    st = np.zeros(64, dtype=np.float32)
    st[:len(state)] = state
    fn = getattr(_emu_lib(), "emu_%s_apply_impulse" % kind.spec["emu"].prefix)
    fn(C.byref(kind.phys), _fp(st), C.c_int(int(link)), _fp(np.ascontiguousarray(point, dtype=np.float32)),
       _fp(np.ascontiguousarray(impulse, dtype=np.float32)))
    return st[:len(state)].copy()


# ------------------------------------------------------------------------------------------------ model / reference
def _O():
    from oracle import oracle as O

    O.build()
    return O


@functools.lru_cache(maxsize=None)
def _table(model):
    from mocca_envs_b200.model_compiler import load_table

    return load_table(os.path.join(ROOT, "mocca_envs_b200", "models", model + ".json"))


class Kind:
    def __init__(self, name):
        O = _O()
        self.name, self.spec = name, KINDS[name]
        self.t = t = _table(self.spec["model"])
        self.A = t["n_dof"]
        self.nu = 6 + self.A
        self.m = O.model_from_table(t)
        self.phys = self.spec["emu"].phys()
        self.vmax = float(self.phys.max_coord_vel)
        self.planar = bool(t.get("planar"))

    def urdf_link(self, name):
        return -1 if name == self.t["base"]["name"] else self.t["link_names"].index(name)

    def movable(self, li):
        """URDF link -> the kernel's link index (the dof of its nearest movable ancestor, -1 = base)."""
        while li >= 0 and self.t["dof_of_link"][li] < 0:
            li = self.t["parent"][li]
        return -1 if li < 0 else self.t["dof_of_link"][li]

    def u(self, row):
        return np.concatenate([row[7:13], row[13 + self.A:13 + 2 * self.A]]).astype(np.float64)

    def point_jacobian(self, c, pos, rot, li, pt):
        """[3][nu]: rows = the oracle's point_jacobian for the directions e_x, e_y, e_z."""
        m = self.m
        J = np.zeros((3, self.nu))
        rel = pt - c
        for k in range(3):
            e = np.eye(3)[k]
            J[k, 0:3] = np.cross(rel, e)
            J[k, 3:6] = e
        link = li
        while link >= 0:
            if m.dof_of_link[link] >= 0:
                aw = rot[link + 1] @ np.array(m.axis[link][:])
                piv = pos[link + 1] - rot[link + 1] @ np.array(m.d_vec[link][:])
                J[:, 6 + m.dof_of_link[link]] = np.cross(aw, pt - piv)
            link = m.parent[link]
        return J

    def loop_rows(self, c, pos, rot):
        """G [6][nu] (btMultiBodyPoint2Point rows: -e_ax on link A, +e_ax on link B) and the pivot gaps p_B - p_A."""
        m = self.m
        G, gaps = [], []
        for k in range(m.n_p2p):
            la, lb = m.p2p_link_a[k], m.p2p_link_b[k]
            pa = pos[la + 1] + rot[la + 1] @ np.array(m.p2p_pivot_a[k][:])
            pb = pos[lb + 1] + rot[lb + 1] @ np.array(m.p2p_pivot_b[k][:])
            JA, JB = self.point_jacobian(c, pos, rot, la, pa), self.point_jacobian(c, pos, rot, lb, pb)
            G.extend(JB[ax] - JA[ax] for ax in range(3))
            gaps.append(pb - pa)
        return (np.array(G), gaps) if G else (None, [])

    def reference(self, row, li, point, impulse):
        """float64 push of the f32 state `row`: dict(du (clamped), lam, M, J, G, gaps, cond)."""
        O = _O()
        row = np.asarray(row, dtype=np.float64)
        s = oracle_state(O, self.A, row)
        pos, rot = O.fk(self.m, s)
        iv, pv = np.array(impulse, dtype=np.float64), np.array(point, dtype=np.float64)
        if self.planar:
            iv[1] = pv[1] = 0.0
        M = O.mass_matrix(self.m, s)
        J = self.point_jacobian(row[0:3], pos, rot, li, pv)
        f = J.T @ iv
        G, gaps = self.loop_rows(row[0:3], pos, rot)
        lam = None
        if G is None:
            du = np.linalg.solve(M, f)
        else:
            ng = len(G)
            K = np.zeros((self.nu + ng, self.nu + ng))
            K[:self.nu, :self.nu], K[:self.nu, self.nu:], K[self.nu:, :self.nu] = M, G.T, G
            sol = np.linalg.solve(K, np.concatenate([f, np.zeros(ng)]))
            du, lam = sol[:self.nu], sol[self.nu:]
        u = self.u(row)
        unew = np.clip(u + du, -self.vmax, self.vmax)
        return dict(du=unew - u, raw=du, lam=lam, M=M, J=J, G=G, gaps=gaps, cond=np.linalg.cond(M), pos=pos,
                    iv=iv, pv=pv)


@functools.lru_cache(maxsize=None)
def _kind(name):
    return Kind(name)


@functools.lru_cache(maxsize=None)
def cases(name, n_states=6, seed=7):
    """Pushes at states of seeded resets plus 1-5 random-action steps (states with a coordinate velocity beyond half of
    max_coord_vel are passed over): on the base and on each of the kind's links, 1-50 N s in a random direction at a
    point within 5 cm of the link frame.  A push whose reference response reaches 90 % of max_coord_vel is halved
    until it does not (the clamp is tested by test_clamp)."""
    from mocca_envs_b200.seeding import mt_state_rows

    kind = _kind(name)
    rng = np.random.RandomState(seed)
    D = 13 + 2 * kind.A
    out, states = [], 0
    for k in range(20 * n_states):
        if states == n_states:
            break
        emu = kind.spec["emu"](mt_state=mt_state_rows([seed * 100 + k])[0])
        emu.reset()
        for _ in range(rng.randint(1, 6)):
            emu.step(rng.uniform(-1, 1, emu.act_dim).astype(np.float32))
        row = emu.state[:D].copy()
        s = oracle_state(_O(), kind.A, row.astype(np.float64))
        if np.abs(kind.u(row)).max() >= 0.5 * kind.vmax or np.linalg.cond(_O().mass_matrix(kind.m, s)) >= COND_MAX:
            continue  # (a light limb already near the clamp; an ill-conditioned M)
        states += 1
        pos, _ = _O().fk(kind.m, s)
        for lname in (kind.t["base"]["name"],) + kind.spec["links"]:
            li = kind.urdf_link(lname)
            pt = (pos[li + 1] + rng.uniform(-0.05, 0.05, 3)).astype(np.float32)
            d = rng.randn(3)
            imp = (rng.uniform(1, 50) * d / np.linalg.norm(d)).astype(np.float32)
            for _ in range(20):
                ref = kind.reference(row, li, pt, imp)
                if np.abs(kind.u(row) + ref["raw"]).max() < 0.9 * kind.vmax:
                    break
                imp = (imp * np.float32(0.5)).astype(np.float32)
            out.append(dict(state=row, li=li, link=kind.movable(li), point=pt, impulse=imp))
    assert states == n_states, (name, states)
    return out


# ------------------------------------------------------------------------------------------------ runners
def run_emu(kind, cs):
    return np.array([emu_push(kind, c["state"], c["link"], c["point"], c["impulse"]) for c in cs])


def _vec(kind, n):
    import torch
    from mocca_envs_b200 import vec_env as V

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return getattr(V, kind.spec["vec"])(n, device="cuda:0", seed=0, **kind.spec.get("kw", {}))


def run_gpu(kind, cs, steps=0):
    """The states after VecEnv.apply_impulse (one env per case); `steps` random-action steps follow, which must stay
    finite."""
    import torch

    env = _vec(kind, len(cs))
    try:
        env.reset()
        env.set_state(torch.tensor(np.stack([c["state"] for c in cs])))
        env.stats(reset=True)
        env.apply_impulse(torch.tensor(np.stack([c["impulse"] for c in cs])),
                          link=torch.tensor([c["link"] for c in cs], dtype=torch.int32),
                          point=torch.tensor(np.stack([c["point"] for c in cs])))
        out = env.get_state().cpu().numpy()
        rng = np.random.RandomState(0)
        for _ in range(steps):
            obs, rew, _, _ = env.step(torch.tensor(rng.uniform(-1, 1, (len(cs), env.act_dim)), dtype=torch.float32))
            assert torch.isfinite(obs).all() and torch.isfinite(rew).all()
        if steps:
            assert env.stats()["nonfinite"] == 0
            assert np.isfinite(env.get_state().cpu().numpy()).all()
    finally:
        env.close()
    return out


def run(kind, cs, backend):
    if backend == "emu":
        return run_emu(kind, cs)
    return run_gpu(kind, cs)


def _du(kind, before, after):
    return kind.u(after) - kind.u(before)


# ------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name", list(KINDS))
def test_vs_reference(name, backend):
    """du equals the float64 reference to 2e-4 of max |du_ref|; pos, quat and q are untouched bit for bit.  On the
    device du also equals the emulation's to max(1e-5, 0.1 cond(M) eps_f32) (see TOL_DEV), and ten env steps after
    the push stay finite."""
    kind = _kind(name)
    cs = cases(name)
    outs = run(kind, cs, backend)
    D = 13 + kind.A
    worst = 0.0
    for i, (c, after) in enumerate(zip(cs, outs)):
        ref = kind.reference(c["state"], c["li"], c["point"], c["impulse"])
        du = _du(kind, c["state"], after)
        scale = np.abs(ref["du"]).max()
        err = np.abs(du - ref["du"]).max() / scale
        assert err < TOL_REF, (name, i, c["li"], err)
        assert np.array_equal(after[0:7], c["state"][0:7]) and np.array_equal(after[13:D], c["state"][13:D]), (name, i)
        worst = max(worst, err)
    if backend == "gpu":
        emu = run_emu(kind, cs)
        eps = float(np.finfo(np.float32).eps)
        dev = 0.0  # worst error in units of the case's tolerance
        for i, (c, a, b) in enumerate(zip(cs, outs, emu)):
            da, db = _du(kind, c["state"], a), _du(kind, c["state"], b)
            err = np.abs(da - db).max() / np.abs(db).max()
            cond = kind.reference(c["state"], c["li"], c["point"], c["impulse"])["cond"]
            tol = max(TOL_DEV, TOL_DEV_COND * cond * eps)
            assert err < tol, (name, i, c["li"], err, cond, tol)
            dev = max(dev, err / tol)
        run_gpu(kind, cs, steps=10)
        print("\n%s gpu: vs reference %.2g, vs emulation %.2g of its tolerance" % (name, worst, dev))
    else:
        print("\n%s emu: vs reference %.2g" % (name, worst))


def _mass_matrices(kind, cs, backend):
    if backend == "emu":
        Ms = []
        for c in cs:
            e = kind.spec["emu"]()
            e.state[:len(c["state"])] = c["state"]
            Ms.append(e.mass_matrix()[0])
        return np.array(Ms, dtype=np.float64)
    import torch

    env = _vec(kind, len(cs))
    try:
        env.set_state(torch.tensor(np.stack([c["state"] for c in cs])))
        return env.mass_matrix().cpu().numpy().astype(np.float64)
    finally:
        env.close()


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name", list(KINDS))
def test_momentum(name, backend):
    """With the kernel's own M at the pre-push state, the base rows of M du are the impulse's momentum about the base
    COM: [(p - c) x i ; i] to 1e-4 |i|.  Cassie: the linear part is exact, the angular part differs by the loop
    closures' pivot-gap term sum (p_B - p_A) x lambda only."""
    kind = _kind(name)
    cs = cases(name)
    outs = run(kind, cs, backend)
    Ms = _mass_matrices(kind, cs, backend)
    worst = 0.0
    for i, (c, after, M) in enumerate(zip(cs, outs, Ms)):
        ref = kind.reference(c["state"], c["li"], c["point"], c["impulse"])
        iv, pv = ref["iv"], ref["pv"]
        h = M @ _du(kind, c["state"], after)
        want_ang = np.cross(pv - c["state"][0:3].astype(np.float64), iv)
        if ref["lam"] is not None:
            for k, gap in enumerate(ref["gaps"]):
                want_ang -= np.cross(gap, ref["lam"][3 * k:3 * k + 3])
        err = max(np.abs(h[0:3] - want_ang).max(), np.abs(h[3:6] - iv).max()) / np.linalg.norm(iv)
        assert err < TOL_MOM, (name, i, c["li"], err, h[0:6], want_ang, iv)
        worst = max(worst, err)
    print("\n%s %s: momentum %.2g" % (name, backend, worst))


@pytest.mark.parametrize("backend", BACKENDS)
def test_cassie_loops_stay_closed(backend):
    """The relative velocity change across each achilles-rod closure, G du, is below 1e-4 of the pushed point's
    velocity change |J du|."""
    kind = _kind("cassie")
    cs = cases("cassie")
    worst = 0.0
    for c, after in zip(cs, run(kind, cs, backend)):
        ref = kind.reference(c["state"], c["li"], c["point"], c["impulse"])
        du = _du(kind, c["state"], after)
        r = np.abs(ref["G"] @ du).max() / np.linalg.norm(ref["J"] @ du)
        assert r < TOL_LOOP, (c["li"], r)
        worst = max(worst, r)
    print("\ncassie %s: |G du| / |J du| %.2g" % (backend, worst))


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name", list(KINDS))
def test_linearity(name, backend):
    """du(i1 + i2) = du(i1) + du(i2) at the same state and point, to float32 rounding."""
    kind = _kind(name)
    rng = np.random.RandomState(3)
    base = cases(name)[::2]
    parts = []
    for c in base:
        i1 = c["impulse"]
        i2 = (np.linalg.norm(i1) * rng.uniform(-0.5, 0.5, 3)).astype(np.float32)
        while np.abs(kind.u(c["state"]) + kind.reference(c["state"], c["li"], c["point"], i1 + i2)["raw"]).max() \
                >= 0.9 * kind.vmax:  # (both parts and their sum stay clear of the clamp)
            i1, i2 = i1 * np.float32(0.5), i2 * np.float32(0.5)
        for imp in (i1, i2, i1 + i2):
            parts.append(dict(c, impulse=imp.astype(np.float32)))
    outs = run(kind, parts, backend)
    worst = 0.0
    for k, c in enumerate(base):
        d1, d2, d12 = (_du(kind, c["state"], outs[3 * k + j]) for j in range(3))
        scale = max(np.abs(d1).max(), np.abs(d2).max(), np.abs(d12).max())
        err = np.abs(d12 - d1 - d2).max() / scale
        assert err < TOL_LIN, (name, k, err)
        worst = max(worst, err)
    print("\n%s %s: linearity %.2g" % (name, backend, worst))


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name", PLANAR)
def test_planar(name, backend):
    """Any 3-D impulse and point keep y, v_y, omega_x, omega_z and quaternion x / z exactly zero, and the result is bit
    for bit the result of the inputs with their y components zeroed."""
    kind = _kind(name)
    rng = np.random.RandomState(5)
    base = cases(name)
    full, proj = [], []
    for c in base:
        imp = c["impulse"] + rng.uniform(-20, 20, 3).astype(np.float32) * np.float32([0, 1, 0])
        pt = c["point"] + np.float32([0, rng.uniform(-0.3, 0.3), 0])
        full.append(dict(c, impulse=imp, point=pt))
        proj.append(dict(c, impulse=imp * np.float32([1, 0, 1]), point=pt * np.float32([1, 0, 1])))
    a, b = run(kind, full + proj, backend).reshape(2, len(base), -1)
    assert np.array_equal(a, b)
    for c, after in zip(base, a):
        assert c["state"][1] == 0 and c["state"][3] == 0 and c["state"][5] == 0
        assert after[1] == 0 and after[11] == 0 and after[7] == 0 and after[9] == 0, after[:13]
        assert after[3] == 0 and after[5] == 0, after[3:7]
        assert not np.array_equal(after, c["state"])


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name", list(KINDS))
def test_untouched(name, backend):
    """Link -2 or NJ, a zero impulse, a NaN or an infinite impulse and a non-finite point leave the env's state bit for
    bit; so does a pure y impulse on a planar model."""
    kind = _kind(name)
    c = cases(name)[1]
    bad = [dict(c, link=-2), dict(c, link=kind.A), dict(c, link=-7),
           dict(c, impulse=np.zeros(3, np.float32)),
           dict(c, impulse=np.float32([np.nan, 1, 1])), dict(c, impulse=np.float32([np.inf, 0, 0])),
           dict(c, point=np.float32([0, np.nan, 0]) if not kind.planar else np.float32([np.nan, 0, 0]))]
    if kind.planar:
        bad.append(dict(c, impulse=np.float32([0, 5, 0])))
    outs = run(kind, bad + [c], backend)
    for k, after in enumerate(outs[:-1]):
        assert np.array_equal(after, c["state"]), (name, k)
    assert not np.array_equal(outs[-1], c["state"])


@pytest.mark.parametrize("backend", BACKENDS)
def test_clamp(backend):
    """A push past max_coord_vel ends at the clamp, as every velocity update of a substep does."""
    kind = _kind("w3d")
    c = dict(cases("w3d")[1], impulse=np.float32([0, 0, 5000]))
    after = run(kind, [c], backend)[0]
    u = kind.u(after)
    ref = kind.reference(c["state"], c["li"], c["point"], c["impulse"])
    assert np.abs(u).max() == np.float32(kind.vmax)
    hit = np.abs(kind.u(c["state"]) + ref["raw"]) > 1.001 * kind.vmax
    assert hit.any() and np.all(np.abs(u[hit]) == np.float32(kind.vmax))


# ------------------------------------------------------------------------------------------------ Python layer
def _bare_vec(cls_name, model, num_envs=1):
    """A VecEnv object without a device handle: enough for link_index and the argument checks of apply_impulse."""
    import torch
    from mocca_envs_b200 import vec_env as V

    env = object.__new__(getattr(V, cls_name))
    env.model = model
    with open(os.path.join(ROOT, "mocca_envs_b200", "models", model + ".json")) as f:
        env.table = json.load(f)
    env.num_envs, env.device, env.nu = num_envs, torch.device("cpu"), 6 + env.table["n_dof"]
    return env


@pytest.mark.parametrize("name", list(KINDS))
def test_link_index(name):
    """link_index maps every URDF link name to the kernel's link index (fixed links folded, the base's name -> -1) and
    raises KeyError for unknown names."""
    kind = _kind(name)
    env = _bare_vec(kind.spec["vec"], kind.spec["model"])
    assert env.link_index(kind.t["base"]["name"]) == -1
    for li, lname in enumerate(kind.t["link_names"]):
        assert env.link_index(lname) == kind.movable(li), lname
    with pytest.raises(KeyError):
        env.link_index("no_such_link")
    if name in ("w3d", "cassie"):
        assert env.link_index({"w3d": "head", "cassie": "vectorNav"}[name]) == -1


def test_apply_impulse_argument_errors():
    env = _bare_vec("Walker3DCustomVecEnv", "walker3d")
    with pytest.raises(ValueError):
        env.apply_impulse([0, 0, 1], link=21)
    with pytest.raises(ValueError):
        env.apply_impulse([0, 0, 1], link=-2)
    with pytest.raises(ValueError):
        env.apply_impulse([0, 0, 1], link=3)  # point=None is the base COM: link -1 only
    import torch

    with pytest.raises(ValueError):
        env.apply_impulse([0, 0, 1], link=torch.tensor([-1]))


@pytest.mark.gpu
def test_facade_push():
    """The N = 1 gym facade takes NumPy inputs; its push equals the VecEnv's on the same state."""
    import torch
    from mocca_envs_b200 import vec_env as V

    g = V.Walker3DCustomEnv(seed=3)
    v = V.Walker3DCustomVecEnv(1, seed=3)
    try:
        g.reset()
        v.reset()
        link = g.link_index("right_foot")
        g.apply_impulse(np.array([3.0, -2.0, 5.0]), link=link, point=np.array([0.1, -0.1, 0.2]))
        v.apply_impulse(torch.tensor([3.0, -2.0, 5.0]), link=link, point=torch.tensor([0.1, -0.1, 0.2]))
        a, b = g.vec.get_state().cpu().numpy(), v.get_state().cpu().numpy()
        assert np.array_equal(a, b)
        g.apply_impulse([0.0, 0.0, 10.0])  # the base, at its COM
        o, r, d, info = g.step(np.zeros(g.action_space.shape))
        assert np.isfinite(o).all()
    finally:
        g.close()
        v.close()
