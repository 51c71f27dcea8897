"""Contact lists of every collision path of Sim::collide, contact by contact, against the float64 oracle.

One stepSimulation of ONE substep from an f32-rounded state: the points the kernel reports (what
mb200_step_physics_points returns, the stand-in for pybullet.getContactPoints) must be the oracle's contact list of
that substep in the same order -- link, partner, point, normal, distance and normal impulse -- and the unused slots
must be empty.  The list decides the constraint rows, the warm-start slots, feet_contact and what the 16-point cap
drops, so a wrong order or a wrong normal on a lightly loaded contact is a bug even when the state after the step
barely moves.

The CPU legs run the kernel source through the lane-loop emulation (tests/emu); the GPU legs (-m gpu) run the same
cases through VecEnv.step_physics_points on the device and also require the device list to equal the emulated one.

Cases are kept out of the regions where float32 and float64 may legitimately disagree: a sampled case is rejected
when the oracle's contact set changes with every contact-breaking threshold moved by +-1e-4, when a joint is within
1e-4 of a limit (a quarter of the range for Mike's locked joints), when the oracle exceeds the 16 contacts or 48 rows
the kernel keeps (a self-contact counting 6 rows there; the caps are not tested here), when a box-vs-bar sample
choice is within 2e-6 of its tie, or when two self-collision core segments cross (gap < 1e-5: in the oracle the pair
is skipped below a 1e-9 gap, while float32 rounding leaves the kernel a gap of ~1e-7 and a contact with an arbitrary
normal -- planar models meet this whenever two limbs overlap)."""
import functools
import os

import numpy as np
import pytest

from tests.emu import emu as E
from tests.helpers import oracle_state, random_states, self_contact_states

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAXC, MAXROW = 16, 48
TOL_GEOM = 2e-5  # point, normal, distance vs the oracle
TOL_IMP = 2e-3  # normal impulse, relative to max(largest impulse of the list, m g dt)
# Cassie's contact rows share the PGS sweeps with the two achilles-rod loop closures, which the float32 solver
# converges less closely in its five iterations
TOL_IMP_CASSIE = 1e-2
TOL_DEV = 1e-5  # device vs emulation geometry

# env kind -> emulation class, VecEnv class (+ kwargs), model, obstacles, whether the kind keeps the ground plane
KINDS = {
    "walker3d": dict(emu=E.EmuW3D, vec="Walker3DCustomVecEnv", model="walker3d", obst=None),
    "child3d": dict(emu=E.EmuChild, vec="Child3DCustomVecEnv", model="child3d", obst=None),
    "walker2d": dict(emu=E.EmuWalker2D, vec="Walker2DCustomVecEnv", model="walker2d", obst=None),
    "crab2d": dict(emu=E.EmuCrab2D, vec="Crab2DCustomVecEnv", model="crab2d", obst=None),
    "cassie": dict(emu=E.EmuCassie, vec="CassieVecEnv", model="cassie", obst=None),
    # the MikeStepperEnv kernel source with the ground plane switched on (the env itself removes it, so this leg
    # exists in the emulation only): the STORE ground pass on a model with exactly NPT = 32 candidates
    "mike_ground": dict(emu=E.EmuMike, vec=None, model="mike", obst=None, ground=1, far_planks=True),
    "stepper": dict(emu=E.EmuStepper, vec="Walker3DStepperVecEnv", model="walker3d", obst="boxes", plank_class=0),
    "plank": dict(emu=E.EmuStepper, vec="Walker3DStepperVecEnv", model="walker3d", obst="boxes", plank_class=1),
    "mike": dict(emu=E.EmuMike, vec="MikeStepperVecEnv", model="mike", obst="boxes", plank_class=0),
    "pillar": dict(emu=E.EmuPillar, vec="Walker3DStepperVecEnv", model="walker3d", obst="boxes", plank_class=2),
    "monkey": dict(emu=E.EmuMonkey, vec="Monkey3DCustomVecEnv", model="monkey3d", obst="bars"),
}
ES_PLANK_CLASS, ES_BOX, EM_BAR = 4, 32, 32
PLANK_NAMES = {0: "LargePlank", 1: "Plank", 2: "Pillar"}


# ------------------------------------------------------------------------------------------------ model / oracle
@functools.lru_cache(maxsize=None)
def _table(model):
    from mocca_envs_b200.model_compiler import load_table

    return load_table(os.path.join(ROOT, "mocca_envs_b200", "models", model + ".json"))


def _O():
    from oracle import oracle as O

    O.build()
    return O


class Kind:
    """The oracle's view of one env kind plus the maps between its contact list and the kernel's."""

    def __init__(self, name):
        O = _O()
        self.name, self.spec = name, KINDS[name]
        self.t = t = _table(self.spec["model"])
        self.A = t["n_dof"]
        self.m = O.model_from_table(t)
        p = O.cassie_params() if name == "cassie" else O.default_params()
        p.substeps = 1
        p.has_ground = self.spec.get("ground", 0 if self.spec["obst"] == "boxes" else 1)
        self.p = p
        self.dt = float(p.dt)
        self.imp_floor = float(t["total_mass"]) * 9.8 * self.dt
        # oracle link -> the dof of its nearest movable ancestor (-1: the base)
        self.movable = {-1: -1}
        for link in range(t["n_links"]):
            k = link
            while k >= 0 and t["dof_of_link"][k] < 0:
                k = t["parent"][k]
            self.movable[link] = -1 if k < 0 else t["dof_of_link"][k]
        # candidate points (sphere centres, capsule end spheres) in the kernel's order: oracle point_id -> index
        self.cands = []  # (geom, end, link, radius)
        for g, geom in enumerate(t["geoms"]):
            if geom["type"] == 2:
                continue
            for e in range(2 if geom["type"] == 1 else 1):
                self.cands.append((g, e, geom["link"], geom["size"][0]))
        self.cand_of_pid = {2 * g + e: i for i, (g, e, _, _) in enumerate(self.cands)}
        self.geom_cands = {g: (self.cand_of_pid[2 * g], self.cand_of_pid.get(2 * g + 1, self.cand_of_pid[2 * g]))
                           for g, _, _, _ in self.cands}
        self.boxgeoms = [g for g, geom in enumerate(t["geoms"]) if geom["type"] == 2]
        self.pairs = t.get("self_pairs", [])

    # ---- obstacles: the record rows (f32) and the oracle's structures built from exactly those numbers
    def oracle_boxes(self, planks, plank_class):
        O = _O()
        boxes = (O.Box * 6)()
        hy = {0: 5.0, 1: 0.375, 2: 0.25}[plank_class]
        for p in range(3):
            c = planks[p, 0:3]
            R = planks[p, 3:12].reshape(3, 3)
            cover = c + R[:, 2] * np.float32(0.125)  # as load_boxes does it, in f32
            for k, (cen, hz) in enumerate(((c, 0.1125), (cover, 0.0125))):
                b = boxes[2 * p + k]
                for i in range(3):
                    b.center[i] = float(cen[i])
                    for j in range(3):
                        b.R[i][j] = float(R[i, j])
                b.half[0], b.half[1], b.half[2] = 0.25, hy, hz
                b.friction, b.stiffness, b.damping = 1.0, 30000.0, 1000.0 + 0.1
                b.id, b.cylinder = 10 + 2 * p + k, int(plank_class == 2)
        return boxes

    def oracle_bars(self, bars):
        O = _O()
        out = (O.Bar * 4)()
        for k in range(4):
            b = out[k]
            for i in range(3):
                b.center[i] = float(bars[k, i])
                b.axis[i] = float(bars[k, 3 + i])
            b.halflen, b.radius, b.friction, b.id = float(bars[k, 6]), float(bars[k, 7]), 0.5, 20 + k
        return out

    def oracle_step(self, case, m=None):
        """The oracle's contact list and rows of the case's one-substep stepSimulation."""
        O = _O()
        s = oracle_state(O, self.A, case["state"].astype(np.float64))
        tau = case["tau"].astype(np.float64)
        m = m or self.m
        if self.spec["obst"] == "bars":
            return O.step_physics_bars(m, self.p, s, tau, self.oracle_bars(case["bars"]))
        boxes = self.oracle_boxes(case["planks"], self.spec["plank_class"]) if self.spec["obst"] == "boxes" else None
        return O.step_physics(m, self.p, s, tau, boxes=boxes)

    def world_points(self, row):
        """World centres of the candidate points and the robot box geoms (centre, rotation, half sizes) at `row`."""
        O = _O()
        pos, rot = O.fk(self.m, oracle_state(O, self.A, row.astype(np.float64)))
        pts = []
        for g, e, link, r in self.cands:
            geom = self.t["geoms"][g]
            loc = np.array(geom["p0"] if e == 0 else geom["p1"])
            pts.append(pos[link + 1] + rot[link + 1] @ loc)  # (fk: rotations local -> world)
        boxes = []
        for g in self.boxgeoms:
            geom = self.t["geoms"][g]
            link = geom["link"]
            x, y, z, w = geom["quat"]
            Rg = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                           [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                           [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
            boxes.append((pos[link + 1] + rot[link + 1] @ np.array(geom["p0"]), rot[link + 1] @ Rg,
                          np.array(geom["size"]), self.m.link_thresh[link + 1]))
        return np.array(pts), boxes


def _signature(c):
    return [(c.point_id[k], c.link[k], c.partner[k], c.link_b[k]) for k in range(c.n)]


def _box_bar_samples(box, bar):
    """box_bar's five sample distances in visiting order (0, -1, +1, -2, +2), each with the distance of its own
    decisions from their ties (inside: the gap between the two shallowest face penetrations; outside: the gap to the
    contact threshold).  A sample outside the threshold has distance inf."""
    cen, R, half, thresh = box
    axis, c, hl, rad = bar[3:6].astype(np.float64), bar[0:3].astype(np.float64), float(bar[6]), float(bar[7])
    t0 = float((cen - c) @ axis)
    out = []
    for k in (0, -1, 1, -2, 2):
        t = min(max(t0 + 0.03 * k, -hl), hl)
        cl = R.T @ (c + t * axis - cen)
        qc = np.clip(cl, -half, half)
        if np.array_equal(qc, cl):
            pens = np.sort(half - np.abs(cl))
            out.append((-pens[0] - rad, pens[1] - pens[0]))
        else:
            ds = float(np.linalg.norm(cl - qc)) - rad
            out.append((ds if ds < thresh else np.inf, abs(thresh - ds)))
    return out


def _box_bar_margin(box, bar):
    """Distance of the oracle's box_bar choices from their ties: the samples' own decisions and, for every sample,
    the gap between its distance and the 'deeper by 1e-5' threshold of the sequential rule."""
    best, margin = np.inf, 1.0
    for ds, m in _box_bar_samples(box, bar):
        margin = min(margin, m)
        if np.isfinite(ds) and np.isfinite(best):
            margin = min(margin, abs(ds - (best - 1e-5)))
        if ds < best - 1e-5:
            best = ds
    return margin


def _seg_gap(a, b):
    """Distance of the segments a and b (the oracle's seg_seg, Ericson 5.1.9, in float64)."""
    d1, d2, r = a[1] - a[0], b[1] - b[0], a[0] - b[0]
    A, Ee, F = d1 @ d1, d2 @ d2, d2 @ r
    s = t = 0.0
    if A <= 1e-12 and Ee <= 1e-12:
        pass
    elif A <= 1e-12:
        t = np.clip(F / Ee, 0, 1)
    else:
        Cc = d1 @ r
        if Ee <= 1e-12:
            s = np.clip(-Cc / A, 0, 1)
        else:
            B = d1 @ d2
            den = A * Ee - B * B
            s = np.clip((B * F - Cc * Ee) / den, 0, 1) if den > 1e-12 else 0.0
            t = (B * s + F) / Ee
            if t < 0:
                t, s = 0.0, np.clip(-Cc / A, 0, 1)
            elif t > 1:
                t, s = 1.0, np.clip((B - Cc) / A, 0, 1)
    return float(np.linalg.norm(a[0] + d1 * s - b[0] - d2 * t))


def _robust(kind, case, c, rows):
    """The case is far enough from every f32 / f64 decision boundary (see the module docstring)."""
    O = _O()
    if c.n > MAXC or rows > MAXROW:
        return False
    A = kind.A
    q = case["state"][13:13 + A].astype(np.float64)
    lo, hi = np.array(kind.t["lower"]), np.array(kind.t["upper"])
    near = np.minimum(1e-4, 0.25 * (hi - lo))  # (Mike's locked joints have a range of 3.5e-5)
    if np.any((lo <= hi) & ((np.abs(q - lo) < near) | (np.abs(q - hi) < near))):
        return False
    # the kernel's row budget counts a self-contact twice
    nself = sum(1 for k in range(c.n) if c.partner[k] >= 1000)
    if rows + 3 * nself > MAXROW:
        return False
    # crossing core segments (gap below 1e-5) have no defined normal: f32 rounding decides whether a contact exists
    pts, _ = kind.world_points(case["state"])
    for ga, gb in kind.pairs:
        ends = []
        for g in (ga, gb):
            i0, i1 = kind.geom_cands[g]
            ends.append((pts[i0], pts[i1]))
        if _seg_gap(ends[0], ends[1]) < 1e-5:
            return False
    sig = _signature(c)
    for sgn in (1.0, -1.0):
        m2 = O.Model.from_buffer_copy(bytes(kind.m))
        for k in range(kind.t["n_links"] + 1):
            m2.link_thresh[k] += sgn * 1e-4
        c2, _ = kind.oracle_step(case, m2)
        if _signature(c2) != sig:
            return False
    if kind.spec["obst"] == "bars" and kind.boxgeoms:
        _, boxes = kind.world_points(case["state"])
        for bar in case["bars"]:
            for box in boxes:
                if _box_bar_margin(box, bar) < 2e-6:
                    return False
    return True


def _accept(kind, case, cases, n):
    """Append the case if it is robust; returns the oracle's (contacts, rows) or None."""
    c, rows = kind.oracle_step(case)
    if c.n == 0 or not _robust(kind, case, c, rows):
        return None
    cases.append(case)
    return c


def _case(kind, row, tau, **obst):
    d = dict(state=np.asarray(row, dtype=np.float32), tau=np.asarray(tau, dtype=np.float32))
    d.update(obst)
    return d


def _pose(kind, rng, spin=0.3, margin=0.2):
    """A random f32 state (joints well inside their limits); planar models stay in the x-z plane."""
    t, A = kind.t, kind.A
    row = random_states(t, rng, 1, spin=spin, margin=margin)[0]
    lo, hi = np.array(t["lower"]), np.array(t["upper"])
    locked = (lo <= hi) & (hi - lo < 1e-3)
    row[13:13 + A][locked] = 0.5 * (lo + hi)[locked]
    if t.get("planar"):
        a = rng.uniform(-0.6, 0.6)
        row[3:7] = [0, np.sin(a / 2), 0, np.cos(a / 2)]
        row[7:10] = [0, spin * rng.randn(), 0]
        row[10:13] = [rng.randn(), 0, rng.randn()]
        row[1] = 0.0
    return row.astype(np.float32)


def _tau(kind, rng, scale=0.3):
    return (scale * np.array(kind.t["gain"]) * rng.uniform(-1, 1, kind.A)).astype(np.float32)


def _lower_to_ground(kind, row, target, depth):
    """Shift the base vertically so that candidate `target`'s sphere reaches `depth` below the plane z = 0."""
    pts, _ = kind.world_points(row)
    r = kind.cands[target][3]
    row = row.copy()
    row[2] = np.float32(row[2] - (pts[target, 2] - r + depth))
    return row


# ------------------------------------------------------------------------------------------------ runners
def run_emu(kind, cases):
    out = []
    for cs in cases:
        emu = kind.spec["emu"]()
        emu.p.substeps = 1
        if "ground" in kind.spec:
            emu.p.has_ground = kind.spec["ground"]
        n = len(cs["state"])
        emu.state[:n] = cs["state"]
        _write_obstacles(kind, cs, emu.rec)
        pts = np.zeros((MAXC, 10), dtype=np.float32)
        rows, nc = emu.step_physics(cs["tau"], points=pts)
        out.append((rows, nc, pts))
    return out


def _write_obstacles(kind, cs, rec):
    if kind.spec.get("far_planks"):
        rec[ES_BOX:ES_BOX + 36] = _far_planks().ravel()
    if kind.spec["obst"] == "boxes":
        rec.view(np.int32)[ES_PLANK_CLASS] = kind.spec["plank_class"]
        rec[ES_BOX:ES_BOX + 36] = cs["planks"].ravel()
    elif kind.spec["obst"] == "bars":
        rec[EM_BAR:EM_BAR + 32] = cs["bars"].ravel()


def run_gpu(kind, cases):
    import torch
    from mocca_envs_b200 import vec_env as V

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    kw = {}
    if kind.spec["obst"] == "boxes":
        kw["plank_class"] = PLANK_NAMES[kind.spec["plank_class"]]
    N = len(cases)
    assert N <= 64
    env = getattr(V, kind.spec["vec"])(N, device="cuda:0", seed=0, physics={"substeps": 1}, **kw)
    try:
        env.reset()
        rec = env.get_record().cpu().numpy()
        for i, cs in enumerate(cases):
            _write_obstacles(kind, cs, rec[i])
        env.set_record(torch.tensor(rec))
        st = np.zeros((N, env.state_dim), dtype=np.float32)
        for i, cs in enumerate(cases):
            st[i, :len(cs["state"])] = cs["state"]
        env.set_state(torch.tensor(st))
        tau = torch.tensor(np.stack([cs["tau"] for cs in cases]))
        rows, nc, pts = env.step_physics_points(tau)
        torch.cuda.synchronize()
        rows, nc, pts = rows.cpu().numpy(), nc.cpu().numpy(), pts.cpu().numpy()
    finally:
        env.close()
    return [(int(rows[i]), int(nc[i]), pts[i]) for i in range(N)]


# ------------------------------------------------------------------------------------------------ comparisons
def check_vs_oracle(kind, cases, outs):
    """Every list equals the oracle's, index by index.  Returns the worst errors (point, normal, distance, impulse
    relative to the list's scale) for the docstrings."""
    worst = np.zeros(4)
    gl = [g["link"] for g in kind.t["geoms"]]
    for i, (cs, (rows, nc, pts)) in enumerate(zip(cases, outs)):
        c, rows_ref = kind.oracle_step(cs)
        where = "%s case %d" % (kind.name, i)
        assert nc == c.n and rows == rows_ref, (where, nc, c.n, rows, rows_ref)
        imp_ref = np.array(c.impulse[:c.n])
        scale = max(np.abs(imp_ref).max(initial=0.0), kind.imp_floor)
        for k in range(c.n):
            o = pts[k]
            assert int(o[8]) == kind.movable[c.link[k]], (where, k, int(o[8]), c.link[k])
            partner = int(o[9])
            if c.partner[k] >= 1000:
                assert partner >= 1000, (where, k, partner)
                ga, gb = kind.pairs[partner - 1000]
                assert (gl[ga], gl[gb]) == (c.link[k], c.link_b[k]), (where, k, partner, c.link[k], c.link_b[k])
                ln = c.dist[k] + kind.t["geoms"][ga]["size"][0] + kind.t["geoms"][gb]["size"][0]
                tol_n = TOL_GEOM / min(1.0, ln)
            else:
                assert partner == c.partner[k], (where, k, partner, c.partner[k])
                tol_n = TOL_GEOM
            e = np.array([np.abs(o[0:3] - np.array(c.pos_a[k][:])).max(),
                          np.abs(o[3:6] - np.array(c.normal[k][:])).max(),
                          abs(o[6] - c.dist[k]), abs(o[7] - c.impulse[k]) / scale])
            assert e[0] < TOL_GEOM and e[1] < tol_n and e[2] < TOL_GEOM, (where, k, e)
            assert e[3] < (TOL_IMP_CASSIE if kind.name == "cassie" else TOL_IMP), (where, k, o[7], c.impulse[k], scale)
            worst = np.maximum(worst, e)
        assert np.all(pts[c.n:, 8] == -2.0), where
        assert not np.any(pts[c.n:, [0, 1, 2, 3, 4, 5, 6, 7, 9]]), where
    return worst


def check_same_lists(a, b):
    """The device list equals the emulated one: counts, order, link and partner exactly, geometry within 1e-5."""
    worst = 0.0
    for i, ((ra, na, pa), (rb, nb, pb)) in enumerate(zip(a, b)):
        assert (ra, na) == (rb, nb), (i, ra, na, rb, nb)
        assert np.array_equal(pa[:, 8:10], pb[:, 8:10]), i
        d = np.abs(pa[:, 0:7] - pb[:, 0:7]).max()
        assert d < TOL_DEV, (i, d)
        worst = max(worst, d)
    return worst


def run_and_check(kind_name, cases, backend):
    kind = Kind(kind_name)
    if backend == "emu":
        worst = check_vs_oracle(kind, cases, run_emu(kind, cases))
        print("\n%s emu: point %.2g normal %.2g dist %.2g impulse %.2g" % ((kind_name,) + tuple(worst)))
        return worst
    dev = run_gpu(kind, cases)
    worst = check_vs_oracle(kind, cases, dev)
    d = check_same_lists(dev, run_emu(kind, cases))
    print("\n%s gpu: point %.2g normal %.2g dist %.2g impulse %.2g; device vs emulation %.2g"
          % ((kind_name,) + tuple(worst) + (d,)))
    return worst


BACKENDS = ["emu", pytest.param("gpu", marks=pytest.mark.gpu)]


# ------------------------------------------------------------------------------------------------ case generators
def _far_planks():
    planks = np.zeros((3, 12), dtype=np.float32)
    planks[:, 0:3] = [[0, 0, -50], [0, 20, -50], [0, -20, -50]]
    planks[:, 3:12] = np.eye(3, dtype=np.float32).ravel()
    return planks


def _far_bars():
    bars = np.zeros((4, 8), dtype=np.float32)
    for k in range(4):
        bars[k] = [10.0 * k, 0, -100, 0, 1, 0, 2.5, 0.015]
    return bars


def _rot(rng, tilt):
    """Rotation (row-major, world from local) of a random yaw and roll / pitch up to `tilt`."""
    from scipy.spatial.transform import Rotation

    return Rotation.from_euler("xyz", [rng.uniform(-tilt, tilt), rng.uniform(-tilt, tilt),
                                       rng.uniform(-np.pi, np.pi)]).as_matrix()


def _place(planks, p, R, local, world):
    """Plank p (base-box frame R) placed so that the local point `local` lands on the world point `world`."""
    planks[p, 0:3] = world - R @ np.asarray(local)
    planks[p, 3:12] = R.ravel()


@functools.lru_cache(maxsize=None)
def ground_cases(name, n, seed):
    """Random poses lowered onto the plane z = 0 until one chosen candidate sphere is 2-10 mm deep; in models with
    more than 32 candidates every other case lowers a candidate of the second ballot pass (index >= 32).  Cassie
    (158 candidates, transformed on the fly in five passes) keeps its standing pose with up to 0.3 rad of tilt and
    lowers a candidate of the third to fifth pass (index >= 64) every other case; states with hull self-contacts are
    skipped (their pairs are tested in test_gpu_cassie)."""
    kind = Kind(name)
    rng = np.random.RandomState(seed)
    npt = len(kind.cands)
    cases = []
    tries = 0
    while len(cases) < n:
        tries += 1
        assert tries < 50 * n, (name, len(cases))
        if name == "cassie":
            from scipy.spatial.transform import Rotation

            A = kind.A
            row = np.zeros(13 + 2 * A)
            row[3:7] = Rotation.from_rotvec(rng.uniform(-0.3, 0.3, 3)).as_quat()
            row[7:10] = 0.2 * rng.randn(3)
            row[10:13] = 0.2 * rng.randn(3)
            lo, hi = np.array(kind.t["lower"]), np.array(kind.t["upper"])
            row[13:13 + A] = np.clip(np.array(kind.t["base_joint_angles"]) + rng.uniform(-0.05, 0.05, A),
                                     lo + 0.01, hi - 0.01)
            row[13 + A:] = 0.3 * rng.randn(A)
            row = row.astype(np.float32)
        else:
            row = _pose(kind, rng)
        hi_pass = 64 if name == "cassie" else 32
        pts, _ = kind.world_points(row)
        bottom = pts[:, 2] - np.array([cd[3] for cd in kind.cands])
        low = np.flatnonzero(bottom < bottom.min() + 0.03)
        if npt > hi_pass and len(cases) % 2 == 0:
            low = low[low >= hi_pass]
        if len(low) == 0:
            continue
        target = int(rng.choice(low))
        row = _lower_to_ground(kind, row, target, rng.uniform(0.002, 0.01))
        case = _case(kind, row, _tau(kind, rng))
        c, rows = kind.oracle_step(case)
        if name == "cassie" and any(c.partner[k] >= 1000 for k in range(c.n)):
            continue
        _accept(kind, case, cases, n)
    return tuple(cases)


def _cands_in_contact(kind, case, partner_lo, partner_hi):
    c, _ = kind.oracle_step(case)
    return [kind.cand_of_pid.get(c.point_id[k], -1) for k in range(c.n) if partner_lo <= c.partner[k] < partner_hi]


BOX_EDGES = ("top", "inside", "edge", "side", "two")


@functools.lru_cache(maxsize=None)
def box_cases(name, n, seed):
    """Planks written into the record around chosen candidate spheres of a random airborne pose (the two other
    planks far away unless the case needs them): a sphere on the top face ("top"), a sphere centre inside the cover
    box (the deepest-axis branch, "inside"), a sphere past the long edge (a normal in the plank's x-z plane, "edge";
    on a Plank past a corner, a normal with three components), a sphere against the side face ("side"), and two
    candidates each on its own plank ("two": contacts on two planks in one pass, listed box-major).  Each case
    records which edge it was built for; the test checks with the oracle that the edge was reached."""
    kind = Kind(name)
    pc = kind.spec["plank_class"]
    hy = {0: 5.0, 1: 0.375}[pc]
    rng = np.random.RandomState(seed)
    cases = []
    tries = 0
    while len(cases) < n:
        tries += 1
        assert tries < 200 * n, (name, len(cases))
        edge = BOX_EDGES[len(cases) % len(BOX_EDGES)]
        row = _pose(kind, rng)
        pts, _ = kind.world_points(row)
        planks = _far_planks()
        target = rng.randint(len(kind.cands))
        r = kind.cands[target][3]
        d = rng.uniform(0.002, 0.008)
        R = _rot(rng, 0.15)
        top = 0.1375
        y = rng.uniform(-0.8, 0.8) * min(hy, 1.0)
        if edge == "top":
            local = [rng.uniform(-0.2, 0.2), y, top + r - d]
        elif edge == "inside":
            local = [rng.uniform(-0.2, 0.2), y, top - rng.uniform(0.003, 0.009)]
        elif edge == "side":
            local = [0.25 + r - d, y, rng.uniform(-0.08, 0.08)]
        elif edge == "edge":
            phi = rng.uniform(0.3, 1.2)
            if pc == 1:  # a corner of the short plank
                th = rng.uniform(0.3, 1.2)
                dirn = np.array([np.cos(phi) * np.cos(th), np.cos(phi) * np.sin(th), np.sin(phi)])
                local = [0.25, hy, top] + (r - d) * dirn
            else:
                local = [0.25 + (r - d) * np.cos(phi), y, top + (r - d) * np.sin(phi)]
        else:
            other = rng.randint(len(kind.cands))
            if np.linalg.norm(pts[other] - pts[target]) < 0.6:
                continue
            R2 = _rot(rng, 0.15)
            r2 = kind.cands[other][3]
            _place(planks, 1, R2, [rng.uniform(-0.2, 0.2), 0.0, top + r2 - rng.uniform(0.002, 0.008)], pts[other])
            local = [rng.uniform(-0.2, 0.2), 0.0, top + r - d]
        _place(planks, 0, R, local, pts[target])
        case = _case(kind, row, _tau(kind, rng), planks=planks.astype(np.float32), edge=edge, target=target)
        c = _accept(kind, case, cases, n)
        if c is not None and not _box_edge_reached(kind, case, c):
            cases.pop()
    return tuple(cases)


def _box_edge_reached(kind, case, c):
    """The oracle's list shows the edge the case was built for (see box_cases)."""
    pid = [2 * kind.cands[case["target"]][0] + kind.cands[case["target"]][1]]
    mine = [k for k in range(c.n) if c.point_id[k] in pid and c.partner[k] in (10, 11)]
    if not mine:
        return False
    R = case["planks"][0, 3:12].reshape(3, 3).astype(np.float64)
    r = kind.cands[case["target"]][3]
    nl = [R.T @ np.array(c.normal[k][:]) for k in mine]
    edge = case["edge"]
    if edge == "inside":
        return any(c.dist[k] < -r for k in mine)
    if edge == "top":
        return any(abs(v[2] - 1) < 1e-9 for v in nl)
    if edge == "side":
        return any(abs(v[0] - 1) < 1e-9 for v in nl)
    if edge == "edge":
        need = 3 if kind.spec["plank_class"] == 1 else 2
        return any(np.sum(np.abs(v) > 0.05) == need for v in nl)
    return len({c.partner[k] // 2 for k in range(c.n) if c.partner[k] < 1000}) >= 2


PILLAR_EDGES = ("side", "cap", "rim", "inside_cap", "inside_side", "axis_out", "axis_in")


@functools.lru_cache(maxsize=None)
def pillar_cases(n, seed):
    """Pillars (capped cylinders of radius 0.25: base half height 0.1125, cover 0.0125 on top) written around a chosen
    candidate sphere of a random airborne pose: against the side wall, on the top cap, over the rim, with the centre
    inside the cover next to the cap (pen_z <= pen_r: cap normal) or inside the base next to the wall (pen_z > pen_r:
    radial normal), and with the centre on the pillar's axis above the cap and inside it."""
    kind = Kind("pillar")
    rng = np.random.RandomState(seed)
    cases = []
    tries = 0
    while len(cases) < n:
        tries += 1
        assert tries < 200 * n, len(cases)
        edge = PILLAR_EDGES[len(cases) % len(PILLAR_EDGES)]
        row = _pose(kind, rng)
        pts, _ = kind.world_points(row)
        planks = _far_planks()
        target = rng.randint(len(kind.cands))
        r = kind.cands[target][3]
        d = rng.uniform(0.002, 0.008)
        th = rng.uniform(-np.pi, np.pi)
        u = np.array([np.cos(th), np.sin(th), 0.0])
        top = 0.1375
        if edge == "side":
            local = (0.25 + r - d) * u + [0, 0, rng.uniform(-0.08, 0.08)]
        elif edge == "cap":
            local = rng.uniform(0.02, 0.18) * u + [0, 0, top + r - d]
        elif edge == "rim":
            phi = rng.uniform(0.3, 1.2)
            local = (0.25 + (r - d) * np.cos(phi)) * u + [0, 0, top + (r - d) * np.sin(phi)]
        elif edge == "inside_cap":
            local = rng.uniform(0.02, 0.18) * u + [0, 0, top - rng.uniform(0.002, 0.008)]
        elif edge == "inside_side":
            local = (0.25 - rng.uniform(0.002, 0.008)) * u + [0, 0, rng.uniform(-0.06, 0.06)]
        elif edge == "axis_out":
            local = np.array([0, 0, top + r - d])
        else:
            local = np.array([0, 0, top - 0.005])
        _place(planks, 0, _rot(rng, 0.15), local, pts[target])
        case = _case(kind, row, _tau(kind, rng), planks=planks.astype(np.float32), edge=edge, target=target)
        c = _accept(kind, case, cases, n)
        if c is not None and not _pillar_edge_reached(kind, case, c):
            cases.pop()
    return tuple(cases)


def _pillar_edge_reached(kind, case, c):
    g, e, _, r = kind.cands[case["target"]]
    mine = [k for k in range(c.n) if c.point_id[k] == 2 * g + e and c.partner[k] in (10, 11)]
    if not mine:
        return False
    R = case["planks"][0, 3:12].reshape(3, 3).astype(np.float64)
    nl = [R.T @ np.array(c.normal[k][:]) for k in mine]
    edge = case["edge"]
    axial = [abs(abs(v[2]) - 1) < 1e-9 for v in nl]
    radial = [abs(v[2]) < 1e-9 for v in nl]
    inside = [c.dist[k] < -r for k in mine]
    if edge in ("side", "inside_side"):
        return any(a and (i == (edge == "inside_side")) for a, i in zip(radial, inside))
    if edge in ("cap", "inside_cap", "axis_out", "axis_in"):
        want_inside = edge in ("inside_cap", "axis_in")
        return any(a and i == want_inside for a, i in zip(axial, inside))
    return any(not a and not b for a, b in zip(axial, radial))


BAR_EDGES = ("grip", "sphere_end", "one_box", "parallel", "box_end", "seven")


def _monkey_reset(seed):
    O = _O()
    o = O.Monkey3DOracle(_table("monkey3d"), seed=seed)
    o.reset()
    bars = np.array([list(b.center) + list(b.axis) + [b.halflen, b.radius] for b in o.e.bars], dtype=np.float32)
    return o.state_vector().astype(np.float32), bars


def _bar(center, axis, halflen, radius):
    axis = np.asarray(axis, dtype=np.float64)
    return np.array(list(center) + list(axis / np.linalg.norm(axis)) + [halflen, radius], dtype=np.float32)


@functools.lru_cache(maxsize=None)
def bar_cases(n, seed):
    """Monkey3D against bars written into the record: the reset grips (both hands' boxes on two bars, the oracle
    env's own layout with the joints moved by up to 0.01 off the closed-finger limits; "grip"), a sphere past the end of a bar (closest point clamped at t = +halflen, "sphere_end"), a bar
    across one hand box ("one_box"), a bar lying along a box face tilted by 1e-4 so that an outer sample is deeper
    by less than 1e-5 (the tie rule keeps the central sample, "parallel"), a bar ending next to a box (outer samples
    clamped at the end, "box_end"), and a bar through both hands with its radius raised until the oracle lists at
    least 7 box contacts on it ("seven": the second pass of six boxes)."""
    kind = Kind("monkey")
    rng = np.random.RandomState(seed)
    cases = []
    tries = 0
    while len(cases) < n:
        tries += 1
        assert tries < 200 * n, len(cases)
        edge = BAR_EDGES[len(cases) % len(BAR_EDGES)]
        tau = _tau(kind, rng, 0.2)
        if edge in ("grip", "seven"):
            row, bars = _monkey_reset(int(rng.randint(1 << 20)))
            A = kind.A
            row[13:13 + A] += rng.uniform(-0.01, 0.01, A).astype(np.float32)
            row[13 + A:] = rng.uniform(-0.2, 0.2, A).astype(np.float32)
        else:
            row = _pose(kind, rng)
            bars = _far_bars()
        pts, boxes = kind.world_points(row)
        rad = np.float32(0.015)
        if edge == "sphere_end":
            target = rng.randint(len(kind.cands))
            r = kind.cands[target][3]
            axis = rng.randn(3)
            axis /= np.linalg.norm(axis)
            perp = np.cross(axis, rng.randn(3))
            perp /= np.linalg.norm(perp)
            beta = rng.uniform(0.2, 1.2)
            gap = r + rad - rng.uniform(0.002, 0.008)
            end = pts[target] - gap * (np.cos(beta) * axis + np.sin(beta) * perp)
            bars[0] = _bar(end - 2.5 * axis, axis, 2.5, rad)
        elif edge in ("one_box", "parallel", "box_end"):
            bi = rng.randint(len(boxes))
            cen, Rb, half, _ = boxes[bi]
            j = int(np.argmin(half))  # the face of the thin side
            a = [k for k in range(3) if k != j]
            sgn = rng.choice([-1.0, 1.0])
            nrm = sgn * Rb[:, j]
            d = rng.uniform(0.002, 0.006)
            if edge == "parallel":
                along = Rb[:, a[int(np.argmax(half[a]))]]
                axis = along - 1e-4 * nrm  # the -t side is closer to the face by 1e-4 per metre
                axis = axis / np.linalg.norm(axis)
                c = cen + (half[j] + rad - d) * nrm
                bars[0] = _bar(c, axis, 2.5, rad)
            else:
                ang = rng.uniform(0, np.pi)
                axis = np.cos(ang) * Rb[:, a[0]] + np.sin(ang) * Rb[:, a[1]]
                off = rng.uniform(-0.5, 0.5) * np.array([half[a[0]], half[a[1]]])
                c = cen + (half[j] + rad - d) * nrm + off[0] * Rb[:, a[0]] + off[1] * Rb[:, a[1]]
                hl = 2.5
                if edge == "box_end":
                    c = c - (hl - rng.uniform(0.0, 0.04)) * axis
                bars[0] = _bar(c, axis, hl, rad)
        elif edge == "seven":
            hands = [[k for k, g in enumerate(kind.boxgeoms) if kind.t["geoms"][g]["link"] in links]
                     for links in ((20, 21), (28, 29))]
            p0 = np.mean([boxes[k][0] for k in hands[0]], axis=0)
            p1 = np.mean([boxes[k][0] for k in hands[1]], axis=0)
            axis = p1 - p0
            found = False
            for radius in np.arange(0.02, 0.16, 0.01):
                bars[3] = _bar(0.5 * (p0 + p1), axis, 0.5 * np.linalg.norm(p1 - p0) + 0.15, radius)
                case = _case(kind, row, tau, bars=bars.copy(), edge=edge)
                c, rows = kind.oracle_step(case)
                nbox = sum(1 for k in range(c.n) if c.partner[k] == 23 and c.point_id[k] // 2 in kind.boxgeoms)
                if nbox >= 7 and c.n <= MAXC:
                    found = True
                    break
            if not found:
                continue
        case = _case(kind, row, tau, bars=bars.copy(), edge=edge, target=target if edge == "sphere_end" else -1)
        c = _accept(kind, case, cases, n)
        if c is not None and not _bar_edge_reached(kind, case, c):
            cases.pop()
    return tuple(cases)


def _bar_edge_reached(kind, case, c):
    edge, bars = case["edge"], case["bars"]
    boxk = [k for k in range(c.n) if 20 <= c.partner[k] < 30 and c.point_id[k] // 2 in kind.boxgeoms]
    sph = [k for k in range(c.n) if 20 <= c.partner[k] < 30 and c.point_id[k] // 2 not in kind.boxgeoms]
    if edge == "grip":
        return len({c.partner[k] for k in boxk}) >= 2
    if edge == "sphere_end":
        g, e, _, _ = kind.cands[case["target"]]
        b = bars[0].astype(np.float64)
        pts, _ = kind.world_points(case["state"])
        return any(c.point_id[k] == 2 * g + e and c.partner[k] == 20 for k in sph) and \
            (pts[case["target"]] - b[0:3]) @ b[3:6] > b[6]
    if edge == "seven":
        return sum(1 for k in boxk if c.partner[k] == 23) >= 7
    if not boxk:
        return False
    if edge == "one_box":
        return True
    _, boxes = kind.world_points(case["state"])
    b = bars[0].astype(np.float64)
    for k in boxk:
        g = c.point_id[k] // 2
        cen, R, half, thresh = boxes[kind.boxgeoms.index(g)]
        t0 = (cen - b[0:3]) @ b[3:6]
        if edge == "box_end" and t0 + 0.06 > b[6]:
            return True
        if edge == "parallel":
            ds = [x[0] for x in _box_bar_samples((cen, R, half, thresh), b)]
            # an outer sample is strictly deeper, yet the oracle kept the central one (its distance)
            if min(ds[1:]) < ds[0] and abs(c.dist[k] - ds[0]) < 1e-12:
                return True
    return False


@functools.lru_cache(maxsize=None)
def self_cases(name, n, seed):
    """Airborne states whose substep lists segment self-contacts (tests.helpers.self_contact_states: random held
    torques from the base pose); Monkey3D's bars are moved out of reach."""
    kind = Kind(name)
    O = _O()
    rng = np.random.RandomState(seed)
    cases = []
    for row in self_contact_states(O, kind.t, rng, 4 * n):
        obst = dict(bars=_far_bars()) if kind.spec["obst"] == "bars" else {}
        _accept(kind, _case(kind, row, _tau(kind, rng), **obst), cases, n)
        if len(cases) == n:
            break
    assert len(cases) == n, (name, len(cases))
    return tuple(cases)


# ------------------------------------------------------------------------------------------------ tests
GROUND = [("walker3d", 24), ("child3d", 16), ("mike_ground", 12), ("walker2d", 12), ("crab2d", 12)]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name,n", GROUND)
def test_ground_store(name, n, backend):
    """Ground plane, STORE path (candidate points staged in shared memory, one ballot pass per 32 of them):
    Walker3D and Child3D (NPT = 34: the oracle lists contacts of candidates 32 and 33, i.e. of the second ballot
    pass), Mike (NPT = 32, the ground pass switched on in the emulation; its env removes the ground, so there is no
    device leg), Walker2D and Crab2D.
    Worst errors (emulation): point 2.0e-7 m, normal 3.1e-7, distance 1.3e-7 m, impulse 2.8e-5 of the scale.
    Device (B200): unmeasured."""
    if backend == "gpu" and KINDS[name]["vec"] is None:
        pytest.skip("the env removes the ground plane on the device")
    kind = Kind(name)
    cases = ground_cases(name, n, 11)
    if len(kind.cands) > 32:
        late = sum(1 for cs in cases if any(k >= 32 for k in _cands_in_contact(kind, cs, 0, 1)))
        assert late >= n // 3, late
    run_and_check(name, cases, backend)


@pytest.mark.parametrize("backend", BACKENDS)
def test_ground_on_the_fly_cassie(backend):
    """Ground plane, on-the-fly path (Cassie: 158 candidates transformed inside the test pass, five ballot passes):
    the oracle lists contacts of candidates in the third to fifth pass (index >= 64) in half the cases, and at least
    one list holds contacts from two different passes.
    Worst errors (emulation): point 2.9e-7 m, normal 0, distance 2.5e-7 m, impulse 6.8e-3 of the scale (hence
    TOL_IMP_CASSIE).  Device (B200): unmeasured."""
    kind = Kind("cassie")
    cases = ground_cases("cassie", 16, 12)
    per = [_cands_in_contact(kind, cs, 0, 1) for cs in cases]
    assert sum(1 for c in per if any(k >= 64 for k in c)) >= 8
    assert len({k // 32 for c in per for k in c}) >= 2
    assert max(len({k // 32 for k in c}) for c in per) >= 2  # one list from two passes
    run_and_check("cassie", cases, backend)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name", ["stepper", "plank", "mike"])
def test_static_boxes(name, backend):
    """Plank boxes (the box-major (box, point) task flattening over the planks in reach): LargePlank and Plank
    (Walker3DStepperEnv) and Mike (MikeStepperEnv), no ground plane.  Every edge of box_cases is reached (checked with
    the oracle per case): top face, centre inside the cover (deepest-axis branch), past an edge (Plank: a corner),
    side face, two planks in one pass.
    Worst errors (emulation): point 3.2e-7 m, normal 4.8e-6, distance 2.9e-7 m, impulse 9.1e-5 of the scale.
    Device (B200): unmeasured."""
    cases = box_cases(name, 20, 13)
    assert {cs["edge"] for cs in cases} == set(BOX_EDGES)
    run_and_check(name, cases, backend)


@pytest.mark.parametrize("backend", BACKENDS)
def test_pillar(backend):
    """Capped cylinders (sphere_cyl, Walker3DStepperEnv with plank_class = "Pillar"): side, cap and rim regions, a
    centre inside with pen_z <= pen_r (cap normal) and with pen_z > pen_r (radial normal), a centre on the axis
    above the cap and inside it -- each reached according to the oracle.
    Worst errors (emulation): point 3.7e-7 m, normal 3.3e-6, distance 1.9e-7 m, impulse 6.3e-6 of the scale.
    Device (B200): unmeasured."""
    cases = pillar_cases(21, 14)
    assert {cs["edge"] for cs in cases} == set(PILLAR_EDGES)
    run_and_check("pillar", cases, backend)


@pytest.mark.parametrize("backend", BACKENDS)
def test_bars(backend):
    """Monkey3D vs bars: sphere / capsule vs bar (sphere_bar and its ballot compaction) at the reset grips and past a
    bar's end (t clamped to +halflen); box vs bar (six boxes x five samples per pass, the 'deeper by 1e-5 wins' rule
    replayed through warp_gather) with one near box, a bar along a box face (an outer sample deeper by less than 1e-5:
    the central one is kept), samples clamped at the bar's end, and >= 7 box contacts on one bar (the second pass,
    base = 6) -- each reached according to the oracle.
    Worst errors (emulation): point 1.0e-6 m, normal 5.3e-6, distance 9.9e-8 m, impulse 2.0e-5 of the scale.
    Device (B200): unmeasured."""
    cases = bar_cases(18, 15)
    assert {cs["edge"] for cs in cases} == set(BAR_EDGES)
    run_and_check("monkey", cases, backend)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name,n", [("walker3d", 16), ("monkey", 12), ("crab2d", 12)])
def test_self_contacts(name, n, backend):
    """Segment self-contacts (collide_self: broad phase ballot, candidate compaction, narrow phase in pair order):
    Walker3D (92 pairs), Monkey3D (87 pairs), Crab2D (9 pairs).  The partner 1000 + p must name the pair of the
    oracle's two links.
    Worst errors (emulation): point 1.6e-7 m, normal 8.5e-7, distance 8.2e-8 m, impulse 2.3e-4 of the scale.
    Device (B200): unmeasured."""
    cases = self_cases(name, n, 16)
    kind = Kind(name)
    assert all(any(k >= 1000 for k in _partners(kind, cs)) for cs in cases)
    run_and_check(name, cases, backend)


def _partners(kind, cs):
    c, _ = kind.oracle_step(cs)
    return [c.partner[k] for k in range(c.n)]


@pytest.mark.gpu
def test_last_pass_at_four_substeps():
    """The points of a 4-substep stepSimulation are those of its LAST collision pass: step_physics_points with
    substeps = 4 from s equals step_physics with substeps = 3 followed by step_physics_points with substeps = 1 from
    the same s, bit for bit (the state crosses HBM in f32 between the calls and load / store copy it unchanged)."""
    import torch
    from mocca_envs_b200.vec_env import Walker3DCustomVecEnv

    cases = ground_cases("walker3d", 24, 11)
    N = len(cases)
    st = torch.tensor(np.stack([cs["state"] for cs in cases]))
    tau = torch.tensor(np.stack([cs["tau"] for cs in cases]))
    envs = {k: Walker3DCustomVecEnv(N, device="cuda:0", seed=0, physics={"substeps": k}) for k in (4, 3, 1)}
    try:
        envs[4].set_state(st)
        _, nc4, p4 = envs[4].step_physics_points(tau)
        envs[3].set_state(st)
        envs[3].step_physics(tau)
        envs[1].set_state(envs[3].get_state())
        _, nc1, p1 = envs[1].step_physics_points(tau)
        torch.cuda.synchronize()
    finally:
        for e in envs.values():
            e.close()
    assert torch.equal(nc4, nc1)
    assert int(nc4.sum()) > 0
    assert torch.equal(p4, p1), float((p4 - p1).abs().max())
