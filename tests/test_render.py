"""Camera images: mb200_render / VecEnv.render / render(mode="rgb_array") for every env kind, against a float64 ray
caster built here and against the laws of the image.

The float64 reference is independent of the kernels and of codegen: link frames from the oracle's forward kinematics,
geoms and hulls from the model JSON (hull face planes from scipy's ConvexHull of the hull vertices), obstacles from
the record's terrain rows (Stepper planks and Pillar stones, Monkey3D bars) and its walk target, and a vectorised NumPy
ray caster with the pixel, depth and segmentation conventions of include/mocca_b200.h.  The CPU tests run the kernel
source through the lane-loop emulation (tests/emu/emu_render.cpp); the GPU tests (-m gpu) render on the device and
require it to equal the emulation.

A pixel is clean when the reference's rays through its centre and through four sub-pixel offsets (+-0.02 px) hit the
same primitive (or all miss), the incidence is |n . d| >= 0.1 and the two closest hits along the centre ray are more
than 1e-3 apart.  Only there is the image a function of the scene rather than of rounding: there seg is equal, depth
is within 1e-4 depth + 1e-5 and RGB within 2 levels (RGB also away from a ground checker edge)."""
import ctypes as C
import functools
import os
import subprocess

import numpy as np
import pytest

from tests.emu import emu as E
from tests.helpers import oracle_state

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TARGET_RADIUS = 0.2  # the walk-target marker (a constant of this library, MB_RENDER_TARGET_RADIUS)
SKY = np.array([178, 204, 230])
LIGHT = np.array([0.40, 0.30, 0.8660254])
AMBIENT = 0.35
COLORS = {"robot": (0.90, 0.55, 0.25), "plank": (0.45, 0.60, 0.85), "bar": (0.80, 0.75, 0.30),
          "target": (0.90, 0.15, 0.15), "ground0": (0.60, 0.64, 0.60), "ground1": (0.36, 0.40, 0.36)}
W = H = 64

KINDS = {
    "w3d": dict(emu=E.EmuW3D, vec="Walker3DCustomVecEnv", model="walker3d", target=True),
    "stepper": dict(emu=E.EmuStepper, vec="Walker3DStepperVecEnv", model="walker3d", curriculum=9),
    "pillar": dict(emu=E.EmuPillar, vec="Walker3DStepperVecEnv", kw=dict(plank_class="Pillar"), model="walker3d",
                   curriculum=5),
    "monkey": dict(emu=E.EmuMonkey, vec="Monkey3DCustomVecEnv", model="monkey3d"),
    "cassie": dict(emu=E.EmuCassie, vec="CassieVecEnv", model="cassie", dist=1.6),
    "child": dict(emu=E.EmuChild, vec="Child3DCustomVecEnv", model="child3d", target=True),
    "mike": dict(emu=E.EmuMike, vec="MikeStepperVecEnv", model="mike", curriculum=3, dist=1.8),
    "walker2d": dict(emu=E.EmuWalker2D, vec="Walker2DCustomVecEnv", model="walker2d", target=True, dist=2.0),
    "crab2d": dict(emu=E.EmuCrab2D, vec="Crab2DCustomVecEnv", model="crab2d", target=True, dist=1.8),
}
STEPPERS = ("stepper", "pillar", "mike")
ES_PLANK_CLASS, ES_PLANKIDX, ES_TERRAIN = 4, 28, 68
EM_BARIDX, EM_TERRAIN = 28, 64
# cameras that frame the robot: (distance, yaw, pitch) about the base position -- the tracking camera and one from
# behind; a kind's "dist" scales the distance (Cassie's thin legs)
CAMERAS = [(2.5, 0.0, -20.0), (2.5, -90.0, -8.0)]
BELOW = (2.5, 60.0, 12.0)  # the stepper kinds have no ground: also from below


def cameras(name):
    f = KINDS[name].get("dist", 2.5) / 2.5
    return [(d * f, y, p) for d, y, p in CAMERAS + ([BELOW] if name in STEPPERS else [])]


# ------------------------------------------------------------------------------------------------ emulation
_EMU_SRC = os.path.join(ROOT, "tests", "emu", "emu_render.cpp")
_EMU_LIB = os.path.join(ROOT, "tests", "emu", "libmb_emu_render.so")


@functools.lru_cache(maxsize=None)
def _emu_lib():
    deps = [_EMU_SRC, os.path.join(ROOT, "mocca_envs_b200", "csrc", "mb_render.cuh")] + E._SRC[1:]
    if not os.path.exists(_EMU_LIB) or any(os.path.getmtime(s) > os.path.getmtime(_EMU_LIB) for s in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                               "-Wno-unused-variable", "-o", _EMU_LIB, _EMU_SRC])
    L = C.CDLL(_EMU_LIB)
    assert L.emu_render_sizeof_phys() == C.sizeof(E.Phys)
    return L


def _fp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def emu_scene(name, state, rec, phys):
    L = _emu_lib()
    out = np.zeros((L.emu_render_rmax(), L.emu_render_stride()), dtype=np.float32)
    st = np.zeros(64, dtype=np.float32)
    st[:len(state)] = state
    nprim = getattr(L, "emu_%s_render_scene" % KINDS[name]["emu"].prefix)(
        C.byref(phys), _fp(st), _fp(np.ascontiguousarray(rec, dtype=np.float32)), _fp(out))
    return nprim, out


def emu_render(name, state, rec, phys, view, proj, w=W, h=H, blank=False):
    """(rgb [h][w][3], depth [h][w], seg [h][w]) of one camera through the emulated kernel source."""
    L = _emu_lib()
    nprim, scene = emu_scene(name, state, rec, phys)
    if blank:
        getattr(L, "emu_%s_render_blank" % KINDS[name]["emu"].prefix)(_fp(scene))
    rgb = np.zeros((h, w, 3), dtype=np.uint8)
    depth = np.zeros((h, w), dtype=np.float32)
    seg = np.zeros((h, w), dtype=np.int32)
    L.emu_render_rays(nprim, _fp(scene), _fp(np.ascontiguousarray(view, dtype=np.float32)),
                      _fp(np.ascontiguousarray(proj, dtype=np.float32)), w, h, _fp(rgb), _fp(depth), _fp(seg))
    return rgb, depth, seg


def cam(target, distance, yaw, pitch, aspect=1.0, near=0.01, far=100.0):
    from mocca_envs_b200.vec_env import camera_matrices

    v, p = camera_matrices(np.asarray(target, dtype=np.float64), distance, yaw, pitch, aspect=aspect, near=near,
                           far=far)
    return v[0].numpy(), p[0].numpy()


# ------------------------------------------------------------------------------------------------ float64 reference
def _O():
    from oracle import oracle as O

    O.build()
    return O


@functools.lru_cache(maxsize=None)
def _table(model):
    from mocca_envs_b200.model_compiler import load_table

    return load_table(os.path.join(ROOT, "mocca_envs_b200", "models", model + ".json"))


def _quat_mat(q):
    from scipy.spatial.transform import Rotation

    return Rotation.from_quat(q).as_matrix()


def movable(t, li):
    """URDF link -> the link index of mb200_apply_impulse (dof of the nearest movable ancestor, -1 = base)."""
    while li >= 0 and t["dof_of_link"][li] < 0:
        li = t["parent"][li]
    return -1 if li < 0 else t["dof_of_link"][li]


def hull_planes(V):
    from scipy.spatial import ConvexHull

    eq = ConvexHull(V).equations
    return np.concatenate([eq[:, :3], -eq[:, 3:]], axis=1)  # n . x <= d inside


def reference_scene(name, state, rec, phys):
    """The float64 scene: a list of primitives dict(kind, seg, cls, ...)."""
    spec = KINDS[name]
    t = _table(spec["model"])
    O = _O()
    m = O.model_from_table(t)
    A = t["n_dof"]
    pos, rot = O.fk(m, oracle_state(O, A, np.asarray(state[:13 + 2 * A], dtype=np.float64)))
    prims = []
    hulls = t.get("hulls", [])
    if hulls:
        for h in hulls:
            li = h["link"]
            V = pos[li + 1] + np.asarray(h["verts"]) @ rot[li + 1].T
            prims.append(dict(kind="hull", planes=hull_planes(V), c=V.mean(0),
                              r=np.linalg.norm(V - V.mean(0), axis=1).max(), seg=100 + movable(t, li), cls="robot"))
    else:
        for g in t["geoms"]:
            li = g["link"]
            Rl, pl = rot[li + 1], pos[li + 1]
            seg = 100 + movable(t, li)
            if g["type"] == 2:
                prims.append(dict(kind="box", c=pl + Rl @ np.array(g["pos"]), R=Rl @ _quat_mat(g["quat"]),
                                  h=np.array(g["size"][:3]), seg=seg, cls="robot"))
            elif g["type"] == 0:
                prims.append(dict(kind="sphere", c=pl + Rl @ np.array(g["p0"]), r=g["size"][0], seg=seg, cls="robot"))
            else:
                prims.append(dict(kind="capsule", a=pl + Rl @ np.array(g["p0"]), b=pl + Rl @ np.array(g["p1"]),
                                  r=g["size"][0], seg=seg, cls="robot"))
    ri = np.asarray(rec, dtype=np.float32).view(np.int32)
    if name in STEPPERS:
        from scipy.spatial.transform import Rotation

        terrain = np.asarray(rec[ES_TERRAIN:ES_TERRAIN + 120], dtype=np.float64).reshape(20, 6)
        cls_ = ri[ES_PLANK_CLASS]
        for p in range(3):
            x, y, z, phi, xt, yt = terrain[ri[ES_PLANKIDX + p]]
            R = Rotation.from_euler("xyz", [xt, yt, phi]).as_matrix()
            base = np.array([x, y, z - 0.1375])
            for cover in (0, 1):
                c = base + cover * 0.125 * R[:, 2]
                hz = 0.0125 if cover else 0.1125
                k = 2 * p + cover
                if name == "pillar":
                    prims.append(dict(kind="cyl", c=c, R=R, rad=0.25, hh=hz, seg=10 + k, cls="plank"))
                else:
                    prims.append(dict(kind="box", c=c, R=R, h=np.array([0.25, 0.375 if cls_ == 1 else 5.0, hz]),
                                      seg=10 + k, cls="plank"))
    if name == "monkey":
        terrain = np.asarray(rec[EM_TERRAIN:EM_TERRAIN + 128], dtype=np.float64).reshape(32, 4)
        for k in range(4):
            x, y, z, phi = terrain[ri[EM_BARIDX + k]]
            ax = np.array([np.sin(phi), -np.cos(phi), 0.0])
            R = np.stack([np.cross(ax, [0, 0, 1.0]) / np.linalg.norm(np.cross(ax, [0, 0, 1.0])), [0, 0, 1.0], ax], 1)
            R[:, 1] = np.cross(R[:, 2], R[:, 0])
            prims.append(dict(kind="cyl", c=np.array([x, y, z]), R=R, rad=0.015, hh=2.5, seg=20 + k, cls="bar"))
    if spec.get("target"):
        prims.append(dict(kind="sphere", c=np.asarray(rec[0:3], dtype=np.float64), r=TARGET_RADIUS, seg=30,
                          cls="target"))
    if phys.has_ground:
        prims.append(dict(kind="plane", seg=0, cls="ground"))
    return prims


def _rays(view, proj, w, h, dx=0.0, dy=0.0):
    """Per pixel (row-major): origin on the near plane, unit direction, length to the far plane, eye z of both ends."""
    V = np.asarray(view, dtype=np.float64).reshape(4, 4).T
    P = np.asarray(proj, dtype=np.float64).reshape(4, 4).T
    inv = np.linalg.inv(P @ V)
    r, c = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    x = (2 * (c.ravel() + 0.5 + dx) / w - 1)
    y = (1 - 2 * (r.ravel() + 0.5 + dy) / h)
    ends = []
    for z in (-1.0, 1.0):
        p = inv @ np.stack([x, y, np.full_like(x, z), np.ones_like(x)])
        ends.append((p[:3] / p[3]).T)
    pn, pf = ends
    d = pf - pn
    L = np.linalg.norm(d, axis=1)
    zn, zf = -(pn @ V[2, :3] + V[2, 3]), -(pf @ V[2, :3] + V[2, 3])
    return pn, d / L[:, None], L, zn, zf


def _sphere(o, d, c, r):
    oc = o - c
    b = (oc * d).sum(1)
    q = oc - b[:, None] * d
    h = r * r - (q * q).sum(1)
    t = -b - np.sqrt(np.maximum(h, 0))
    t = np.where((h >= 0) & (t > 0), t, np.inf)
    n = (oc + t[:, None] * d) / r
    return t, n


def _capsule(o, d, a, b, r):
    ba = b - a
    baba = ba @ ba
    oa = o - a
    bard, baoa = d @ ba, oa @ ba
    A = baba - bard ** 2
    w, v = np.cross(oa, ba), np.cross(d, ba)
    B = (v * w).sum(1)
    Cc = (w * w).sum(1) - r * r * baba
    h = B * B - A * Cc
    with np.errstate(divide="ignore", invalid="ignore"):
        t = (-B - np.sqrt(np.maximum(h, 0))) / A
    y = baoa + t * bard
    ok = (A > 1e-12 * baba) & (h >= 0) & (t > 0) & (y > 0) & (y < baba)
    t = np.where(ok, t, np.inf)
    n = (oa + t[:, None] * d - (y / baba)[:, None] * ba) / r
    for e in (a, b):
        te, ne = _sphere(o, d, e, r)
        better = te < t
        t, n = np.where(better, te, t), np.where(better[:, None], ne, n)
    return t, n


def _local(o, d, c, R):
    return (o - c) @ R, d @ R


def _box(o, d, c, R, hh):
    ol, dl = _local(o, d, c, R)
    with np.errstate(divide="ignore", invalid="ignore"):
        t1, t2 = (-hh - ol) / dl, (hh - ol) / dl
    lo, hi = np.minimum(t1, t2), np.maximum(t1, t2)
    lo = np.where(np.isnan(lo), -np.inf, lo)
    hi = np.where(np.isnan(hi), np.inf, hi)
    ax = lo.argmax(1)
    tn, tf = lo.max(1), hi.min(1)
    t = np.where((tn <= tf) & (tn > 0), tn, np.inf)
    sg = -np.sign(dl[np.arange(len(o)), ax])
    n = R[:, ax].T * sg[:, None]
    return t, n


def _cyl(o, d, c, R, rad, hh):
    ol, dl = _local(o, d, c, R)
    a = dl[:, 0] ** 2 + dl[:, 1] ** 2
    with np.errstate(divide="ignore", invalid="ignore"):
        s = -(ol[:, 0] * dl[:, 0] + ol[:, 1] * dl[:, 1]) / a
        qx, qy = ol[:, 0] + s * dl[:, 0], ol[:, 1] + s * dl[:, 1]
        h = rad * rad - (qx * qx + qy * qy)
        ts = s - np.sqrt(np.maximum(h, 0) / a)
    z = ol[:, 2] + ts * dl[:, 2]
    ts = np.where((a > 1e-20) & (h >= 0) & (ts > 0) & (np.abs(z) <= hh), ts, np.inf)
    ns = np.stack([(ol[:, 0] + ts * dl[:, 0]) / rad, (ol[:, 1] + ts * dl[:, 1]) / rad, np.zeros(len(o))], 1)
    zc = np.where(dl[:, 2] > 0, -hh, hh)
    with np.errstate(divide="ignore", invalid="ignore"):
        tc = (zc - ol[:, 2]) / dl[:, 2]
    x, y = ol[:, 0] + tc * dl[:, 0], ol[:, 1] + tc * dl[:, 1]
    tc = np.where((tc > 0) & (x * x + y * y <= rad * rad), tc, np.inf)
    nc = np.stack([np.zeros(len(o)), np.zeros(len(o)), -np.sign(dl[:, 2])], 1)
    cap = tc < ts
    t = np.where(cap, tc, ts)
    with np.errstate(invalid="ignore"):
        n = np.where(cap[:, None], nc, ns) @ R.T
    return t, n


def _hull(o, d, planes):
    den = d @ planes[:, :3].T
    dist = planes[:, 3][None, :] - o @ planes[:, :3].T
    with np.errstate(divide="ignore", invalid="ignore"):
        tt = dist / den
    ent = np.where(den < 0, tt, -np.inf)
    ext = np.where(den > 0, tt, np.inf)
    outside_par = ((den == 0) & (dist < 0)).any(1)
    face = ent.argmax(1)
    tn, tf = ent.max(1), ext.min(1)
    t = np.where((tn <= tf) & (tn > 0) & ~outside_par, tn, np.inf)
    return t, planes[face, :3]


def _hits(prims, o, d):
    """[n_prim][n_ray] hit distances and [n_prim][n_ray][3] outward normals."""
    T, N = [], []
    for p in prims:
        k = p["kind"]
        if k == "plane":
            with np.errstate(divide="ignore", invalid="ignore"):
                t = -o[:, 2] / d[:, 2]
            t = np.where(t > 0, t, np.inf)
            n = np.zeros_like(o)
            n[:, 2] = np.where(o[:, 2] >= 0, 1.0, -1.0)
        elif k == "sphere":
            t, n = _sphere(o, d, p["c"], p["r"])
        elif k == "capsule":
            t, n = _capsule(o, d, p["a"], p["b"], p["r"])
        elif k == "box":
            t, n = _box(o, d, p["c"], p["R"], p["h"])
        elif k == "cyl":
            t, n = _cyl(o, d, p["c"], p["R"], p["rad"], p["hh"])
        else:
            t, n = _hull(o, d, p["planes"])
        T.append(t)
        N.append(n)
    return np.array(T), np.array(N)


def reference_render(prims, view, proj, w=W, h=H):
    """dict(rgb, depth, seg, clean, edge, robot) of the float64 ray caster."""
    def cast(dx, dy):
        o, d, L, zn, zf = _rays(view, proj, w, h, dx, dy)
        T, N = _hits(prims, o, d)
        T = np.where(T < L[None, :], T, np.inf)
        idx = T.argmin(0)
        t = T[idx, np.arange(len(o))]
        hit = np.isfinite(t)
        idx = np.where(hit, idx, -1)
        n = N[np.maximum(idx, 0), np.arange(len(o))]
        p = o + np.where(hit, t, 0)[:, None] * d
        tile = (np.floor(p[:, 0]).astype(np.int64) + np.floor(p[:, 1]).astype(np.int64)) & 1
        return dict(o=o, d=d, L=L, zn=zn, zf=zf, T=T, idx=idx, t=t, hit=hit, n=n, tile=tile)

    c = cast(0.0, 0.0)
    subs = [cast(dx, dy) for dx, dy in ((0.02, 0), (-0.02, 0), (0, 0.02), (0, -0.02))]
    n_ray = len(c["t"])
    seg = np.full(n_ray, -1)
    seg[c["hit"]] = np.array([prims[i]["seg"] for i in c["idx"][c["hit"]]])
    depth = np.where(c["hit"], c["zn"] + np.where(c["hit"], c["t"], 0) * (c["zf"] - c["zn"]) / c["L"], c["zf"])
    same = np.all([s["idx"] == c["idx"] for s in subs], axis=0)
    inc = np.abs((c["n"] * c["d"]).sum(1))
    Ts = np.sort(c["T"], axis=0)
    with np.errstate(invalid="ignore"):
        gap = Ts[1] - Ts[0] if len(prims) > 1 else np.full(n_ray, np.inf)
    gap = np.where(np.isnan(gap), np.inf, gap)
    clean = same & (~c["hit"] | ((inc >= 0.1) & (gap > 1e-3)))
    ground = np.array([c["hit"][i] and prims[c["idx"][i]]["cls"] == "ground" for i in range(n_ray)])
    edge = ground & ~np.all([s["tile"] == c["tile"] for s in subs], axis=0)
    rgb = np.tile(SKY, (n_ray, 1)).astype(np.float64)
    for i in np.nonzero(c["hit"])[0]:
        cls = prims[c["idx"][i]]["cls"]
        base = np.array(COLORS["ground%d" % c["tile"][i]] if cls == "ground" else COLORS[cls])
        n = c["n"][i] * (-1.0 if n_dot(c["n"][i], c["d"][i]) > 0 else 1.0)
        k = AMBIENT + (1 - AMBIENT) * max(n_dot(n, LIGHT), 0.0)
        rgb[i] = np.floor(np.minimum(base * k, 1.0) * 255 + 0.5)
    robot = seg >= 99
    return dict(rgb=rgb.reshape(h, w, 3), depth=depth.reshape(h, w), seg=seg.reshape(h, w), idx=c["idx"].reshape(h, w),
                clean=clean.reshape(h, w), edge=edge.reshape(h, w), robot=robot.reshape(h, w))


def n_dot(a, b):
    return float(np.dot(a, b))


# ------------------------------------------------------------------------------------------------ states
@functools.lru_cache(maxsize=None)
def states(name, n=2, seed=3):
    """(state, rec) of seeded resets plus a few random-action steps (Monkey3D: at reset, gripping a bar)."""
    from mocca_envs_b200.seeding import mt_state_rows

    spec = KINDS[name]
    rng = np.random.RandomState(seed)
    out = []
    for k in range(n):
        kw = dict(curriculum=spec["curriculum"]) if "curriculum" in spec else {}
        emu = spec["emu"](mt_state=mt_state_rows([seed * 100 + k])[0], **kw)
        emu.reset()
        for _ in range(0 if name == "monkey" else rng.randint(2, 8)):
            emu.step(rng.uniform(-1, 1, emu.act_dim).astype(np.float32))
        out.append((emu.state.copy(), emu.rec.copy(), emu.p))
    return out


def check_against_reference(name, img, ref):
    """seg / depth / RGB of `img` equal the reference's on clean pixels; the comparison is not vacuous."""
    rgb, depth, seg = img
    clean = ref["clean"]
    assert clean.mean() >= 0.90, (name, clean.mean())
    assert ref["robot"].mean() >= 0.02, (name, ref["robot"].mean())
    bad = clean & (seg != ref["seg"])
    assert not bad.any(), (name, int(bad.sum()), np.argwhere(bad)[:5])
    dtol = 1e-4 * ref["depth"] + 1e-5
    derr = np.abs(depth - ref["depth"])
    assert (derr[clean] <= dtol[clean]).all(), (name, float((derr - dtol)[clean].max()))
    ok = clean & ~ref["edge"]
    rerr = np.abs(rgb.astype(np.int64) - ref["rgb"]).max(-1)
    assert (rerr[ok] <= 2).all(), (name, int(rerr[ok].max()))


# ------------------------------------------------------------------------------------------------ CPU tests
@pytest.mark.parametrize("name", list(KINDS))
def test_emulation_vs_reference(name):
    """Every kind, a tracking camera and one from behind and below, at seeded states: the emulated kernel source
    equals the float64 ray caster on clean pixels (>= 90 % of each frame, >= 2 % robot pixels)."""
    for state, rec, phys in states(name):
        prims = reference_scene(name, state, rec, phys)
        if name in ("stepper", "mike"):
            terrain = rec[ES_TERRAIN:ES_TERRAIN + 120].reshape(20, 6)
            assert np.abs(terrain[:, 4:6]).max() > 0.05, "the curriculum draws tilted planks"
        for dist, yaw, pitch in cameras(name):
            view, proj = cam(state[0:3], dist, yaw, pitch)
            img = emu_render(name, state, rec, phys, view, proj)
            check_against_reference(name, img, reference_render(prims, view, proj))


def _out_of_view(name):
    state, rec, phys = states(name)[0]
    st = state.copy()
    st[0:3] = [1000.0, 1000.0, 50.0]  # the robot far away (set_state); the scene keeps its ground
    return st, rec, phys


def test_analytic_ground_pin():
    """Straight down from height h over the empty ground: seg 0 and depth h everywhere (to 1e-6 h), and the
    checkerboard flips exactly at integer world x / y (within half a pixel)."""
    st, rec, phys = _out_of_view("w3d")
    rec = rec.copy()
    rec[0:3] = [1000.0, -1000.0, 1.0]  # the target too
    for h in (1.7, 4.0):
        cx, cy = 0.3, -0.45
        # looking along -z with +y up on the image: view = lookAt(eye, eye - z, up = y)
        view, proj = cam([cx, cy, 0.0], h, 0.0, -90.0 + 1e-9)
        rgb, depth, seg = emu_render("w3d", st, rec, phys, view, proj)
        assert (seg == 0).all()
        np.testing.assert_allclose(depth, h, rtol=1e-6)
        # world x, y of every pixel centre on the ground (exact pinhole geometry)
        o, d, L, zn, zf = _rays(view, proj, W, H)
        t = -o[:, 2] / d[:, 2]
        p = (o + t[:, None] * d).reshape(H, W, 3)
        half = 0.5 * 2 * h * np.tan(np.deg2rad(30.0)) / W
        tile = (np.floor(p[..., 0]) + np.floor(p[..., 1])).astype(np.int64) & 1
        frac_x, frac_y = p[..., 0] - np.round(p[..., 0]), p[..., 1] - np.round(p[..., 1])
        away = (np.abs(frac_x) > half) & (np.abs(frac_y) > half)
        dark = rgb[..., 0] < 128
        assert away.mean() > 0.5
        assert (dark[away] == (tile[away] == 1)).all()


def test_seg_codes():
    """Every code the header states appears: the plank covers and bases, every bar, the target marker, every robot
    link of each kind (but a link whose spheres all lie inside another sphere: Mike's shoulders and butt sit inside its
    waist), and each of Cassie's 16 hulls under its link's code."""
    for name in KINDS:
        t = _table(KINDS[name]["model"])
        links, hulls_seen = set(), set()
        for state, rec, phys in states(name):
            prims = reference_scene(name, state, rec, phys)
            for dist, yaw, pitch in CAMERAS + [(2.0, 90.0, -10.0), (2.0, 180.0, -60.0), (1.5, 45.0, 30.0)]:
                view, proj = cam(state[0:3], dist, yaw, pitch)
                seg = emu_render(name, state, rec, phys, view, proj, 96, 96)[2]
                links |= set(np.unique(seg).tolist())
                if t.get("hulls"):  # which hull the reference hits, where the kernel shows that hull's link code
                    ref = reference_render(prims, view, proj, 96, 96)
                    for k, p in enumerate(prims[:16]):
                        if ((ref["idx"] == k) & (seg == p["seg"])).any():
                            hulls_seen.add(k)
        geoms = [h["link"] for h in t.get("hulls", [])] or [g["link"] for g in t["geoms"]]
        want = {100 + movable(t, li) for li in geoms}
        if not t.get("hulls"):
            def enclosed(g):
                return g["type"] == 0 and any(
                    h is not g and h["type"] == 0 and
                    np.linalg.norm(_geom_centre(t, g) - _geom_centre(t, h)) + g["size"][0] <= h["size"][0]
                    for h in t["geoms"])
            hidden = {c for c in want if all(enclosed(g) for g in t["geoms"] if 100 + movable(t, g["link"]) == c)}
            want -= hidden
        assert want <= links, (name, sorted(want - links))
        assert not {c for c in links if c >= 99} - want, name
        if t.get("hulls"):
            assert hulls_seen == set(range(16)), ("Cassie hulls not seen", sorted(set(range(16)) - hulls_seen))
    # obstacles and the target, from cameras aimed at them
    st, rec, phys = _out_of_view("stepper")
    state0, rec0, _ = states("stepper")[0]
    terrain = rec0[ES_TERRAIN:ES_TERRAIN + 120].reshape(20, 6)
    idx = rec0.view(np.int32)[ES_PLANKIDX:ES_PLANKIDX + 3]
    codes = set()
    for p in range(3):
        x, y, z = terrain[idx[p], 0:3]
        for yaw, pitch in ((90.0, -5.0), (0.0, -60.0)):
            view, proj = cam([x, y, z - 0.1], 1.2, yaw, pitch)
            codes |= set(np.unique(emu_render("stepper", st, rec0, phys, view, proj)[2]).tolist())
    assert {10, 11, 12, 13, 14, 15} <= codes, codes
    st, rec, phys = _out_of_view("monkey")
    _, recm, _ = states("monkey")[0]
    terrain = recm[EM_TERRAIN:EM_TERRAIN + 128].reshape(32, 4)
    idx = recm.view(np.int32)[EM_BARIDX:EM_BARIDX + 4]
    codes = set()
    for k in range(4):
        view, proj = cam(terrain[idx[k], 0:3], 0.3, 0.0, -80.0)
        codes |= set(np.unique(emu_render("monkey", st, recm, phys, view, proj)[2]).tolist())
    assert {20, 21, 22, 23} <= codes, codes
    st, rec, phys = _out_of_view("w3d")
    rec = rec.copy()
    rec[0:3] = [2.0, 1.0, 1.0]
    view, proj = cam(rec[0:3], 2.0, 0.0, -10.0)
    assert 30 in np.unique(emu_render("w3d", st, rec, phys, view, proj)[2])


def _geom_centre(t, g):
    """A sphere geom's centre in the base frame at the zero pose (codegen's link frames)."""
    from mocca_envs_b200 import codegen

    r = codegen.reduce_table(t)
    k = [p["geom"] for p in r["points"]].index(t["geoms"].index(g))
    o = r["points"][k]["owner"]
    off = np.zeros(3) if o < 0 else _pivot(r, o)
    return off + np.asarray(r["points"][k]["pos"])


def _pivot(r, j):
    p = np.zeros(3)
    while j >= 0:
        p += np.asarray(r["joff"][j])
        j = r["jparent"][j]
    return p


def test_codegen_hull_planes():
    """The generated hull planes: every hull vertex lies inside every plane of its hull (to 1e-6), and every plane
    touches at least 3 vertices."""
    from mocca_envs_b200 import codegen

    r = codegen.reduce_table(_table("cassie"))
    assert len(r["hulls"]) == 16
    for h in r["hulls"]:
        V, P = np.asarray(h["verts"]), h["planes"]
        s = V @ P[:, :3].T - P[:, 3][None, :]
        assert s.max() <= 1e-6
        assert ((np.abs(s) <= 1e-6).sum(0) >= 3).all()
        np.testing.assert_allclose(np.linalg.norm(P[:, :3], axis=1), 1.0, atol=1e-12)


def test_blank_and_null_outputs():
    """An id outside the batch renders a blank frame (sky, depth = far, seg -1); NULL outputs are skipped."""
    state, rec, phys = states("w3d")[0]
    view, proj = cam(state[0:3], 2.5, 0.0, -20.0, far=50.0)
    rgb, depth, seg = emu_render("w3d", state, rec, phys, view, proj, blank=True)
    assert (seg == -1).all() and (rgb == SKY).all()
    far = float(np.float64(proj[14]) / (np.float64(proj[10]) + 1.0))  # the far plane of the float32 matrix
    assert abs(far - 50.0) < 0.05
    np.testing.assert_allclose(depth, far, rtol=1e-5)
    L = _emu_lib()
    nprim, scene = emu_scene("w3d", state, rec, phys)
    d = np.zeros((H, W), dtype=np.float32)
    L.emu_render_rays(nprim, _fp(scene), _fp(view), _fp(proj), W, H, None, _fp(d), None)
    assert np.array_equal(d, emu_render("w3d", state, rec, phys, view, proj)[1])


def test_camera_matrices():
    """camera_matrices puts the eye at target + distance (cos p sin y, -cos p cos y, -sin p), looks at the target with
    the stated up vector, and builds the OpenGL perspective projection."""
    from mocca_envs_b200.vec_env import camera_matrices

    rng = np.random.RandomState(0)
    for _ in range(10):
        tgt = rng.uniform(-3, 3, 3)
        dist, yaw, pitch = rng.uniform(0.5, 5), rng.uniform(-180, 180), rng.uniform(-80, 80)
        v, p = camera_matrices(tgt, dist, yaw, pitch, fov=50.0, aspect=1.5, near=0.1, far=30.0)
        V = v[0].double().numpy().reshape(4, 4).T
        y, pp = np.deg2rad(yaw), np.deg2rad(pitch)
        eye = tgt + dist * np.array([np.cos(pp) * np.sin(y), -np.cos(pp) * np.cos(y), -np.sin(pp)])
        np.testing.assert_allclose(V @ np.append(eye, 1.0), [0, 0, 0, 1], atol=2e-5)
        np.testing.assert_allclose(V @ np.append(tgt, 1.0), [0, 0, -dist, 1], atol=2e-5 * max(1, dist))
        up = np.array([np.sin(pp) * np.sin(y), -np.sin(pp) * np.cos(y), np.cos(pp)])
        np.testing.assert_allclose(V[1, :3], up, atol=1e-6)  # the image's up axis in world
        P = p[0].double().numpy().reshape(4, 4).T
        for z in (-0.1, -30.0):  # near and far planes map to NDC z = -1 / +1
            q = P @ np.array([0, 0, z, 1.0])
            assert abs(q[2] / q[3] - (-1 if z == -0.1 else 1)) < 1e-5
        np.testing.assert_allclose(P[0, 0] * 1.5, P[1, 1], rtol=1e-6)
        np.testing.assert_allclose(P[1, 1], 1 / np.tan(np.deg2rad(25.0)), rtol=1e-6)


# ------------------------------------------------------------------------------------------------ GPU tests
def _vec(name, n, seed=0):
    import torch
    from mocca_envs_b200 import vec_env as V

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return getattr(V, KINDS[name]["vec"])(n, device="cuda:0", seed=seed, **KINDS[name].get("kw", {}))


def _load(env, cases):
    import torch

    env.reset()
    st = env.get_state().cpu().numpy()
    rc = env.get_record().cpu().numpy()
    for i, (state, rec, _) in enumerate(cases):
        st[i] = state[:st.shape[1]]
        rc[i] = rec[:rc.shape[1]]
    env.set_state(torch.tensor(st))
    env.set_record(torch.tensor(rc))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(KINDS))
def test_device_vs_emulation(name):
    """The device renders what the emulation renders (seg equal on >= 99.9 % of the kind's pixels, depth to 1e-5
    relative where seg is equal) and meets the float64 reference like the emulation.  (Where two primitives meet, the
    device's FMA contraction and the emulation's separate roundings can pick different sides of the seam.)"""
    import torch

    cases = states(name)
    env = _vec(name, len(cases))
    same_px = total_px = 0
    try:
        _load(env, cases)
        for dist, yaw, pitch in cameras(name):
            vs, ps = zip(*[cam(c[0][0:3], dist, yaw, pitch) for c in cases])
            out = env.render(width=W, height=H, view=torch.tensor(np.stack(vs)), proj=torch.tensor(np.stack(ps)))
            for i, (state, rec, phys) in enumerate(cases):
                img = tuple(out[k][i].cpu().numpy() for k in ("rgb", "depth", "seg"))
                emu = emu_render(name, state, rec, phys, vs[i], ps[i])
                same = img[2] == emu[2]
                same_px += int(same.sum())
                total_px += same.size
                np.testing.assert_allclose(img[1][same], emu[1][same], rtol=1e-5)
                check_against_reference(name, img, reference_render(reference_scene(name, state, rec, phys), vs[i],
                                                                    ps[i]))
    finally:
        env.close()
    assert same_px >= 0.999 * total_px, (name, same_px / total_px)


@pytest.mark.gpu
def test_render_has_no_side_effects():
    """Two batches, same seed, 60 steps; one renders after every step.  Observations, rewards, dones, truncations,
    state, record, RNG streams and statistics stay bit-identical.  The Walker3D and Stepper batches pass through
    auto-resets (asserted); Monkey3D's episodes do not end within 60 random steps, so its leg checks steps only."""
    import torch

    for name in ("w3d", "stepper", "monkey"):
        a, b = _vec(name, 64, seed=5), _vec(name, 64, seed=5)
        try:
            oa, ob = a.reset(), b.reset()
            g = torch.Generator(device="cuda:0").manual_seed(1)
            resets = 0
            for _ in range(60):
                act = torch.rand(64, a.act_dim, device="cuda:0", generator=g) * 4 - 2  # large: episodes end
                ra, rb = a.step(act), b.step(act)
                b.render(width=32, height=24)
                b.render(env_ids=torch.tensor([3, 1, 99, -1]), width=17, height=9, outputs=("seg",))
                for x, y in zip(ra[:3], rb[:3]):
                    assert torch.equal(x, y)
                assert torch.equal(ra[3]["TimeLimit.truncated"], rb[3]["TimeLimit.truncated"])
                resets += int(ra[2].sum())
            assert resets > 0 or name == "monkey", name
            # (bitwise: the record's int fields, e.g. -1, read as float NaN)
            assert torch.equal(a.get_state().view(torch.int32), b.get_state().view(torch.int32))
            assert torch.equal(a.get_record().view(torch.int32), b.get_record().view(torch.int32))
            assert np.array_equal(a.get_rng(), b.get_rng())
            assert a.stats() == b.stats()
        finally:
            a.close()
            b.close()


@pytest.mark.gpu
def test_subset_and_full_batch():
    """At 16 384 envs, env_ids in an arbitrary order with repeats: every frame equals the frame of that env rendered
    alone; the full batch (env_ids=None) likewise."""
    import torch

    n = 16384
    env = _vec("w3d", n, seed=2)
    try:
        env.reset()
        g = torch.Generator(device="cuda:0").manual_seed(0)
        for _ in range(5):
            env.step(torch.rand(n, env.act_dim, device="cuda:0", generator=g) * 2 - 1)
        ids = torch.randint(0, n, (300,), generator=torch.Generator().manual_seed(1))
        ids = torch.cat([ids, ids[:20], torch.tensor([n - 1, 0, 0])])
        sub = env.render(env_ids=ids, width=24, height=20)
        full = env.render(width=24, height=20)
        for j in list(range(0, len(ids), 7)) + [len(ids) - 1]:
            one = env.render(env_ids=ids[j:j + 1], width=24, height=20)
            for k in ("rgb", "depth", "seg"):
                assert torch.equal(sub[k][j], one[k][0]), (j, k)
                assert torch.equal(full[k][int(ids[j])], one[k][0]), (j, k)
        assert (full["seg"] >= 99).float().mean() > 0.02
    finally:
        env.close()


@pytest.mark.gpu
def test_gym_facade_rgb_array():
    """render("rgb_array") returns an (H, W, 3) uint8 frame for every env id and the Pillar variant; "human"
    raises NotImplementedError; the metadata names rgb_array."""
    from mocca_envs_b200 import vec_env as V

    facades = [(V.Walker3DCustomEnv, {}), (V.Walker3DStepperEnv, {}), (V.Walker3DStepperEnv, dict(plank_class="Pillar")),
               (V.Monkey3DCustomEnv, {}), (V.CassieEnv, {}), (V.Child3DCustomEnv, {}), (V.MikeStepperEnv, {}),
               (V.Walker2DCustomEnv, {}), (V.Crab2DCustomEnv, {})]
    for cls, kw in facades:
        env = cls(seed=0, **kw)
        try:
            env.reset()
            env.step(env.action_space.sample())
            frame = env.render("rgb_array", width=80, height=60)
            assert isinstance(frame, np.ndarray) and frame.shape == (60, 80, 3) and frame.dtype == np.uint8
            assert len(np.unique(frame.reshape(-1, 3), axis=0)) > 3
            assert env.render().shape == (240, 320, 3)
            assert cls.metadata["render.modes"] == ["rgb_array"]
            with pytest.raises(NotImplementedError):
                env.render("human")
        finally:
            env.close()


@pytest.mark.gpu
def test_argument_errors():
    """Bad width, height or count: an error with a message; NULL outputs are skipped; out-of-range ids are blank."""
    import torch

    env = _vec("w3d", 4)
    try:
        env.reset()
        for w, h in ((0, 8), (8, 0), (2049, 8), (8, 2049)):
            with pytest.raises(RuntimeError, match="width and height"):
                env.render(width=w, height=h)
        with pytest.raises(RuntimeError, match="count"):
            env.render(env_ids=torch.zeros(0, dtype=torch.int32))
        with pytest.raises(ValueError):
            env.render(outputs=("normals",))
        out = env.render(env_ids=[5, -1, 2], width=16, height=8, outputs=("depth", "seg"))
        assert set(out) == {"depth", "seg"}
        # depth = far of the tracking camera's float32 projection matrix (far = P[14] / (P[10] + 1))
        from mocca_envs_b200.vec_env import TRACKING_CAMERA, camera_matrices

        p = camera_matrices([0.0, 0.0, 0.0], aspect=2.0, **TRACKING_CAMERA)[1][0].double()
        far = float(p[14] / (p[10] + 1.0))
        assert abs(far - TRACKING_CAMERA["far"]) < 1e-3 * TRACKING_CAMERA["far"]
        assert (out["seg"][0:2] == -1).all()
        assert torch.allclose(out["depth"][0:2].double(), torch.tensor(far, device="cuda:0", dtype=torch.float64),
                              rtol=1e-5)
        full = env.render(env_ids=[2], width=16, height=8)
        assert torch.equal(full["seg"][0], out["seg"][2]) and torch.equal(full["depth"][0], out["depth"][2])
    finally:
        env.close()
