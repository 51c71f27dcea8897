"""Reduce a Bullet-convention model table (model_compiler.py) to the kernel's articulation tables and emit
them as a C header (``csrc/generated/<robot>_model.h``) consumed by the CUDA kernels.

Kernel-side representation (all constant, derived at q = 0):

* joints j = 0..NJ-1  : the revolute links in PyBullet joint order (== action order, robots.py:163-172).
  ``jparent`` (-1 = base), the joint frame's pose in its parent joint frame (``joff``, ``jrot``), the axis.
  Frames sit at the joint pivots; fixed links between revolute links are folded into these constants.
* bodies b = 0..NB-1  : every Bullet link with mass (base first, DFS order) attached to its owner joint frame:
  COM offset, inertia (symmetric 3x3 in owner axes), mass.  Kept un-merged because Bullet's velocity damping is
  per link and non-linear in |v| (SURVEY App. G).
* points              : contact candidates -- sphere centres and both capsule end-sphere centres.
* generalised coordinates u = [omega_world, v_baseCOM_world, qd] (PyBullet/btMultiBody order), NU = 6 + NJ.
* render geoms         : the collision geometry as mb200_render draws it (sphere, capsule, box in the owner joint
  frame) and the face planes of the mesh hulls; read by the render kernels only.
"""
from __future__ import annotations

import os

import numpy as np

from .model_compiler import JOINT_REVOLUTE, GEOM_SPHERE, GEOM_CAPSULE, GEOM_BOX, load_table, quat_to_mat


def reduce_table(t: dict) -> dict:
    nl = t["n_links"]
    parent = t["parent"]
    # pose of every Bullet link COM frame in the base frame at q = 0
    Rl = [np.eye(3)] * (nl + 1)
    pl = [np.zeros(3)] * (nl + 1)
    piv = [np.zeros(3)] * (nl + 1)
    for i in range(nl):
        Rz = quat_to_mat(t["rot_parent_to_this"][i])  # parent -> this
        p = parent[i] + 1
        Rl[i + 1] = Rl[p] @ Rz.T
        piv[i + 1] = pl[p] + Rl[p] @ np.array(t["e_vec"][i])
        pl[i + 1] = piv[i + 1] + Rl[i + 1] @ np.array(t["d_vec"][i])

    jlink = [i for i in range(nl) if t["joint_type"][i] == JOINT_REVOLUTE]
    nj = len(jlink)
    joint_of_link = {l: j for j, l in enumerate(jlink)}

    def owner_joint(link):  # nearest revolute ancestor-or-self, -1 = base
        l = link
        while l >= 0:
            if l in joint_of_link:
                return joint_of_link[l]
            l = parent[l]
        return -1

    def frame(j):  # joint frame in base coords at q = 0: origin at the pivot, axes parallel to the base's (round 2:
        # every zero-pose rotation between consecutive joint frames is then the identity, and the kinematics is one
        # Rodrigues rotation per joint about the axis as it points at q = 0 -- no per-joint constant rotation)
        if j < 0:
            return np.eye(3), np.zeros(3)
        return np.eye(3), piv[jlink[j] + 1]

    jparent, joff, jrot, jaxis, jlevel, janc = [], [], [], [], [], []
    for j, l in enumerate(jlink):
        pj = owner_joint(parent[l])
        Rp, op = frame(pj)
        Rj, oj = frame(j)
        jparent.append(pj)
        joff.append(Rp.T @ (oj - op))
        jrot.append(Rp.T @ Rj)
        ax_ = Rl[l + 1] @ np.array(t["axis"][l], dtype=np.float64)
        ax_ = np.where(np.abs(ax_) < 1e-15, 0.0, ax_)
        jaxis.append(ax_ / np.linalg.norm(ax_))
        jlevel.append(0 if pj < 0 else jlevel[pj] + 1)
        janc.append((1 << j) | (0 if pj < 0 else janc[pj]))

    bodies = []
    masses = [t["base"]["mass"]] + t["mass"]
    inertias = [t["base"]["inertia"]] + t["inertia"]
    names = [t["base"]["name"]] + t["link_names"]
    for li in range(nl + 1):
        if masses[li] <= 0:
            continue
        link = li - 1
        oj = owner_joint(link) if link >= 0 else -1
        Ro, oo = frame(oj)
        Rrel = Ro.T @ Rl[li]
        I = Rrel @ np.diag(inertias[li]) @ Rrel.T
        bodies.append(dict(name=names[li], link=link, owner=oj, com=Ro.T @ (pl[li] - oo), mass=masses[li],
                           inertia=[I[0, 0], I[1, 1], I[2, 2], I[0, 1], I[0, 2], I[1, 2]]))
    nb = len(bodies)
    # subtree body ranges (bodies are in DFS order -> contiguous)
    bstart, bend = [], []
    for j in range(nj):
        idx = [k for k, b in enumerate(bodies) if b["owner"] >= 0 and (janc[b["owner"]] >> j) & 1]
        assert idx == list(range(idx[0], idx[-1] + 1)), "subtree bodies must be contiguous"
        bstart.append(idx[0])
        bend.append(idx[-1] + 1)

    # body forest for the leaf-to-root accumulation of the composite inertias: parent = the latest previous body whose
    # owner joint is the base, the same joint, or an ancestor of the body's owner.  The composite of joint j is then the
    # accumulated record of body bstart(j) -- asserted: its descendants are exactly the range [bstart(j), bend(j)).
    bparent = []
    for k, b in enumerate(bodies):
        cand = [k2 for k2 in range(k) if bodies[k2]["owner"] < 0 or
                (b["owner"] >= 0 and (janc[b["owner"]] >> bodies[k2]["owner"]) & 1)]
        bparent.append(cand[-1] if cand else -1)
    assert bparent[0] == -1 and all(pb >= 0 for pb in bparent[1:]), "body 0 must be the base"
    desc = [{k} for k in range(nb)]
    for k in range(nb - 1, 0, -1):
        desc[bparent[k]] |= desc[k]
    assert desc[0] == set(range(nb))
    for j in range(nj):
        assert desc[bstart[j]] == set(range(bstart[j], bend[j])), "joint %d: subtree is not one body's subtree" % j

    thresh = [t["base"]["contact_threshold"]] + t["contact_threshold"]
    foot_links = t["foot_links"]
    palm_links = t.get("palm_links", [])
    points = []
    xboxes = []  # robot box geoms (Monkey3D fingers / hands): collide with the monkey bars only
    for gi, g in enumerate(t["geoms"]):
        if g["type"] == GEOM_BOX:
            link = g["link"]
            oj = owner_joint(link) if link >= 0 else -1
            Ro, oo = frame(oj)
            cw = pl[link + 1] + Rl[link + 1] @ np.array(g["pos"])
            Rg = Rl[link + 1] @ quat_to_mat(g["quat"])
            xboxes.append(dict(geom=gi, link=link, owner=oj, pos=Ro.T @ (cw - oo), rot=(Ro.T @ Rg).reshape(9),
                               half=g["size"], friction=g["friction"], thresh=thresh[link + 1],
                               foot=foot_links.index(link) if link in foot_links else -1))
            continue
        if g["type"] not in (GEOM_SPHERE, GEOM_CAPSULE):
            continue
        link = g["link"]
        oj = owner_joint(link) if link >= 0 else -1
        Ro, oo = frame(oj)
        ends = [g["p0"]] if g["type"] == GEOM_SPHERE else [g["p0"], g["p1"]]
        for e, pe in enumerate(ends):
            pw = pl[link + 1] + Rl[link + 1] @ np.array(pe)
            points.append(dict(geom=gi, end=e, link=link, owner=oj, pos=Ro.T @ (pw - oo), radius=g["size"][0],
                               friction=g["friction"], thresh=thresh[link + 1],
                               foot=foot_links.index(link) if link in foot_links else
                               (2 + palm_links.index(link) if link in palm_links else -1)))
    foot_body = [[b["link"] for b in bodies].index(f) for f in foot_links]
    # self-collision candidate pairs (model_compiler.self_collision_pairs): candidate-point indices of the two core
    # segments (a sphere is a zero-length segment), the smaller breaking threshold, the product friction
    # (btManifoldResult::calculateCombinedFriction) and which feet the two links are (Stepper feet_contact)
    pts_of_geom = {}
    for k, pnt in enumerate(points):
        pts_of_geom.setdefault(pnt["geom"], []).append(k)
    spairs = []
    for ga, gb in t.get("self_pairs", []):
        pa, pb = pts_of_geom[ga], pts_of_geom[gb]
        A, B = points[pa[0]], points[pb[0]]
        feet = sum(1 << f for f in range(2) for x in (A, B) if x["foot"] == f)
        half = lambda ids: 0.5 * float(np.linalg.norm(np.asarray(points[ids[0]]["pos"]) - np.asarray(points[ids[-1]]["pos"])))
        reach = half(pa) + half(pb) + A["radius"] + B["radius"] + min(A["thresh"], B["thresh"])
        spairs.append(dict(reach=reach * (1 + 1e-5) + 1e-6, pack=pa[0] | (pa[-1] << 8) | (pb[0] << 16) | (pb[-1] << 24), thresh=min(A["thresh"], B["thresh"]),
                           mu=A["friction"] * B["friction"], own_a=A["owner"], own_b=B["owner"], feet=feet))
        assert A["owner"] != B["owner"]
    # mesh-hull self-collision (Cassie, urdf_compiler.hull_collision_pairs): hull vertices and bounding spheres in the
    # owner joint frames; the pairs ride in the same sp_* tables as the segment pairs (pack = hull a | hull b << 8)
    hulls = []
    for h in t.get("hulls", []):
        link = h["link"]
        oj = owner_joint(link)
        Ro, oo = frame(oj)
        vw = [Ro.T @ (pl[link + 1] + Rl[link + 1] @ np.array(v) - oo) for v in h["verts"]]
        c = np.mean(vw, axis=0)
        # bounding capsule for the broad phase: principal axis of the vertices, radius = largest distance to it
        V = np.array(vw) - c
        u = np.linalg.eigh(V.T @ V)[1][:, -1]
        tt = V @ u
        seg = (c + tt.min() * u, c + tt.max() * u)
        crad = float(np.linalg.norm(V - np.outer(tt, u), axis=1).max())
        hulls.append(dict(link=link, owner=oj, verts=vw, center=c, radius=max(float(np.linalg.norm(v - c)) for v in vw),
                          seg=seg, crad=crad,
                          thresh=thresh[link + 1], friction=t["link_friction"][link + 1],
                          foot=foot_links.index(link) if link in foot_links else -1))
    for ha, hb in t.get("hull_pairs", []):
        A, B = hulls[ha], hulls[hb]
        assert not spairs or "hull" in spairs[0], "a model has segment pairs or hull pairs, not both"
        feet = sum(1 << f for f in range(2) for x in (A, B) if x["foot"] == f)
        th = min(A["thresh"], B["thresh"])
        spairs.append(dict(hull=1, reach=(A["crad"] + B["crad"] + th + 2 * t["hull_margin"]) * (1 + 1e-5) + 1e-6,
                           pack=ha | (hb << 8), thresh=th, mu=A["friction"] * B["friction"], own_a=A["owner"],
                           own_b=B["owner"], feet=feet))
        assert A["owner"] != B["owner"]
    # render geoms (mb200_render): every sphere / capsule / box in its owner joint frame.  A model with mesh hulls
    # (Cassie) is drawn as its hulls; its geoms are the hull-vertex contact spheres and are not drawn.
    rgeoms = []
    for g in ([] if hulls else t["geoms"]):
        link = g["link"]
        oj = owner_joint(link) if link >= 0 else -1
        Ro, oo = frame(oj)
        loc = lambda v: Ro.T @ (pl[link + 1] + Rl[link + 1] @ np.array(v) - oo)
        if g["type"] == GEOM_BOX:
            rgeoms.append(dict(type=2, owner=oj, a=loc(g["pos"]), b=loc(g["pos"]), r=0.0,
                               rot=(Ro.T @ Rl[link + 1] @ quat_to_mat(g["quat"])).reshape(9), half=g["size"][:3]))
        elif g["type"] in (GEOM_SPHERE, GEOM_CAPSULE):
            p1 = g["p0"] if g["type"] == GEOM_SPHERE else g["p1"]
            rgeoms.append(dict(type=0 if g["type"] == GEOM_SPHERE else 1, owner=oj, a=loc(g["p0"]), b=loc(p1),
                               r=g["size"][0], rot=np.eye(3).reshape(9), half=[0.0, 0.0, 0.0]))
    for h in hulls:
        h["planes"] = hull_planes(h["verts"])
    # ancestor chains (root -> self) packed 5 bits per entry, and the compact (chain-ordered) factor layout:
    # row i of L stores only its support [base block | ancestors root->parent | diagonal]
    chains = []
    for j in range(nj):
        c = [j]
        while jparent[c[0]] >= 0:
            c.insert(0, jparent[c[0]])
        chains.append(c)
    jdepth = [len(c) - 1 for c in chains]
    assert max(jdepth) + 1 <= 12 and nj <= 32
    chainpack = [sum(a << (5 * t) for t, a in enumerate(c)) for c in chains]
    rowlen = [i + 1 for i in range(6)] + [6 + jdepth[j] + 1 for j in range(nj)]
    rowoff = [sum(rowlen[:i]) for i in range(6 + nj)]
    rowmask_rt = [(1 << i) - 1 for i in range(6)] + [0x3F | ((janc[j] & ~(1 << j)) << 6) for j in range(nj)]
    palm_body = [[b["link"] for b in bodies].index(f) for f in palm_links]
    # loop closures (Cassie): pivots re-expressed in the owner joint frames of the two links
    p2p = []
    for c in t.get("p2p", []):
        sides = []
        for link, pivot in ((c["link_a"], c["pivot_a"]), (c["link_b"], c["pivot_b"])):
            oj = owner_joint(link)
            Ro, oo = frame(oj)
            pw = pl[link + 1] + Rl[link + 1] @ np.array(pivot)
            sides.append(dict(owner=oj, pos=Ro.T @ (pw - oo)))
        p2p.append(dict(sides=sides, max_impulse=c["max_impulse"]))
    dof_of_rev_link = {l: j for j, l in enumerate(jlink)}
    extras = {}
    if "ordered_dofs" in t:
        pd = t["powered_joint_inds"] + t["spring_joint_inds"]
        extras = dict(ordered=t["ordered_dofs"], pd_dof=[t["ordered_dofs"][k] for k in pd], pd_ordered=pd,
                      pd_kp=t["pd_kp"], pd_kd=t["pd_kd"], npowered=len(t["powered_joint_inds"]))
    return dict(name=t["name"], nj=nj, nb=nb, nu=6 + nj, npt=len(points), nlevel=max(jlevel) + 1,
                xboxes=xboxes, palm_body=palm_body, rgeoms=rgeoms, p2p=p2p, extras=extras, spairs=spairs, hulls=hulls,
                hull_margin=t.get("hull_margin", 0.0),
                jparent=jparent, joff=joff, jrot=jrot, jaxis=jaxis, jlevel=jlevel, janc=janc,
                lower=t["lower"], upper=t["upper"], gain=t["gain"], damping=t["damping"], armature=t["armature"],
                bodies=bodies, bstart=bstart, bend=bend, bparent=bparent, points=points, foot_body=foot_body,
                nfeet=len(foot_links), base_joint_angles=t["base_joint_angles"], base_position=t["base_position"],
                right=t["right_joint_indices"], left=t["left_joint_indices"], neg=t["negation_joint_indices"],
                jdepth=jdepth, chainpack=chainpack, rowlen=rowlen, rowoff=rowoff, rowmask_rt=rowmask_rt,
                lsize=sum(rowlen), maxsup=max(rowlen))


def hull_planes(verts) -> np.ndarray:
    """Face planes [k][4] = (n, d), |n| = 1, of the convex hull of `verts`: n . x <= d inside.  Coplanar facets of
    scipy's triangulation are merged, so each plane is one face."""
    from scipy.spatial import ConvexHull

    V = np.asarray(verts, dtype=np.float64)
    planes = []
    for eq in ConvexHull(V).equations:  # n . x + off <= 0 inside, |n| = 1
        n, d = eq[:3], -eq[3]
        if not any(np.abs(n - p[:3]).max() < 1e-9 and abs(d - p[3]) < 1e-9 for p in planes):
            planes.append(np.concatenate([n, [d]]))
    return np.array(planes)


def _f(v) -> str:
    s = "%.9g" % float(v)
    if "." not in s and "e" not in s and "n" not in s:
        s += ".0"
    return s + "f"


def _farr(name, rows, width=None):
    rows = np.asarray(rows, dtype=np.float64)
    if rows.ndim == 1:
        body = ", ".join(_f(v) for v in rows)
        return "MB_TABLE float %s[%d] = {%s};\n" % (name, len(rows), body)
    body = ",\n  ".join("{" + ", ".join(_f(v) for v in r) + "}" for r in rows)
    return "MB_TABLE float %s[%d][%d] = {\n  %s};\n" % (name, rows.shape[0], rows.shape[1], body)


def _darr(name, vals):
    vals = list(vals) or [0.0]
    return "MB_TABLE double %s[%d] = {%s};\n" % (name, len(vals), ", ".join("%.17g" % float(v) for v in vals))


def _iarr(name, vals, ctype="int"):
    vals = list(vals) or [-1 if ctype == "int" else 0]  # zero-length arrays are not C
    fmt = "%du" if ctype == "unsigned" else "%d"
    return "MB_TABLE %s %s[%d] = {%s};\n" % (ctype, name, len(vals), ", ".join(fmt % v for v in vals))


def emit_header(t: dict, prefix: str) -> str:
    r = reduce_table(t)
    P = prefix
    out = []
    out.append("// GENERATED by mocca_envs_b200/codegen.py from mocca_envs_b200/models/%s.json -- do not edit.\n" % r["name"])
    out.append("// Source model: reference mocca_envs/%s.\n" % t["source"])
    out.append("#pragma once\n#include \"../mb_tables.h\"\n\n")
    out.append(_iarr(P + "_jparent", r["jparent"]))
    out.append(_iarr(P + "_janc", r["janc"], "unsigned"))
    out.append(_iarr(P + "_jdepth", r["jdepth"]))
    out.append(_iarr(P + "_rowoff", r["rowoff"]))
    out.append(_iarr(P + "_rowlen", r["rowlen"]))
    out.append(_iarr(P + "_rowmask", r["rowmask_rt"], "unsigned"))
    # uniform-indexed copies in constant memory (one LDC instead of a global load in the sequential loops)
    out.append(_iarr(P + "_c_rowoff", r["rowoff"]).replace("MB_TABLE", "MB_CTABLE"))
    out.append(_iarr(P + "_c_rowlen", r["rowlen"]).replace("MB_TABLE", "MB_CTABLE"))
    # facoff[k][t]: offset of the compact row that entry t of row k updates (its column index' own row)
    maxoff = r["maxsup"] - 1
    fac = []
    for k in range(r["nu"]):
        cols = sorted(j for j in range(k) if (r["rowmask_rt"][k] >> j) & 1)
        fac.append([r["rowoff"][c] for c in cols] + [0] * (maxoff - len(cols)))
    # fcol[k][t]: generalised coordinate whose column sits in slot t of compact row k
    fcol = []
    for k in range(r["nu"]):
        cols = sorted(j for j in range(k) if (r["rowmask_rt"][k] >> j) & 1)
        fcol.append(cols + [0] * (maxoff - len(cols)))
    # Affine form of the two tables (round 2): the rows along a chain are stored like a packed dense triangle, so for the
    # pair (t, s) with packed index p = t (t + 1) / 2 + s the update lands at  p + delta_k(t)  and slot t belongs to column
    # t + cdelta_k(t), where both deltas are piecewise constant in t with one step per branch point the chain passes
    # after leaving the first-stored path: fstep[k][i] = (t_i, increment of delta, increment of cdelta), t_i = 15 = unused.
    fsteps = []
    for k in range(r["nu"]):
        nk = r["rowlen"][k] - 1
        dd_ = [fac[k][tt] - tt * (tt + 1) // 2 for tt in range(nk)]
        dc_ = [fcol[k][tt] - tt for tt in range(nk)]
        st_, pd_, pc_ = [], 0, 0
        for tt in range(nk):
            if dd_[tt] != pd_ or dc_[tt] != pc_:
                st_.append((tt, dd_[tt] - pd_, dc_[tt] - pc_))
                pd_, pc_ = dd_[tt], dc_[tt]
        fsteps.append(st_)
    nsteps = max(1, max(len(x) for x in fsteps))
    assert nsteps <= 2, "factorize() supports two steps per pivot row"
    for i in range(nsteps):
        out.append(_iarr(P + "_c_ft%d" % (i + 1), [x[i][0] if len(x) > i else 15 for x in fsteps]).replace("MB_TABLE", "MB_CTABLE"))
        out.append(_iarr(P + "_c_fd%d" % (i + 1), [x[i][1] if len(x) > i else 0 for x in fsteps]).replace("MB_TABLE", "MB_CTABLE"))
        out.append(_iarr(P + "_c_fc%d" % (i + 1), [x[i][2] if len(x) > i else 0 for x in fsteps]).replace("MB_TABLE", "MB_CTABLE"))
    # lane-indexed variant (global memory) for setup_rows(): the support of a constraint row on coordinate k is row k's
    # support PLUS k itself (slot nk), so the steps are taken over t = 0 .. nk inclusive
    rsteps = []
    for k in range(r["nu"]):
        nk = r["rowlen"][k] - 1
        cols_ = fcol[k][:nk] + [k]
        offs_ = fac[k][:nk] + [r["rowoff"][k]]
        st_, pd_, pc_ = [], 0, 0
        for tt in range(nk + 1):
            dd_, dc_ = offs_[tt] - tt * (tt + 1) // 2, cols_[tt] - tt
            if dd_ != pd_ or dc_ != pc_:
                st_.append((tt, dd_ - pd_, dc_ - pc_))
                pd_, pc_ = dd_, dc_
        rsteps.append(st_)
    assert max(len(x) for x in rsteps) <= 2, "setup_rows() supports two steps per row"
    r["rsteps"] = max(1, max(len(x) for x in rsteps))
    for i in range(2):
        out.append(_iarr(P + "_ft%d" % (i + 1), [x[i][0] if len(x) > i else 15 for x in rsteps]))
        out.append(_iarr(P + "_fd%d" % (i + 1), [x[i][1] if len(x) > i else 0 for x in rsteps]))
        out.append(_iarr(P + "_fc%d" % (i + 1), [x[i][2] if len(x) > i else 0 for x in rsteps]))
    r["fsteps"] = nsteps
    r["fsteps_list"] = fsteps
    # per coordinate: depth in the joint tree (-1 for the six base coordinates) and its ancestors' coordinate
    # indices by level, 5 bits each (levels 0-5 in word 0, 6-11 in word 1)
    cdepth = [-1] * 6 + list(r["jdepth"])
    anc0, anc1 = [0] * 6, [0] * 6
    for j in range(r["nj"]):
        c = [j]
        while r["jparent"][c[0]] >= 0:
            c.insert(0, r["jparent"][c[0]])
        w0 = sum((6 + a) << (5 * t) for t, a in enumerate(c[:6]))
        w1 = sum((6 + a) << (5 * t) for t, a in enumerate(c[6:12]))
        anc0.append(w0)
        anc1.append(w1)
    out.append(_iarr(P + "_cdepth", cdepth))
    out.append(_iarr(P + "_canc0", anc0, "unsigned"))
    out.append(_iarr(P + "_canc1", anc1, "unsigned"))
    # Chain-walk kinematics (round 2): lane 3 * ch + c carries row c of the rotation (and component c of every vector)
    # down the ch-th root-to-leaf chain in registers; kin[step][ch] = the joint met at that step, its pivot offset in
    # the parent frame, its axis, and whether this chain is the one that stores the joint (shared prefixes are walked
    # by every chain that contains them, stored by the first).  Chain NCH is the idle one of the unused lanes.
    leaves = [j for j in range(r["nj"]) if j not in r["jparent"]]
    kchains = []
    for lf in leaves:
        c = [lf]
        while r["jparent"][c[0]] >= 0:
            c.insert(0, r["jparent"][c[0]])
        kchains.append(c)
    assert len(kchains) <= 10, "three lanes per chain"
    seen = set()
    krec = []
    for st in range(r["nlevel"]):
        row = []
        for c in kchains + [[]]:
            if st < len(c):
                j = c[st]
                row.append((j, list(r["joff"][j]), list(r["jaxis"][j]), 0 if j in seen else 1))
                seen.add(j)
            else:
                row.append((0, [0.0, 0.0, 0.0], [0.0, 0.0, 1.0], 0))
        krec.append(row)
    assert seen == set(range(r["nj"]))
    out.append("MB_TABLE MbKinRec %s_kin[%d][%d] = {\n  %s};\n" % (P, r["nlevel"], len(kchains) + 1, ",\n  ".join(
        "{" + ", ".join("{%d, {%s}, {%s}, %d}" % (j, ", ".join(_f(v) for v in off), ", ".join(_f(v) for v in ax), fl)
                        for j, off, ax, fl in row) + "}" for row in krec)))
    r["nch"] = len(kchains)
    # float32 limits exactly as robots.py:126-130 builds them (weight = f32(upper - lower), bias = f32(lower))
    out.append(_farr(P + "_lower", r["lower"]))
    out.append(_farr(P + "_upper", r["upper"]))
    out.append(_farr(P + "_weight", [np.float32(u - l) for u, l in zip(r["upper"], r["lower"])]))
    out.append(_farr(P + "_gain", r["gain"]))
    out.append(_farr(P + "_damping", r["damping"]))
    out.append(_farr(P + "_armature", r["armature"]))
    out.append(_iarr(P + "_bstart", r["bstart"]))
    out.append(_iarr(P + "_bend", r["bend"]))
    out.append(_iarr(P + "_bowner", [b["owner"] for b in r["bodies"]]))
    out.append(_farr(P + "_bcom", [b["com"] for b in r["bodies"]]))
    out.append(_farr(P + "_bmass", [b["mass"] for b in r["bodies"]]))
    out.append(_farr(P + "_binertia", [b["inertia"] for b in r["bodies"]]))
    out.append(_iarr(P + "_powner", [p["owner"] for p in r["points"]]))
    out.append(_iarr(P + "_pfoot", [p["foot"] for p in r["points"]]))
    out.append(_iarr(P + "_pid", [2 * p["geom"] + p["end"] for p in r["points"]]))
    out.append(_farr(P + "_ppos", [p["pos"] for p in r["points"]]))
    out.append(_farr(P + "_pradius", [p["radius"] for p in r["points"]]))
    out.append(_farr(P + "_pfriction", [p["friction"] for p in r["points"]]))
    out.append(_farr(P + "_pthresh", [p["thresh"] for p in r["points"]]))
    out.append(_iarr(P + "_foot_body", r["foot_body"]))
    sides = [sd for c in r["p2p"] for sd in c["sides"]]
    out.append(_iarr(P + "_lc_owner", [sd["owner"] for sd in sides]))
    out.append(_farr(P + "_lc_pos", [sd["pos"] for sd in sides] or [[0, 0, 0]]))
    out.append(_farr(P + "_lc_maximp", [c["max_impulse"] for c in r["p2p"]] or [0]))
    sp = r["spairs"]
    out.append(_iarr(P + "_sp_pack", [x["pack"] for x in sp] or [0], "unsigned"))
    out.append(_iarr(P + "_sp_own", [(x["own_a"] + 1) | ((x["own_b"] + 1) << 8) | (x["feet"] << 16) for x in sp] or [0]))
    out.append(_farr(P + "_sp_thresh", [x["thresh"] for x in sp] or [0]))
    out.append(_farr(P + "_sp_mu", [x["mu"] for x in sp] or [0]))
    out.append(_farr(P + "_sp_reach", [x["reach"] for x in sp] or [0]))
    hl = r["hulls"] or [dict(owner=-1, verts=[np.zeros(3)] * 32, center=np.zeros(3), radius=0.0,
                             seg=(np.zeros(3), np.zeros(3)))]
    out.append(_iarr(P + "_hown", [h["owner"] for h in hl]))
    out.append(_farr(P + "_hcen", [list(h["center"]) + [h["radius"]] for h in hl]))
    out.append(_farr(P + "_hseg", [list(h["seg"][0]) + list(h["seg"][1]) for h in hl]))
    out.append("MB_TABLE float %s_hv[%d][32][3] = {\n%s};\n" % (P, len(hl), ",\n".join(
        "  {" + ", ".join("{%s, %s, %s}" % tuple(_f(x) for x in v) for v in h["verts"]) + "}" for h in hl)))
    ex = r["extras"]
    out.append(_iarr(P + "_ordered", ex.get("ordered", [])))
    out.append(_iarr(P + "_pd_dof", ex.get("pd_dof", [])))
    out.append(_iarr(P + "_pd_ordered", ex.get("pd_ordered", [])))
    out.append(_farr(P + "_pd_kp", ex.get("pd_kp", [0])))
    out.append(_farr(P + "_pd_kd", ex.get("pd_kd", [0])))
    out.append(_iarr(P + "_palm_body", r["palm_body"] or [-1]))
    xb = r["xboxes"] or [dict(owner=-1, foot=-1, pos=[0, 0, 0], rot=np.eye(3).reshape(9), half=[0, 0, 0], friction=0,
                              thresh=0)]
    out.append(_iarr(P + "_xowner", [b["owner"] for b in xb]))
    out.append(_iarr(P + "_xfoot", [b["foot"] for b in xb]))
    out.append(_iarr(P + "_xpid", [2 * b.get("geom", 0) for b in xb]))
    out.append(_farr(P + "_xpos", [b["pos"] for b in xb]))
    out.append(_farr(P + "_xrot", [b["rot"] for b in xb]))
    out.append(_farr(P + "_xhalf", [b["half"] for b in xb]))
    out.append(_farr(P + "_xfriction", [b["friction"] for b in xb]))
    out.append(_farr(P + "_xthresh", [b["thresh"] for b in xb]))
    out.append(_darr(P + "_base_angles", r["base_joint_angles"]))
    out.append(_iarr(P + "_right", r["right"]))
    out.append(_iarr(P + "_left", r["left"]))
    out.append(_iarr(P + "_neg", r["neg"]))
    # render tables (mb200_render only): geoms in their owner joint frames, the hulls' face planes (n, d) in the same
    # frames, hull h owning planes [hpl_off[h], hpl_off[h + 1]).  Constant memory, declared behind every other table:
    # the physics kernels' global-table addresses (constant bank 4) and constant tables keep their slots.
    rg = r["rgeoms"] or [dict(type=-1, owner=-1, a=[0, 0, 0], b=[0, 0, 0], r=0, rot=np.eye(3).reshape(9), half=[0, 0, 0])]
    out.append(_iarr(P + "_rg_type", [g["type"] for g in rg]).replace("MB_TABLE", "MB_CTABLE"))
    out.append(_iarr(P + "_rg_owner", [g["owner"] for g in rg]).replace("MB_TABLE", "MB_CTABLE"))
    out.append(_farr(P + "_rg_a", [g["a"] for g in rg]).replace("MB_TABLE", "MB_CTABLE"))
    out.append(_farr(P + "_rg_b", [g["b"] for g in rg]).replace("MB_TABLE", "MB_CTABLE"))
    out.append(_farr(P + "_rg_r", [g["r"] for g in rg]).replace("MB_TABLE", "MB_CTABLE"))
    out.append(_farr(P + "_rg_rot", [g["rot"] for g in rg]).replace("MB_TABLE", "MB_CTABLE"))
    out.append(_farr(P + "_rg_half", [g["half"] for g in rg]).replace("MB_TABLE", "MB_CTABLE"))
    hpl = [p for h in r["hulls"] for p in h["planes"]] or [[0.0, 0.0, 1.0, 0.0]]
    hoff = [0]
    for h in r["hulls"]:
        hoff.append(hoff[-1] + len(h["planes"]))
    out.append(_iarr(P + "_hpl_off", hoff).replace("MB_TABLE", "MB_CTABLE"))
    out.append(_farr(P + "_hpl", hpl).replace("MB_TABLE", "MB_CTABLE"))
    # support of row i of the mass matrix / its L^T L factor (columns j < i): base block + ancestors
    rowmask = []
    for i in range(r["nu"]):
        if i < 6:
            rowmask.append((1 << i) - 1)
        else:
            j = i - 6
            rowmask.append(0x3F | (((r["janc"][j] & ~(1 << j))) << 6))
    out.append("\nstruct %s_Model {\n" % P)
    out.append("  MB_HD static constexpr unsigned rowmask_c(int i) {\n    return " +
               " ".join("i == %d ? %du :" % (i, m) for i, m in enumerate(rowmask)) + " 0u;\n  }\n")
    out.append("  enum { NJ = %d, NB = %d, NU = %d, NPT = %d, NLEVEL = %d, NFEET = %d, NMIRROR = %d, NNEG = %d,\n"
               "         LSIZE = %d, MAXSUP = %d, NXBOX = %d, NLOOP = %d, NORDERED = %d, NPD = %d, NPOWERED = %d, NSELF = %d,\n"
               "         NHULL = %d, SELF_HULLS = %d };  // the self-collision pairs are mesh-hull pairs (hull-vs-hull narrow phase)\n"
               % (r["nj"], r["nb"], r["nu"], r["npt"], r["nlevel"], r["nfeet"], len(r["right"]), len(r["neg"]),
                  r["lsize"], r["maxsup"], len(r["xboxes"]), len(r["p2p"]), len(ex.get("ordered", [])),
                  len(ex.get("pd_dof", [])), ex.get("npowered", 0), len(sp),
                  len(r["hulls"]), int(bool(r["hulls"]) and bool(sp))))
    out.append("  enum { NRG = %d, NHPL = %d };  // render geoms, hull face planes (mb200_render)\n"
               % (len(r["rgeoms"]), len(hpl) if r["hulls"] else 0))
    out.append("  MB_HD static const float* hpl() { return &%s_hpl[0][0]; }\n" % P)
    out.append("  MB_HD static float hull_margin() { return %s; }\n" % _f(r["hull_margin"]))
    out.append("  MB_HD static int hown(int i) { return %s_hown[i]; }\n" % P)
    out.append("  MB_HD static float hcen(int i, int k) { return %s_hcen[i][k]; }\n" % P)
    out.append("  MB_HD static float hseg(int i, int k) { return %s_hseg[i][k]; }\n" % P)
    out.append("  MB_HD static float hv(int h, int v, int k) { return %s_hv[h][v][k]; }\n" % P)
    out.append("  enum { NCH = %d };  // root-to-leaf chains of the kinematics walk (kin[step][chain], chain NCH = idle)\n" % r["nch"])
    out.append("  MB_HD static const MbKinRec* kin(int step, int ch) { return &%s_kin[step][ch]; }\n" % P)
    out.append("  enum { FSTEPS = %d };  // steps of the affine factorisation addressing (c_ft / c_fd / c_fc)\n" % r["fsteps"])
    # compile-time copies for the unrolled factorisation (template-indexed: every per-pivot scalar becomes an immediate)
    out.append("  static constexpr int k_rowoff[%d] = {%s};\n" % (r["nu"], ", ".join(str(v) for v in r["rowoff"])))
    out.append("  static constexpr int k_bparent[%d] = {%s};\n" % (r["nb"], ", ".join(str(max(v, 0)) for v in r["bparent"])))
    out.append("  static constexpr int k_rowlen[%d] = {%s};\n" % (r["nu"], ", ".join(str(v) for v in r["rowlen"])))
    for i in range(2):
        for nm, col, dflt in (("ft", 0, 15), ("fd", 1, 0), ("fc", 2, 0)):
            out.append("  static constexpr int k_%s%d[%d] = {%s};\n" % (nm, i + 1, r["nu"], ", ".join(
                str(x[i][col] if len(x) > i else dflt) for x in r["fsteps_list"])))
    for i in range(r["fsteps"]):
        for nm in ("ft", "fd", "fc"):
            out.append("  MB_HD static int c_%s%d(int k) { return %s_c_%s%d[k]; }\n" % (nm, i + 1, P, nm, i + 1))
    out.append("  enum { RSTEPS = %d };  // steps of the affine chain addressing of a constraint row (ft / fd / fc)\n" % r["rsteps"])
    for i in range(2):
        for nm in ("ft", "fd", "fc"):
            out.append("  MB_HD static int %s%d(int k) { return %s_%s%d[k]; }\n" % (nm, i + 1, P, nm, i + 1))
    if r["fsteps"] < 2:
        out.append("  MB_HD static int c_ft2(int) { return 15; }\n  MB_HD static int c_fd2(int) { return 0; }\n"
                   "  MB_HD static int c_fc2(int) { return 0; }\n")
    out.append("  MB_HD static int c_rowoff(int i) { return %s_c_rowoff[i]; }\n" % P)
    out.append("  MB_HD static int c_rowlen(int i) { return %s_c_rowlen[i]; }\n" % P)
    for fld, ctype in [("jparent", "int"), ("janc", "unsigned"), ("bstart", "int"), ("bend", "int"),
                       ("jdepth", "int"), ("rowoff", "int"), ("rowlen", "int"), ("rowmask", "unsigned"),
                       ("cdepth", "int"), ("canc0", "unsigned"), ("canc1", "unsigned"),
                       ("bowner", "int"), ("powner", "int"), ("pfoot", "int"), ("pid", "int"), ("foot_body", "int"),
                       ("palm_body", "int"), ("xowner", "int"), ("xfoot", "int"), ("xpid", "int"),
                       ("lc_owner", "int"), ("ordered", "int"), ("pd_dof", "int"), ("pd_ordered", "int"),
                       ("right", "int"), ("left", "int"), ("neg", "int"), ("sp_pack", "unsigned"), ("sp_own", "int"),
                       ("rg_type", "int"), ("rg_owner", "int"), ("hpl_off", "int")]:
        out.append("  MB_HD static %s %s(int i) { return %s_%s[i]; }\n" % (ctype, fld, P, fld))
    out.append("  MB_HD static double base_angles(int i) { return %s_base_angles[i]; }\n" % P)
    for fld in ["lower", "upper", "weight", "gain", "damping", "armature", "bmass", "pradius", "pfriction", "pthresh",
                "xfriction", "xthresh", "lc_maximp", "pd_kp", "pd_kd", "sp_thresh", "sp_mu", "sp_reach", "rg_r"]:
        out.append("  MB_HD static float %s(int i) { return %s_%s[i]; }\n" % (fld, P, fld))
    for fld in ["bcom", "binertia", "ppos", "xpos", "xrot", "xhalf", "lc_pos", "rg_a", "rg_b", "rg_rot", "rg_half"]:
        out.append("  MB_HD static float %s(int i, int k) { return %s_%s[i][k]; }\n" % (fld, P, fld))
    out.append("  MB_HD static float base_x() { return %s; }\n" % _f(r["base_position"][0]))
    out.append("  MB_HD static float base_y() { return %s; }\n" % _f(r["base_position"][1]))
    out.append("  MB_HD static float base_z() { return %s; }\n" % _f(r["base_position"][2]))
    # base orientation of the start pose (robots.py:276,311-323; xyzw), the env's termination height
    # (env_locomotion.py:44,320) and the stepper env's robot_init_position (env_locomotion.py:339,845)
    bq = t.get("base_orientation", [0.0, 0.0, 0.0, 1.0])
    out.append("  MB_HD static float base_quat(int k) { return k == 0 ? %s : (k == 1 ? %s : (k == 2 ? %s : %s)); }\n"
               % tuple(_f(v) for v in bq))
    out.append("  MB_HD static float term_height() { return %s; }\n" % _f(t.get("termination_height", 0.7)))
    # Walker2DCustomEnv / Crab2DCustomEnv (env_locomotion.py:285-310): done is forced to False, reset() returns zeros
    # in the two target slots
    out.append("  MB_HD static constexpr bool planar_env() { return %s; }\n" % ("true" if t.get("planar") else "false"))
    sp = t.get("stepper_init_position", [0.3, 0.0, 1.32])
    out.append("  MB_HD static float stepper_x() { return %s; }\n" % _f(sp[0]))
    out.append("  MB_HD static float stepper_y() { return %s; }\n" % _f(sp[1]))
    out.append("  MB_HD static float stepper_z() { return %s; }\n" % _f(sp[2]))
    out.append("};\n")
    return "".join(out)


def emit_all(repo_root: str):
    gen = os.path.join(repo_root, "mocca_envs_b200", "csrc", "generated")
    os.makedirs(gen, exist_ok=True)
    models = os.path.join(repo_root, "mocca_envs_b200", "models")
    for name, prefix in (("walker3d", "W3D"), ("monkey3d", "MK3D"), ("cassie", "CAS"), ("child3d", "CH3D"),
                         ("mike", "MIKE"), ("walker2d", "W2D"), ("crab2d", "CR2D")):
        t = load_table(os.path.join(models, name + ".json"))
        with open(os.path.join(gen, name + "_model.h"), "w") as f:
            f.write(emit_header(t, prefix))
