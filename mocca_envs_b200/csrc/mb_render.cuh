// mb_render.cuh -- camera images of an env batch by ray casting the collision geometry (mb200_render).
//
// Two passes, so that the warp-per-env physics code stays apart from the pixel code:
//   1. mb_render_scene<Env> (one warp per camera, the kind's k_render_scene_<kind>): the env's state through the
//      existing load_state / kinematics_pose / load_obstacles, then one world-space primitive per lane into the
//      camera's slice of the scene buffer, [MB_RMAX][MB_RSTRIDE] floats.
//   2. mb_render_pixel (one thread per pixel, the kind-independent k_render_rays in mb200.cu): the closest hit of the
//      pixel's ray over the camera's primitives, flat Lambert shading, RGB / depth / segmentation.
// Both are plain MB_HD code: the CPU emulation (tests/emu/emu_render.cpp) runs the same source.
#pragma once
#include "mb_env.cuh"

#define MB_RMAX 34    /* primitives per camera: Monkey3D's 29 geoms + 4 bars + the ground */
#define MB_RSTRIDE 24 /* floats per primitive */
#define MB_RENDER_TARGET_RADIUS 0.2f /* the walk-target marker sphere (a constant of this library) */
#define MB_RENDER_MAXDIM 2048

// primitive record, MB_RSTRIDE floats:
//   [0..3]   bounding sphere: centre, radius (< 0: empty slot)
//   [4..7]   type, seg code, colour class (int bits), hull: plane count (int bits)
//   [8..16]  R: local -> world rotation, row-major (column k = local axis k in world); capsule: [8..10] = end 1
//   [17..19] centre / origin of the local frame; capsule: end 0
//   [20..22] box: half extents; cylinder: radius, half height (about local z); hull: [20..21] = plane pointer
//   [23]     sphere / capsule radius
enum { MB_RP_NONE = 0, MB_RP_PLANE, MB_RP_SPHERE, MB_RP_CAPSULE, MB_RP_BOX, MB_RP_CYL, MB_RP_HULL };
enum { MB_RC_ROBOT = 0, MB_RC_GROUND, MB_RC_PLANK, MB_RC_BAR, MB_RC_TARGET };
enum { MB_SEG_SKY = -1, MB_SEG_GROUND = 0, MB_SEG_BOX = 10, MB_SEG_BAR = 20, MB_SEG_TARGET = 30, MB_SEG_LINK = 100 };

MB_HD float mb_ibits(int v) {
  float f;
  memcpy(&f, &v, 4);
  return f;
}
MB_HD int mb_fbits(float f) {
  int v;
  memcpy(&v, &f, 4);
  return v;
}

// which optional scene parts an env template has (the walk target: the Walker3DCustomEnv template)
template <class Env> struct MbRenderTraits { enum { TARGET = 0 }; };
template <class M> struct MbRenderTraits<W3DEnv<M>> { enum { TARGET = 1 }; };

template <class Env> struct MbRenderLayout {
  typedef typename Env::Model M;
  enum {
    NOBST = (Env::OBST & (MB_OBST_BOXES | MB_OBST_CYLS)) ? MB_MAXBOX : ((Env::OBST & MB_OBST_BARS) ? MB_MAXBAR : 0),
    HULL0 = M::NRG, OBST0 = HULL0 + M::NHULL, TARGET0 = OBST0 + NOBST,
    GROUND = TARGET0 + MbRenderTraits<Env>::TARGET, NPRIM = GROUND + 1
  };
};

MB_HD void mb_render_empty(float* e) {
  for (int k = 0; k < MB_RSTRIDE; ++k) e[k] = 0.0f;
  e[3] = -1.0f;
  e[4] = mb_ibits(MB_RP_NONE);
}

// a rigid frame of the robot in world coordinates: owner joint o (-1 = base)
template <class M> MB_HD void mb_render_frame(const WarpMem<M>& S, int o, const float** R, float* org) {
  *R = o < 0 ? S.Rb : S.w.k.jR[o];
  for (int k = 0; k < 3; ++k) org[k] = S.pos[k] + (o < 0 ? 0.0f : S.w.k.jp[o][k]);
}

// primitive i of the env's scene (after load_state / kinematics_pose / load_obstacles)
template <class Env> MB_HD void mb_render_prim(const typename Env::Mem& S, const MbPhysics& P, const float* rec, int i,
                                              float* e) {
  typedef typename Env::Model M;
  typedef MbRenderLayout<Env> Lay;
  mb_render_empty(e);
  const float* R;
  float org[3];
  if (i < Lay::HULL0) {  // robot geom
    const int o = M::rg_owner(i), ty = M::rg_type(i);
    mb_render_frame<M>(S, o, &R, org);
    const float a[3] = {M::rg_a(i, 0), M::rg_a(i, 1), M::rg_a(i, 2)};
    float aw[3];
    mb_matvec(R, a, aw);
    for (int k = 0; k < 3; ++k) e[17 + k] = org[k] + aw[k];
    e[5] = mb_ibits(MB_SEG_LINK + o);
    e[6] = mb_ibits(MB_RC_ROBOT);
    if (ty == 2) {  // box
      float Rg[9];
      for (int k = 0; k < 9; ++k) Rg[k] = M::rg_rot(i, k);
      mb_matmul(R, Rg, e + 8);
      const float hx = M::rg_half(i, 0), hy = M::rg_half(i, 1), hz = M::rg_half(i, 2);
      e[20] = hx; e[21] = hy; e[22] = hz;
      e[4] = mb_ibits(MB_RP_BOX);
      for (int k = 0; k < 3; ++k) e[k] = e[17 + k];
      e[3] = sqrtf(hx * hx + hy * hy + hz * hz);
    } else {
      const float r = M::rg_r(i);
      e[23] = r;
      if (ty == 0) {
        e[4] = mb_ibits(MB_RP_SPHERE);
        for (int k = 0; k < 3; ++k) e[k] = e[17 + k];
        e[3] = r;
      } else {
        const float b[3] = {M::rg_b(i, 0), M::rg_b(i, 1), M::rg_b(i, 2)};
        float bw[3];
        mb_matvec(R, b, bw);
        float hl = 0.0f;
        for (int k = 0; k < 3; ++k) {
          e[8 + k] = org[k] + bw[k];
          e[k] = 0.5f * (e[17 + k] + e[8 + k]);
          hl += (e[8 + k] - e[17 + k]) * (e[8 + k] - e[17 + k]);
        }
        e[4] = mb_ibits(MB_RP_CAPSULE);
        e[3] = 0.5f * sqrtf(hl) + r;
      }
    }
  } else if (i < Lay::OBST0) {  // mesh hull: its planes stay in the owner joint frame
    const int h = i - Lay::HULL0, o = M::hown(h);
    mb_render_frame<M>(S, o, &R, org);
    for (int k = 0; k < 9; ++k) e[8 + k] = R[k];
    for (int k = 0; k < 3; ++k) e[17 + k] = org[k];
    const float c[3] = {M::hcen(h, 0), M::hcen(h, 1), M::hcen(h, 2)};
    float cw[3];
    mb_matvec(R, c, cw);
    for (int k = 0; k < 3; ++k) e[k] = org[k] + cw[k];
    e[3] = M::hcen(h, 3);
    const int p0 = M::hpl_off(h);
    const float* planes = M::hpl() + 4 * p0;
    memcpy(e + 20, &planes, sizeof(planes));
    e[4] = mb_ibits(MB_RP_HULL);
    e[5] = mb_ibits(MB_SEG_LINK + o);
    e[6] = mb_ibits(MB_RC_ROBOT);
    e[7] = mb_ibits(M::hpl_off(h + 1) - p0);
  } else if (i < Lay::TARGET0) {  // static obstacles as load_obstacles staged them for collision
    const int k = i - Lay::OBST0;
    if (Env::OBST & (MB_OBST_BOXES | MB_OBST_CYLS)) {
      if (k >= S.nbox) return;
      const float* bx = S.rc.box[k];
      for (int c = 0; c < 3; ++c) e[c] = e[17 + c] = bx[c];
      for (int c = 0; c < 9; ++c) e[8 + c] = bx[3 + c];
      if (Env::OBST & MB_OBST_CYLS) {  // capped cylinder about local z: radius bx[12], half height bx[14]
        e[4] = mb_ibits(MB_RP_CYL);
        e[20] = bx[12]; e[21] = bx[14];
        e[3] = sqrtf(bx[12] * bx[12] + bx[14] * bx[14]);
      } else {
        e[4] = mb_ibits(MB_RP_BOX);
        e[20] = bx[12]; e[21] = bx[13]; e[22] = bx[14];
        e[3] = sqrtf(bx[12] * bx[12] + bx[13] * bx[13] + bx[14] * bx[14]);
      }
      e[5] = mb_ibits(MB_SEG_BOX + k);
      e[6] = mb_ibits(MB_RC_PLANK);
    } else {
      if (k >= S.nbar) return;
      const float* bar = S.rc.bar[k];  // centre, unit axis, half length, radius: a capped cylinder
      float p[3], q[3];
      mb_plane_space(bar + 3, p, q);
      for (int c = 0; c < 3; ++c) {
        e[c] = e[17 + c] = bar[c];
        e[8 + 3 * c] = p[c]; e[9 + 3 * c] = q[c]; e[10 + 3 * c] = bar[3 + c];
      }
      e[4] = mb_ibits(MB_RP_CYL);
      e[20] = bar[7]; e[21] = bar[6];
      e[3] = sqrtf(bar[6] * bar[6] + bar[7] * bar[7]);
      e[5] = mb_ibits(MB_SEG_BAR + k);
      e[6] = mb_ibits(MB_RC_BAR);
    }
  } else if (i < Lay::GROUND) {  // walk target marker
    for (int c = 0; c < 3; ++c) e[c] = e[17 + c] = rec[ER_TX + c];
    e[3] = e[23] = MB_RENDER_TARGET_RADIUS;
    e[4] = mb_ibits(MB_RP_SPHERE);
    e[5] = mb_ibits(MB_SEG_TARGET);
    e[6] = mb_ibits(MB_RC_TARGET);
  } else if (P.has_ground) {  // the plane z = 0 (no bounding sphere)
    e[3] = 0.0f;
    e[4] = mb_ibits(MB_RP_PLANE);
    e[5] = mb_ibits(MB_SEG_GROUND);
    e[6] = mb_ibits(MB_RC_GROUND);
  }
}

// pass 1 for one env: its world-space primitive list, MbRenderLayout<Env>::NPRIM records into `out`
template <class Env> MB_HD void mb_render_scene(typename Env::Mem& S, const MbPhysics& P, const float* state,
                                               const float* rec, float* out) {
  typedef MbRenderLayout<Env> Lay;
  static_assert(Lay::NPRIM <= MB_RMAX, "MB_RMAX is below the primitive count of an env kind");
  Env::load_state(S, state);
  Sim<typename Env::Model>::kinematics_pose(S, P);
  Env::load_obstacles(S, rec);
  MB_LANES(l)
    for (int i = l; i < Lay::NPRIM; i += 32) {
      float e[MB_RSTRIDE];
      mb_render_prim<Env>(S, P, rec, i, e);
      for (int k = 0; k < MB_RSTRIDE; ++k) out[(size_t)i * MB_RSTRIDE + k] = e[k];
    }
  MB_END
}

// pass 1 for an id outside the batch: no primitive at all (a blank frame)
MB_HD void mb_render_blank(float* out, int nprim) {
  MB_LANES(l)
    for (int i = l; i < nprim; i += 32) mb_render_empty(out + (size_t)i * MB_RSTRIDE);
  MB_END
}

// ------------------------------------------------------------------------------------------------ pass 2
// A camera: inverse of proj * view (column-major OpenGL matrices, as pybullet.computeViewMatrix /
// computeProjectionMatrixFOV return them), inverted in double precision, and the view matrix's third row (eye-space z).
struct MbCamera {
  double inv[16];  // column-major (proj * view)^-1
  double vz[4];    // eye z = vz . (x, y, z, 1)
  int ok;          // 0: singular or non-finite matrices (the frame is blank, depth NaN)
};

MB_HD void mb_render_camera(const float* view, const float* proj, MbCamera* cam) {
  double m[16];
  for (int c = 0; c < 4; ++c)
    for (int r = 0; r < 4; ++r) {
      double s = 0.0;
      for (int k = 0; k < 4; ++k) s += (double)proj[4 * k + r] * (double)view[4 * c + k];
      m[4 * c + r] = s;
    }
  for (int k = 0; k < 4; ++k) cam->vz[k] = (double)view[4 * k + 2];
  // Gauss-Jordan with partial pivoting on [m | I] (column-major m[4 * c + r])
  double a[4][8];
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 8; ++c) a[r][c] = c < 4 ? m[4 * c + r] : (c - 4 == r ? 1.0 : 0.0);
  bool ok = true;
  for (int c = 0; c < 4; ++c) {
    int p = c;
    for (int r = c + 1; r < 4; ++r)
      if (fabs(a[r][c]) > fabs(a[p][c])) p = r;
    if (!(fabs(a[p][c]) > 1e-300)) { ok = false; break; }
    if (p != c)
      for (int k = 0; k < 8; ++k) { const double t = a[c][k]; a[c][k] = a[p][k]; a[p][k] = t; }
    const double iv = 1.0 / a[c][c];
    for (int k = 0; k < 8; ++k) a[c][k] *= iv;
    for (int r = 0; r < 4; ++r)
      if (r != c) {
        const double f = a[r][c];
        for (int k = 0; k < 8; ++k) a[r][k] -= f * a[c][k];
      }
  }
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) {
      cam->inv[4 * c + r] = a[r][4 + c];
      ok = ok && fabs(a[r][4 + c]) <= 1.7e308 && fabs(cam->vz[c]) <= 1.7e308;
    }
  cam->ok = ok ? 1 : 0;
}

#define MB_RENDER_SKY_R 178
#define MB_RENDER_SKY_G 204
#define MB_RENDER_SKY_B 230
#define MB_RENDER_AMBIENT 0.35f

// base colour of a class (ground: the two checkerboard tiles)
MB_HD void mb_render_color(int cls, int tile, float* c) {
  switch (cls) {
    case MB_RC_ROBOT: c[0] = 0.90f; c[1] = 0.55f; c[2] = 0.25f; break;
    case MB_RC_GROUND:
      if (tile) { c[0] = 0.36f; c[1] = 0.40f; c[2] = 0.36f; } else { c[0] = 0.60f; c[1] = 0.64f; c[2] = 0.60f; }
      break;
    case MB_RC_PLANK: c[0] = 0.45f; c[1] = 0.60f; c[2] = 0.85f; break;
    case MB_RC_BAR: c[0] = 0.80f; c[1] = 0.75f; c[2] = 0.30f; break;
    default: c[0] = 0.90f; c[1] = 0.15f; c[2] = 0.15f; break;
  }
}

// Ray-primitive tests.  The ray is o + t d, |d| = 1, o near the primitive (mb_render_pixel moves it to the entry of
// the bounding sphere, so no test subtracts two large numbers).  A hit is an entry through the outside of the
// primitive at t > 0; each returns t (or -1) and the outward normal at the hit.
MB_HD float mb_ray_sphere(const float* o, const float* d, const float* c, float r, float* n) {
  const float oc[3] = {o[0] - c[0], o[1] - c[1], o[2] - c[2]};
  const float b = mb_dot3(oc, d);
  const float q[3] = {oc[0] - b * d[0], oc[1] - b * d[1], oc[2] - b * d[2]};
  const float h = r * r - mb_dot3(q, q);
  if (h < 0.0f) return -1.0f;
  const float t = -b - sqrtf(h);
  if (!(t > 0.0f)) return -1.0f;
  for (int k = 0; k < 3; ++k) n[k] = (oc[k] + t * d[k]) / r;
  return t;
}

MB_HD float mb_ray_capsule(const float* o, const float* d, const float* pa, const float* pb, float r, float* n) {
  const float ba[3] = {pb[0] - pa[0], pb[1] - pa[1], pb[2] - pa[2]};
  const float oa[3] = {o[0] - pa[0], o[1] - pa[1], o[2] - pa[2]};
  const float baba = mb_dot3(ba, ba), bard = mb_dot3(ba, d), baoa = mb_dot3(ba, oa);
  float best = -1.0f;
  const float a = baba - bard * bard;
  if (a > 1e-12f * baba) {  // the side: |(oa + t d) x ba|^2 = r^2 |ba|^2, written without cancellation
    float w[3], v[3];
    mb_cross(oa, ba, w);
    mb_cross(d, ba, v);
    const float B = mb_dot3(v, w), Cc = mb_dot3(w, w) - r * r * baba;
    const float h = B * B - a * Cc;
    if (h >= 0.0f) {
      const float t = (-B - sqrtf(h)) / a;
      const float y = baoa + t * bard;
      if (t > 0.0f && y > 0.0f && y < baba) {
        const float s = y / baba;
        for (int k = 0; k < 3; ++k) n[k] = (oa[k] + t * d[k] - s * ba[k]) / r;
        return t;
      }
    }
  }
  // the end spheres
  float n2[3];
  const float ta = mb_ray_sphere(o, d, pa, r, n);
  const float tb = mb_ray_sphere(o, d, pb, r, n2);
  best = ta;
  if (tb > 0.0f && (best < 0.0f || tb < best)) {
    best = tb;
    n[0] = n2[0]; n[1] = n2[1]; n[2] = n2[2];
  }
  return best;
}

// slabs in the box frame (R columns = box axes, c = centre, h = half extents)
MB_HD float mb_ray_box(const float* o, const float* d, const float* R, const float* c, const float* h, float* n) {
  const float w[3] = {o[0] - c[0], o[1] - c[1], o[2] - c[2]};
  float tn = -3.0e38f, tf = 3.0e38f;
  int ax = -1;
  float sg = 0.0f;
  for (int k = 0; k < 3; ++k) {
    const float ol = R[k] * w[0] + R[3 + k] * w[1] + R[6 + k] * w[2];
    const float dl = R[k] * d[0] + R[3 + k] * d[1] + R[6 + k] * d[2];
    if (fabsf(dl) < 1e-20f) {
      if (fabsf(ol) > h[k]) return -1.0f;
      continue;
    }
    const float inv = 1.0f / dl;
    float t1 = (-h[k] - ol) * inv, t2 = (h[k] - ol) * inv;
    if (t1 > t2) { const float t = t1; t1 = t2; t2 = t; }
    if (t1 > tn) { tn = t1; ax = k; sg = dl > 0.0f ? -1.0f : 1.0f; }
    if (t2 < tf) tf = t2;
  }
  if (ax < 0 || !(tn <= tf) || !(tn > 0.0f)) return -1.0f;
  for (int k = 0; k < 3; ++k) n[k] = sg * R[3 * k + ax];
  return tn;
}

// capped cylinder about the local z axis (R column 2), radius rad, half height hh
MB_HD float mb_ray_cyl(const float* o, const float* d, const float* R, const float* c, float rad, float hh, float* n) {
  const float w[3] = {o[0] - c[0], o[1] - c[1], o[2] - c[2]};
  float ol[3], dl[3];
  for (int k = 0; k < 3; ++k) {
    ol[k] = R[k] * w[0] + R[3 + k] * w[1] + R[6 + k] * w[2];
    dl[k] = R[k] * d[0] + R[3 + k] * d[1] + R[6 + k] * d[2];
  }
  float best = -1.0f, nl[3] = {0.0f, 0.0f, 0.0f};
  const float a = dl[0] * dl[0] + dl[1] * dl[1];
  if (a > 1e-20f) {  // side
    const float b = ol[0] * dl[0] + ol[1] * dl[1];
    // closest approach to the axis, then back off: no cancellation of two large squares
    const float s = -b / a;
    const float qx = ol[0] + s * dl[0], qy = ol[1] + s * dl[1];
    const float h = rad * rad - (qx * qx + qy * qy);
    if (h >= 0.0f) {
      const float t = s - sqrtf(h / a);
      const float z = ol[2] + t * dl[2];
      if (t > 0.0f && fabsf(z) <= hh) {
        best = t;
        nl[0] = (ol[0] + t * dl[0]) / rad; nl[1] = (ol[1] + t * dl[1]) / rad; nl[2] = 0.0f;
      }
    }
  }
  if (fabsf(dl[2]) > 1e-20f) {  // the cap that faces the ray
    const float zc = dl[2] > 0.0f ? -hh : hh;
    const float t = (zc - ol[2]) / dl[2];
    const float x = ol[0] + t * dl[0], y = ol[1] + t * dl[1];
    if (t > 0.0f && x * x + y * y <= rad * rad && (best < 0.0f || t < best)) {
      best = t;
      nl[0] = 0.0f; nl[1] = 0.0f; nl[2] = dl[2] > 0.0f ? -1.0f : 1.0f;
    }
  }
  if (best > 0.0f) mb_matvec(R, nl, n);
  return best;
}

// convex polytope: planes (n, dd) in the frame (R, c), n . x <= dd inside; Cyrus-Beck clipping
MB_HD float mb_ray_hull(const float* o, const float* d, const float* R, const float* c, const float* planes, int np,
                        float* n) {
  const float w[3] = {o[0] - c[0], o[1] - c[1], o[2] - c[2]};
  float ol[3], dl[3];
  for (int k = 0; k < 3; ++k) {
    ol[k] = R[k] * w[0] + R[3 + k] * w[1] + R[6 + k] * w[2];
    dl[k] = R[k] * d[0] + R[3 + k] * d[1] + R[6 + k] * d[2];
  }
  float tn = -3.0e38f, tf = 3.0e38f;
  int face = -1;
  for (int p = 0; p < np; ++p) {
    const float* pl = planes + 4 * p;
    const float den = pl[0] * dl[0] + pl[1] * dl[1] + pl[2] * dl[2];
    const float dist = pl[3] - (pl[0] * ol[0] + pl[1] * ol[1] + pl[2] * ol[2]);  // > 0 inside
    if (den == 0.0f) {
      if (dist < 0.0f) return -1.0f;
    } else if (den < 0.0f) {  // entering
      const float t = dist / den;
      if (t > tn) { tn = t; face = p; }
    } else {
      const float t = dist / den;
      if (t < tf) tf = t;
    }
    if (tn > tf) return -1.0f;
  }
  if (face < 0 || !(tn > 0.0f)) return -1.0f;
  mb_matvec(R, planes + 4 * face, n);
  return tn;
}

// one pixel of one camera: `prims` = the camera's nprim records (pass 1)
MB_HD void mb_render_pixel(const MbCamera& cam, const float* prims, int nprim, int W, int H, int row, int col,
                           uint8_t* rgb, float* depth, int* seg) {
  if (!cam.ok) {
    if (rgb) { rgb[0] = MB_RENDER_SKY_R; rgb[1] = MB_RENDER_SKY_G; rgb[2] = MB_RENDER_SKY_B; }
    if (depth) *depth = NAN;
    if (seg) *seg = MB_SEG_SKY;
    return;
  }
  // the pixel's ray from the near plane (NDC z = -1) to the far plane (z = +1), in double
  const double x = 2.0 * (col + 0.5) / W - 1.0, y = 1.0 - 2.0 * (row + 0.5) / H;
  double pn[4], pf[4];
  for (int r = 0; r < 4; ++r) {
    const double b = cam.inv[r] * x + cam.inv[4 + r] * y + cam.inv[12 + r];
    pn[r] = b - cam.inv[8 + r];
    pf[r] = b + cam.inv[8 + r];
  }
  for (int r = 0; r < 3; ++r) { pn[r] /= pn[3]; pf[r] /= pf[3]; }
  const double dd[3] = {pf[0] - pn[0], pf[1] - pn[1], pf[2] - pn[2]};
  const double len = sqrt(dd[0] * dd[0] + dd[1] * dd[1] + dd[2] * dd[2]);
  const double zn = -(cam.vz[0] * pn[0] + cam.vz[1] * pn[1] + cam.vz[2] * pn[2] + cam.vz[3]);
  const double zf = -(cam.vz[0] * pf[0] + cam.vz[1] * pf[1] + cam.vz[2] * pf[2] + cam.vz[3]);
  const float o[3] = {(float)pn[0], (float)pn[1], (float)pn[2]};
  const float d[3] = {(float)(dd[0] / len), (float)(dd[1] / len), (float)(dd[2] / len)};
  const float tmax = (float)len;
  float best = tmax, nb[3] = {0.0f, 0.0f, 1.0f};
  int hit = -1;
  for (int i = 0; i < nprim; ++i) {
    const float* e = prims + (size_t)i * MB_RSTRIDE;
    const int ty = mb_fbits(e[4]);
    float t = -1.0f, n[3];
    if (ty == MB_RP_PLANE) {
      if (d[2] != 0.0f) {
        t = -o[2] / d[2];
        n[0] = 0.0f; n[1] = 0.0f; n[2] = o[2] >= 0.0f ? 1.0f : -1.0f;
      }
    } else if (ty != MB_RP_NONE) {
      // bounding sphere: skip what the ray misses or what lies behind the best hit so far
      const float oc[3] = {e[0] - o[0], e[1] - o[1], e[2] - o[2]};
      const float s = mb_dot3(oc, d);
      const float q[3] = {oc[0] - s * d[0], oc[1] - s * d[1], oc[2] - s * d[2]};
      const float rb = e[3] * 1.001f + 1e-5f;
      if (mb_dot3(q, q) > rb * rb || s + rb <= 0.0f || s - rb >= best) continue;
      // move the origin to the entry of the bounding sphere
      const float s0 = fmaxf(s - rb, 0.0f);
      const float os[3] = {o[0] + s0 * d[0], o[1] + s0 * d[1], o[2] + s0 * d[2]};
      if (ty == MB_RP_SPHERE) t = mb_ray_sphere(os, d, e + 17, e[23], n);
      else if (ty == MB_RP_CAPSULE) t = mb_ray_capsule(os, d, e + 17, e + 8, e[23], n);
      else if (ty == MB_RP_BOX) t = mb_ray_box(os, d, e + 8, e + 17, e + 20, n);
      else if (ty == MB_RP_CYL) t = mb_ray_cyl(os, d, e + 8, e + 17, e[20], e[21], n);
      else {
        const float* planes;
        memcpy(&planes, e + 20, sizeof(planes));
        t = mb_ray_hull(os, d, e + 8, e + 17, planes, mb_fbits(e[7]), n);
      }
      if (t > 0.0f) t += s0;
    }
    if (t > 0.0f && t < best) {
      best = t;
      hit = i;
      nb[0] = n[0]; nb[1] = n[1]; nb[2] = n[2];
    }
  }
  if (hit < 0) {
    if (rgb) { rgb[0] = MB_RENDER_SKY_R; rgb[1] = MB_RENDER_SKY_G; rgb[2] = MB_RENDER_SKY_B; }
    if (depth) *depth = (float)zf;
    if (seg) *seg = MB_SEG_SKY;
    return;
  }
  const float* e = prims + (size_t)hit * MB_RSTRIDE;
  if (depth) *depth = (float)(zn + (double)best * ((zf - zn) / len));
  if (seg) *seg = mb_fbits(e[5]);
  if (rgb) {
    const int cls = mb_fbits(e[6]);
    int tile = 0;
    if (cls == MB_RC_GROUND) {
      const float px = o[0] + best * d[0], py = o[1] + best * d[1];
      tile = ((int)floorf(px) + (int)floorf(py)) & 1;
    }
    float c[3];
    mb_render_color(cls, tile, c);
    // one fixed directional light (unit vector towards the light) plus ambient
    const float L[3] = {0.40f, 0.30f, 0.8660254f};
    const float s = mb_dot3(nb, d) > 0.0f ? -1.0f : 1.0f;  // the side the ray sees
    const float lam = fmaxf(s * mb_dot3(nb, L), 0.0f);
    const float k = MB_RENDER_AMBIENT + (1.0f - MB_RENDER_AMBIENT) * lam;
    for (int j = 0; j < 3; ++j) rgb[j] = (uint8_t)(fminf(c[j] * k, 1.0f) * 255.0f + 0.5f);
  }
}
