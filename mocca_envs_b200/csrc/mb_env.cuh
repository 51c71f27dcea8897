// mb_env.cuh -- env layer fused around the simulator core: action -> torque, frame_skip substeps,
// observation / reward / termination, gym TimeLimit, auto-reset with NumPy-compatible MT19937 streams.
//
// Restates (per environment, one warp each):
//   WalkerBase.apply_action / calc_state / reset      reference mocca_envs/robots.py:31-95,179-227
//   Walker3DCustomEnv.reset/step/calc_*               reference mocca_envs/env_locomotion.py:67-222
//   gym TimeLimit(max_episode_steps=1000)             reference mocca_envs/__init__.py:52-56
#pragma once
#include "mb_core.cuh"

// ---- HBM record layout (array-of-records: one warp streams its env's record with coalesced 128 B lines) ----
#define MB_STATE_STRIDE 64 /* floats: pos3 quat4 omega3 vel3 q[NJ] qd[NJ] */
#define MB_REC_STRIDE 32   /* floats/ints, see ER_* (Walker3DCustomEnv) */
#define MB_REC_STRIDE_STEPPER 192 /* ER_* + ES_* (Walker3DStepperEnv) */
#define MB_MT_STRIDE 640   /* uint32: 624 state words + [624] position */
enum {
  ER_TX = 0, ER_TY, ER_TZ,      // walk_target
  ER_DIST, ER_ANGLE, ER_STOP,   // randomize_target() draws
  ER_CLOSE,                     // close_count (int)
  ER_LINPOT,                    // linear_potential
  ER_ELAPSED,                   // TimeLimit counter (int)
  ER_FEET0, ER_FEET1,           // feet_contact
  ER_ALIASED,                   // robot RNG still aliased to env RNG (int)  -- env_base.py:93 quirk Q1
  ER_EPRET, ER_EPLEN,           // running episode return / length (float, int)
  ER_MIRRORED,                  // robots.py:182-188 (int)
  ER_ROWS,                      // diagnostics: constraint rows accumulated (float)
  ER_CONTACTS,                  // diagnostics: contact points accumulated (float)
  ER_BODYX,                     // body_xyz[0] of the previous calc_state (eval mode, env_locomotion.py:115-116)
  ER_EVAL,                      // eval_mode (int)
  ER_LAST_EPRET, ER_LAST_EPLEN, // return / length of the last finished episode
  ER_OVERFLOW,                  // contact/row cap hits (int)
};

enum {  // CassieEnv additions (env_cassie.py:285-479)
  EC_POTENTIAL = 22,  // potential = -distance / control_step (kept for inspection; f32 ulp at -33333 is 4e-3)
  EC_PREVX, EC_PREVY, // body x, y at the previous calc_potential: the progress reward is formed from exact differences
  EC_JVEL = 32,       // [14] low-pass joint velocity of the ordered joints (env_cassie.py:319,451-453,467-468)
};
#define MB_REC_STRIDE_CASSIE 64

enum {  // Monkey3DCustomEnv additions (env_locomotion.py:1136-1516)
  EM_NEXT = 22,      // next_step_index (int)
  EM_FREEFALL,       // free_fall_count (int)
  EM_TIMESTEP,       // timestep (int)
  EM_SWING,          // swing_leg (int)
  EM_PIVOT,          // pivot_leg (int)
  EM_SWINGPOT,       // swing_potential
  EM_BARIDX,         // [4] terrain row shown by each physical bar (int)
  EM_BAR = 32,       // [4][8] bar centre, unit axis, half length, radius
  EM_TERRAIN = 64,   // [32][4] x y z phi
};
#define MB_REC_STRIDE_MONKEY 192

enum {  // Walker3DStepperEnv additions (env_locomotion.py:330-840)
  ES_NEXT = 22,       // next_step_index (int)
  ES_COUNT,           // target_reached_count (int)
  ES_STOP,            // stop_on_next_step (int)
  ES_SETSTOP,         // set_stop_on_next_step (int)
  ES_TIMESTEP,        // timestep (int)
  ES_CURRIC,          // curriculum 0..9 (int)
  ES_PLANKIDX,        // [3] terrain row shown by each physical plank (int)
  ES_STEPS_REACHED = 31,  // info["steps_reached"] of the last step, -1 = not reported (int)
  ES_GAIN_CURRIC = 6,     // curriculum the applied_gain was taken from at reset (env_locomotion.py:489) (int)
  ES_PLANK_CLASS = 4,     // plank_class kwarg (env_locomotion.py:342,356-357): 0 LargePlank, 1 Plank, 2 Pillar (the
                          // library launches the PILLAR instantiation for 2) (int; ER_ANGLE unused here)
  ES_RANDOM_REWARD = 3,   // random_reward kwarg (env_locomotion.py:355,528-547) (int; ER_DIST is unused by this env)
  ES_BOX = 32,        // [3][12] plank base-box centre + axes
  ES_TERRAIN = 68,    // [20][6] x y z phi x_tilt y_tilt
};

// ---- physics parameters (host): the reference's Bullet world.  P is mb200_physics (include/mocca_b200.h) or
// MbPhysics, which carries the same public fields.
template <class P> inline void mb_default_physics(P* p) {
  p->dt = 1.0f / 240.0f; p->substeps = 4; p->iterations = 5; p->gravity = 9.8f; p->erp_contact = 0.9f;
  p->erp_joint = 0.2f; p->linear_slop = 1e-5f; p->lin_damping = 0.04f; p->ang_damping = 0.04f;
  p->max_coord_vel = 100.0f; p->limit_max_impulse = 100.0f; p->split_threshold = -0.04f;
  p->residual_threshold = 1e-7f; p->ground_friction = 0.8f; p->has_ground = 1; p->self_collision = 1;
  p->warmstart = 0.0f;
}
// public parameters -> the solver's; the obstacle contacts start out like the ground's (an env's fix_physics may
// change them)
template <class P> inline void mb_to_internal(const P& p, MbPhysics* q) {
  q->dt = p.dt; q->substeps = p.substeps; q->iterations = p.iterations; q->gravity = p.gravity;
  q->erp_contact = p.erp_contact; q->erp_joint = p.erp_joint; q->linear_slop = p.linear_slop;
  q->lin_damping = p.lin_damping; q->ang_damping = p.ang_damping; q->max_coord_vel = p.max_coord_vel;
  q->limit_max_impulse = p.limit_max_impulse; q->split_threshold = p.split_threshold;
  q->residual_threshold = p.residual_threshold; q->ground_friction = p.ground_friction; q->has_ground = p.has_ground;
  q->box_friction = 1.0f; q->box_erp = p.erp_contact; q->box_cfm = 0.0f; q->bar_friction = 0.5f;
  q->self_collision = p.self_collision;
  q->warmstart = p.warmstart > 0.0f ? p.warmstart : 0.0f;
}

// A key mb200_set_param accepts for an env (Env::PARAMS, ended by a null key): the int record field it sets to
// (int)value for every env.
struct MbParam {
  const char* key;
  int field;
  bool boolean;                                // the scalar setter stores value != 0
  const char* (*check)(float v, float first);  // error for value v of a batch whose first value is `first`, or null
  const char* (*variant)(float first);         // the kernel variant ("" / "pillar") the batch's values select, or null
};

struct MbStats {  // per-device accumulators, all-reduced across ranks by the host (NCCL) when asked
  unsigned long long episodes;
  unsigned long long steps_reached_sum;  // info["steps_reached"] summed over finished episodes (Stepper, Monkey)
  unsigned long long nonfinite;
  unsigned long long overflow;
  double ret_sum;
  double len_sum;
};

// one warp per env adds to the per-device statistics; the CPU emulation runs one env at a time
MB_HD void mb_stat_add(unsigned long long* s, unsigned long long v) {
#ifdef __CUDACC__
  atomicAdd(s, v);
#else
  *s += v;
#endif
}
MB_HD void mb_stat_add(double* s, double v) {
#ifdef __CUDACC__
  atomicAdd(s, v);
#else
  *s += v;
#endif
}

// warm-start impulses of an env (HBM, MbPhysics::warmstart > 0): zeroed at every reset
MB_HD void mb_clear_warm(float* warm) {
  if (MB_UNLIKELY(warm != nullptr)) {
    MB_LANES(l)
      for (int i = l; i < MB_NWARM; i += 32) warm[i] = 0.0f;
    MB_END
  }
}

MB_HD int& rec_i(float* rec, int k) { return reinterpret_cast<int*>(rec)[k]; }
MB_HD int rec_i(const float* rec, int k) { return reinterpret_cast<const int*>(rec)[k]; }

// The end of every env's step(), after the env has written obs, its own record fields and its reward: gym
// TimeLimit(1000), the episode / diagnostics record, reward / done / truncated, the terminal observation, the episode
// statistics and the auto-reset (VecEnv convention: on done obs becomes the first observation of the next episode).
// Per-env differences are compile-time properties of Env: CREDIT_STEPS_REACHED adds `steps_reached` to
// MbStats::steps_reached_sum at an episode end, and the record's INFO_FIELD (if any) keeps the finished episode's
// value across the reset.  nonfinite: the state went non-finite (it ended the episode); anybad: non-finite actions.
template <class Env>
MB_HD void mb_step_epilogue(typename Env::Mem& S, const MbPhysics& P, float* rec, uint32_t* mt_env, uint32_t* mt_robot,
                            float* obs, float reward, int env_done, int nonfinite, int steps_reached, int rows,
                            int ncsum, int overflow, unsigned anybad, float* rew, uint8_t* done, uint8_t* trunc,
                            float* final_obs, MbStats* stats) {
  const int elapsed = rec_i(rec, ER_ELAPSED) + 1;
  int truncated = 0, any_done = env_done;
  if (elapsed >= 1000) { truncated = !env_done; any_done = 1; }
  const float epret = rec[ER_EPRET] + reward;
  const int eplen = rec_i(rec, ER_EPLEN) + 1;
  MB_LANES(l)
    if (l == 0) {
      rec_i(rec, ER_ELAPSED) = elapsed;
      rec[ER_EPRET] = epret; rec_i(rec, ER_EPLEN) = eplen;
      rec[ER_ROWS] += (float)rows; rec[ER_CONTACTS] += (float)ncsum; S.step_rows = rows;
      if (MB_UNLIKELY(overflow > 0)) {  // contacts / rows dropped at MB_MAXC / MB_MAXROW: per env and per device
        rec_i(rec, ER_OVERFLOW) += overflow;
        mb_stat_add(&stats->overflow, (unsigned long long)overflow);
      }
      *rew = reward; *done = (uint8_t)any_done; *trunc = (uint8_t)truncated;
    }
  MB_END
  if (any_done) {
    if (final_obs) {
      MB_LANES(l)
        for (int i = l; i < Env::OBS; i += 32) final_obs[i] = obs[i];
      MB_END
    }
    MB_LANES(l)
      if (l == 0) {
        rec[ER_LAST_EPRET] = epret; rec_i(rec, ER_LAST_EPLEN) = eplen;
        mb_stat_add(&stats->episodes, 1ull);
        mb_stat_add(&stats->ret_sum, (double)epret);
        mb_stat_add(&stats->len_sum, (double)eplen);
        if constexpr (Env::CREDIT_STEPS_REACHED)
          mb_stat_add(&stats->steps_reached_sum, (unsigned long long)steps_reached);
        if (nonfinite) mb_stat_add(&stats->nonfinite, 1ull);
      }
    MB_END
    if constexpr (Env::INFO_FIELD >= 0) {
      const int keep = rec_i(rec, Env::INFO_FIELD);
      Env::reset(S, P, rec, mt_env, mt_robot, obs);
      MB_LANES(l)
        if (l == 0) rec_i(rec, Env::INFO_FIELD) = keep;  // info of the finished episode stays readable
      MB_END
    } else {
      Env::reset(S, P, rec, mt_env, mt_robot, obs);
    }
  }
  if (anybad) {
    MB_LANES(l)
      if (l == 0) mb_stat_add(&stats->nonfinite, 1ull);
    MB_END
  }
}

// One stepSimulation of an env: the joint torques tau (nullptr = zero) held over the substeps, the static obstacles of
// its record.  `points` (nullptr = off) receives the contact points of the last collision pass (what getContactPoints
// reports after stepSimulation).  Returns the constraint rows; *contacts = the contacts of the last pass.
template <class Env>
MB_HD int mb_physics_step(typename Env::Mem& S, const MbPhysics& P, float* state, const float* rec, const float* tau,
                          float* points, int* contacts) {
  typedef typename Env::Model M;
  Env::load_state(S, state);
  MB_LANES(l)
    if (l < M::NJ) S.tau[l] = tau ? tau[l] : 0.0f;
  MB_END
  int rows = 0, nc = 0, overflow = 0;
  typename Sim<M>::LaneConst C;
  Sim<M>::init_lane_const(C);
#pragma unroll 1
  for (int k = 0; k < P.substeps; ++k) {
    Env::load_obstacles(S, rec);
    rows += Sim<M>::template substep<Env::OBST>(S, P, C, &nc, &overflow, k,
                                                points && k == P.substeps - 1 ? points : nullptr);
  }
  Env::store_state(S, state);
  *contacts = nc;
  return rows;
}

// The mass matrix (S.L, read with mb_Lget) and S.rhs = -bias with zero applied torque, at `state`
template <class Env> MB_HD void mb_mass_matrix(typename Env::Mem& S, const MbPhysics& P, const float* state) {
  typedef typename Env::Model M;
  Env::load_state(S, state);
  MB_LANES(l)
    S.tau[l] = 0.0f;
  MB_END
  typename Sim<M>::LaneConst C;
  Sim<M>::init_lane_const(C);
  Sim<M>::kinematics(S, P, C, true);
  Sim<M>::bodies(S, P);
  Sim<M>::mass_matrix_and_rhs(S);
}

// z -= Y_G (Y_G^T Y_G)^-1 Y_G^T z: the part of the push in z = L du space that would open a loop closure is removed, so
// that G du = Y_G^T z = 0 afterwards.  g[i] is loop multiplier i's row Y = L^-T G_i^T, lane-indexed (the sum of its two
// compact parts).  Y_G^T Y_G = G M^-1 G^T exactly, coupling term included (Bullet's PGS denominator drops it; this
// projection is not a PGS row and needs the exact Gram matrix).  Every lane holds the 6x6 system and solves it alike.
template <int NG>
MB_HD void mb_project_loops(const LaneVar<float>* g, LaneVar<float>& z) {
  float A[NG][NG], b[NG];
#pragma unroll
  for (int i = 0; i < NG; ++i) {
    LaneVar<float> t;
#pragma unroll
    for (int j = 0; j <= i; ++j) {
      MB_LANES(l)
        t[l] = g[i][l] * g[j][l];
      MB_END_REG
      A[i][j] = warp_sum(t);
    }
    MB_LANES(l)
      t[l] = g[i][l] * z[l];
    MB_END_REG
    b[i] = warp_sum(t);
  }
  // Cholesky A = R R^T in place (lower triangle), then R R^T lambda = b
#pragma unroll
  for (int k = 0; k < NG; ++k) {
    float d = A[k][k];
#pragma unroll
    for (int s = 0; s < k; ++s) d -= A[k][s] * A[k][s];
    const float rinv = d > 0.0f ? 1.0f / sqrtf(d) : 0.0f;  // (a degenerate loop row takes no multiplier)
    A[k][k] = rinv;
#pragma unroll
    for (int i = k + 1; i < NG; ++i) {
      float v = A[i][k];
#pragma unroll
      for (int s = 0; s < k; ++s) v -= A[i][s] * A[k][s];
      A[i][k] = v * rinv;
    }
  }
#pragma unroll
  for (int i = 0; i < NG; ++i) {
#pragma unroll
    for (int s = 0; s < i; ++s) b[i] -= A[i][s] * b[s];
    b[i] *= A[i][i];
  }
#pragma unroll
  for (int i = NG - 1; i >= 0; --i) {
#pragma unroll
    for (int s = i + 1; s < NG; ++s) b[i] -= A[s][i] * b[s];
    b[i] *= A[i][i];
  }
  MB_LANES(l)
#pragma unroll
    for (int i = 0; i < NG; ++i) z[l] = fmaf(-b[i], g[i][l], z[l]);
  MB_END_REG
}

// An instantaneous linear impulse (N s, world frame) at the world point `point` rigidly attached to `link` (-1 = the
// base, j = the movable frame of dof j), between two env steps:  du = M(q)^-1 J(point)^T impulse, u = [omega_w, v_w, qd],
// clamped to +-max_coord_vel like every velocity update of a substep.  Cassie's loop closures are kept closed
// (du = M^-1 (J^T impulse - G^T lambda) with G du = 0, mb_project_loops).  Planar models push with the y components of
// impulse and point set to zero: what their slide-x / slide-z / hinge-y root transmits.  Positions, q and everything
// outside `state` are untouched; so is the whole env for a link outside [-1, NJ), a zero impulse or a non-finite input.
// The push is one synthetic contact-normal row through row_build: its Y = L^-T J^T is the push itself in z space.
template <class Env>
MB_HD void mb_apply_impulse(typename Env::Mem& S, const MbPhysics& P, float* state, int link, const float* point,
                            const float* impulse) {
  typedef typename Env::Model M;
  typedef Sim<M> Q;
  float iv[3] = {impulse[0], impulse[1], impulse[2]}, pv[3] = {point[0], point[1], point[2]};
  if (M::planar_env()) { iv[1] = 0.0f; pv[1] = 0.0f; }
  const float mag = sqrtf(mb_dot3(iv, iv));
  bool ok = link >= -1 && link < M::NJ && mag > 0.0f && mb_finite(mag);
  for (int k = 0; k < 3; ++k) ok = ok && mb_finite(pv[k]);
  if (!ok) return;
  Env::load_state(S, state);
  MB_LANES(l)
    S.tau[l] = 0.0f;
  MB_END
  typename Q::LaneConst C;
  Q::init_lane_const(C);
  Q::kinematics(S, P, C, true);
  Q::loop_pivots(S);  // (reads jR / jp: the rows below overwrite them)
  Q::bodies(S, P);
  Q::mass_matrix_and_rhs(S);
  Q::template factorize<false>(S, C);
  MB_LANES(l)
    if (l == 0) {
      const float inv = 1.0f / mag;
      for (int k = 0; k < 3; ++k) { S.cP[0][k] = pv[k] - S.pos[k]; S.cn[0][k] = iv[k] * inv; }
      S.cdist[0] = 0.0f; S.cmu[0] = 0.0f; S.cerp[0] = 0.0f; S.ccfm[0] = 0.0f;
      S.clink[0] = link; S.cfoot[0] = 0; S.cpartner[0] = 0;
    }
  MB_END
  // rows: the loop closures [0, NLC) (no limit rows), then the push as contact slot 0
  MB_LANES(l)
    if (l <= Q::NLC) Q::row_build(S, P, 0, 1, 0, l);
  MB_END
  LaneVar<float> z;
  const unsigned sup = S.rc.r.r_mask[Q::NLC] & MB_ROW_SUP;
  MB_LANES(l)
    z[l] = ((sup >> l) & 1u) ? S.w.Yc[Q::NLC][C.tl[l]] * mag : 0.0f;
  MB_END_REG
  if constexpr (M::NLOOP > 0) {
    LaneVar<float> g[Q::NLC / 2];
#pragma unroll
    for (int i = 0; i < Q::NLC / 2; ++i) {
      const unsigned sa = S.rc.r.r_mask[2 * i] & MB_ROW_SUP, sb = S.rc.r.r_mask[2 * i + 1] & MB_ROW_SUP;
      MB_LANES(l)
        g[i][l] = (((sa >> l) & 1u) ? S.w.Yc[2 * i][C.tl[l]] : 0.0f) +
                  (((sb >> l) & 1u) ? S.w.Yc[2 * i + 1][C.tl[l]] : 0.0f);
      MB_END_REG
    }
    mb_project_loops<Q::NLC / 2>(g, z);
  }
  Q::template solve_L<false>(S, C, z);
  MB_LANES(l)
    if (l < M::NU) S.u[l] = fminf(fmaxf(S.u[l] + z[l], -P.max_coord_vel), P.max_coord_vel);
  MB_END
  Env::store_state(S, state);
}

// ------------------------------------------------------------------------------------------------ MT19937
// NumPy legacy RandomState stream, warp-cooperative.  mt[0..623] state words, mt[624] position.
MB_HD void mt_twist(uint32_t* mt) {
  for (int g = 0; g < 624; g += 32) {
    LaneVar<uint32_t> nv;
    MB_LANES(l)
      const int k = g + l;
      nv[l] = 0;
      if (k < 624) {
        const uint32_t y = (mt[k] & 0x80000000u) | (mt[(k + 1) % 624] & 0x7fffffffu);
        nv[l] = mt[(k + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
      }
    MB_END
    MB_LANES(l)
      const int k = g + l;
      if (k < 624) mt[k] = nv[l];
    MB_END
  }
}
MB_HD uint32_t mt_temper(uint32_t y) {
  y ^= (y >> 11);
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  y ^= (y >> 18);
  return y;
}
MB_HD void mt_fill(uint32_t* mt, uint32_t* out, int count) {
  int pos = (int)mt[624];
  int produced = 0;
  while (produced < count) {
    if (pos >= 624) { mt_twist(mt); pos = 0; }
    int take = 624 - pos;
    if (take > count - produced) take = count - produced;
    MB_LANES(l)
      for (int i = l; i < take; i += 32) out[produced + i] = mt_temper(mt[pos + i]);
    MB_END
    pos += take;
    produced += take;
  }
  MB_LANES(l)
    if (l == 0) mt[624] = (uint32_t)pos;
  MB_END
}
// RandomState.random_sample(): 53-bit double from two 32-bit outputs (SURVEY App. A.6)
MB_HD double mt_double(const uint32_t* w) { return ((double)(w[0] >> 5) * 67108864.0 + (double)(w[1] >> 6)) / 9007199254740992.0; }

// ------------------------------------------------------------------------------------------------ Walker3DCustom
struct W3DObsScalars {
  float height, vx, vy, vz, roll, pitch, yaw;
  int joints_at_limit;
  int nonfinite;
};

// pybullet.getEulerFromQuaternion (reference bullet_utils.py:83-84)
MB_HD void mb_euler(const float* qin, float* rpy) {
  const float len = sqrtf(qin[0] * qin[0] + qin[1] * qin[1] + qin[2] * qin[2] + qin[3] * qin[3]);
  const float q0 = qin[0] / len, q1 = qin[1] / len, q2 = qin[2] / len, q3 = qin[3] / len;
  // (products that feed sums are rounded on their own / fused explicitly: left to the compiler, the contraction of
  // a * b + c * d came out differently in the device-buffer and the host-buffer instantiation of one step kernel)
  const float sqx = MB_FMUL(q0, q0), sqy = MB_FMUL(q1, q1), sqz = MB_FMUL(q2, q2), squ = MB_FMUL(q3, q3);
  const float sarg = -2.0f * fmaf(q0, q2, -MB_FMUL(q3, q1));
  if (sarg <= -0.99999f) { rpy[0] = 0; rpy[1] = -0.5f * MB_PI_F; rpy[2] = 2 * atan2f(q0, -q1); }
  else if (sarg >= 0.99999f) { rpy[0] = 0; rpy[1] = 0.5f * MB_PI_F; rpy[2] = 2 * atan2f(-q0, q1); }
  else {
    rpy[0] = atan2f(2 * fmaf(q1, q2, MB_FMUL(q3, q0)), squ - sqx - sqy + sqz);
    rpy[1] = asinf(sarg);
    rpy[2] = atan2f(2 * fmaf(q0, q1, MB_FMUL(q3, q2)), squ + sqx - sqy - sqz);
  }
}
MB_HD float mb_clip5(float x) { return fminf(fmaxf(x, -5.0f), 5.0f); }

// mirrored base pose (robots.py:182-188): joint j of a mirrored robot takes the base angle of joint *src times the
// returned sign (+-1)
template <class M> MB_HD float mb_mirror_joint(int j, int mirrored, int* src) {
  *src = j;
  float sign = 1.0f;
  if (mirrored) {
    for (int k = 0; k < M::NMIRROR; ++k) {
      if (M::right(k) == j) *src = M::left(k);
      if (M::left(k) == j) *src = M::right(k);
    }
    for (int k = 0; k < M::NNEG; ++k)
      if (M::neg(k) == j) sign = -1.0f;
  }
  return sign;
}

// WalkerBase.reset pose of joint j (robots.py:182-194): the mirrored base angle plus +-0.1 rad noise from the robot
// words wr (wr[0..1] drew the mirror coin, joint j's uniform is wr[2 + 2 j]), clipped to +-0.95 normalised
template <class M> MB_HD float mb_reset_joint(int j, int mirrored, const uint32_t* wr) {
  int src;
  const float sign = mb_mirror_joint<M>(j, mirrored, &src);
  const double ang = sign * M::base_angles(src);
  const double ds = -0.1 + (0.1 - -0.1) * mt_double(wr + 2 + 2 * j);
  const double bias = (double)M::lower(j), weight = (double)M::weight(j);
  double ps = 2 * (ang + ds - bias) / weight - 1;
  ps = ps > 0.95 ? 0.95 : (ps < -0.95 ? -0.95 : ps);
  return (float)(weight * (ps + 1) / 2 + bias);
}

template <class M> struct W3DEnv {
  typedef WarpMem<M> Mem;
  typedef Sim<M> S_;
  typedef M Model;
  enum { NJ = M::NJ, NU = M::NU, OBS = 6 + 2 * M::NJ + M::NFEET + 2, ROBOT_OBS = 6 + 2 * M::NJ + M::NFEET,
         REC_STRIDE = MB_REC_STRIDE, OBST = 0, ACT = M::NJ, INFO_FIELD = -1, CREDIT_STEPS_REACHED = 0 };
  // the env's kind configuration (host): its own public physics defaults, what it fixes after the caller's
  // parameters, and the keys of mb200_set_param
  template <class P> static void default_physics(P&) {}
  static void fix_physics(MbPhysics&) {}
  static constexpr MbParam PARAMS[] = {{"eval_mode", ER_EVAL, true, nullptr, nullptr}, {}};
  MB_HD static void load_obstacles(WarpMem<M>&, const float*) {}

  // HBM <-> shared
  MB_HD static void load_state(Mem& S, const float* st) {
    MB_LANES(l)
      if (l == 0) { S.nbox = 0; S.nbar = 0; }
      for (int i = l; i < 13 + 2 * NJ; i += 32) {
        const float v = st[i];
        if (i < 3) S.pos[i] = v;
        else if (i < 7) S.quat[i - 3] = v;
        else if (i < 13) S.u[i - 7] = v;
        else if (i < 13 + NJ) S.q[i - 13] = v;
        else S.u[6 + i - 13 - NJ] = v;
      }
    MB_END
  }
  MB_HD static void store_state(const Mem& S, float* st) {
    MB_LANES(l)
      for (int i = l; i < 13 + 2 * NJ; i += 32) {
        float v;
        if (i < 3) v = S.pos[i];
        else if (i < 7) v = S.quat[i - 3];
        else if (i < 13) v = S.u[i - 7];
        else if (i < 13 + NJ) v = S.q[i - 13];
        else v = S.u[6 + i - 13 - NJ];
        st[i] = v;
      }
    MB_END
  }

  // robots.py:42-95 calc_state: writes robot_state (clipped to +-5) into obs[0 .. ROBOT_OBS) and returns the
  // unclipped scalars the reward needs.  Requires kinematics(S, P, false) at the current pose.
  MB_HD static W3DObsScalars observe(Mem& S, const float* rec, float* obs, const LaneVar<float>& araw, float* s1,
                                     float* s2) {
    W3DObsScalars o;
    LaneVar<float> e1, e2;
    LaneVar<int> atl, bad;
    MB_LANES(l)
      e1[l] = 0.0f; e2[l] = 0.0f; atl[l] = 0; bad[l] = 0;
      if (l < NJ) {
        const float q = S.q[l], qd = S.u[6 + l];
        const float nrm = 2.0f * (q - M::lower(l)) / M::weight(l) - 1.0f;
        const float sp = 0.1f * qd;
        obs[6 + l] = mb_clip5(nrm);
        obs[6 + NJ + l] = mb_clip5(sp);
        atl[l] = fabsf(nrm) > 0.99f;
        bad[l] = !(mb_finite(nrm) && mb_finite(sp));
        const float a = araw[l];
        e1[l] = fabsf(a * sp);
        e2[l] = a * a;
      }
    MB_END
    o.joints_at_limit = mb_popc(warp_ballot(atl));
    *s1 = warp_sum(e1);
    *s2 = warp_sum(e2);
    float rpy[3];
    mb_euler(S.quat, rpy);
    o.roll = rpy[0]; o.pitch = rpy[1]; o.yaw = rpy[2];
    const float cy = cosf(-o.yaw), sy = sinf(-o.yaw);
    o.vx = cy * S.u[3] - sy * S.u[4];
    o.vy = sy * S.u[3] + cy * S.u[4];
    o.vz = S.u[5];
    float minz = 1e30f;
    for (int f = 0; f < M::NFEET; ++f) {
      const int b = M::foot_body(f), ow = M::bowner(b);
      const float* R = S.w.k.jR[ow];
      const float z = S.w.k.jp[ow][2] + R[6] * M::bcom(b, 0) + R[7] * M::bcom(b, 1) + R[8] * M::bcom(b, 2);
      minz = fminf(minz, z);
    }
    o.height = -minz;  // body_z - min(feet_z), both relative to the base COM
    o.nonfinite = warp_ballot(bad) != 0u ||
                  !(mb_finite(o.height) && mb_finite(o.vx) && mb_finite(o.vy) && mb_finite(o.vz) && mb_finite(o.roll) &&
                    mb_finite(o.pitch));
    MB_LANES(l)
      if (l == 0) {
        obs[0] = mb_clip5(o.height); obs[1] = mb_clip5(o.vx); obs[2] = mb_clip5(o.vy); obs[3] = mb_clip5(o.vz);
        obs[4] = mb_clip5(o.roll); obs[5] = mb_clip5(o.pitch);
        obs[6 + 2 * NJ] = rec[ER_FEET0];
        obs[6 + 2 * NJ + 1] = rec[ER_FEET1];
      }
    MB_END
    return o;
  }

  // env_locomotion.py:143-158
  MB_HD static void potential(const Mem& S, const float* rec, float yaw, float scene_dt, float* dist, float* ang,
                              float* linpot) {
    const float dx = rec[ER_TX] - S.pos[0], dy = rec[ER_TY] - S.pos[1];
    *ang = atan2f(dy, dx) - yaw;
    *dist = sqrtf(dx * dx + dy * dy);
    *linpot = -(*dist) / scene_dt;
  }
  MB_HD static void target_obs(float dist, float ang, float* obs) {  // env_locomotion.py:124-129
    const float s_ = dist * sinf(ang), c_ = dist * cosf(ang);
    MB_LANES(l)
      if (l == 0) {
        obs[ROBOT_OBS] = s_ / (1.0f + fabsf(s_));
        obs[ROBOT_OBS + 1] = c_ / (1.0f + fabsf(c_));
      }
    MB_END
  }

  // env_locomotion.py:67-74 -- consumes target_words() words of the env stream: two uniforms (2 words each) and the
  // choice (1 word); in eval mode the uniforms are not drawn and the choice is the first word
  MB_HD static int target_words(const float* rec) { return rec_i(rec, ER_EVAL) ? 1 : 5; }
  MB_HD static void randomize_target(float* rec, const uint32_t* w, double* dist, double* angle) {
    const bool ev = rec_i(rec, ER_EVAL) != 0;
    if (ev) { *dist = 4.0; *angle = 0.0; }
    else {
      *dist = 3.0 + (5.0 - 3.0) * mt_double(w);
      const double lo = -3.14159265358979323846 / 2, hi = 3.14159265358979323846 / 2;
      *angle = lo + (hi - lo) * mt_double(w + 2);
    }
    const float stop = (w[ev ? 0 : 4] & 1u) ? 60.0f : 30.0f;
    MB_LANES(l)
      if (l == 0) { rec[ER_DIST] = (float)*dist; rec[ER_ANGLE] = (float)*angle; rec[ER_STOP] = stop; }
    MB_END
  }

  // Walker3DCustomEnv.reset (env_locomotion.py:79-109) + WalkerBase.reset (robots.py:179-210)
  MB_HD static void reset(Mem& S, const MbPhysics& P, float* rec, uint32_t* mt_env, uint32_t* mt_robot, float* obs) {
    mb_clear_warm(S.warm);  // (robot reset: the cached contact impulses die with the episode)
    uint32_t* w = reinterpret_cast<uint32_t*>(S.rc.scratch);
    const int aliased = rec_i(rec, ER_ALIASED);
    const int nrobot = 2 + 2 * NJ, nt = target_words(rec);
    if (aliased) mt_fill(mt_env, w, nt + nrobot);
    else { mt_fill(mt_env, w, nt); mt_fill(mt_robot, w + nt, nrobot); }
    double dist, angle;
    randomize_target(rec, w, &dist, &angle);
    const uint32_t* wr = w + nt;
    const int mirrored = mt_double(wr) < 0.5;
    MB_LANES(l)
      if (l == 0) {
        rec[ER_TX] = (float)(dist * cos(angle)); rec[ER_TY] = (float)(dist * sin(angle)); rec[ER_TZ] = 1.0f;
        rec_i(rec, ER_CLOSE) = 0; rec_i(rec, ER_ELAPSED) = 0; rec[ER_FEET0] = 0.0f; rec[ER_FEET1] = 0.0f;
        rec_i(rec, ER_MIRRORED) = mirrored; rec[ER_EPRET] = 0.0f; rec_i(rec, ER_EPLEN) = 0;
      }
      if (l < NJ) S.q[l] = mb_reset_joint<M>(l, mirrored, wr);
      if (l < NU) S.u[l] = 0.0f;
      if (l == 31) {
        S.pos[0] = M::base_x(); S.pos[1] = M::base_y(); S.pos[2] = M::base_z();
        // "quat = quat or self.base_orientation" (robots.py:199): the un-mirrored attribute
        S.quat[0] = M::base_quat(0); S.quat[1] = M::base_quat(1); S.quat[2] = M::base_quat(2); S.quat[3] = M::base_quat(3);
      }
    MB_END
    typename S_::LaneConst C;
    S_::init_lane_const(C);
    S_::kinematics(S, P, C, false);
    LaneVar<float> zero;
    MB_LANES(l)
      zero[l] = 0.0f;
    MB_END
    float s1, s2;
    W3DObsScalars o = observe(S, rec, obs, zero, &s1, &s2);
    float d, a, lp;
    potential(S, rec, o.yaw, P.dt * P.substeps, &d, &a, &lp);
    MB_LANES(l)
      if (l == 0) { rec[ER_LINPOT] = lp; rec[ER_BODYX] = S.pos[0]; }
    MB_END
    if (M::planar_env()) {
      // Walker2DCustomEnv.reset (env_locomotion.py:289-299): np.concatenate((robot_state, [0], [0]))
      MB_LANES(l)
        if (l == 0) { obs[ROBOT_OBS] = 0.0f; obs[ROBOT_OBS + 1] = 0.0f; }
      MB_END
    } else {
      target_obs(d, a, obs);
    }
  }

  // Walker3DCustomEnv.step (env_locomotion.py:111-141) for one env; obs/reward/done follow the VecEnv
  // convention: on done the env is reset in place and obs is the first observation of the next episode
  // (the terminal observation goes to final_obs when that pointer is non-null).
  MB_HD static void step(Mem& S, const MbPhysics& P, float* state, float* rec, uint32_t* mt_env, uint32_t* mt_robot,
                         const float* act, float* obs, float* rew, uint8_t* done, uint8_t* trunc, float* final_obs,
                         MbStats* stats) {
    load_state(S, state);
    LaneVar<float> araw;
    LaneVar<int> badact;
    MB_LANES(l)
      araw[l] = 0.0f; badact[l] = 0;
      if (l < NJ) {
        float a = act[l];
        if (!mb_finite(a)) { a = 0.0f; badact[l] = 1; }  // reference asserts (robots.py:32); we count and zero
        araw[l] = a;
        const float ac = fminf(fmaxf(a, -1.0f), 1.0f);
        // torque is applied once and held for all substeps, as is PyBullet's -damping*qd (SURVEY App. B.2)
        S.tau[l] = M::gain(l) * ac - M::damping(l) * S.u[6 + l];
      }
    MB_END
    const unsigned anybad = warp_ballot(badact);
    int rows = 0, nc = 0, overflow = 0, ncsum = 0;
    typename S_::LaneConst C;
    S_::init_lane_const(C);
#pragma unroll 1
    for (int k = 0; k < P.substeps; ++k) {
      rows += S_::template substep<0>(S, P, C, &nc, &overflow, k);
      ncsum += nc;
    }
    // feet_contact from the last collision pass (robots.py:74-86 via getContactPoints)
    float fc0 = 0.0f, fc1 = 0.0f;
    for (int k = 0; k < nc; ++k) {
      if (S.cpartner[k] == 0 && mb_foot(S.cfoot[k]) == 0) fc0 = 1.0f;
      if (S.cpartner[k] == 0 && mb_foot(S.cfoot[k]) == 1) fc1 = 1.0f;
    }
    const float prev_bodyx = rec[ER_BODYX];
    const int eval_mode = rec_i(rec, ER_EVAL);
    MB_LANES(l)
      if (l == 0) {
        rec[ER_FEET0] = fc0; rec[ER_FEET1] = fc1;
        if (eval_mode) { rec[ER_TX] = prev_bodyx + 4.0f; rec[ER_TY] = 0.0f; rec[ER_TZ] = 1.0f; }
      }
    MB_END
    S_::kinematics(S, P, C, false);
    float s1, s2;
    W3DObsScalars o = observe(S, rec, obs, araw, &s1, &s2);
    int env_done = o.nonfinite ? 1 : 0;
    const float old_lp = rec[ER_LINPOT];
    float dist, ang, lp;
    const float scene_dt = P.dt * P.substeps;
    potential(S, rec, o.yaw, scene_dt, &dist, &ang, &lp);
    const float progress = lp - old_lp;
    float posture = 0.0f;
    if (!(-0.2f < o.pitch && o.pitch < 0.4f)) posture = fabsf(o.pitch);
    if (!(-0.4f < o.roll && o.roll < 0.4f)) posture += fabsf(o.roll);
    const float energy = 4.5f * (s1 / NJ) + 0.225f * (s2 / NJ);
    const float joints_pen = 0.1f * o.joints_at_limit;
    const float height_obs = mb_clip5(o.height);
    const float tall = height_obs > M::term_height() ? 2.0f : -1.0f;  // env_locomotion.py:44,195,320
    if (tall < 0.0f) env_done = 1;
    // Walker2DCustomEnv.step (env_locomotion.py:301-305) overwrites done with False: only the TimeLimit ends an
    // episode (the reward keeps the -1 "tall bonus").  A non-finite state still resets here (the reference would
    // stay broken for the rest of the episode).
    if (M::planar_env()) env_done = o.nonfinite ? 1 : 0;
    float target_bonus = 0.0f;
    int close = rec_i(rec, ER_CLOSE);
    if (dist < 0.15f) { close += 1; target_bonus = 2.0f; }
    if ((float)close >= rec[ER_STOP]) {
      // env_locomotion.py:214-222 -- re-sample the target mid-episode from the env stream
      close = 0;
      uint32_t* w = reinterpret_cast<uint32_t*>(S.rc.scratch);
      mt_fill(mt_env, w, target_words(rec));
      double nd, na;
      randomize_target(rec, w, &nd, &na);
      MB_LANES(l)
        if (l == 0) { rec[ER_TX] += (float)(nd * cos(na)); rec[ER_TY] += (float)(nd * sin(na)); }
      MB_END
      potential(S, rec, o.yaw, scene_dt, &dist, &ang, &lp);
    }
    const float reward = progress + target_bonus - energy + tall - posture - joints_pen;
    target_obs(dist, ang, obs);
    MB_LANES(l)
      if (l == 0) { rec_i(rec, ER_CLOSE) = close; rec[ER_LINPOT] = lp; rec[ER_BODYX] = S.pos[0]; }
    MB_END
    mb_step_epilogue<W3DEnv>(S, P, rec, mt_env, mt_robot, obs, reward, env_done, o.nonfinite, 0, rows, ncsum, overflow,
                             anybad, rew, done, trunc, final_obs, stats);
    store_state(S, state);
  }
};

// ================================================================================================ Stepper
// Walker3DStepperEnv (reference env_locomotion.py:330-840) with 3 recycled LargePlanks (bullet_objects.py:47-103).
// PILLAR: plank_class = "Pillar" (bullet_objects.py:86-90): the stones are capped cylinders of radius step_radius = 0.25
// with the planks' heights; a separate instantiation so that the default kernel's hot loop carries no dead branch.
template <class M, bool PILLAR = false> struct StepperEnv {
  typedef WarpMem<M> Mem;
  typedef Sim<M> S_;
  typedef W3DEnv<M> B_;
  typedef M Model;
  enum { NJ = M::NJ, NU = M::NU, ROBOT_OBS = 6 + 2 * M::NJ + M::NFEET, OBS = ROBOT_OBS + 15, NSTEPS = 20,
         REC_STRIDE = MB_REC_STRIDE_STEPPER, OBST = PILLAR ? MB_OBST_CYLS : MB_OBST_BOXES, ACT = M::NJ,
         INFO_FIELD = ES_STEPS_REACHED, CREDIT_STEPS_REACHED = 1 };
  template <class P> static void default_physics(P&) {}
  // remove_ground=True (env_locomotion.py:359); planks: lateralFriction 1.0, contactStiffness 30000, contactDamping
  // 1000 (bullet_objects.py:64-72) -> per-contact erp / cfm (SURVEY App. B.4); Bullet sums both bodies' contact
  // damping and a link's default is 0.1
  static void fix_physics(MbPhysics& p) {
    p.has_ground = 0;
    const float kp = 30000.0f, kd = 1000.0f + 0.1f, denom = p.dt * kp + kd;
    p.box_friction = 1.0f;
    p.box_erp = p.dt * kp / denom;
    p.box_cfm = 1.0f / denom;
  }
  static const char* check_curriculum(float v, float) {
    return v >= 0.0f && v <= 9.0f ? nullptr : "mb200_set_param: curriculum must be in [0, 9]";
  }
  static const char* check_plank_class(float v, float first) {
    if (!(v == 0.0f || v == 1.0f || v == 2.0f))
      return "mb200_set_param: plank_class must be 0 (LargePlank), 1 (Plank) or 2 (Pillar)";
    // Pillar runs its own kernel instantiation: the whole batch or none of it
    if ((v == 2.0f) != (first == 2.0f))
      return "mb200_set_param: plank_class 2 (Pillar) cannot be mixed with other classes in one batch";
    return nullptr;
  }
  static const char* plank_variant(float first) { return first == 2.0f ? "pillar" : ""; }
  static constexpr MbParam PARAMS[] = {{"curriculum", ES_CURRIC, false, check_curriculum, nullptr},
                                       {"plank_class", ES_PLANK_CLASS, false, check_plank_class, plank_variant},
                                       {"random_reward", ES_RANDOM_REWARD, false, nullptr, nullptr},
                                       {}};
  MB_HD static void load_obstacles(Mem& S, const float* rec) { load_boxes(S, rec); }
  MB_HD static void load_state(Mem& S, const float* st) { B_::load_state(S, st); }
  MB_HD static void store_state(const Mem& S, float* st) { B_::store_state(S, st); }

  MB_HD static float lin10(float a, float b, int i) { return i >= 9 ? b : a + i * ((b - a) / 9.0f); }

  // plank p -> two boxes in shared memory (base, cover): bullet_objects.py:98-103 scaled by 2*step_radius = 0.5
  MB_HD static void load_boxes(Mem& S, const float* rec) {
    MB_LANES(l)
      if (l < 6) {
        const int p = l >> 1, cover = l & 1;
        const float* b = rec + ES_BOX + 12 * p;
        float* bx = S.rc.box[l];
#pragma unroll
        for (int k = 0; k < 12; ++k) bx[k] = b[k];
        if (cover) { bx[0] += b[3 + 2] * 0.125f; bx[1] += b[3 + 5] * 0.125f; bx[2] += b[3 + 8] * 0.125f; }
        // plank_large.urdf: box 1 x 20 x (0.45 | 0.05), plank.urdf: 1 x 1.5 x (0.45 | 0.05); globalScaling 2 * 0.25
        // pillar.urdf: cylinders radius 1, length 0.9 / 0.1, globalScaling step_radius = 0.25 (bx[13] bounds the cull)
        bx[12] = 0.25f;
        bx[13] = PILLAR ? 0.25f : (rec_i(rec, ES_PLANK_CLASS) == 1 ? 0.375f : 5.0f);
        bx[14] = cover ? 0.0125f : 0.1125f;
        bx[15] = 0.0f;
      }
      if (l == 0) S.nbox = 6;
    MB_END
  }

  // BaseStep.set_position via set_step_state (env_locomotion.py:461-465, bullet_objects.py:77-83):
  // base box centre = pos + (0, 0, -0.1375) (not rotated, quirk Q15), R = euler(x_tilt, y_tilt, phi)
  MB_HD static void place_plank(float* rec, int info, int plank) {
    MB_LANES(l)
      if (l == 0) {
        const float* t = rec + ES_TERRAIN + 6 * info;
        const float roll = t[4], pitch = t[5], yaw = t[3];
        const float cr = cosf(roll * 0.5f), sr = sinf(roll * 0.5f), cp = cosf(pitch * 0.5f), sp = sinf(pitch * 0.5f);
        const float cy = cosf(yaw * 0.5f), sy = sinf(yaw * 0.5f);
        const float q[4] = {sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy, cr * cp * sy - sr * sp * cy,
                            cr * cp * cy + sr * sp * sy};
        float* b = rec + ES_BOX + 12 * plank;
        b[0] = t[0]; b[1] = t[1]; b[2] = t[2] - 0.1375f;
        mb_quat_to_mat(q, b + 3);
        rec_i(rec, ES_PLANKIDX + plank) = info;
      }
    MB_END
  }

  // delta_to_k_targets (env_locomotion.py:712-759): writes obs[ROBOT_OBS .. +15) and walk_target
  MB_HD static void targets(const Mem& S, float* rec, float yaw, float* obs) {
    const int N = rec_i(rec, ES_NEXT), stop = rec_i(rec, ES_STOP);
    MB_LANES(l)
      if (l < 3) {
        int idx = stop ? (l == 0 ? N - 1 : N) : N - 1 + l;
        if (idx > NSTEPS - 1) idx = NSTEPS - 1;
        const float* t = rec + ES_TERRAIN + 6 * idx;
        const float dx = t[0] - S.pos[0], dy = t[1] - S.pos[1], dz = t[2] - S.pos[2];
        const float ang = atan2f(dy, dx) - yaw, d = sqrtf(dx * dx + dy * dy);
        float* o = obs + ROBOT_OBS + 5 * l;
        o[0] = sinf(ang) * d; o[1] = cosf(ang) * d; o[2] = dz; o[3] = t[4]; o[4] = t[5];
        if (l == 2) { rec[ER_TX] = t[0]; rec[ER_TY] = t[1]; rec[ER_TZ] = t[2]; }
      }
    MB_END
  }

  // generate_step_placements (env_locomotion.py:395-441) in float64 from 200 words of the env stream
  MB_HD static void generate_terrain(Mem& S, float* rec, const uint32_t* w, double* dbuf) {
    const int c = rec_i(rec, ES_CURRIC);
    const double PI_D = 3.14159265358979323846, D2R = PI_D / 180;
    const double ratio = c / 9.0;
    const double dist_hi = c >= 9 ? 1.25 : 0.65 + c * ((1.25 - 0.65) / 9.0);
    const double yaw_lo = -20 * ratio * D2R, yaw_hi = 20 * ratio * D2R;
    const double pit_lo = -30 * ratio * D2R + PI_D / 2, pit_hi = 30 * ratio * D2R + PI_D / 2;
    const double til_lo = -15 * ratio * D2R, til_hi = 15 * ratio * D2R;
    double* dphi = dbuf;            // [20]
    double* dx = dbuf + 20;         // [20]
    double* dy = dbuf + 40;
    double* dz = dbuf + 60;
    double* tilt = dbuf + 80;       // [40] x_tilt, y_tilt
    MB_LANES(l)
      if (l < NSTEPS) {
        double dr = 0.65 + (dist_hi - 0.65) * mt_double(w + 2 * l);
        double dp = yaw_lo + (yaw_hi - yaw_lo) * mt_double(w + 40 + 2 * l);
        double dt = pit_lo + (pit_hi - pit_lo) * mt_double(w + 80 + 2 * l);
        double xt = til_lo + (til_hi - til_lo) * mt_double(w + 120 + 2 * l);
        double yt = til_lo + (til_hi - til_lo) * mt_double(w + 160 + 2 * l);
        if (l == 0) { dr = 0.0; dp = 0.0; dt = PI_D / 2; }
        if (l == 1 || l == 2) { dr = 0.75; dp = 0.0; dt = PI_D / 2; }
        if (l < 3) { xt = 0.0; yt = 0.0; }
        dphi[l] = dp; dx[l] = dr; dy[l] = dt; tilt[l] = xt; tilt[20 + l] = yt;
      }
    MB_END
    MB_LANES(l)
      if (l < NSTEPS) {
        double phi = 0.0;
        for (int j = 0; j <= l; ++j) phi += dphi[j];  // np.cumsum order
        const double dr = dx[l], dt = dy[l];
        double ddx = dr * sin(dt) * cos(phi);
        const double ddy = dr * sin(dt) * sin(phi);
        const double ddz = dr * cos(dt);
        if (l >= 2) {
          const double ax = fabs(ddx), mx = ax > 0.25 * 2.5 ? ax : 0.25 * 2.5;
          const double sg = ddx > 0 ? 1.0 : (ddx < 0 ? -1.0 : 0.0);
          ddx = sg * (mx < 1.25 ? mx : 1.25);
        }
        dz[l] = ddz;
        rec[ES_TERRAIN + 6 * l + 3] = (float)phi;
        rec[ES_TERRAIN + 6 * l + 4] = (float)tilt[l];
        rec[ES_TERRAIN + 6 * l + 5] = (float)tilt[20 + l];
        tilt[l] = ddx;        // reuse: dx increments
        tilt[20 + l] = ddy;   //        dy increments
      }
    MB_END
    MB_LANES(l)
      if (l < NSTEPS) {
        double x = 0.0, y = 0.0, z = 0.0;
        for (int j = 0; j <= l; ++j) { x += tilt[j]; y += tilt[20 + j]; z += dz[j]; }
        rec[ES_TERRAIN + 6 * l + 0] = (float)x;
        rec[ES_TERRAIN + 6 * l + 1] = (float)y;
        rec[ES_TERRAIN + 6 * l + 2] = (float)z;
      }
    MB_END
  }

  // Walker3DStepperEnv.reset (env_locomotion.py:481-513)
  MB_HD static void reset(Mem& S, const MbPhysics& P, float* rec, uint32_t* mt_env, uint32_t* mt_robot, float* obs) {
    mb_clear_warm(S.warm);  // (robot reset: the cached contact impulses die with the episode)
    // 44 robot words + 200 terrain words; the row storage is free between steps and serves as scratch
    uint32_t* w = reinterpret_cast<uint32_t*>(&S.w);
    double* dbuf = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(w + 256) + 7) & ~(uintptr_t)7);
    const int aliased = rec_i(rec, ER_ALIASED);
    const int nrobot = 2 + 2 * NJ;
    if (aliased) mt_fill(mt_env, w, nrobot + 200);
    else { mt_fill(mt_robot, w, nrobot); mt_fill(mt_env, w + nrobot, 200); }
    const int mirrored = mt_double(w) < 0.5;
    MB_LANES(l)
      if (l == 0) {
        rec_i(rec, ER_ELAPSED) = 0; rec[ER_FEET0] = 0.0f; rec[ER_FEET1] = 0.0f;
        rec_i(rec, ER_MIRRORED) = mirrored; rec[ER_EPRET] = 0.0f; rec_i(rec, ER_EPLEN) = 0;
        rec_i(rec, ES_TIMESTEP) = 0; rec_i(rec, ES_COUNT) = 0; rec_i(rec, ES_STOP) = 0; rec_i(rec, ES_SETSTOP) = 0;
        rec_i(rec, ES_NEXT) = 1; rec_i(rec, ES_STEPS_REACHED) = -1;
        rec_i(rec, ES_GAIN_CURRIC) = rec_i(rec, ES_CURRIC);
      }
      if (l < NJ) S.q[l] = mb_reset_joint<M>(l, mirrored, w);
      if (l < NU) S.u[l] = 0.0f;
      if (l == 31) {
        S.pos[0] = M::stepper_x(); S.pos[1] = M::stepper_y(); S.pos[2] = M::stepper_z();  // robot_init_position, env_locomotion.py:339,845
        S.quat[0] = 0.0f; S.quat[1] = 0.0f; S.quat[2] = 0.0f; S.quat[3] = 1.0f;
      }
    MB_END
    generate_terrain(S, rec, w + nrobot, dbuf);
    for (int k = 0; k < 3; ++k) place_plank(rec, k, k);
    typename S_::LaneConst C;
    S_::init_lane_const(C);
    S_::kinematics(S, P, C, false);
    LaneVar<float> zero;
    MB_LANES(l)
      zero[l] = 0.0f;
    MB_END
    float s1, s2;
    W3DObsScalars o = B_::observe(S, rec, obs, zero, &s1, &s2);
    targets(S, rec, o.yaw, obs);
    float d, a, lp;
    B_::potential(S, rec, o.yaw, P.dt * P.substeps, &d, &a, &lp);
    MB_LANES(l)
      if (l == 0) rec[ER_LINPOT] = lp;
    MB_END
  }

  // Walker3DStepperEnv.step (env_locomotion.py:515-568)
  MB_HD static void step(Mem& S, const MbPhysics& P, float* state, float* rec, uint32_t* mt_env, uint32_t* mt_robot,
                         const float* act, float* obs, float* rew, uint8_t* done, uint8_t* trunc, float* final_obs,
                         MbStats* stats) {
    B_::load_state(S, state);
    const int cur_c = rec_i(rec, ES_CURRIC);  // terminal height follows the attribute immediately (:628)
    const float applied_gain = lin10(1.0f, 1.2f, rec_i(rec, ES_GAIN_CURRIC));  // gain is latched at reset (:489)
    LaneVar<float> araw;
    LaneVar<int> badact;
    MB_LANES(l)
      araw[l] = 0.0f; badact[l] = 0;
      if (l < NJ) {
        float a = act[l];
        if (!mb_finite(a)) { a = 0.0f; badact[l] = 1; }
        araw[l] = a;
        const float ac = fminf(fmaxf(a, -1.0f), 1.0f);
        S.tau[l] = M::gain(l) * (applied_gain * ac) - M::damping(l) * S.u[6 + l];
      }
    MB_END
    const unsigned anybad = warp_ballot(badact);
    int rows = 0, nc = 0, overflow = 0, ncsum = 0;
    typename S_::LaneConst C;
    S_::init_lane_const(C);
#pragma unroll 1
    for (int k = 0; k < P.substeps; ++k) {
      load_boxes(S, rec);  // the obstacle staging area is reused by the constraint rows of every substep
      rows += S_::template substep<OBST>(S, P, C, &nc, &overflow, k);
      ncsum += nc;
    }
    const int timestep = rec_i(rec, ES_TIMESTEP) + 1;
    int next = rec_i(rec, ES_NEXT);
    int set_stop = (next == 6 || next == 7 || next == 13 || next == 14) ? 1 : 0;
    // foot contacts from the last collision pass: any partner; target = cover of plank next % 3
    const int cover_id = 10 + 2 * (next % 3) + 1;
    float fc0 = 0.0f, fc1 = 0.0f;
    int reached = 0;
    for (int k = 0; k < nc; ++k) {
      if (mb_foot(S.cfoot[k]) == 0) fc0 = 1.0f;
      if (mb_foot(S.cfoot[k]) == 1) fc1 = 1.0f;
      if (mb_foot(S.cfoot[k]) >= 0 && S.cpartner[k] == cover_id) reached = 1;
      if (M::NSELF > 0 && S.cpartner[k] >= 1000) {
        // "contact = 1.0 if contact_ids" (env_locomotion.py:645-646): a self-contact of the foot link counts too
        const int feet = M::sp_own(S.cpartner[k] - 1000) >> 16;
        if (feet & 1) fc0 = 1.0f;
        if (feet & 2) fc1 = 1.0f;
      }
    }
    S_::kinematics(S, P, C, false);
    float s1, s2;
    W3DObsScalars o = B_::observe(S, rec, obs, araw, &s1, &s2);  // foot contacts lag one step (quirk Q6)
    int env_done = o.nonfinite ? 1 : 0;
    const int cur_index = next;
    // calc_feet_state (env_locomotion.py:632-674)
    float fdist[2];
    for (int f = 0; f < 2; ++f) {
      const int b = M::foot_body(f), ow = M::bowner(b);
      const float* R = S.w.k.jR[ow];
      const float fx = S.pos[0] + S.w.k.jp[ow][0] + R[0] * M::bcom(b, 0) + R[1] * M::bcom(b, 1) + R[2] * M::bcom(b, 2);
      const float fy = S.pos[1] + S.w.k.jp[ow][1] + R[3] * M::bcom(b, 0) + R[4] * M::bcom(b, 1) + R[5] * M::bcom(b, 2);
      const float dx = fx - rec[ES_TERRAIN + 6 * next], dy = fy - rec[ES_TERRAIN + 6 * next + 1];
      fdist[f] = sqrtf(dx * dx + dy * dy);
    }
    int count = rec_i(rec, ES_COUNT), stop = rec_i(rec, ES_STOP);
    int place_info = -1, place_plank_id = 0;
    if (reached) {
      count += 1;
      if (count > 120) { stop = 0; set_stop = 0; }
      if (count >= 2) {
        if (!stop) {
          next += 1;
          count = 0;
          if (next >= 3) { place_plank_id = next % 3; place_info = next < NSTEPS - 1 ? next : NSTEPS - 1; }
        }
        stop = set_stop;
      }
      if (next >= NSTEPS) next -= 1;
    }
    MB_LANES(l)
      if (l == 0) {
        rec[ER_FEET0] = fc0; rec[ER_FEET1] = fc1;
        rec_i(rec, ES_NEXT) = next; rec_i(rec, ES_COUNT) = count; rec_i(rec, ES_STOP) = stop;
        rec_i(rec, ES_SETSTOP) = set_stop; rec_i(rec, ES_TIMESTEP) = timestep;
      }
    MB_END
    if (place_info >= 0) place_plank(rec, place_info, place_plank_id);
    // calc_base_reward (env_locomotion.py:598-630)
    const float old_lp = rec[ER_LINPOT];
    float dist, ang, lp;
    const float scene_dt = P.dt * P.substeps;
    B_::potential(S, rec, o.yaw, scene_dt, &dist, &ang, &lp);
    const float progress = lp - old_lp;
    float posture = 0.0f;
    if (!(-0.2f < o.pitch && o.pitch < 0.4f)) posture = fabsf(o.pitch);
    if (!(-0.4f < o.roll && o.roll < 0.4f)) posture += fabsf(o.roll);
    const float energy = 4.5f * (s1 / NJ) + 0.225f * (s2 / NJ);
    const float joints_pen = 0.1f * o.joints_at_limit;
    const float tall = mb_clip5(o.height) > lin10(0.75f, 0.45f, cur_c) ? 2.0f : -1.0f;
    if (tall < 0.0f) env_done = 1;
    // calc_step_reward (env_locomotion.py:676-693); 2.718 is the reference's literal (quirk Q13)
    float step_bonus = 0.0f;
    if (reached && count == 1 && next != NSTEPS - 1)
      step_bonus = 50.0f * powf(2.718f, -fminf(fdist[0], fdist[1]) / 0.25f);
    float target_bonus = 0.0f;
    if ((next == NSTEPS - 1 || stop) && dist < 0.15f) target_bonus = 2.0f;
    targets(S, rec, o.yaw, obs);
    if (cur_index != next) B_::potential(S, rec, o.yaw, scene_dt, &dist, &ang, &lp);
    float reward = progress - energy + step_bonus + target_bonus + tall - posture - joints_pen;
    if (rec_i(rec, ES_RANDOM_REWARD)) {
      // np.dot(np_random.uniform(0.8, 1.2, 8), [progress, -energy, step_bonus, target_bonus, -speed_penalty * 0,
      // tall_bonus, -posture_penalty, -joints_penalty]) (env_locomotion.py:532-547): eight draws of the env stream
      // per step, the fifth multiplies zero
      uint32_t* w = reinterpret_cast<uint32_t*>(S.rc.scratch);
      mt_fill(mt_env, w, 16);
      const float term[8] = {progress, -energy, step_bonus, target_bonus, 0.0f, tall, -posture, -joints_pen};
      double acc = 0.0;
      for (int i = 0; i < 8; ++i) acc += (0.8 + (1.2 - 0.8) * mt_double(w + 2 * i)) * (double)term[i];
      reward = (float)acc;
    }
    MB_LANES(l)
      if (l == 0) {
        rec[ER_LINPOT] = lp;
        rec_i(rec, ES_STEPS_REACHED) = (env_done || timestep == 999) ? next : -1;
      }
    MB_END
    mb_step_epilogue<StepperEnv>(S, P, rec, mt_env, mt_robot, obs, reward, env_done, o.nonfinite, next, rows, ncsum,
                                 overflow, anybad, rew, done, trunc, final_obs, stats);
    B_::store_state(S, state);
  }
};

// ================================================================================================ Monkey3D
// Monkey3DCustomEnv (reference env_locomotion.py:1136-1516) with 4 recycled MonkeyBars (bullet_objects.py:148-187).
// btMatrix3x3::getRotation of a row-major local->world rotation (xyzw)
MB_HD void mb_mat_to_quat(const float* R, float* q) {
  const float tr = R[0] + R[4] + R[8];
  if (tr > 0.0f) {
    float s = sqrtf(tr + 1.0f);
    q[3] = s * 0.5f;
    s = 0.5f / s;
    q[0] = (R[7] - R[5]) * s; q[1] = (R[2] - R[6]) * s; q[2] = (R[3] - R[1]) * s;
  } else {
    const int i = R[0] < R[4] ? (R[4] < R[8] ? 2 : 1) : (R[0] < R[8] ? 2 : 0);
    const int j = (i + 1) % 3, k = (i + 2) % 3;
    float s = sqrtf(R[4 * i] - R[4 * j] - R[4 * k] + 1.0f);
    float t[4];
    t[i] = s * 0.5f;
    s = 0.5f / s;
    t[3] = (R[3 * k + j] - R[3 * j + k]) * s; t[j] = (R[3 * j + i] + R[3 * i + j]) * s;
    t[k] = (R[3 * k + i] + R[3 * i + k]) * s;
    q[0] = t[0]; q[1] = t[1]; q[2] = t[2]; q[3] = t[3];
  }
}

template <class M> struct MonkeyEnv {
  typedef WarpMem<M> Mem;
  typedef Sim<M> S_;
  typedef W3DEnv<M> B_;
  typedef M Model;
  enum { NJ = M::NJ, NU = M::NU, ROBOT_OBS = 6 + 2 * M::NJ + M::NFEET, OBS = ROBOT_OBS + 15, NSTEPS = 32, NBARS = 4,
         REC_STRIDE = MB_REC_STRIDE_MONKEY, OBST = MB_OBST_BARS, ACT = M::NJ, INFO_FIELD = -1,
         CREDIT_STEPS_REACHED = 1 };
  template <class P> static void default_physics(P&) {}
  static void fix_physics(MbPhysics&) {}
  static constexpr MbParam PARAMS[] = {{}};
  MB_HD static void load_obstacles(Mem& S, const float* rec) { load_bars(S, rec); }
  MB_HD static void load_state(Mem& S, const float* st) { B_::load_state(S, st); }
  MB_HD static void store_state(const Mem& S, float* st) { B_::store_state(S, st); }

  MB_HD static void load_bars(Mem& S, const float* rec) {
    MB_LANES(l)
      S.rc.bar[l >> 3][l & 7] = rec[EM_BAR + l];
      if (l == 0) S.nbar = NBARS;
    MB_END
  }

  // set_step_state (env_locomotion.py:1244-1248): cylinder axis = euler(90 deg, 0, phi) applied to local z
  MB_HD static void place_bar(float* rec, int info, int bar) {
    MB_LANES(l)
      if (l == 0) {
        const float* t = rec + EM_TERRAIN + 4 * info;
        float* b = rec + EM_BAR + 8 * bar;
        b[0] = t[0]; b[1] = t[1]; b[2] = t[2];
        b[3] = sinf(t[3]); b[4] = -cosf(t[3]); b[5] = 0.0f;
        b[6] = 2.5f;    // bar_length / 2 (env_locomotion.py:1143)
        b[7] = 0.015f;  // step_radius (env_locomotion.py:1148)
        rec_i(rec, EM_BARIDX + bar) = info;
      }
    MB_END
  }

  // palm link pose relative to the base COM (BodyPart.pose() of right_palm / left_palm, env_locomotion.py:1269-1272)
  MB_HD static void palm_rel(const Mem& S, int h, float* p) {
    const int b = M::palm_body(h), ow = M::bowner(b);
    const float* R = S.w.k.jR[ow];
    const float c[3] = {M::bcom(b, 0), M::bcom(b, 1), M::bcom(b, 2)};
    mb_matvec(R, c, p);
    p[0] += S.w.k.jp[ow][0]; p[1] += S.w.k.jp[ow][1]; p[2] += S.w.k.jp[ow][2];
  }
  MB_HD static void foot_rel(const Mem& S, int f, float* p) {
    const int b = M::foot_body(f), ow = M::bowner(b);
    const float* R = S.w.k.jR[ow];
    const float c[3] = {M::bcom(b, 0), M::bcom(b, 1), M::bcom(b, 2)};
    mb_matvec(R, c, p);
    p[0] += S.w.k.jp[ow][0]; p[1] += S.w.k.jp[ow][1]; p[2] += S.w.k.jp[ow][2];
  }

  // calc_potential (env_locomotion.py:1351-1364): only swing_potential is used by the reward
  MB_HD static float swing_potential(const Mem& S, const float* rec, int swing, float scene_dt) {
    float p[3];
    palm_rel(S, swing == 0 ? 0 : 1, p);
    // (target - base) - palm_rel: both differences are small, no cancellation at 20 m altitude
    const float dx = (rec[ER_TX] - S.pos[0]) - p[0], dy = (rec[ER_TY] - S.pos[1]) - p[1];
    const float dz = (rec[ER_TZ] - S.pos[2]) - p[2];
    return -sqrtf(dx * dx + dy * dy + dz * dz) / scene_dt;
  }

  // delta_to_k_targets(k=2) (env_locomotion.py:1489-1516): obs[ROBOT_OBS .. +6) and walk_target
  MB_HD static void targets(const Mem& S, float* rec, float yaw, float* obs) {
    const int N = rec_i(rec, EM_NEXT);
    MB_LANES(l)
      if (l < 2) {
        int idx = N + l;
        if (idx > NSTEPS - 1) idx = NSTEPS - 1;
        const float* t = rec + EM_TERRAIN + 4 * idx;
        const float dx = t[0] - S.pos[0], dy = t[1] - S.pos[1], dz = t[2] - S.pos[2];
        const float ang = atan2f(dy, dx) - yaw, d = sqrtf(dx * dx + dy * dy);
        float* o = obs + ROBOT_OBS + 3 * l;
        o[0] = sinf(ang) * d; o[1] = cosf(ang) * d; o[2] = dz;
        if (l == 0) { rec[ER_TX] = t[0]; rec[ER_TY] = t[1]; rec[ER_TZ] = t[2]; }
      }
    MB_END
  }

  // get_observation_component tail (env_locomotion.py:1268-1281)
  MB_HD static void tail_obs(const Mem& S, const float* rec, float* obs) {
    const int swing = rec_i(rec, EM_SWING), pivot = rec_i(rec, EM_PIVOT);
    const int h = swing == 0 ? 0 : 1;
    float p[3], q[4];
    palm_rel(S, h, p);
    mb_mat_to_quat(S.w.k.jR[M::bowner(M::palm_body(h))], q);
    MB_LANES(l)
      if (l == 0) {
        float* o = obs + ROBOT_OBS + 6;
        o[0] = (float)swing; o[1] = (float)pivot;
        o[2] = (rec[ER_TX] - S.pos[0]) - p[0]; o[3] = (rec[ER_TY] - S.pos[1]) - p[1];
        o[4] = (rec[ER_TZ] - S.pos[2]) - p[2];
        o[5] = q[0]; o[6] = q[1]; o[7] = q[2]; o[8] = q[3];
      }
    MB_END
  }

  // generate_step_placements (env_locomotion.py:1183-1228), n_steps = 32, yaw_limit = pitch_limit = 0:
  // 96 float64 draws (192 words) of the env stream; rows 0 / 1 are pinned to the rear / front hand
  MB_HD static void generate_terrain(const Mem& S, float* rec, const uint32_t* w, double* dbuf, int mirrored) {
    const double PI_D = 3.14159265358979323846, D2R = PI_D / 180;
    double* dx = dbuf;        // [32]
    double* dy = dbuf + 32;
    double* dz = dbuf + 64;
    float f0[3], f1[3];
    foot_rel(S, 0, f0);
    foot_rel(S, 1, f1);
    const double fx[2] = {(double)S.pos[0] + f0[0], (double)S.pos[0] + f1[0]};
    const double fy[2] = {(double)S.pos[1] + f0[1], (double)S.pos[1] + f1[1]};
    const double fz[2] = {(double)S.pos[2] + f0[2], (double)S.pos[2] + f1[2]};
    const int i0 = fx[1] < fx[0] ? 1 : 0, j0 = fx[1] > fx[0] ? 1 : 0;
    MB_LANES(l)
      {
        const double dr = 0.3 + (0.5 - 0.3) * mt_double(w + 2 * l);
        const double dth = (90 - 0) * D2R + ((90 + 0) * D2R - (90 - 0) * D2R) * mt_double(w + 128 + 2 * l);
        const double deg = l == 0 ? -10.0 : (l == NSTEPS - 1 ? 10.0 : ((l & 1) ? 20.0 : -20.0));
        const double bp = (D2R * deg) * (mirrored ? -1.0 : 1.0);  // phi = cumsum(0) = 0
        double x = dr * sin(dth) * cos(0.0 + bp);
        const double ax = fabs(x), mx = ax > 0.015 * 2.5 ? ax : 0.015 * 2.5;
        const double sg = x > 0 ? 1.0 : (x < 0 ? -1.0 : 0.0);
        x = sg * (mx < 0.5 ? mx : 0.5);
        double y = dr * sin(dth) * sin(0.0 + bp);
        double z = dr * cos(dth);
        if (l == 0) { x = fx[i0] + 0.04; y = fy[i0]; z = fz[i0] + (-20 + 0.04); }
        if (l == 1) { x = fx[j0] - fx[i0] + 0.01; y = fy[j0] - fy[i0]; z = fz[j0] - fz[i0] - 0.02; }
        dx[l] = x; dy[l] = y; dz[l] = z;
      }
    MB_END
    MB_LANES(l)
      {
        double x = 0.0, y = 0.0, z = 0.0;
        for (int j = 0; j <= l; ++j) { x += dx[j]; y += dy[j]; z += dz[j]; }
        rec[EM_TERRAIN + 4 * l + 0] = (float)x;
        rec[EM_TERRAIN + 4 * l + 1] = (float)y;
        rec[EM_TERRAIN + 4 * l + 2] = (float)(z + 20);
        rec[EM_TERRAIN + 4 * l + 3] = 0.0f;
        if (l == 0) { rec_i(rec, EM_SWING) = i0; rec_i(rec, EM_PIVOT) = j0; }
      }
    MB_END
  }

  // Monkey3DCustomEnv.reset (env_locomotion.py:1283-1316); robot.reset(random_pose=False) still draws the coin
  MB_HD static void reset(Mem& S, const MbPhysics& P, float* rec, uint32_t* mt_env, uint32_t* mt_robot, float* obs) {
    mb_clear_warm(S.warm);  // (robot reset: the cached contact impulses die with the episode)
    uint32_t* w = reinterpret_cast<uint32_t*>(S.L);  // 2 + 192 words; the factor storage is free between steps
    // kinematics(with_vel = false) writes jR / jp / js only: the body scratch behind them is free for the doubles
    double* dbuf = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(&S.w.k.u2) + 7) & ~(uintptr_t)7);
    static_assert(sizeof(S.L) >= 200 * sizeof(uint32_t), "factor storage too small for the reset scratch");
    static_assert(sizeof(S.w.k.u2) >= 97 * sizeof(double), "body scratch too small for the terrain doubles");
    const int aliased = rec_i(rec, ER_ALIASED);
    if (aliased) mt_fill(mt_env, w, 2 + 192);
    else { mt_fill(mt_robot, w, 2); mt_fill(mt_env, w + 2, 192); }
    const int mirrored = mt_double(w) < 0.5;
    MB_LANES(l)
      if (l == 0) {
        rec_i(rec, ER_ELAPSED) = 0; rec[ER_FEET0] = 0.0f; rec[ER_FEET1] = 0.0f;
        rec_i(rec, ER_MIRRORED) = mirrored; rec[ER_EPRET] = 0.0f; rec_i(rec, ER_EPLEN) = 0;
        rec_i(rec, EM_TIMESTEP) = 0; rec_i(rec, EM_FREEFALL) = 0; rec_i(rec, EM_NEXT) = 2;
      }
      if (l < NJ) {
        int src;
        const float sign = mb_mirror_joint<M>(l, mirrored, &src);
        S.q[l] = sign * (float)M::base_angles(src);
      }
      // base_velocity (3, 0, -1) (env_locomotion.py:1154): every lane writes its own coordinate (racecheck: no second
      // writer for u[3..5])
      if (l < NU) S.u[l] = l == 3 ? 3.0f : (l == 5 ? -1.0f : 0.0f);
      if (l == 31) {
        S.pos[0] = 0.0f; S.pos[1] = 0.0f; S.pos[2] = 20.0f;  // initial_height (env_locomotion.py:1142,1153)
        S.quat[0] = 0.0f; S.quat[1] = 0.0f; S.quat[2] = 0.0f; S.quat[3] = 1.0f;
      }
    MB_END
    typename S_::LaneConst C;
    S_::init_lane_const(C);
    S_::kinematics(S, P, C, false);
    generate_terrain(S, rec, w + 2, dbuf, mirrored);
    for (int k = 0; k < NBARS; ++k) place_bar(rec, k, k);
    LaneVar<float> zero;
    MB_LANES(l)
      zero[l] = 0.0f;
    MB_END
    float s1, s2;
    W3DObsScalars o = B_::observe(S, rec, obs, zero, &s1, &s2);
    targets(S, rec, o.yaw, obs);
    const float sp = swing_potential(S, rec, rec_i(rec, EM_SWING), P.dt * P.substeps);
    MB_LANES(l)
      if (l == 0) rec[EM_SWINGPOT] = sp;
    MB_END
    tail_obs(S, rec, obs);
  }

  // Monkey3DCustomEnv.step (env_locomotion.py:1318-1349)
  MB_HD static void step(Mem& S, const MbPhysics& P, float* state, float* rec, uint32_t* mt_env, uint32_t* mt_robot,
                         const float* act, float* obs, float* rew, uint8_t* done, uint8_t* trunc, float* final_obs,
                         MbStats* stats) {
    B_::load_state(S, state);
    int swing = rec_i(rec, EM_SWING), pivot = rec_i(rec, EM_PIVOT);
    const int jswing = swing == 0 ? 17 : 22, jpivot = pivot == 0 ? 17 : 22;
    LaneVar<float> araw;
    LaneVar<int> badact;
    MB_LANES(l)
      araw[l] = 0.0f; badact[l] = 0;
      if (l < NJ) {
        float a = act[l];
        if (!mb_finite(a)) { a = 0.0f; badact[l] = 1; }
        // the finger joints are scripted: swing hand opens, pivot hand closes (env_locomotion.py:1322-1323)
        if (l == jswing) a = 1.0f;
        if (l == jpivot) a = -1.0f;
        araw[l] = a;
        const float ac = fminf(fmaxf(a, -1.0f), 1.0f);
        S.tau[l] = M::gain(l) * ac - M::damping(l) * S.u[6 + l];
      }
    MB_END
    const unsigned anybad = warp_ballot(badact);
    int rows = 0, nc = 0, overflow = 0, ncsum = 0;
    typename S_::LaneConst C;
    S_::init_lane_const(C);
#pragma unroll 1
    for (int k = 0; k < P.substeps; ++k) {
      load_bars(S, rec);  // the obstacle staging area is reused by the constraint rows of every substep
      rows += S_::template substep<MB_OBST_BARS>(S, P, C, &nc, &overflow, k);
      ncsum += nc;
    }
    const int timestep = rec_i(rec, EM_TIMESTEP) + 1;
    int next = rec_i(rec, EM_NEXT);
    const int cur_index = next;
    // calc_feet_state (env_locomotion.py:1404-1452) on the contact list of the last collision pass
    const int target_id = 20 + (next % NBARS);
    float fc[2] = {0.0f, 0.0f};
    int palm_hit[2] = {0, 0};
    for (int k = 0; k < nc; ++k) {
      const int f = mb_foot(S.cfoot[k]);
      if (f == 0 || f == 1) fc[f] = 1.0f;
      if ((f == 2 || f == 3) && S.cpartner[k] == target_id) palm_hit[f - 2] = 1;
    }
    S_::kinematics(S, P, C, false);
    // next_step / p_xyz are bound before the loop over the feet and stay stale if the index advances at i == 0
    const float tpx = rec[EM_TERRAIN + 4 * next], tpy = rec[EM_TERRAIN + 4 * next + 1];
    int reached = 0, place_info = -1, place_id = 0;
    float foot_dist = 0.0f;
    for (int i = 0; i < 2; ++i) {
      if (i != swing) continue;
      float fp[3];
      foot_rel(S, swing, fp);
      const float dx = (S.pos[0] - tpx) + fp[0], dy = (S.pos[1] - tpy) + fp[1];
      foot_dist = sqrtf(dx * dx + dy * dy);
      reached = palm_hit[swing == 0 ? 0 : 1];
      if (!reached) continue;
      next = next + 1 > NSTEPS - 1 ? NSTEPS - 1 : next + 1;
      if (next >= NBARS) {  // update_steps (env_locomotion.py:1255-1266)
        if (place_info >= 0) place_bar(rec, place_info, place_id);
        place_id = next % NBARS;
        place_info = next;
      }
      pivot = swing;
      swing = (swing + 1) % 2;
    }
    MB_LANES(l)
      if (l == 0) {
        rec[ER_FEET0] = fc[0]; rec[ER_FEET1] = fc[1];
        rec_i(rec, EM_NEXT) = next; rec_i(rec, EM_SWING) = swing; rec_i(rec, EM_PIVOT) = pivot;
        rec_i(rec, EM_TIMESTEP) = timestep;
      }
    MB_END
    if (place_info >= 0) place_bar(rec, place_info, place_id);
    float s1, s2;
    W3DObsScalars o = B_::observe(S, rec, obs, araw, &s1, &s2);
    int env_done = o.nonfinite ? 1 : 0;
    // calc_base_reward (env_locomotion.py:1366-1402): the swing progress and the free-fall test are what survives
    // the zero weights in step()
    const float scene_dt = P.dt * P.substeps;
    const float old_sp = rec[EM_SWINGPOT];
    float sp = swing_potential(S, rec, swing, scene_dt);
    const float progress = sp - old_sp;
    int freefall = rec_i(rec, EM_FREEFALL);
    if (freefall > 30) env_done = 1;
    const float step_bonus = reached ? 50.0f * expf(-foot_dist / 0.25f) : 0.0f;  // env_locomotion.py:1454-1458
    targets(S, rec, o.yaw, obs);
    const int airborne = (fc[0] + fc[1]) == 0.0f;
    freefall = airborne ? freefall + 1 : 0;
    if (cur_index != next) sp = swing_potential(S, rec, swing, scene_dt);
    const float reward = progress + step_bonus - fc[swing];
    if (timestep > 180 && next <= 2) env_done = 1;
    tail_obs(S, rec, obs);
    MB_LANES(l)
      if (l == 0) { rec[EM_SWINGPOT] = sp; rec_i(rec, EM_FREEFALL) = freefall; }
    MB_END
    mb_step_epilogue<MonkeyEnv>(S, P, rec, mt_env, mt_robot, obs, reward, env_done, o.nonfinite, next, rows, ncsum,
                                overflow, anybad, rew, done, trunc, final_obs, stats);
    B_::store_state(S, state);
  }
};

// ================================================================================================ Cassie
// CassieEnv-v0 (reference env_cassie.py:285-479; its defects fixed by intent, SURVEY App. D Q7-Q9): 10 residual PD
// targets, 50 x { low-pass joint velocity, PD torque, clip, one 0.6 ms Bullet step with two point-to-point loop
// closures } per env step.  No random draws: reset restores the saved state (env_cassie.py:363-378).
template <class M> struct CassieEnv {
  typedef WarpMem<M> Mem;
  typedef Sim<M> S_;
  typedef W3DEnv<M> B_;
  typedef M Model;
  enum { NJ = M::NJ, NU = M::NU, NO = M::NORDERED, ROBOT_OBS = 6 + 2 * M::NORDERED, OBS = ROBOT_OBS + 2,
         ACT = M::NPOWERED, REC_STRIDE = MB_REC_STRIDE_CASSIE, OBST = 0, LLC_FRAME_SKIP = 50, INFO_FIELD = -1,
         CREDIT_STEPS_REACHED = 0 };
  MB_HD static void load_obstacles(Mem&, const float*) {}
  MB_HD static void load_state(Mem& S, const float* st) { B_::load_state(S, st); }
  MB_HD static void store_state(const Mem& S, float* st) { B_::store_state(S, st); }
  static constexpr float CONTROL_STEP = 0.03f;  // env_cassie.py:287
  MB_HD static float control_step() { return CONTROL_STEP; }
  // sim_frame_skip 1 (env_cassie.py:287-289, env_base.py:81): one stepSimulation = one substep, LLC_FRAME_SKIP of them
  // per env step
  template <class P> static void default_physics(P& p) {
    p.dt = CONTROL_STEP / LLC_FRAME_SKIP;
    p.substeps = 1;
  }
  static void fix_physics(MbPhysics&) {}
  static constexpr MbParam PARAMS[] = {{}};

  // Joint.current_relative_position + to_radians (bullet_utils.py:212-215, env_cassie.py:204-212): lane k < 14
  MB_HD static float rad_angle(const Mem& S, int k, float* nrm_out) {
    const int d = M::ordered(k);
    const float lo = M::lower(d), hi = M::upper(d), mid = 0.5f * (lo + hi);
    const float nrm = 2.0f * (S.q[d] - mid) / (hi - lo);
    *nrm_out = nrm;
    return (hi - lo) * (nrm + 1.0f) * 0.5f + lo;
  }

  // Cassie.calc_state + CassieEnv.get_obs (env_cassie.py:238-276,416-431).  Needs kinematics(S, P, C, false).
  // Returns body_z - min(feet_z) and whether the state is finite.
  MB_HD static float observe(Mem& S, const float* rec, float* obs, int* nonfinite) {
    LaneVar<int> bad;
    MB_LANES(l)
      bad[l] = 0;
      if (l < NO) {
        float nrm;
        rad_angle(S, l, &nrm);
        const float sp = S.u[6 + M::ordered(l)];
        obs[6 + l] = nrm;
        obs[6 + NO + l] = sp;
        bad[l] = !(mb_finite(nrm) && mb_finite(sp));
      }
    MB_END
    float rpy[3];
    mb_euler(S.quat, rpy);
    const float cy = cosf(-rpy[2]), sy = sinf(-rpy[2]);
    const float vx = cy * S.u[3] - sy * S.u[4], vy = sy * S.u[3] + cy * S.u[4], vz = S.u[5];
    const float dz = S.pos[2] - M::base_z();  // initial_z is the reset height (env_cassie.py:252-254)
    float minz = 1e30f;
    for (int f = 0; f < M::NFEET; ++f) {
      const int b = M::foot_body(f), ow = M::bowner(b);
      const float* R = S.w.k.jR[ow];
      minz = fminf(minz, S.w.k.jp[ow][2] + R[6] * M::bcom(b, 0) + R[7] * M::bcom(b, 1) + R[8] * M::bcom(b, 2));
    }
    *nonfinite = warp_ballot(bad) != 0u ||
                 !(mb_finite(dz) && mb_finite(vx) && mb_finite(vy) && mb_finite(vz) && mb_finite(rpy[0]) && mb_finite(rpy[1]));
    // get_obs: R_z(-dtheta) walk_target, walk_target = (1000, 0, 0)
    const float tx = rec[ER_TX], ty = rec[ER_TY];
    const float dth = atan2f(ty - S.pos[1], tx - S.pos[0]) - rpy[2];
    const float cs = cosf(-dth), sn = sinf(-dth);
    MB_LANES(l)
      if (l == 0) {
        obs[0] = dz; obs[1] = vx; obs[2] = vy; obs[3] = vz; obs[4] = rpy[0]; obs[5] = rpy[1];
        obs[ROBOT_OBS] = cs * tx - sn * ty;
        obs[ROBOT_OBS + 1] = sn * tx + cs * ty;
      }
    MB_END
    return -minz;  // feet relative to the base COM
  }

  MB_HD static float potential(const Mem& S, const float* rec) {  // env_cassie.py:348-354
    const float dx = rec[ER_TX] - S.pos[0], dy = rec[ER_TY] - S.pos[1];
    return -sqrtf(dy * dy + dx * dx) / control_step();
  }

  MB_HD static void reset(Mem& S, const MbPhysics& P, float* rec, uint32_t*, uint32_t*, float* obs) {
    mb_clear_warm(S.warm);  // (robot reset: the cached contact impulses die with the episode)
    MB_LANES(l)
      if (l == 0) {
        rec[ER_TX] = 1000.0f; rec[ER_TY] = 0.0f; rec[ER_TZ] = 0.0f;
        rec_i(rec, ER_ELAPSED) = 0; rec[ER_EPRET] = 0.0f; rec_i(rec, ER_EPLEN) = 0;
      }
      if (l < NO) rec[EC_JVEL + l] = 0.0f;
      if (l < NJ) S.q[l] = (float)M::base_angles(l);
      if (l < NU) S.u[l] = 0.0f;
      if (l == 31) {
        // the saved state holds the base INERTIAL frame at base_position, identity orientation
        // (resetBasePositionAndOrientation, env_cassie.py:104-106)
        S.pos[0] = M::base_x(); S.pos[1] = M::base_y(); S.pos[2] = M::base_z();
        S.quat[0] = 0.0f; S.quat[1] = 0.0f; S.quat[2] = 0.0f; S.quat[3] = 1.0f;
      }
    MB_END
    typename S_::LaneConst C;
    S_::init_lane_const(C);
    S_::kinematics(S, P, C, false);
    int nonfinite;
    observe(S, rec, obs, &nonfinite);
    const float pot = potential(S, rec);
    MB_LANES(l)
      if (l == 0) { rec[EC_POTENTIAL] = pot; rec[EC_PREVX] = S.pos[0]; rec[EC_PREVY] = S.pos[1]; }
    MB_END
  }

  MB_HD static void step(Mem& S, const MbPhysics& P, float* state, float* rec, uint32_t* mt_env, uint32_t* mt_robot,
                         const float* act, float* obs, float* rew, uint8_t* done, uint8_t* trunc, float* final_obs,
                         MbStats* stats) {
    B_::load_state(S, state);
    // PD targets, one lane per PD joint: base angle + residual action for the 10 powered joints, 0 for the two
    // knee_to_shin "springs" (env_cassie.py:434-443)
    // (the PD gains, targets and index maps are re-read from the tables in every substep instead of living in eight
    // registers across the 50-substep loop: the Cassie kernel is register-starved in its constraint solver, round 2)
    LaneVar<float> jvel, jpos0;
    LaneVar<int> badact;
    MB_LANES(l)
      badact[l] = l < M::NPOWERED && !mb_finite(act[l]);
      float nrm;
      jpos0[l] = l < NO ? rad_angle(S, l, &nrm) : 0.0f;
      jvel[l] = l < NO ? rec[EC_JVEL + l] : 0.0f;  // lane k < 14 holds ordered joint k
    MB_END
    const unsigned anybad = warp_ballot(badact);
    int rows = 0, nc = 0, overflow = 0, ncsum = 0;
    typename S_::LaneConst C;
    S_::init_lane_const(C);
#pragma unroll 1
    for (int it = 0; it < LLC_FRAME_SKIP; ++it) {
      // jvel <- 0.8 jvel + 0.2 joint_speeds (env_cassie.py:319,451-453); the filtered value of PD joint l lives in
      // lane pd_ordered(l) and is fetched through shared memory
      MB_LANES(l)
        if (l < NO) {
          jvel[l] = (1.0f - 0.2f) * jvel[l] + 0.2f * S.u[6 + M::ordered(l)];
          S.rc.scratch[l] = jvel[l];
        }
        if (l < NJ) S.tau[l] = -M::damping(l) * S.u[6 + l];  // PyBullet's joint damping, once per stepSimulation
      MB_END
      MB_LANES(l)
        if (l < M::NPD) {
          const int pdo = M::pd_ordered(l), pdd = M::pd_dof(l);
          float target = 0.0f;
          if (l < M::NPOWERED) {
            const float a = act[l];
            target = (float)M::base_angles(pdd) + (mb_finite(a) ? a : 0.0f);
          }
          const float lim = M::gain(pdd);
          float nrm;
          const float q = rad_angle(S, pdo, &nrm);
          const float verr = fminf(fmaxf(0.0f - S.rc.scratch[pdo], -5.0f), 5.0f);  // env_cassie.py:380-393
          const float t = M::pd_kp(l) * (target - q) + M::pd_kd(l) * verr;
          S.tau[pdd] += fminf(fmaxf(t, -lim), lim);                                // apply_action clip (:225-230)
        }
      MB_END
      rows += S_::template substep<0>(S, P, C, &nc, &overflow, it);
      ncsum += nc;
    }
    S_::kinematics(S, P, C, false);
    MB_LANES(l)
      if (l < NO) {  // jvel = (jpos_end - jpos_start) / control_step (env_cassie.py:467-468)
        float nrm;
        rec[EC_JVEL + l] = (rad_angle(S, l, &nrm) - jpos0[l]) / control_step();
      }
    MB_END
    int nonfinite;
    const float height = observe(S, rec, obs, &nonfinite);
    int env_done = nonfinite ? 1 : 0;
    // compute_rewards (env_cassie.py:401-414)
    // progress = potential_new - potential_old = -(d_new - d_old) / control_step with the target 1000 m away:
    // d_new - d_old = (d_new^2 - d_old^2) / (d_new + d_old), the squares' difference factored through the exact
    // position differences (the potentials themselves only resolve 4e-3 in f32)
    const float pot = potential(S, rec);
    const float dxn = rec[ER_TX] - S.pos[0], dyn = rec[ER_TY] - S.pos[1];
    const float dxo = rec[ER_TX] - rec[EC_PREVX], dyo = rec[ER_TY] - rec[EC_PREVY];
    const float dn = sqrtf(dxn * dxn + dyn * dyn), dold = sqrtf(dxo * dxo + dyo * dyo);
    const float num = (rec[EC_PREVX] - S.pos[0]) * (dxn + dxo) + (rec[EC_PREVY] - S.pos[1]) * (dyn + dyo);
    const float progress = (dn + dold) > 0.0f ? -(num / (dn + dold)) / control_step() : 0.0f;
    const float tall = height > 0.6f ? 2.0f : -1.0f;
    if (tall < 0.0f) env_done = 1;
    const float reward = tall + progress;
    MB_LANES(l)
      if (l == 0) { rec[EC_POTENTIAL] = pot; rec[EC_PREVX] = S.pos[0]; rec[EC_PREVY] = S.pos[1]; }
    MB_END
    mb_step_epilogue<CassieEnv>(S, P, rec, mt_env, mt_robot, obs, reward, env_done, nonfinite, 0, rows, ncsum, overflow,
                                anybad, rew, done, trunc, final_obs, stats);
    B_::store_state(S, state);
  }
};
