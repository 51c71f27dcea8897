/*
 * mocca_b200.h -- C ABI of libmocca_b200.so, the B200-native batched replacement for the mocca_envs hot path.
 *
 * The reference has no FFI of its own for this path: its "plugin API" is the gym.Env protocol implemented by
 * EnvBase subclasses, and all arithmetic is reached through pybullet (SURVEY.md section 8b).  Every entry point
 * below cites the reference interface it replaces.  Conventions:
 *   - plain pointers and sizes only; *_dev pointers are DEVICE pointers owned by the caller (e.g. torch tensors),
 *     *_host pointers are host memory; the library owns only the opaque handle and its internal state arrays;
 *   - row-major [n_envs, dim] float32 at the boundary;
 *   - return 0 on success, negative on error, message via mb200_last_error(); no exceptions cross the ABI;
 *   - asynchronous on the given cudaStream_t (passed as void*; NULL = default stream) unless stated;
 *   - no CPU fallback: mb200_create fails unless the device is compute capability 10.x (sm_100a code only).
 */
#ifndef MOCCA_B200_H
#define MOCCA_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mb200_env mb200_env;

/* Physics constants of the reference's Bullet world; mb200_default_physics() fills the reference values. */
typedef struct mb200_physics {
  float dt;                 /* 1/240  env_base.py:81 (control_step / llc_frame_skip / sim_frame_skip)      */
  int substeps;             /* 4      bullet_utils.py:346-350 numSubSteps = frame_skip                     */
  int iterations;           /* 5      bullet_utils.py:340 numSolverIterations                             */
  float gravity;            /* 9.8    env_base.py:80, bullet_utils.py:344                                 */
  float erp_contact;        /* 0.9    bullet_utils.py:345 setDefaultContactERP                            */
  float erp_joint;          /* 0.2    Bullet m_erp (joint-limit rows)                                     */
  float linear_slop;        /* 1e-5   PyBullet world default                                              */
  float lin_damping;        /* 0.04   btMultiBody default linear damping                                  */
  float ang_damping;        /* 0.04   btMultiBody default angular damping                                 */
  float max_coord_vel;      /* 100    btMultiBody m_maxCoordinateVelocity                                 */
  float limit_max_impulse;  /* 100    btMultiBodyConstraint m_maxAppliedImpulse                           */
  float split_threshold;    /* -0.04  m_splitImpulsePenetrationThreshold (limit rows)                     */
  float residual_threshold; /* 1e-7   m_leastSquaresResidualThreshold (PGS early exit)                    */
  float ground_friction;    /* 0.8    bullet_utils.py:371 changeDynamics(lateralFriction=0.8)             */
  int has_ground;           /* 1      bullet_utils.py:361-371 plane_stadium.sdf (0 = remove_ground)       */
  int self_collision;       /* 1      robots.py:259-264, env_cassie.py:81-85 URDF_USE_SELF_COLLISION |
                                      ..._EXCLUDE_ALL_PARENTS: Walker3D / Monkey3D sphere and capsule geoms (closest points
                                      of segments), Cassie's mesh hulls (GJK on 32-vertex link hulls, left vs right leg) */
  float warmstart;          /* 0      Bullet-version switch (SURVEY App. B.3, OQ11): multibody contact warm starting.
                                      0 = off (btMultiBodyConstraintSolver disables it); f > 0 = every contact normal row
                                      starts from f x the impulse its candidate point carried in the previous substep
                                      (m_warmstartingFactor), across env steps too (per-env impulses kept in HBM)   */
} mb200_physics;

void mb200_default_physics(mb200_physics* p);
/* the same with the env's own timing: CassieEnv-v0 runs dt = 0.03 / 50 with one substep per stepSimulation and 50
 * PD-controlled stepSimulations per env step (env_cassie.py:287-289,450-465) */
void mb200_default_physics_for(const char* env_id, mb200_physics* p);

/* gym.make("mocca_envs:<env_id>") x n_envs  (reference mocca_envs/__init__.py:18-116, env_base.py:16-42).
 * env_id: "Walker3DCustomEnv-v0" (__init__.py:52-56), "Walker3DStepperEnv-v0" (__init__.py:58-62),
 * "Monkey3DCustomEnv-v0" (__init__.py:94-98; env_locomotion.py:1136-1516), "CassieEnv-v0" (__init__.py:18-22;
 * env_cassie.py:285-479), "Child3DCustomEnv-v0" (__init__.py:45-49; env_locomotion.py:317-327),
 * "MikeStepperEnv-v0" (__init__.py:64-68; env_locomotion.py:843-851), "Walker2DCustomEnv-v0" (__init__.py:106-110;
 * env_locomotion.py:285-310) or "Crab2DCustomEnv-v0" (__init__.py:112-116; env_locomotion.py:312-314).
 * physics may be NULL (reference values). */
int mb200_create(const char* env_id, int n_envs, int device, const mb200_physics* physics, mb200_env** out);
/* EnvBase.close (env_base.py:44-47) */
void mb200_destroy(mb200_env* env);

/* observation_space.shape[0], action_space.shape[0] (robots.py:22-29, env_locomotion.py:58-60); state_dim is the
 * width of the get/set_state vector [pos3 quat4(xyzw) omega3 vel3 q qd]; nu = 6 + action dim. */
int mb200_dims(const mb200_env* env, int* n_envs, int* obs_dim, int* act_dim, int* state_dim, int* nu);

/* EnvBase.seed (env_base.py:164-166): mt_host is [n_envs][625] uint32 -- the 624 MT19937 key words of
 * numpy.random.RandomState(gym_seed_words(seed_i)) followed by its position (624).  at_construction != 0 also
 * binds the robot's stream to the env's (env_base.py:93); later calls rebind only the env stream (quirk Q1).
 * Synchronous. */
int mb200_seed(mb200_env* env, const uint32_t* mt_host, int at_construction);

/* Env.reset (env_locomotion.py:79-109) for every env whose mask byte is non-zero (mask_dev NULL = all). */
int mb200_reset(mb200_env* env, const uint8_t* mask_dev, float* obs_dev, void* stream);

/* The same with HOST buffers (mask_host NULL = all; only the rows of the envs that were reset are written).
 * Synchronous.  This is what the gym facade's reset() needs when the caller holds no device memory. */
int mb200_reset_host(mb200_env* env, const uint8_t* mask_host, float* obs_host, void* stream);

/* Env.step (env_locomotion.py:111-141) for all envs, fused with gym TimeLimit and VecEnv auto-reset:
 * where done is set, obs is the first observation of the next episode and, if final_obs_dev is not NULL, the
 * terminal observation is written there.  trunc = info["TimeLimit.truncated"]. */
int mb200_step(mb200_env* env, const float* act_dev, float* obs_dev, float* rew_dev, uint8_t* done_dev,
               uint8_t* trunc_dev, float* final_obs_dev, void* stream);

/* Same call with HOST buffers (what a gym/SubprocVecEnv user holds); returns when the results are in the buffers.
 * Pinned buffers (cudaHostAlloc / cudaHostRegister, e.g. torch pin_memory): the step kernel reads the actions from and
 * stores obs/reward/done/trunc into the mapped host memory itself, so the transfers overlap the launch.  Pageable
 * buffers: H2D of the actions, the step kernel, D2H of the results through device staging buffers.
 * MB200_HOST_DIRECT=0 in the environment forces the staged path, =1 keeps only the result stores direct. */
int mb200_step_host(mb200_env* env, const float* act_host, float* obs_host, float* rew_host, uint8_t* done_host,
                    uint8_t* trunc_host, void* stream);

/* The integer part of the info dict of the last mb200_step / mb200_step_host, one int per env:
 * info["steps_reached"] of Walker3DStepperEnv / MikeStepperEnv (env_locomotion.py:505-506; -1 where the step did not
 * report it, i.e. the episode did not end), -1 for the other envs (their info dicts are empty; Cassie's reward terms
 * are recomputed by the host mirror).  mb200_info copies device-to-device on the stream; mb200_info_host is
 * synchronous. */
int mb200_info(mb200_env* env, int* info_dev, void* stream);
int mb200_info_host(mb200_env* env, int* info_host, void* stream);

/* resetJointState / resetBasePositionAndOrientation / resetBaseVelocity and the matching getters
 * (robots.py:212-216, bullet_utils.py:100-146,157-175): rows are [pos3 quat4 omega3 vel3 q[A] qd[A]]. */
int mb200_get_state(mb200_env* env, float* state_dev, void* stream);
int mb200_set_state(mb200_env* env, const float* state_dev, void* stream);
/* per-env bookkeeping record (walk_target, potentials, counters, terrain ...), mb200_record_stride() 4-byte words
 * per env, see ER_* / ES_* in csrc/mb_env.cuh; used by tests and checkpointing. */
int mb200_record_stride(const mb200_env* env);
int mb200_get_record(mb200_env* env, float* rec_dev, void* stream);
int mb200_set_record(mb200_env* env, const float* rec_dev, void* stream);
/* the env / robot MT19937 streams (np_random of env_base.py:164-166 and robots.py:182,192), [n_envs][2][640] uint32
 * on the HOST: 624 key words, position, padding.  With get/set_state and get/set_record this is the complete
 * checkpoint of a batch: a restored batch continues bit-exactly.  Synchronous. */
int mb200_rng_words(const mb200_env* env);
int mb200_get_rng(mb200_env* env, uint32_t* mt_host);
int mb200_set_rng(mb200_env* env, const uint32_t* mt_host);

/* The contact impulses kept for warm starting (mb200_physics.warmstart > 0), [n_envs][mb200_warm_width()] float32 on the
 * device, one slot per contact candidate id: the fourth part of a checkpoint when the switch is on.  Width 0 = off. */
int mb200_warm_width(const mb200_env* env);
int mb200_get_warm(mb200_env* env, float* warm_dev, void* stream);
int mb200_set_warm(mb200_env* env, const float* warm_dev, void* stream);

/* stepSimulation only (bullet_utils.py:352-353): hold tau_dev [n][nu - 6] over `substeps` substeps, no env logic.
 * Outputs per env: rows_dev (constraint rows summed over the substeps) and contacts_dev (contact points of the
 * last substep); either may be NULL. */
int mb200_step_physics(mb200_env* env, const float* tau_dev, int* rows_dev, int* contacts_dev, void* stream);

/* The same stepSimulation, also returning what pybullet.getContactPoints reports afterwards (robots.py:74-86 reads it
 * for feet_contact; bullet_utils.py:177-181): the contact points of the LAST collision pass with the normal impulse the
 * solver applied to each.  points_dev is [n][mb200_max_contact_points()][mb200_contact_point_width()] float32:
 * {world position on the robot link (3), contact normal on the partner pointing to the link (3), distance, normal
 * impulse, robot link index, partner}.  The link index is the dof index of the movable frame that carries the geom:
 * a fixed link is folded into its nearest movable ancestor, -1 is the base and -2 an unused slot (so it is not the URDF
 * link index pybullet reports when the model has fixed links).  The partner is 0 for the ground plane, 10 + k for
 * plank box k (plank k / 2: k even = base box, k odd = cover), 20 + k for bar k and 1000 + p for a self-contact, where
 * p indexes the env kind's self-collision pair table (the model's "self_pairs", geom A then geom B; the point is on A's
 * link and the normal points from B to A).  Unused slots are zero apart from their link index.  Parity /
 * golden-vector entry point; the env step kernels do not produce it. */
int mb200_max_contact_points(void);
int mb200_contact_point_width(void);
int mb200_step_physics_points(mb200_env* env, const float* tau_dev, int* rows_dev, int* contacts_dev, float* points_dev,
                              void* stream);

/* pybullet.calculateMassMatrix / calculateInverseDynamics analogues at the current state, in PyBullet's
 * generalised coordinates u = [omega_world, v_world, qd]:  M_dev [n][nu][nu];  tau = M acc + C + G, [n][nu]. */
int mb200_mass_matrix(mb200_env* env, float* M_dev, void* stream);
int mb200_inverse_dynamics(mb200_env* env, const float* acc_dev, float* tau_dev, void* stream);

/* A push between two env steps: env i receives the instantaneous linear impulse impulse_dev[i] (N s, world frame) at the
 * world point point_dev[i], rigidly attached to link link_dev[i] (shapes [n], [n][3], [n][3], device memory).  The
 * generalised velocity u = [omega_world, v_world, qd] (the coordinates of mb200_mass_matrix) changes by
 *   du = M(q)^-1 J(point)^T impulse,
 * then u is clamped to +-max_coord_vel as in every substep.  Positions, quaternion, q, the record, the RNG streams and
 * the warm-start impulses are untouched; contacts and joint limits do not act at the instant of the push (the next
 * substep's rows react to the new velocity).  A force F held over one env step is, to first order, the impulse
 * F * control_step; this is not pybullet.applyExternalForce.  The observation the caller holds is the pre-push one.
 * Link index: -1 = the base, j = the movable frame of dof j with fixed links folded into their nearest movable ancestor
 * (the link index of mb200_step_physics_points).  Any other index (e.g. -2), an all-zero impulse or a non-finite
 * impulse or point leaves that env untouched, bit for bit.
 * CassieEnv-v0: the response keeps the two achilles-rod loop closures closed: du = M^-1 (J^T impulse - G^T lambda) with
 * G du = 0 (G = the six point-to-point rows).  Walker2D / Crab2D: the y components of impulse and point are taken as
 * zero (what the planar root transmits), so the motion stays exactly in the x-z plane. */
int mb200_apply_impulse(mb200_env* env, const int* link_dev, const float* point_dev, const float* impulse_dev,
                        void* stream);

/* Camera images (pybullet.getCameraImage(width, height, viewMatrix, projectionMatrix) for a batch): for each of `count`
 * cameras, env env_ids_dev[i] (device memory, [count]; NULL = envs 0..count-1) in its current state -- the state the
 * last reset / step / set_state / apply_impulse left, i.e. after an auto-reset the first state of the new episode.
 * An id outside [0, n_envs) gives a blank frame (sky colour, depth = far, seg = -1).
 *   view_dev, proj_dev: [count][16] float32, column-major OpenGL 4x4 matrices exactly as pybullet.computeViewMatrix*
 *     and computeProjectionMatrixFOV return them (the same camera can be passed to both).  proj * view is inverted in
 *     double precision once per camera; a singular or non-finite product gives a blank frame with depth NaN.
 *   The ray of pixel (row r, column c) runs through NDC x = 2 (c + 0.5) / W - 1, y = 1 - 2 (r + 0.5) / H from the near
 *     plane to the far plane; row 0 is the top row, as in getCameraImage.  1 <= width, height <= 2048, count >= 1.
 * Outputs (device memory; any may be NULL, it is then not written):
 *   rgb_dev   [count][H][W][3] uint8;
 *   depth_dev [count][H][W] float32: eye-space distance along the view axis in metres (far where nothing is hit).
 *     Not PyBullet's nonlinear depth buffer: that is  buf = far (depth - near) / (depth (far - near)).
 *   seg_dev   [count][H][W] int32: -1 sky; 0 ground, 10 + k plank box k (k = 2 p base / 2 p + 1 cover of plank p, the
 *     Pillar stones likewise), 20 + k bar k (the partner codes of mb200_step_physics_points); 30 the walk target;
 *     100 + link for a robot link, link as mb200_apply_impulse and the contact list index it (99 = the base, fixed
 *     links folded into their movable ancestor).
 * Scene: the collision geometry only (no visual meshes): the robot's spheres, capsules and boxes; CassieEnv-v0's link
 * hulls as convex polytopes (its hull-vertex contact spheres are not drawn, so a Cassie link without a hull, e.g. the
 * pelvis, is invisible); the ground plane where physics.has_ground is set; the Stepper / Mike planks as the base and
 * cover boxes (or the Pillar cylinders) and Monkey3D's four bars, as the collision pass stages them; for the
 * Walker3DCustomEnv template (Walker3D, Child3D, Walker2D, Crab2D) the walk target as a sphere of radius 0.2 m (a
 * constant of this library).  Shading is flat and deterministic: one colour per class, a 1 m checkerboard on the
 * ground, Lambert shading from one fixed directional light plus ambient; no shadows, no anti-aliasing.
 * Rendering reads the state and the record and writes only its outputs (state, record, RNG streams, warm-start impulses,
 * statistics and observations are untouched); asynchronous on `stream`.  The handle owns the scene scratch buffer: one
 * handle's renders on different streams must not overlap. */
int mb200_render(mb200_env* env, const int* env_ids_dev, int count, const float* view_dev, const float* proj_dev,
                 int width, int height, uint8_t* rgb_dev, float* depth_dev, int32_t* seg_dev, void* stream);

/* EnvBase.set_env_params analogue (env_base.py:103-106): "eval_mode" (Walker3DCustomEnv, env_locomotion.py:76-77),
 * "curriculum" 0..9 (Walker3DStepperEnv, env_locomotion.py:362-369; takes effect at the next reset like the
 * reference, whose terrain / gain / terminal height are read in reset() and step()), "random_reward" 0 / 1
 * and "plank_class" 0 = LargePlank / 1 = Plank / 2 = Pillar (Walker3DStepperEnv constructor kwargs,
 * env_locomotion.py:355-357, 528-547; bullet_objects.py:86-103; Pillar launches its own kernel instantiation, so it
 * is set for the whole batch or not at all).  The array variant sets one value per env
 * (values_host[count], count == n_envs).  Synchronous. */
int mb200_set_param(mb200_env* env, const char* key, float value);
int mb200_set_param_array(mb200_env* env, const char* key, const float* values_host, int count);

/* Episode statistics accumulated on the device since the last call with reset != 0 (synchronous):
 * out = {episodes, sum_return, sum_length, nonfinite_events, cap_overflows, sum_steps_reached (Stepper), 0, 0}. */
int mb200_stats(mb200_env* env, double out[8], int reset);

/* number of kernel launches issued through this handle (bench.py's gpu_launches) */
long long mb200_launch_count(const mb200_env* env);

/* FP32 FMA throughput of `device` in TFLOP/s (synchronous probe kernel, ~10 ms): the measured denominator of the
 * CUDA-core roofline bench.py reports for this path. */
int mb200_measure_fp32_peak(int device, double* tflops_out);

const char* mb200_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
