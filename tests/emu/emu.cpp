// Lane-loop emulation of the kernel source (mb_core.cuh / mb_env.cuh compiled by g++ with MB_LANES as a
// 32-iteration loop).  DEBUG/TEST HARNESS ONLY: lets the exact kernel source be diffed against the CPU oracle on
// a box without a GPU.  Never loaded by the mocca_envs_b200 package; the product path is libmocca_b200.so.
#include <string.h>

#include "../../mocca_envs_b200/csrc/generated/walker3d_model.h"
#include "../../mocca_envs_b200/csrc/generated/monkey3d_model.h"
#include "../../mocca_envs_b200/csrc/generated/cassie_model.h"
#include "../../mocca_envs_b200/csrc/generated/child3d_model.h"
#include "../../mocca_envs_b200/csrc/generated/mike_model.h"
#include "../../mocca_envs_b200/csrc/generated/walker2d_model.h"
#include "../../mocca_envs_b200/csrc/generated/crab2d_model.h"
#include "../../mocca_envs_b200/csrc/mb_env.cuh"

static void default_phys(MbPhysics* p) {
  p->dt = 1.0f / 240.0f; p->substeps = 4; p->iterations = 5; p->gravity = 9.8f; p->erp_contact = 0.9f;
  p->erp_joint = 0.2f; p->linear_slop = 1e-5f; p->lin_damping = 0.04f; p->ang_damping = 0.04f;
  p->max_coord_vel = 100.0f; p->limit_max_impulse = 100.0f; p->split_threshold = -0.04f;
  p->residual_threshold = 1e-7f; p->ground_friction = 0.8f; p->has_ground = 1;
  p->box_friction = 1.0f; p->box_erp = 0.9f; p->box_cfm = 0.0f; p->bar_friction = 0.5f;
  p->self_collision = 1;
  p->warmstart = 0.0f;
}

extern "C" {
int emu_sizeof_phys() { return (int)sizeof(MbPhysics); }
void emu_default_phys(MbPhysics* p) { default_phys(p); }

// ---- Walker3DStepperEnv (also Mike, Pillar)
void emu_stepper_phys(MbPhysics* p) {
  default_phys(p);
  p->has_ground = 0;
  const float kp = 30000.0f, kd = 1000.0f + 0.1f, denom = p->dt * kp + kd;
  p->box_friction = 1.0f; p->box_erp = p->dt * kp / denom; p->box_cfm = 1.0f / denom;
}

// ---- CassieEnv
void emu_cassie_phys(MbPhysics* p) {
  default_phys(p);
  p->dt = 0.03f / 50.0f;
  p->substeps = 1;
}

// emu_<PFX>_rec_stride / _reset / _step / _step_physics / _mass_matrix of one env kind.
// step: stats_out[6] = the step's MbStats in the order of mb200_stats (episodes, ret_sum, len_sum, nonfinite,
// overflow, steps_reached_sum).  step_physics: one stepSimulation with the obstacles of `rec`; `warm` [MB_NWARM] plays
// the env's HBM warm-start impulses, `points` [MB_MAXC][MB_POINT_WIDTH] receives the contact points of the last
// collision pass (see Sim::substep); nullptr switches either off.
#define EMU_ENV(PFX, ENV)                                                                                             \
  int emu_##PFX##_rec_stride() { return (int)ENV::REC_STRIDE; }                                                       \
  void emu_##PFX##_reset(const MbPhysics* p, float* state, float* rec, uint32_t* mt_env, uint32_t* mt_robot,         \
                         float* obs) {                                                                                \
    static ENV::Mem S;                                                                                                \
    memset(&S, 0, sizeof(S));                                                                                         \
    ENV::reset(S, *p, rec, mt_env, mt_robot, obs);                                                                    \
    ENV::store_state(S, state);                                                                                       \
  }                                                                                                                   \
  void emu_##PFX##_step(const MbPhysics* p, float* state, float* rec, uint32_t* mt_env, uint32_t* mt_robot,          \
                        const float* act, float* obs, float* rew, uint8_t* done, uint8_t* trunc, float* final_obs,   \
                        double* stats_out) {                                                                          \
    static ENV::Mem S;                                                                                                \
    memset(&S, 0, sizeof(S));                                                                                         \
    MbStats st;                                                                                                       \
    memset(&st, 0, sizeof(st));                                                                                       \
    ENV::step(S, *p, state, rec, mt_env, mt_robot, act, obs, rew, done, trunc, final_obs, &st);                       \
    stats_out[0] = (double)st.episodes; stats_out[1] = st.ret_sum; stats_out[2] = st.len_sum;                         \
    stats_out[3] = (double)st.nonfinite; stats_out[4] = (double)st.overflow;                                          \
    stats_out[5] = (double)st.steps_reached_sum;                                                                      \
  }                                                                                                                   \
  void emu_##PFX##_step_physics(const MbPhysics* p, float* state, const float* rec, const float* tau, float* warm,    \
                                float* points, int* rows, int* contacts) {                                            \
    typedef Sim<ENV::Model> Sim_;                                                                                     \
    static ENV::Mem S;                                                                                                \
    memset(&S, 0, sizeof(S));                                                                                         \
    S.warm = warm;                                                                                                    \
    ENV::load_state(S, state);                                                                                        \
    for (int j = 0; j < ENV::NJ; ++j) S.tau[j] = tau[j];                                                              \
    int r = 0, nc = 0, ov = 0;                                                                                        \
    Sim_::LaneConst C;                                                                                                \
    Sim_::init_lane_const(C);                                                                                         \
    for (int k = 0; k < p->substeps; ++k) {                                                                           \
      ENV::load_obstacles(S, rec);                                                                                    \
      r += Sim_::substep<ENV::OBST>(S, *p, C, &nc, &ov, k, k == p->substeps - 1 ? points : nullptr);                  \
    }                                                                                                                 \
    ENV::store_state(S, state);                                                                                       \
    *rows = r;                                                                                                        \
    *contacts = nc;                                                                                                   \
  }                                                                                                                   \
  void emu_##PFX##_mass_matrix(const MbPhysics* p, const float* state, float* Mout, float* bias) {                   \
    typedef Sim<ENV::Model> Sim_;                                                                                     \
    static ENV::Mem S;                                                                                                \
    memset(&S, 0, sizeof(S));                                                                                         \
    ENV::load_state(S, state);                                                                                        \
    Sim_::LaneConst C;                                                                                                \
    Sim_::init_lane_const(C);                                                                                         \
    Sim_::kinematics(S, *p, C, true);                                                                                 \
    Sim_::bodies(S, *p);                                                                                              \
    Sim_::mass_matrix_and_rhs(S);                                                                                     \
    const int NU = ENV::NU;                                                                                           \
    for (int i = 0; i < NU; ++i) {                                                                                    \
      for (int j = 0; j < NU; ++j) Mout[i * NU + j] = mb_Lget<ENV::Model>(S.L, i, j);                                 \
      bias[i] = -S.rhs[i];                                                                                            \
    }                                                                                                                 \
  }

typedef W3DEnv<W3D_Model> W3DKind;
typedef StepperEnv<W3D_Model> StepperKind;
typedef StepperEnv<W3D_Model, true> PillarKind;  // plank_class = "Pillar"
typedef MonkeyEnv<MK3D_Model> MonkeyKind;
typedef CassieEnv<CAS_Model> CassieKind;
typedef W3DEnv<CH3D_Model> ChildKind;  // Child3DCustomEnv-v0
typedef StepperEnv<MIKE_Model> MikeKind;  // MikeStepperEnv-v0
typedef W3DEnv<W2D_Model> Walker2DKind;
typedef W3DEnv<CR2D_Model> Crab2DKind;
EMU_ENV(w3d, W3DKind)
EMU_ENV(stepper, StepperKind)
EMU_ENV(pillar, PillarKind)
EMU_ENV(monkey, MonkeyKind)
EMU_ENV(cassie, CassieKind)
EMU_ENV(child, ChildKind)
EMU_ENV(mike, MikeKind)
EMU_ENV(walker2d, Walker2DKind)
EMU_ENV(crab2d, Crab2DKind)
}
