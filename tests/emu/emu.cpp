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

extern "C" {
int emu_sizeof_phys() { return (int)sizeof(MbPhysics); }

// emu_<PFX>_phys / _rec_stride / _reset / _step / _step_physics / _mass_matrix of one env kind.
// phys: the solver parameters mb200_create gives the kind when the caller passes none.
// step: stats_out[6] = the step's MbStats in the order of mb200_stats (episodes, ret_sum, len_sum, nonfinite,
// overflow, steps_reached_sum).  step_physics: one stepSimulation with the obstacles of `rec`; `warm` [MB_NWARM] plays
// the env's HBM warm-start impulses, `points` [MB_MAXC][MB_POINT_WIDTH] receives the contact points of the last
// collision pass; nullptr switches either off.
#define EMU_ENV(PFX, ENV)                                                                                             \
  void emu_##PFX##_phys(MbPhysics* q) {                                                                               \
    MbPhysics p;                                                                                                      \
    mb_default_physics(&p);                                                                                           \
    ENV::default_physics(p);                                                                                          \
    mb_to_internal(p, q);                                                                                             \
    ENV::fix_physics(*q);                                                                                             \
  }                                                                                                                   \
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
    static ENV::Mem S;                                                                                                \
    memset(&S, 0, sizeof(S));                                                                                         \
    S.warm = warm;                                                                                                    \
    *rows = mb_physics_step<ENV>(S, *p, state, rec, tau, points, contacts);                                           \
  }                                                                                                                   \
  void emu_##PFX##_mass_matrix(const MbPhysics* p, const float* state, float* Mout, float* bias) {                   \
    static ENV::Mem S;                                                                                                \
    memset(&S, 0, sizeof(S));                                                                                         \
    mb_mass_matrix<ENV>(S, *p, state);                                                                                \
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
