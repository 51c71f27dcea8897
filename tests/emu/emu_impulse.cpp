// Lane-loop emulation of mb_apply_impulse (the body of the k_apply_impulse_* kernels), one env kind per entry point:
// emu_<PFX>_apply_impulse(phys, state, link, point[3], impulse[3]) pushes `state` in place.  Built beside emu.cpp
// (same compiler flags, same MbPhysics from emu_<PFX>_phys) by tests/test_impulse.py.  TEST HARNESS ONLY.
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
int emu_impulse_sizeof_phys() { return (int)sizeof(MbPhysics); }

#define EMU_IMPULSE(PFX, ENV)                                                                                        \
  void emu_##PFX##_apply_impulse(const MbPhysics* p, float* state, int link, const float* point,                     \
                                 const float* impulse) {                                                             \
    static ENV::Mem S;                                                                                                \
    memset(&S, 0, sizeof(S));                                                                                         \
    mb_apply_impulse<ENV>(S, *p, state, link, point, impulse);                                                        \
  }

typedef W3DEnv<W3D_Model> W3DKind;
typedef StepperEnv<W3D_Model> StepperKind;
typedef StepperEnv<W3D_Model, true> PillarKind;
typedef MonkeyEnv<MK3D_Model> MonkeyKind;
typedef CassieEnv<CAS_Model> CassieKind;
typedef W3DEnv<CH3D_Model> ChildKind;
typedef StepperEnv<MIKE_Model> MikeKind;
typedef W3DEnv<W2D_Model> Walker2DKind;
typedef W3DEnv<CR2D_Model> Crab2DKind;
EMU_IMPULSE(w3d, W3DKind)
EMU_IMPULSE(stepper, StepperKind)
EMU_IMPULSE(pillar, PillarKind)
EMU_IMPULSE(monkey, MonkeyKind)
EMU_IMPULSE(cassie, CassieKind)
EMU_IMPULSE(child, ChildKind)
EMU_IMPULSE(mike, MikeKind)
EMU_IMPULSE(walker2d, Walker2DKind)
EMU_IMPULSE(crab2d, Crab2DKind)
}
