// Emulation of mb200_render's two passes, the same source as the kernels: emu_<PFX>_render_scene(phys, state, rec,
// out) runs mb_render_scene (the body of k_render_scene_<kind>) for one env with the lane loop and returns the kind's
// primitive count; emu_render_rays loops mb_render_pixel (the body of k_render_rays) over every pixel of one camera.
// Built beside emu.cpp (same compiler flags, MbPhysics from emu_<PFX>_phys) by tests/test_render.py.  TEST HARNESS ONLY.
#include <math.h>
#include <string.h>

#include "../../mocca_envs_b200/csrc/generated/walker3d_model.h"
#include "../../mocca_envs_b200/csrc/generated/monkey3d_model.h"
#include "../../mocca_envs_b200/csrc/generated/cassie_model.h"
#include "../../mocca_envs_b200/csrc/generated/child3d_model.h"
#include "../../mocca_envs_b200/csrc/generated/mike_model.h"
#include "../../mocca_envs_b200/csrc/generated/walker2d_model.h"
#include "../../mocca_envs_b200/csrc/generated/crab2d_model.h"
#include "../../mocca_envs_b200/csrc/mb_render.cuh"

extern "C" {
int emu_render_sizeof_phys() { return (int)sizeof(MbPhysics); }
int emu_render_rmax() { return MB_RMAX; }
int emu_render_stride() { return MB_RSTRIDE; }

// out: [MB_RMAX][MB_RSTRIDE]; returns the kind's primitive count
#define EMU_RENDER(PFX, ENV)                                                                                         \
  int emu_##PFX##_render_scene(const MbPhysics* p, const float* state, const float* rec, float* out) {              \
    static ENV::Mem S;                                                                                                \
    memset(&S, 0, sizeof(S));                                                                                         \
    mb_render_scene<ENV>(S, *p, state, rec, out);                                                                     \
    return MbRenderLayout<ENV>::NPRIM;                                                                                \
  }                                                                                                                   \
  void emu_##PFX##_render_blank(float* out) { mb_render_blank(out, MbRenderLayout<ENV>::NPRIM); }

typedef W3DEnv<W3D_Model> W3DKind;
typedef StepperEnv<W3D_Model> StepperKind;
typedef StepperEnv<W3D_Model, true> PillarKind;
typedef MonkeyEnv<MK3D_Model> MonkeyKind;
typedef CassieEnv<CAS_Model> CassieKind;
typedef W3DEnv<CH3D_Model> ChildKind;
typedef StepperEnv<MIKE_Model> MikeKind;
typedef W3DEnv<W2D_Model> Walker2DKind;
typedef W3DEnv<CR2D_Model> Crab2DKind;
EMU_RENDER(w3d, W3DKind)
EMU_RENDER(stepper, StepperKind)
EMU_RENDER(pillar, PillarKind)
EMU_RENDER(monkey, MonkeyKind)
EMU_RENDER(cassie, CassieKind)
EMU_RENDER(child, ChildKind)
EMU_RENDER(mike, MikeKind)
EMU_RENDER(walker2d, Walker2DKind)
EMU_RENDER(crab2d, Crab2DKind)

// one camera: scene [nprim][MB_RSTRIDE] from a scene pass, view / proj [16]; outputs [H][W](3), each may be NULL
void emu_render_rays(int nprim, const float* scene, const float* view, const float* proj, int W, int H, uint8_t* rgb,
                     float* depth, int* seg) {
  MbCamera cam;
  mb_render_camera(view, proj, &cam);
  for (int r = 0; r < H; ++r)
    for (int c = 0; c < W; ++c) {
      const size_t px = (size_t)r * W + c;
      uint8_t p3[3];
      float dp;
      int sg;
      mb_render_pixel(cam, scene, nprim, W, H, r, c, p3, &dp, &sg);
      if (rgb) { rgb[3 * px] = p3[0]; rgb[3 * px + 1] = p3[1]; rgb[3 * px + 2] = p3[2]; }
      if (depth) depth[px] = dp;
      if (seg) seg[px] = sg;
    }
}
}
