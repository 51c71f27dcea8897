"""Loader for libmocca_b200.so (the C ABI in include/mocca_b200.h).  There is NO CPU fallback: importing the
package works anywhere, but creating an env fails loudly unless the CUDA library is built and a B200 is present."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MB200_LIB") or os.path.join(_HERE, "libmocca_b200.so")
CSRC = os.path.join(_HERE, "csrc")
# one translation unit per env kind (csrc/kinds/<kind>.cu = model table + MB_DEFINE_KIND) + the C ABI (mb200.cu)
KINDS = {
    "walker3d_custom": "walker3d", "walker3d_stepper": "walker3d", "walker3d_stepper_pillar": "walker3d",
    "monkey3d_custom": "monkey3d", "cassie": "cassie", "child3d_custom": "child3d", "walker2d_custom": "walker2d",
    "crab2d_custom": "crab2d", "mike_stepper": "mike", "mike_stepper_pillar": "mike",
}
COMMON = [os.path.join(CSRC, f) for f in ("mb_core.cuh", "mb_env.cuh", "mb_kind.cuh", "mb_tables.h")] + [
    os.path.join(os.path.dirname(_HERE), "include", "mocca_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]
BUILD_DIR = os.path.join(_HERE, "build")

SYMBOLS = [
    "mb200_default_physics", "mb200_default_physics_for", "mb200_create", "mb200_destroy", "mb200_dims", "mb200_seed", "mb200_reset",
    "mb200_reset_host", "mb200_info", "mb200_info_host", "mb200_step_physics_points", "mb200_max_contact_points",
    "mb200_contact_point_width", "mb200_warm_width", "mb200_get_warm", "mb200_set_warm",
    "mb200_step", "mb200_step_host", "mb200_get_state", "mb200_set_state", "mb200_get_record", "mb200_set_record",
    "mb200_rng_words", "mb200_get_rng", "mb200_set_rng", "mb200_step_physics", "mb200_mass_matrix", "mb200_inverse_dynamics",
    "mb200_apply_impulse", "mb200_render", "mb200_set_param",
    "mb200_set_param_array", "mb200_record_stride", "mb200_stats",
    "mb200_launch_count", "mb200_measure_fp32_peak", "mb200_last_error",
]


class Physics(C.Structure):
    """mb200_physics (include/mocca_b200.h)."""
    _fields_ = [("dt", C.c_float), ("substeps", C.c_int), ("iterations", C.c_int), ("gravity", C.c_float),
                ("erp_contact", C.c_float), ("erp_joint", C.c_float), ("linear_slop", C.c_float),
                ("lin_damping", C.c_float), ("ang_damping", C.c_float), ("max_coord_vel", C.c_float),
                ("limit_max_impulse", C.c_float), ("split_threshold", C.c_float), ("residual_threshold", C.c_float),
                ("ground_friction", C.c_float), ("has_ground", C.c_int), ("self_collision", C.c_int),
                ("warmstart", C.c_float)]


def _units():
    """(source, object, dependencies) of every translation unit."""
    units = [(os.path.join(CSRC, "mb200.cu"), os.path.join(BUILD_DIR, "mb200.o"), COMMON)]
    for kind, model in KINDS.items():
        units.append((os.path.join(CSRC, "kinds", kind + ".cu"), os.path.join(BUILD_DIR, kind + ".o"),
                      COMMON + [os.path.join(CSRC, "generated", model + "_model.h")]))
    return units


def build(force: bool = False, verbose: bool = False, defines=(), lib_path: str | None = None,
          build_dir: str | None = None) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU): the translation units in
    parallel, then one link.  `defines` / `lib_path` / `build_dir` build an A/B variant beside the product library."""
    from concurrent.futures import ThreadPoolExecutor

    out = lib_path or LIB_PATH
    bdir = build_dir or BUILD_DIR
    os.makedirs(bdir, exist_ok=True)
    todo, objs = [], []
    for src, obj, deps in _units():
        obj = os.path.join(bdir, os.path.basename(obj))
        objs.append(obj)
        stale = (not os.path.exists(obj)) or any(
            os.path.exists(d) and os.path.getmtime(d) > os.path.getmtime(obj) for d in [src] + deps)
        if force or stale:
            todo.append((src, obj))

    def compile_one(so):
        cmd = ["nvcc"] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) + [
            "-c", "-o", so[1], so[0]]
        subprocess.check_call(cmd)

    if todo:
        with ThreadPoolExecutor(max_workers=min(len(todo), os.cpu_count() or 4)) as ex:
            list(ex.map(compile_one, todo))
    if todo or not os.path.exists(out):
        subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out] + objs)
    return out


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libmocca_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'`; "
                "there is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp, ip = C.c_void_p, C.c_int
        L.mb200_last_error.restype = C.c_char_p
        L.mb200_launch_count.restype = C.c_longlong
        L.mb200_launch_count.argtypes = [vp]
        L.mb200_default_physics.argtypes = [C.POINTER(Physics)]
        L.mb200_default_physics_for.argtypes = [C.c_char_p, C.POINTER(Physics)]
        L.mb200_create.argtypes = [C.c_char_p, ip, ip, C.POINTER(Physics), C.POINTER(vp)]
        L.mb200_destroy.argtypes = [vp]
        L.mb200_destroy.restype = None
        L.mb200_dims.argtypes = [vp] + [C.POINTER(ip)] * 5
        L.mb200_seed.argtypes = [vp, vp, ip]
        L.mb200_reset.argtypes = [vp, vp, vp, vp]
        L.mb200_reset_host.argtypes = [vp, vp, vp, vp]
        L.mb200_info.argtypes = [vp, vp, vp]
        L.mb200_info_host.argtypes = [vp, vp, vp]
        L.mb200_step.argtypes = [vp] * 8
        L.mb200_step_host.argtypes = [vp] * 7
        L.mb200_warm_width.argtypes = [vp]
        for f in ("mb200_get_state", "mb200_set_state", "mb200_get_record", "mb200_set_record", "mb200_mass_matrix",
                  "mb200_get_warm", "mb200_set_warm"):
            getattr(L, f).argtypes = [vp, vp, vp]
        L.mb200_step_physics.argtypes = [vp, vp, vp, vp, vp]
        L.mb200_step_physics_points.argtypes = [vp, vp, vp, vp, vp, vp]
        L.mb200_rng_words.argtypes = [vp]
        L.mb200_get_rng.argtypes = [vp, vp]
        L.mb200_set_rng.argtypes = [vp, vp]
        L.mb200_inverse_dynamics.argtypes = [vp, vp, vp, vp]
        L.mb200_apply_impulse.argtypes = [vp, vp, vp, vp, vp]
        L.mb200_render.argtypes = [vp, vp, ip, vp, vp, ip, ip, vp, vp, vp, vp]
        L.mb200_set_param.argtypes = [vp, C.c_char_p, C.c_float]
        L.mb200_set_param_array.argtypes = [vp, C.c_char_p, vp, ip]
        L.mb200_record_stride.argtypes = [vp]
        L.mb200_stats.argtypes = [vp, C.POINTER(C.c_double), ip]
        L.mb200_measure_fp32_peak.argtypes = [ip, C.POINTER(C.c_double)]
        _lib = L
    return _lib


def check(rc: int):
    if rc != 0:
        raise RuntimeError("libmocca_b200: " + lib().mb200_last_error().decode())
