"""The C-ABI library loads and exports every symbol include/mocca_b200.h declares; no CPU fallback exists."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_exported():
    from mocca_envs_b200 import _lib

    _lib.build()
    L = C.CDLL(_lib.LIB_PATH)
    hdr = open(os.path.join(ROOT, "include", "mocca_b200.h")).read()
    declared = set(re.findall(r"\b(mb200_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    for sym in declared:
        assert hasattr(L, sym), sym
    assert declared == set(_lib.SYMBOLS)


def test_create_fails_loudly_without_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from mocca_envs_b200 import _lib

    L = _lib.lib()
    h = C.c_void_p()
    rc = L.mb200_create(b"Walker3DCustomEnv-v0", 4, 0, None, C.byref(h))
    assert rc != 0 and h.value is None
    assert len(L.mb200_last_error()) > 0
    rc = L.mb200_create(b"NoSuchEnv-v0", 4, 0, None, C.byref(h))
    assert rc != 0 and b"unsupported env id" in L.mb200_last_error()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "mocca_envs_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("CPU oracle", "").replace("the oracle", "").lower() or f in (
                    "seeding.py",), (f, "product code must not reference oracle/")


def test_generated_header_is_current():
    """csrc/generated/walker3d_model.h matches what codegen emits from the committed JSON table."""
    from mocca_envs_b200 import codegen
    from mocca_envs_b200.model_compiler import load_table

    t = load_table(os.path.join(ROOT, "mocca_envs_b200", "models", "walker3d.json"))
    want = codegen.emit_header(t, "W3D")
    have = open(os.path.join(ROOT, "mocca_envs_b200", "csrc", "generated", "walker3d_model.h")).read()
    assert want == have


def test_device_and_host_step_kernels_round_alike():
    """mb200_step and mb200_step_host run two instantiations of each step kernel whose outputs are compared bit for bit on
    the GPU (tests/test_gpu_f3.py).  Checked here without a GPU: per source line both kernels carry the same multiset of
    FFMA / FMUL / FADD / MUFU opcodes with the same negation pattern, i.e. the compiler contracted every a * b + c * d the
    same way round in both (it once did not: mb_euler, round 2)."""
    import importlib.util
    import shutil

    from mocca_envs_b200 import _lib

    if not (shutil.which("cuobjdump") and shutil.which("nvdisasm")) or not os.path.exists(_lib.LIB_PATH):
        pytest.skip("CUDA binary utilities or the built library are not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("sass_fp_diff", os.path.join(root, "tools", "sass_fp_diff.py"))
    tool = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tool)
    cubins = tool.extract(_lib.LIB_PATH)
    kinds = [k for k in cubins if re.fullmatch(r"_Z\d+k_step_\w+_host8StepArgs", k)]
    assert len(kinds) == len(_lib.KINDS)
    for kh in kinds:
        name = re.fullmatch(r"_Z\d+(k_step_\w+)_host8StepArgs", kh).group(1)
        kd = "_Z%d%s8StepArgs" % (len(name), name)
        assert kd in cubins, kd
        assert tool.differences(cubins, kd, kh) == [], name
