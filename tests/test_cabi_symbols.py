"""CPU-side checks of the drop-in boundary: the library builds/loads and exports every symbol
include/ndi_b200.h declares; the product path fails loudly without a GPU (no CPU fallback)."""
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "ndi_b200.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ndi_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_and_exports_every_declared_symbol():
    from ndarray_interp_b200 import build
    so = build.build()
    out = subprocess.check_output(["nm", "-D", "--defined-only", so], text=True)
    exported = set(re.findall(r" T (ndi_[a-z0-9_]+)", out))
    declared = _declared()
    assert len(declared) >= 25
    missing = [s for s in declared if s not in exported]
    assert not missing, f"declared in ndi_b200.h but not exported: {missing}"


def test_ctypes_signatures_cover_the_header():
    from ndarray_interp_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared()
    lib = _lib.load()                      # types every entry point; AttributeError if one is missing
    assert b"sm_100a" in lib.ndi_version_string()


def test_no_torch_types_in_the_abi():
    src = open(HEADER).read()
    assert "torch" not in src.lower().replace("no torch", "") and "at::" not in src and "Tensor" not in src


def test_product_does_not_touch_the_oracle():
    """the product package must never import / link / call anything under oracle/"""
    pkg = os.path.join(ROOT, "ndarray_interp_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                for pat in (r"libndi_oracle", r"oracle_py", r"\bora_[a-z]", r"from\s+oracle", r"import\s+oracle",
                            r"#include[^\n]*oracle", r"oracle/"):
                    assert not re.search(pat, text), f"{f} uses the oracle ({pat})"
    out = subprocess.check_output(["ldd", os.path.join(pkg, "libndi_b200.so")], text=True)
    assert "oracle" not in out


def test_fails_loudly_without_a_gpu():
    import ctypes as C

    from ndarray_interp_b200 import _lib
    from ndarray_interp_b200.interp1d import Interp1D
    n = C.c_int32(0)
    if _lib.load().ndi_device_count(C.byref(n)) == _lib.OK and n.value >= 1:
        pytest.skip("a CUDA device is visible: only meaningful on a machine without a GPU")
    with pytest.raises(_lib.NdiLibraryError, match="no CPU fallback"):
        Interp1D.builder(np.array([1.0, 2.0, 3.0])).build()


def test_packed_f32x2_products_are_not_contracted_into_fma():
    """ptxas 12.9 fuses mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (one rounding where the reference rounds twice; found
    by the GPU parity tests).  The kernels therefore add products per half with scalar adds (csrc/ndi_device.cuh).
    Here, without a GPU: in the built library every packed FMA of the thin-row kernels is one of the two explicit
    fmas of the exact division (as many FFMA2 as FMUL2 in lerp / bilerp, none at all in the cubic form)."""
    import shutil
    so = os.path.join(ROOT, "ndarray_interp_b200", "libndi_b200.so")
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")

    def counts(kernel):
        sass = subprocess.check_output([tool, "-sass", "-fun", kernel, so], text=True, stderr=subprocess.DEVNULL)
        return {op: len(re.findall(r"\b" + op + r"\b", sass)) for op in ("FFMA2", "FMUL2", "FADD2")}
    lin = counts("_ZN3ndi22interp1d_linear_kernelIfLi4ELi4EEEvNS_5Eval1IT_EE")
    pair = counts("_ZN3ndi27interp1d_linear_pair_kernelIfLi4EEEvNS_5Eval1IT_EE")
    bil = counts("_ZN3ndi24interp2d_bilinear_kernelIfLi4ELi8ELb1EEEvNS_5Eval2IT_EE")
    cub = counts("_ZN3ndi21interp1d_cubic_kernelIfLi4ELi8EEEvNS_5Eval1IT_EE")
    for c in (lin, pair, bil):
        assert c["FMUL2"] > 0 and c["FFMA2"] == c["FMUL2"], c      # per pair of columns: q0 = a r, m dq | two fmas of div_by
        assert c["FADD2"] * 2 <= c["FMUL2"], c                      # only the subtractions are packed adds
    assert cub["FMUL2"] > 0 and cub["FFMA2"] == 0 and cub["FADD2"] == 0, cub
