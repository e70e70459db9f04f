"""Derivatives (NOT in the reference), CPU side: the specification in tests/deriv_oracle.cpp against scipy and exact
arithmetic, the packed-f32 SASS of the new kernels, and the C++ program that exercises the mirror's derivative methods."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import deriv_oracle as D
from oracle import oracle_py as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
scipy_interp = pytest.importorskip("scipy.interpolate")


def _rel_err(got, ref):
    """max over elements of |got - ref| / max(|ref|, max |ref| of the column)"""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    scale = np.maximum(np.abs(ref), np.max(np.abs(ref), axis=0, keepdims=True))
    scale = np.where(scale == 0, 1.0, scale)
    return float(np.max(np.abs(got - ref) / scale))


def _grid(n, uniform, dtype, rng):
    g = np.linspace(0.0, 3.0, n) if uniform else np.cumsum(rng.uniform(0.5, 1.5, n))
    return g.astype(dtype)


BCS = ["natural", "clamped", "periodic", "individual", "not-a-knot"]


def _case(bc, n, w, dtype, rng):
    x = _grid(n, bc == "not-a-knot", dtype, rng)      # NotAKnot: uniform grids only (DESIGN.md section 2)
    y = rng.normal(size=(n, w)).astype(dtype)
    if bc == "periodic":
        y[-1] = y[0]
    v1, v2 = rng.normal(size=w).astype(dtype), rng.normal(size=w).astype(dtype)
    spec = {"natural": {"kind": "Natural"}, "clamped": {"kind": "Clamped"}, "periodic": {"kind": "Periodic"},
            "not-a-knot": {"kind": "NotAKnot"},
            "individual": {"kind": "Individual", "rows": [{"kind": "Mixed", "left": {"kind": "FirstDeriv", "value": float(a)},
                                                          "right": {"kind": "SecondDeriv", "value": float(b)}}
                                                         for a, b in zip(v1, v2)]}}[bc]
    return x, y, spec, v1, v2


def _scipy(bc, x, y, v1, v2, q, nu):
    x64, y64 = x.astype(np.float64), y.astype(np.float64)
    if bc == "individual":
        return np.stack([scipy_interp.CubicSpline(x64, y64[:, c], bc_type=((1, float(v1[c])), (2, float(v2[c]))))(q, nu)
                         for c in range(y.shape[1])], axis=1)
    return scipy_interp.CubicSpline(x64, y64, bc_type=bc)(q.astype(np.float64), nu)


@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-12), (np.float32, 1e-5)])
@pytest.mark.parametrize("bc", BCS)
@pytest.mark.parametrize("n", [5, 50, 400])
def test_cubic_deriv_oracle_matches_scipy(bc, n, dtype, tol):
    rng = np.random.default_rng(n * 7 + len(bc))
    w = 3
    x, y, spec, v1, v2 = _case(bc, n, w, dtype, rng)
    st, a, b = O.spline_build(x, y, spec)
    assert st == O.ST_OK
    inside = rng.uniform(x[0], x[-1], 200).astype(dtype)
    q = np.concatenate([inside, x, [x[0], x[-1]]]).astype(dtype)        # knots and both ends
    if bc == "periodic":
        mode, outside = 2, np.array([x[0] - 0.3, x[-1] + 0.7, x[-1] + 3.1], dtype)
    else:
        mode, outside = 1, np.array([x[0] - 0.25, x[-1] + 0.25], dtype)
    q = np.concatenate([q, outside]).astype(dtype)
    for order in (1, 2):
        st, got, bad = D.cubic_deriv(x, y, a, b, q, mode, order)
        assert st == O.ST_OK and bad == -1
        qref = q.astype(np.float64)
        if bc == "periodic":                  # scipy wraps as well, but in f64: wrap as the library does, in dtype
            x0, xn = x[0], x[-1]
            wrapped = np.where((q < x0) | (q > xn), np.mod(q - x0, xn - x0) + x0, q).astype(dtype)
            qref = wrapped.astype(np.float64)
        ref = _scipy(bc, x, y, v1, v2, qref, order)
        err = _rel_err(got, ref)
        assert err <= tol, (bc, n, order, err)


def test_cubic_deriv_errors_and_order():
    x = np.arange(6.0)
    y = np.random.default_rng(1).normal(size=(6, 2))
    st, a, b = O.spline_build(x, y, {"kind": "Natural"})
    q = np.array([0.5, 1.5, 7.0, np.nan])
    st, out, bad = D.cubic_deriv(x, y, a, b, q, 0, 1)
    assert st == O.ST_OUT_OF_BOUNDS and bad == 2 and np.all(out[2:] == 0)
    st, out, bad = D.cubic_deriv(x, y, a, b, q, 1, 2)
    assert st == O.ST_NAN_QUERY and bad == 3
    assert D.cubic_deriv(x, y, a, b, q[:1], 0, 3)[0] == O.ST_INVALID_ARGUMENT


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_linear_slope_oracle_is_the_correctly_rounded_quotient(dtype):
    rng = np.random.default_rng(3)
    x = np.cumsum(rng.uniform(0.1, 2.0, 40)).astype(dtype)
    y = rng.normal(size=(40, 5)).astype(dtype)
    y[7, 0], y[8, 0] = dtype(0.0), -dtype(0.0)            # -0 numerator: the quotient keeps its sign
    q = np.concatenate([rng.uniform(x[0], x[-1], 300), x, [x[7] + (x[8] - x[7]) / 2]]).astype(dtype)
    st, got, _ = D.linear_deriv(x, y, q, False)
    assert st == O.ST_OK
    idx = np.clip(np.searchsorted(x, q, side="right") - 1, 0, len(x) - 2)
    ref = (y[idx + 1] - y[idx]) / (x[idx + 1] - x[idx])[:, None]          # numpy: one rounding per op, in dtype
    assert got.dtype == dtype and np.array_equal(got.view(np.uint8), ref.astype(dtype).view(np.uint8))
    assert np.signbit(got[-1, 0]) and got[-1, 0] == 0


@pytest.mark.parametrize("dtype", [np.int32, np.int64, np.uint32, np.uint64])
def test_linear_slope_oracle_integers_wrap_and_truncate(dtype):
    bits = np.dtype(dtype).itemsize * 8
    signed = np.issubdtype(dtype, np.signedinteger)
    info = np.iinfo(dtype)
    rng = np.random.default_rng(bits + signed)
    x = np.cumsum(rng.integers(1, 50, 30)).astype(dtype)
    y = rng.integers(info.min // 2 if signed else info.max // 4, info.max, size=(30, 4), dtype=dtype)
    q = np.concatenate([rng.integers(int(x[0]), int(x[-1]), 200), x]).astype(dtype)
    st, got, _ = D.linear_deriv(x, y, q, False)
    assert st == O.ST_OK
    mod = 1 << bits

    def wrap(v):
        v %= mod
        return v - mod if signed and v >= mod // 2 else v
    for i, xv in enumerate(q.tolist()):
        k = min(max(int(np.searchsorted(x, xv, side="right")) - 1, 0), len(x) - 2)
        d = wrap(int(x[k + 1]) - int(x[k]))
        for c in range(y.shape[1]):
            num = wrap(int(y[k + 1, c]) - int(y[k, c]))
            quo = abs(num) // abs(d) * (1 if (num >= 0) == (d >= 0) else -1)      # truncating division
            assert int(got[i, c]) == wrap(quo), (i, c)


def test_packed_f32x2_products_in_the_derivative_kernels_are_not_contracted():
    """as test_cabi_symbols.py::test_packed_f32x2_products_are_not_contracted_into_fma for the value kernels: every sum or
    difference that takes a packed product is done per half, so no FFMA2 appears; the packed adds are the two (order 1)
    or one (order 2) subtractions of loaded values per pair of columns, the packed products four per pair"""
    from ndarray_interp_b200 import build
    so = build.build()
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")

    def counts(kernel):
        sass = subprocess.check_output([tool, "-sass", "-fun", kernel, so], text=True, stderr=subprocess.DEVNULL)
        return {op: len(re.findall(r"\b" + op + r"\b", sass)) for op in ("FFMA2", "FMUL2", "FADD2")}
    for lpq in (8, 32):
        for order, adds in ((1, 2), (2, 1)):
            c = counts(f"_ZN3ndi27interp1d_cubic_deriv_kernelIfLi4ELi{lpq}ELi{order}EEEvNS_5Eval1IT_EE")
            assert c["FMUL2"] > 0 and c["FFMA2"] == 0, (lpq, order, c)
            assert c["FADD2"] * 4 == c["FMUL2"] * adds, (lpq, order, c)


def _build_cpp():
    from ndarray_interp_b200.build import build
    build()
    pkg = os.path.join(ROOT, "ndarray_interp_b200")
    exe = os.path.join(ROOT, "tests", "cpp", "test_deriv.bin")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "test_deriv.cpp"),
           "-o", exe, "-L", pkg, "-lndi_b200", "-Wl,-rpath," + pkg, "-Wl,-rpath,/usr/local/cuda/lib64"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return exe


def test_cpp_deriv_program_compiles_and_links():
    assert os.path.exists(_build_cpp())


@pytest.mark.gpu
def test_cpp_deriv_program_runs():
    r = subprocess.run([_build_cpp()], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert " 0 failures" in r.stdout
