"""Definite integrals (NOT in the reference), CPU side: the specification in tests/integral_oracle.cpp against scipy's
PPoly.integrate, exact rational arithmetic and np.trapezoid, the precision of the cumulative table on a long f32 grid,
and the packed-f32 SASS of the new kernels."""
import math
import os
import re
import shutil
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import integral_oracle as I
from oracle import oracle_py as O
from test_deriv_cpu import BCS, _case

scipy_interp = pytest.importorskip("scipy.interpolate")


def _ppoly(x, y, a, b, periodic):
    """the spline (1-t) yl + t yr + t(1-t)(a(1-t) + b t) as a scipy PPoly in powers of (x - x[i]), in f64"""
    x, y, a, b = (np.asarray(v, np.float64) for v in (x, y, a, b))
    h = np.diff(x)[:, None]
    yl, yr = y[:-1], y[1:]
    c = np.stack([(a - b) / h ** 3, (b - 2 * a) / h ** 2, (yr - yl + a) / h, yl])
    return scipy_interp.PPoly(c, x, extrapolate="periodic" if periodic else True)


def _pairs(x, dtype, rng, periodic):
    x0, xn = float(x[0]), float(x[-1])
    P = xn - x0
    lo = rng.uniform(x0, xn, 24)
    hi = rng.uniform(x0, xn, 24)
    pairs = list(zip(lo, hi)) + list(zip(hi[:8], lo[:8]))                     # random and reversed pairs
    pairs += [(float(x[i]), float(x[j])) for i, j in ((0, len(x) - 1), (1, len(x) - 2), (len(x) - 1, 0))]   # knots, ends
    if periodic:                                                               # several periods, both directions
        pairs += [(x0 - 0.3 * P, xn + 2.6 * P), (xn + 3.2 * P, x0 - 0.1 * P), (x0 + 0.4 * P, x0 + 4.4 * P), (xn + 0.2 * P, xn + 0.9 * P)]
    else:                                                                      # extrapolated bounds
        pairs += [(x0 - 0.25, xn + 0.25), (x0 - 0.2, x0 + 0.1), (xn + 0.3, xn - 0.1)]
    arr = np.array(pairs, dtype=dtype)
    return arr[:, 0].copy(), arr[:, 1].copy()


@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-12), (np.float32, 1e-5)])
@pytest.mark.parametrize("bc", BCS)
@pytest.mark.parametrize("n", [3, 5, 50, 400])
def test_cubic_integral_oracle_matches_scipy(bc, n, dtype, tol):
    rng = np.random.default_rng(n * 11 + len(bc))
    x, y, spec, v1, v2 = _case(bc, n, 3, dtype, rng)
    st, a, b = O.spline_build(x, y, spec)
    assert st == O.ST_OK
    periodic = bc == "periodic"
    lo, hi = _pairs(x, dtype, rng, periodic)
    st, got, bad, bound = I.integrate(x, y, a, b, lo, hi, 2 if periodic else 1)
    assert st == O.ST_OK and bad == -1
    pp = _ppoly(x, y, a, b, periodic)
    ref = np.stack([pp.integrate(float(l), float(h)) for l, h in zip(lo, hi)])
    P = float(x[-1]) - float(x[0])
    col = P * np.max(np.abs(y.astype(np.float64)), axis=0)                  # sum of h_i max|y| of the column
    span = np.maximum(1.0, np.abs(hi.astype(np.float64) - lo.astype(np.float64)) / P)[:, None]
    scale = np.maximum(np.abs(ref), col[None, :] * span)
    err = float(np.max(np.abs(got.astype(np.float64) - ref) / scale))
    assert err <= tol, (bc, n, err)
    # equal bounds: exactly zero; reversed bounds: exactly the negative
    st, z, _, _ = I.integrate(x, y, a, b, lo, lo, 2 if periodic else 1)
    assert np.all(z == 0) and not np.any(np.signbit(z))
    st, r, _, _ = I.integrate(x, y, a, b, hi, lo, 2 if periodic else 1)
    assert np.array_equal(r, -got)


def test_cubic_full_period_is_the_last_table_row():
    rng = np.random.default_rng(5)
    x, y, spec, _, _ = _case("periodic", 40, 4, np.float64, rng)
    st, a, b = O.spline_build(x, y, spec)
    cum = I.table(x, y, a, b)
    P = x[-1] - x[0]
    lo = np.array([x[0], x[0] - 3 * P, x[-1] + 5 * P])
    st, got, _, _ = I.integrate(x, y, a, b, lo, lo + P, 2)
    assert st == O.ST_OK and np.allclose(got, cum[-1][None, :], rtol=1e-12, atol=1e-12 * np.abs(cum).max())


def test_integral_errors_report_the_bound():
    x = np.arange(6.0)
    y = np.random.default_rng(1).normal(size=(6, 2))
    st, a, b = O.spline_build(x, y, {"kind": "Natural"})
    lo = np.array([0.5, 1.5, 2.0, 7.0])
    hi = np.array([1.0, 9.0, np.nan, np.nan])
    st, out, bad, bound = I.integrate(x, y, a, b, lo, hi, 0)
    assert (st, bad, bound) == (O.ST_OUT_OF_BOUNDS, 1, 1) and np.all(out[1:] == 0)
    st, out, bad, bound = I.integrate(x, y, a, b, lo, hi, 1)
    assert (st, bad, bound) == (O.ST_NAN_QUERY, 2, 1)
    st, out, bad, bound = I.integrate(x, y, None, None, lo[3:], hi[3:], 0)     # both bounds fail: lo is reported
    assert (st, bad, bound) == (O.ST_OUT_OF_BOUNDS, 0, 0)
    st, out, bad, bound = I.integrate(x, y, a, b, np.array([1.0, np.inf]), np.array([2.0, 1.0]), 2)
    assert (st, bad, bound) == (O.ST_NAN_QUERY, 1, 0)


def _exact_linear(x, y, lo, hi):
    """the integral of the piecewise linear interpolant through the f64 knots, in rationals (extrapolating the edges)"""
    X = [Fraction(float(v)) for v in x]
    Y = [Fraction(float(v)) for v in y]

    def f(i, t):
        return Y[i] + (Y[i + 1] - Y[i]) * (t - X[i]) / (X[i + 1] - X[i])

    def F(u):                                  # antiderivative from x[0]
        u = Fraction(float(u))
        i = min(max(int(np.searchsorted(x, float(u), side="right")) - 1, 0), len(x) - 2)
        s = sum(((X[k + 1] - X[k]) * (Y[k] + Y[k + 1]) / 2 for k in range(i)), Fraction(0))
        return s + (u - X[i]) * (f(i, X[i]) + f(i, u)) / 2
    return float(F(hi) - F(lo))


def test_linear_integral_oracle_against_rationals_and_trapezoid():
    rng = np.random.default_rng(2)
    x = np.cumsum(rng.uniform(0.2, 1.5, 7))
    y = rng.normal(size=(7, 2))
    lo = np.concatenate([rng.uniform(x[0], x[-1], 12), [x[0], x[2], x[0] - 0.5]])
    hi = np.concatenate([rng.uniform(x[0], x[-1], 12), [x[-1], x[2], x[-1] + 0.5]])
    st, got, _, _ = I.integrate(x, y, None, None, lo, hi, 1)
    assert st == O.ST_OK
    scale = (x[-1] - x[0]) * np.abs(y).max()
    for q in range(len(lo)):
        for c in range(2):
            assert abs(got[q, c] - _exact_linear(x, y[:, c], lo[q], hi[q])) <= 1e-13 * scale, (q, c)
    st, knots, _, _ = I.integrate(x, y, None, None, np.full(7, x[0]), x, 0)
    ref = np.stack([np.trapezoid(y[: i + 1], x[: i + 1], axis=0) for i in range(7)])
    assert np.allclose(knots, ref, rtol=0, atol=1e-14 * scale)


def test_f32_table_on_a_long_grid_is_within_one_ulp_of_the_exact_sum():
    """n = 65536 f32: h (y[i] + y[i+1]) * 0.5 is exact in double for f32 inputs, so the exact prefix sums are rationals;
    the table, accumulated in double and rounded once, is within 1 ulp of them rounded to f32"""
    rng = np.random.default_rng(9)
    n = 65536
    x = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(np.float32)
    y = (rng.normal(size=n) + 3.0).astype(np.float32)
    cum = I.table(x, y)
    h = np.diff(x).astype(np.float64)                                       # f32 differences, exact in f64
    e = h * (y[:-1].astype(np.float64) + y[1:].astype(np.float64)) * 0.5   # exact: 24 + 25 bit mantissas
    acc, exact = Fraction(0), [0.0]
    for v in e.tolist():
        acc += Fraction(v)
        exact.append(acc)
    ref = np.array([np.float32(float(v)) for v in exact], dtype=np.float32)
    ulp = np.abs(cum.view(np.int32).astype(np.int64) - ref.view(np.int32).astype(np.int64))
    assert ulp.max() <= 1, int(ulp.max())
    assert math.isclose(float(cum[-1]), float(exact[-1]), rel_tol=1e-7)


def test_packed_f32x2_products_in_the_integral_kernels_are_not_contracted():
    """every sum that takes a packed product is done per half (ndi_device.cuh: ptxas fuses mul.rn.f32x2 + add.rn.f32x2),
    so the f32 integral kernels contain packed products but no FFMA2"""
    from ndarray_interp_b200 import build
    so = build.build()
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    sass = subprocess.check_output([tool, "-sass", so], text=True, stderr=subprocess.DEVNULL)
    seen = 0
    for fn, body in re.findall(r"Function : (\S+)\n(.*?)(?=\n\s+Function : |\Z)", sass, re.S):
        if "integral_kernelIf" not in fn:
            continue
        seen += 1
        assert "FFMA2" not in body, fn
        if re.search(r"integral_kernelIfLi[24]E", fn):
            assert re.search(r"\bFMUL2\b", body), fn
    assert seen == 2 * 3 * 6, seen            # cubic and linear, V = 1, 2, 4, six lanes-per-query counts


def _build_cpp():
    from ndarray_interp_b200.build import build
    build()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "ndarray_interp_b200")
    exe = os.path.join(root, "tests", "cpp", "test_integral.bin")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(root, "include"), os.path.join(root, "tests", "cpp", "test_integral.cpp"),
           "-o", exe, "-L", pkg, "-lndi_b200", "-Wl,-rpath," + pkg, "-Wl,-rpath,/usr/local/cuda/lib64"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return exe


def test_cpp_integral_program_compiles_and_links():
    assert os.path.exists(_build_cpp())


@pytest.mark.gpu
def test_cpp_integral_program_runs():
    r = subprocess.run([_build_cpp()], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert " 0 failures" in r.stdout
