"""The specification of ndi_interp1d_hermite_build (tests/hermite_oracle.cpp) against scipy, without a GPU: in f64 the
knot slopes of PCHIP, Akima and makima are scipy's bit for bit -- all n of them, taken from the dydx scipy hands to
CubicHermiteSpline.__init__ --, and the interpolant agrees with scipy's to 1e-12 (f64) / 1e-5 (f32) of the column's
scale.  Also: given slopes against CubicHermiteSpline, PCHIP's monotonicity, the SASS of the new kernels and the C++
mirror program."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import scipy.interpolate as si

import deriv_oracle as D
import hermite_oracle as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def scipy_slopes(monkeypatch):
    """the dydx PchipInterpolator / Akima1DInterpolator pass to CubicHermiteSpline.__init__ (.c[2] misses d[n-1])"""
    seen = {}
    orig = si.CubicHermiteSpline.__init__

    def wrapped(self, x, y, dydx, *args, **kw):
        seen["d"] = np.array(dydx, copy=True)
        return orig(self, x, y, dydx, *args, **kw)
    monkeypatch.setattr(si.CubicHermiteSpline, "__init__", wrapped)

    def slopes(kind, x, y):
        if kind == H.PCHIP:
            f = si.PchipInterpolator(x, y)
        else:
            f = si.Akima1DInterpolator(x, y, method="akima" if kind == H.AKIMA else "makima")
        return seen["d"].reshape(y.shape), f
    return slopes


def _case(rng, t):
    n = int([2, 3, 4, 5, rng.integers(6, 80)][t % 5])
    w = int(rng.integers(1, 5))
    x = np.cumsum(rng.uniform(0.05, 2.0, n)) if t % 4 else np.arange(n) * 0.25
    y = rng.standard_normal((n, w))
    k = t % 6
    if k == 1:
        y = np.round(y)                                            # plateaus
    elif k == 2:
        y = np.cumsum(np.abs(y) * (rng.uniform(size=(n, w)) < 0.6), axis=0)   # monotone with flat runs
    elif k == 3:
        y = np.cumsum(np.sign(rng.standard_normal((n, w))), axis=0)           # sign changes, equal slopes
    elif k == 4:
        y = np.repeat((np.arange(n) // 3)[:, None], w, axis=1) * 1.0          # exact ties: Akima's fallback
    elif k == 5 and w > 1:
        y[:, 0] *= 1e12                                            # the global maximum M decides the other columns
    return x, y


def _bits(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


@pytest.mark.parametrize("kind", [H.PCHIP, H.AKIMA, H.MAKIMA])
def test_f64_slopes_are_scipys_bit_for_bit(kind, scipy_slopes):
    rng = np.random.default_rng(100 + kind)
    for t in range(300):
        x, y = _case(rng, t)
        want, _ = scipy_slopes(kind, x, y)
        d, _, _ = H.hermite(x, y, kind)
        assert _bits(d, want), (kind, t, len(x), y.shape)


@pytest.mark.parametrize("kind", [H.PCHIP, H.AKIMA, H.MAKIMA])
def test_one_column_slopes_and_a_column_scaled_by_1e12(kind, scipy_slopes):
    rng = np.random.default_rng(7 + kind)
    for n in (2, 3, 4, 5, 17):
        x = np.cumsum(rng.uniform(0.1, 1.0, n))
        y = rng.standard_normal(n)
        want, _ = scipy_slopes(kind, x, y)
        assert _bits(H.hermite(x, y, kind)[0], want)
    # a nearly straight column next to one 1e12 times larger: with the table's maximum the small column's f12 falls
    # below 1e-9 M and takes the fallback, with its own maximum it would not
    x = np.arange(12) * 1.0
    small = 1e-3 * x + 1e-9 * rng.standard_normal(12)
    y = np.stack([small, 1e12 * rng.standard_normal(12)], axis=1)
    want, _ = scipy_slopes(kind, x, y)
    d, _, _ = H.hermite(x, y, kind)
    assert _bits(d, want)
    if kind != H.PCHIP:
        alone, _, _ = H.hermite(x, np.ascontiguousarray(y[:, :1]), kind)
        assert not _bits(alone[:, 0], d[:, 0])


def test_nan_in_the_data():
    """scipy refuses non-finite data, the device build does not: a NaN reaches PCHIP's slopes only at the knots next to
    it (sign(NaN) never equals a sign, so those interior knots get 0), and it makes Akima's M NaN, so every knot of
    every column takes the fallback 0.5 (m[i+1] + m[i-2]), as numpy's comparison with NaN would"""
    rng = np.random.default_rng(3)
    x = np.cumsum(rng.uniform(0.5, 1.5, 15))
    y = rng.standard_normal((15, 3))
    y[6, 1] = np.nan
    d, _, _ = H.hermite(x, y, H.PCHIP)
    for c in (0, 2):
        assert _bits(d[:, c], H.hermite(x, np.ascontiguousarray(y[:, c]), H.PCHIP)[0])
    assert np.all(d[5:8, 1] == 0)
    for kind in (H.AKIMA, H.MAKIMA):
        d, _, _ = H.hermite(x, y, kind)
        m = np.diff(y[:, 0]) / np.diff(x)
        mp = np.concatenate([[0, 0], m, [0, 0]])
        mp[1] = 2 * mp[2] - mp[3]
        mp[0] = 2 * mp[1] - mp[2]
        mp[-2] = 2 * mp[-3] - mp[-4]
        mp[-1] = 2 * mp[-2] - mp[-3]
        assert _bits(d[:, 0], 0.5 * (mp[3:] + mp[:-3]))


@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-12), (np.float32, 1e-5)])
@pytest.mark.parametrize("kind", [H.PCHIP, H.AKIMA, H.MAKIMA])
def test_values_match_scipys_interpolant(kind, dtype, tol, scipy_slopes):
    from oracle import oracle_py as O
    rng = np.random.default_rng(11 + kind)
    for t in range(40):
        x, y = _case(rng, t)
        _, f = scipy_slopes(kind, x, y)
        xd, yd = x.astype(dtype), y.astype(dtype)
        _, a, b = H.hermite(xd, yd, kind)
        q = np.sort(rng.uniform(xd[0], xd[-1], 200)).astype(dtype)
        st, got, _ = O.interp1d_cubic(xd, yd, a, b, q, 0)
        assert st == 0
        scale = np.maximum(np.max(np.abs(y), axis=0), 1e-300)
        err = np.max(np.abs(got - f(q.astype(np.float64))) / scale)
        assert err <= tol, (kind, t, err)


def test_given_slopes_against_cubic_hermite_spline():
    from oracle import oracle_py as O
    rng = np.random.default_rng(21)
    for n in (2, 3, 9, 100):
        x = np.cumsum(rng.uniform(0.1, 2.0, n))
        y = rng.standard_normal((n, 3))
        dydx = rng.standard_normal((n, 3))
        d, a, b = H.hermite(x, y, H.GIVEN, dydx)
        assert _bits(d, dydx)
        f = si.CubicHermiteSpline(x, y, dydx)
        q = rng.uniform(x[0], x[-1], 300)
        _, got, _ = O.interp1d_cubic(x, y, a, b, q, 0)
        assert np.max(np.abs(got - f(q))) <= 1e-12 * max(1.0, np.max(np.abs(y)), np.max(np.abs(dydx)) * np.max(np.diff(x)))
        st, der, _ = D.cubic_deriv(x, y, a, b, x[:-1], 0, 1)
        assert np.max(np.abs(der - dydx[:-1])) <= 1e-12 * max(1.0, np.max(np.abs(dydx)))


def test_pchip_is_monotone_on_monotone_data():
    from oracle import oracle_py as O
    rng = np.random.default_rng(31)
    for dtype in (np.float32, np.float64):
        x = np.cumsum(rng.uniform(0.1, 3.0, 60)).astype(dtype)
        y = np.cumsum(np.abs(rng.standard_normal((60, 4))) * (rng.uniform(size=(60, 4)) < 0.5), axis=0).astype(dtype)
        _, a, b = H.hermite(x, y, H.PCHIP)
        q = np.linspace(x[0], x[-1], 20000).astype(dtype)
        _, v, _ = O.interp1d_cubic(x, y, a, b, q, 0)
        # up to the rounding of the evaluation itself (a few ulp of the column's scale)
        slack = -4 * np.finfo(dtype).eps * np.max(np.abs(y), axis=0)
        assert np.all(np.diff(v.astype(np.float64), axis=0) >= slack), dtype


def test_bad_arguments_are_refused():
    x = np.arange(4.0)
    y = np.zeros((4, 2))
    for kind, d in ((4, None), (H.GIVEN, None), (H.PCHIP, np.zeros((4, 2)))):
        with pytest.raises(ValueError):
            H.hermite(x, y, kind, d)


def test_new_kernels_have_no_fused_packed_multiply_add():
    """-fmad=false keeps scalar products and sums apart; ptxas fuses PACKED products and sums (FFMA2), so the f32
    kernels must not contain any FFMA2 (they pack nothing: one rounding per operation, as the specification)"""
    from ndarray_interp_b200 import build
    so = build.build()
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    sass = subprocess.check_output([tool, "-sass", so], text=True, stderr=subprocess.DEVNULL)
    funcs = re.split(r"\n\s+Function : ", sass)
    hermite = [f for f in funcs if f.startswith("_ZN3ndi21hermite_coeffs_kernel") or f.startswith("_ZN3ndi22hermite_f12_max_kernel")]
    assert len(hermite) == 24, len(hermite)                       # 4 kinds x 2 types x 2 widths + 2 x 2 x 2 max passes
    for f in hermite:
        assert not re.search(r"\bFFMA2\b", f), f.split("\n", 1)[0]


def _build_cpp():
    from ndarray_interp_b200.build import build
    build()
    pkg = os.path.join(ROOT, "ndarray_interp_b200")
    exe = os.path.join(ROOT, "tests", "cpp", "test_hermite.bin")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "test_hermite.cpp"),
           "-o", exe, "-L", pkg, "-lndi_b200", "-Wl,-rpath," + pkg, "-Wl,-rpath,/usr/local/cuda/lib64"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return exe


def test_cpp_hermite_program_compiles_and_links():
    assert os.path.exists(_build_cpp())


@pytest.mark.gpu
def test_cpp_hermite_program_runs():
    r = subprocess.run([_build_cpp()], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert " 0 failures" in r.stdout
