"""Shape-preserving cubics built on the GPU (NOT in the reference): ndi_interp1d_hermite_build for PCHIP, Akima,
makima and given slopes, through the Python mirror and the C ABI.  The coefficients must be bit-identical to the
specification in tests/hermite_oracle.cpp, and the value, derivative and integral calls on such a handle bit-identical
to their specifications applied to those coefficients."""
import ctypes as C

import numpy as np
import pytest

import deriv_oracle as D
import hermite_oracle as H
import integral_oracle as I
from ndarray_interp_b200 import BuilderError
from ndarray_interp_b200 import _lib as L
from ndarray_interp_b200.interp1d import (Akima, CubicHermite, CubicSpline, HermiteStrategy, Interp1D, Interp1DBuilder,
                                          Pchip)
from oracle import oracle_py as O
from test_deriv_gpu import _ndev

pytestmark = pytest.mark.gpu

KINDS = [H.PCHIP, H.AKIMA, H.MAKIMA, H.GIVEN]
NAMES = {H.PCHIP: "pchip", H.AKIMA: "akima", H.MAKIMA: "makima", H.GIVEN: "given"}
CASES = ["random", "plateaus", "monotone", "signs", "ties", "scaled", "nan"]
WIDTHS = [1, 2, 3, 4, 5, 8, 31, 64, 1024, 4099]
SIZES = [2, 3, 4, 5, 33, 1000, 4097]


def _same(a, b):
    """bit-identical, except that a NaN may carry any payload (the CPU and the GPU make different NaNs)"""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint8), b[~nb].view(np.uint8))


def _grid(n, uniform, rng, dtype):
    return (np.arange(n) * 0.5 + 1.0 if uniform else np.cumsum(rng.uniform(0.1, 2.0, n))).astype(dtype)


def _data(case, n, w, rng, dtype):
    y = rng.standard_normal((n, w))
    if case == "plateaus":
        y = np.round(y)
    elif case == "monotone":
        y = np.cumsum(np.abs(y) * (rng.uniform(size=(n, w)) < 0.7), axis=0)
    elif case == "signs":
        y = np.cumsum(np.sign(rng.standard_normal((n, w))), axis=0) * 0.5
    elif case == "ties":
        y = np.repeat(np.arange(n)[:, None] // 3, w, axis=1).astype(float)     # equal neighbouring slopes: Akima's fallback
    elif case == "scaled":
        y[:, 0] *= 1e12                                    # the global maximum of f12 decides the other columns
    elif case == "nan":
        y[n // 2, w // 2] = np.nan
    return y.astype(dtype)


def _builder(kind, dydx=None, extrapolate=False):
    if kind == H.PCHIP:
        s = Pchip.new()
    elif kind == H.GIVEN:
        s = CubicHermite.new(dydx)
    else:
        s = Akima.new().method("akima" if kind == H.AKIMA else "makima")
    return s.extrapolate(extrapolate)


def _build(x, y, kind, rng, extrapolate=False):
    dydx = rng.standard_normal(y.shape).astype(y.dtype) if kind == H.GIVEN else None
    ip = Interp1DBuilder.new(y).x(x).strategy(_builder(kind, dydx, extrapolate)).build()
    return ip, dydx


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("w", WIDTHS)
def test_coefficients_bit_identical_to_the_specification(dtype, w):
    rng = np.random.default_rng(w * 7 + np.dtype(dtype).itemsize)
    for j, n in enumerate(SIZES):
        if n * w > 5_000_000:
            continue
        for kind in KINDS:
            case = CASES[(j + kind + w) % len(CASES)]
            x = _grid(n, (j + kind) % 2 == 0, rng, dtype)
            y = _data(case, n, w, rng, dtype)
            ip, dydx = _build(x, y.reshape((n,) + ((w,) if w > 1 else ())), kind, rng)
            a, b = ip.strategy.coefficients(ip)
            _, wa, wb = H.hermite(x, y, kind, None if dydx is None else dydx.reshape(n, w))
            assert _same(a.reshape(n - 1, w), wa) and _same(b.reshape(n - 1, w), wb), (NAMES[kind], n, case)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("case", CASES)
def test_every_data_case_on_every_width_class(kind, case):
    rng = np.random.default_rng(kind * 31 + CASES.index(case))
    for dtype in (np.float32, np.float64):
        for n, w in ((5, 1), (33, 3), (64, 4), (40, 8), (17, 33)):
            x = _grid(n, False, rng, dtype)
            y = _data(case, n, w, rng, dtype)
            ip, dydx = _build(x, y, kind, rng)
            a, b = ip.strategy.coefficients(ip)
            _, wa, wb = H.hermite(x, y, kind, dydx)
            assert _same(a, wa) and _same(b, wb), (NAMES[kind], case, n, w, dtype)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n", [2, 3, 4, 5, 200])
def test_value_derivative_and_integral_calls_on_hermite_handles(dtype, n):
    """n == 2 included: the first handles with cubic coefficients and two knots"""
    rng = np.random.default_rng(n + np.dtype(dtype).itemsize)
    for kind in KINDS:
        for w in (1, 4, 37):
            x = _grid(n, kind % 2 == 1, rng, dtype)
            y = _data("random", n, w, rng, dtype)
            ip, dydx = _build(x, y, kind, rng, extrapolate=True)
            _, a, b = H.hermite(x, y, kind, dydx)
            q = np.concatenate([rng.uniform(x[0], x[-1], 500), x, [x[0] - 0.7, x[-1] + 1.3]]).astype(dtype)
            st, want, _ = O.interp1d_cubic(x, y, a, b, q, 1)
            assert st == 0 and _same(ip.interp_array(q), want), (NAMES[kind], w)
            for order in (1, 2):
                st, want, _ = D.cubic_deriv(x, y, a, b, q, 1, order)
                assert st == 0 and _same(ip.interp_array_deriv(q, order), want), (NAMES[kind], w, order)
            lo = rng.uniform(x[0] - 0.5, x[-1] + 0.5, 300).astype(dtype)
            hi = rng.uniform(x[0] - 0.5, x[-1] + 0.5, 300).astype(dtype)
            st, want, _, _ = I.integrate(x, y, a, b, lo, hi, 1)
            assert st == 0 and _same(ip.interp_array_integral(lo, hi), want), (NAMES[kind], w)
            # the table the integral calls read, built at n == 2 too
            cum = ip.interp_array_integral(np.full(n, x[0]), x)
            assert _same(cum[:-1], I.table(x, y, a, b)[:-1])


def test_given_slopes_from_device_pointers():
    import torch
    rng = np.random.default_rng(5)
    for dtype, tdt in ((np.float32, torch.float32), (np.float64, torch.float64)):
        n, w = 300, 6
        x = _grid(n, False, rng, dtype)
        y = _data("random", n, w, rng, dtype)
        dydx = rng.standard_normal((n, w)).astype(dtype)
        ip = Interp1DBuilder.new(y).x(x).strategy(Pchip.new()).build()
        dev = torch.from_numpy(dydx).to("cuda")
        torch.cuda.synchronize()
        assert L.check(L.load().ndi_interp1d_hermite_build(ip._handle(), L.HERMITE_GIVEN, C.c_void_p(dev.data_ptr()),
                                                           L.DEVICE_POINTERS)) == L.OK
        a, b = ip.strategy.coefficients(ip)
        _, wa, wb = H.hermite(x, y, H.GIVEN, dydx)
        assert _same(a, wa) and _same(b, wb)
        # an odd offset into a device buffer: no 16-byte alignment, the single-column path
        big = torch.from_numpy(np.concatenate([[0.0], dydx.reshape(-1)]).astype(dtype)).to("cuda")
        torch.cuda.synchronize()
        L.check(L.load().ndi_interp1d_hermite_build(ip._handle(), L.HERMITE_GIVEN,
                                                    C.c_void_p(big.data_ptr() + np.dtype(dtype).itemsize), L.DEVICE_POINTERS))
        a, b = ip.strategy.coefficients(ip)
        assert _same(a, wa) and _same(b, wb)


def _status(h, kind, dydx, flags=0):
    return L.load().ndi_interp1d_hermite_build(h, kind, dydx, flags)


def test_error_statuses_and_a_failed_build_keeps_the_coefficients():
    rng = np.random.default_rng(9)
    x = _grid(20, False, rng, np.float64)
    y = _data("random", 20, 3, rng, np.float64)
    ip = Interp1DBuilder.new(y).x(x).strategy(Pchip.new()).build()
    h = ip._handle()
    a0, b0 = ip.strategy.coefficients(ip)
    d = np.zeros((20, 3))
    assert _status(h, 4, None) == L.INVALID_ARGUMENT
    assert _status(h, -1, None) == L.INVALID_ARGUMENT
    assert _status(h, L.HERMITE_GIVEN, None) == L.INVALID_ARGUMENT
    assert _status(h, L.HERMITE_PCHIP, L.ptr(d)) == L.INVALID_ARGUMENT
    assert _status(None, L.HERMITE_PCHIP, None) == L.INVALID_ARGUMENT
    a1, b1 = ip.strategy.coefficients(ip)
    assert _same(a0, a1) and _same(b0, b1)
    lv = C.c_int32(0)
    L.check(L.load().ndi_interp1d_build_info(h, C.byref(lv)))
    assert lv.value == L.BUILD_INFO_HERMITE + L.HERMITE_PCHIP
    for dt in (np.int32, np.int64, np.uint32, np.uint64):
        hi = C.c_void_p()
        xi, yi = np.arange(5).astype(dt), np.arange(10).astype(dt).reshape(5, 2)
        L.check(L.load().ndi_interp1d_create(L.dtype_code(np.dtype(dt)), L.ptr(xi), 5, L.ptr(yi), 2, L.ASSUME_VALID,
                                             C.byref(hi)))
        assert _status(hi, L.HERMITE_PCHIP, None) == L.UNSUPPORTED_DTYPE
        L.load().ndi_interp1d_destroy(hi)
    with pytest.raises(TypeError):
        Interp1DBuilder.new(np.arange(5)).strategy(Pchip.new()).build()
    with pytest.raises(BuilderError.ShapeError):
        Interp1DBuilder.new(y).x(x).strategy(CubicHermite.new(np.zeros((20, 2)))).build()
    with pytest.raises(BuilderError.NotEnoughData):
        Interp1DBuilder.new(np.array([1.0])).strategy(Akima.new()).build()


def test_build_info_rebuild_and_integral_table_drop():
    rng = np.random.default_rng(13)
    n, w = 50, 4
    x = _grid(n, False, rng, np.float64)
    y = _data("random", n, w, rng, np.float64)
    ip = Interp1DBuilder.new(y).x(x).strategy(CubicSpline.new().extrapolate(True)).build()
    h = ip._handle()
    lo, hi = np.array([x[1]]), np.array([x[-3]])
    ip.prepare_integral()
    out, bad, bound = np.zeros((1, w)), C.c_int64(-1), C.c_int32(-1)
    assert L.load().ndi_interp1d_cubic_integral(h, L.ptr(lo), L.ptr(hi), 1, 1, L.ptr(out), C.byref(bad), C.byref(bound)) == 0
    for kind in (H.AKIMA, H.MAKIMA, H.PCHIP):
        assert _status(h, kind, None) == L.OK
        lv = C.c_int32(0)
        L.check(L.load().ndi_interp1d_build_info(h, C.byref(lv)))
        assert lv.value == L.BUILD_INFO_HERMITE + kind
        assert L.load().ndi_interp1d_cubic_integral(h, L.ptr(lo), L.ptr(hi), 1, 1, L.ptr(out), C.byref(bad),
                                                    C.byref(bound)) == L.NO_INTEGRAL
        a, b = ip.strategy.coefficients(ip)
        _, wa, wb = H.hermite(x, y, kind)
        assert _same(a, wa) and _same(b, wb)
        L.check(L.load().ndi_interp1d_integral_build(h, L.INTEGRAL_CUBIC))
    # a spline build replaces Hermite coefficients again
    L.check(L.load().ndi_interp1d_spline_build(h, 0, None, None, None, None, None))
    a, b = ip.strategy.coefficients(ip)
    lv = C.c_int32(0)
    L.check(L.load().ndi_interp1d_build_info(h, C.byref(lv)))
    assert lv.value < L.BUILD_INFO_HERMITE
    _, wa, _ = H.hermite(x, y, H.PCHIP)
    assert not _same(a, wa)
    # the mirror builds the dropped table again on first use
    p = Interp1DBuilder.new(y).x(x).strategy(Pchip.new().extrapolate(True)).build()
    _, pa, pb = H.hermite(x, y, H.PCHIP)
    _, want, _, _ = I.integrate(x, y, pa, pb, lo, hi, 1)
    assert _same(p.integrate(lo, hi), want)
    assert isinstance(p.strategy, HermiteStrategy) and p.strategy.build_info(p) == L.BUILD_INFO_HERMITE


def test_clone_to_device_and_group_calls():
    rng = np.random.default_rng(17)
    n, w = 400, 8
    x = _grid(n, False, rng, np.float64)
    y = _data("monotone", n, w, rng, np.float64)
    ip = Interp1DBuilder.new(y).x(x).strategy(Akima.new().method("makima").extrapolate(True)).build()
    _, a, b = H.hermite(x, y, H.MAKIMA)
    clone = C.c_void_p()
    L.check(L.load().ndi_interp1d_clone_to_device(ip._handle(), 0, C.byref(clone)))
    ca, cb = np.zeros_like(a), np.zeros_like(b)
    L.check(L.load().ndi_interp1d_spline_coeffs(clone, L.ptr(ca), L.ptr(cb)))
    L.load().ndi_interp1d_destroy(clone)
    assert _same(ca, a) and _same(cb, b)
    q = rng.uniform(x[0], x[-1], 40000)
    lo, hi = q[:-1].copy(), q[1:].copy()
    ip.prepare_integral()
    grp = ip.replicate(list(range(max(1, min(_ndev(), 2)))))
    _, want, _ = O.interp1d_cubic(x, y, a, b, q, 1)
    assert _same(grp.interp_array(q), want)
    _, want, _ = D.cubic_deriv(x, y, a, b, q, 1, 1)
    assert _same(grp.interp_array_deriv(q, 1), want)
    _, want, _, _ = I.integrate(x, y, a, b, lo, hi, 1)
    assert _same(grp.interp_array_integral(lo, hi), want)


@pytest.mark.skipif(_ndev() < 2, reason="needs two GPUs")
def test_clone_to_a_second_device():
    rng = np.random.default_rng(19)
    x = _grid(300, False, rng, np.float32)
    y = _data("plateaus", 300, 5, rng, np.float32)
    ip = Interp1DBuilder.new(y).x(x).strategy(Pchip.new()).build()
    _, a, b = H.hermite(x, y, H.PCHIP)
    clone = C.c_void_p()
    L.check(L.load().ndi_interp1d_clone_to_device(ip._handle(), 1, C.byref(clone)))
    ca, cb = np.zeros_like(a), np.zeros_like(b)
    L.check(L.load().ndi_interp1d_spline_coeffs(clone, L.ptr(ca), L.ptr(cb)))
    L.load().ndi_interp1d_destroy(clone)
    assert _same(ca, a) and _same(cb, b)


def test_unchecked_constructor_and_the_mirror_match_the_c_calls():
    rng = np.random.default_rng(23)
    n = 64
    x = _grid(n, False, rng, np.float64)
    y = _data("signs", n, 3, rng, np.float64).reshape(n, 3)
    ip = Interp1D.new_unchecked(x, y, Pchip.new().build(x, y))
    _, a, b = H.hermite(x, y, H.PCHIP)
    q = rng.uniform(x[0], x[-1], 100)
    out, bad = np.zeros((100, 3)), C.c_int64(-1)
    L.check(L.load().ndi_interp1d_cubic(ip._handle(), L.ptr(q), 100, 0, L.ptr(out), C.byref(bad)))
    assert _same(ip.interp_array(q), out)
    _, want, _ = O.interp1d_cubic(x, y, a, b, q, 0)
    assert _same(out, want)


def test_one_built_strategy_binds_to_several_interpolators():
    """a built strategy may be handed to more than one interpolator, as a CubicSplineStrategy can; given slopes too"""
    rng = np.random.default_rng(37)
    n = 40
    x = _grid(n, False, rng, np.float64)
    y = _data("random", n, 2, rng, np.float64)
    dydx = rng.standard_normal((n, 2))
    for kind in KINDS:
        strat = _builder(kind, dydx).build(x, y)
        _, wa, wb = H.hermite(x, y, kind, dydx if kind == H.GIVEN else None)
        for _ in range(2):
            ip = Interp1D.new_unchecked(x, y, strat)
            a, b = ip.strategy.coefficients(ip)
            assert _same(a, wa) and _same(b, wb), NAMES[kind]


def test_c2_size_pchip_sampled():
    """4096 x 1024 f64 PCHIP, the C2 shape, against the specification on sampled columns"""
    rng = np.random.default_rng(29)
    n, w = 4096, 1024
    x = np.cumsum(rng.uniform(0.5, 1.5, n))
    y = np.cumsum(rng.standard_normal((n, w)), axis=0)
    ip = Interp1DBuilder.new(y).x(x).strategy(Pchip.new()).build()
    a, b = ip.strategy.coefficients(ip)
    cols = np.sort(rng.choice(w, 48, replace=False))
    _, wa, wb = H.hermite(x, np.ascontiguousarray(y[:, cols]), H.PCHIP)
    assert _same(a[:, cols], wa) and _same(b[:, cols], wb)
