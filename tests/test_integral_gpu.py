"""Definite integrals on the GPU (NOT in the reference): ndi_interp1d_integral_build, ndi_interp1d_cubic_integral /
ndi_interp1d_linear_integral and their _dev and group forms, through the Python mirror, compared bit for bit with the
specification in tests/integral_oracle.cpp applied to the coefficients the handle itself holds.  Each bound is handled
as the value call handles a query: the first failing bound (lo before hi), rows at and after its query untouched."""
import ctypes as C

import numpy as np
import pytest

import integral_oracle as I
from ndarray_interp_b200 import InterpolateError
from ndarray_interp_b200 import _lib as L
from ndarray_interp_b200.errors import Panic, rust_debug
from ndarray_interp_b200.interp1d import Interp1D, Interp1DBuilder, Interp1DStrategy, Linear
from test_deriv_gpu import BOUNDARIES, SENTINEL, SOLVERS, WIDTHS, _bits_equal, _ndev, _out_buffer, _spline

pytestmark = pytest.mark.gpu


def _pairs(kind, x, nq, rng, dtype):
    """(lo, hi): consecutive sorted bins, dense pairs inside one interval, or random pairs (reversed ones included)"""
    if kind == "bins":
        e = np.sort(rng.uniform(x[0], x[-1], nq + 1)).astype(dtype)
        lo, hi = e[:-1].copy(), e[1:].copy()
    elif kind == "dense":
        e = np.sort(rng.uniform(x[3], x[4], nq + 1)).astype(dtype)
        lo, hi = e[:-1].copy(), e[1:].copy()
    else:
        lo = rng.uniform(x[0], x[-1], nq).astype(dtype)
        hi = rng.uniform(x[0], x[-1], nq).astype(dtype)
    k = min(len(x) - 1, nq)
    lo[:k], hi[:k] = x[:k], x[1:k + 1]                     # knot to knot
    lo[k // 2] = hi[k // 2]                                # equal bounds
    return lo, hi


def _extend(lo, hi, x, mode, dtype):
    P = float(x[-1] - x[0])
    if mode == 1:
        lo[-3:] = np.array([x[0] - 1.5, x[-1] + 0.5, x[5]], dtype)
        hi[-3:] = np.array([x[-1] + 2.25, x[2], x[-1] + 3.0], dtype)
    elif mode == 2:
        lo[-4:] = np.array([x[0] - 2.3 * P, x[-1] + 5.1 * P, x[7], x[3]], dtype)
        hi[-4:] = np.array([x[-1] + 3.7 * P, x[0] - 0.4 * P, x[7] + P, x[3] - 4 * P], dtype)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("w", WIDTHS)
def test_cubic_integral_bits_equal_the_oracle_on_the_handles_coefficients(dtype, w):
    rng = np.random.default_rng(w + 3 * (dtype == np.float32))
    n = 300
    nq = 2000 if w < 1000 else 1200
    x = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(dtype)
    y = rng.normal(size=(n, w)).astype(dtype)
    y[-1] = y[0]
    for i, kind in enumerate(BOUNDARIES):
        solver = ["auto"] + SOLVERS
        ip = _spline(x, y, kind, True, solver[(i + w) % 4], rng)
        a, b = ip.strategy.coefficients(ip)
        mode = 2 if kind == "Periodic" else 1
        lo, hi = _pairs(["bins", "dense", "random"][(i + w) % 3], x, nq, rng, dtype)
        _extend(lo, hi, x, mode, dtype)
        st, want, _, _ = I.integrate(x, y, a, b, lo, hi, mode)
        assert st == 0
        got = ip.interp_array_integral(lo, hi)
        assert _bits_equal(got, want), (kind, w)
        z = got[np.nonzero(lo == hi)[0]]
        assert np.all(z == 0)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_cubic_integral_every_search_mode_and_extrapolation_mode(dtype):
    from ndarray_interp_b200.interp1d import BoundaryCondition, CubicSpline
    rng = np.random.default_rng(11)
    n, w, nq = 200, 16, 5000
    x = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(dtype)
    y = rng.normal(size=(n, w)).astype(dtype)
    y[-1] = y[0]
    for kind, extrapolate, mode in (("Natural", False, 0), ("Natural", True, 1), ("Periodic", True, 2)):
        ip = Interp1DBuilder.new(y).x(x).strategy(CubicSpline.new().boundary(getattr(BoundaryCondition, kind))
                                                  .extrapolate(extrapolate)).build()
        a, b = ip.strategy.coefficients(ip)
        lo, hi = _pairs("bins", x, nq, rng, dtype)
        if mode:
            _extend(lo, hi, x, mode, dtype)
        _, want, _, _ = I.integrate(x, y, a, b, lo, hi, mode)
        for sm in range(6):
            L.check(L.load().ndi_interp1d_set_search_mode(ip._handle(), sm))
            assert _bits_equal(ip.interp_array_integral(lo, hi), want), (kind, sm)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("w", [1, 2, 3, 4, 8, 16, 33, 100, 1025])     # 16 - 64-byte rows: the pair-table widths
def test_linear_integral_bits_equal_the_oracle(dtype, w):
    rng = np.random.default_rng(w * 13 + np.dtype(dtype).itemsize)
    n, nq = 120, 3000
    x = np.cumsum(rng.uniform(0.25, 2.0, n)).astype(dtype)
    y = rng.normal(size=(n, w)).astype(dtype)
    for extrapolate in (False, True):
        ip = Interp1DBuilder.new(y).x(x).strategy(Linear.new().extrapolate(extrapolate)).build()
        for kind in ("bins", "random"):
            lo, hi = _pairs(kind, x, nq, rng, dtype)
            if extrapolate:
                _extend(lo, hi, x, 1, dtype)
            st, want, _, _ = I.integrate(x, y, None, None, lo, hi, int(extrapolate))
            assert st == 0
            assert _bits_equal(ip.interp_array_integral(lo, hi), want), (w, extrapolate, kind)


@pytest.mark.parametrize("n,w", [(3, 5), (31, 4), (32, 4), (33, 4), (65, 3), (1025, 8), (65536, 1), (40, 1025)])
def test_table_shapes_around_the_block_size(n, w):
    """C[i] (i < n-1) is observable exactly as the integral from x[0] to the knot x[i], where t = 0 makes F vanish; the
    last knot is the end of interval n-2 (t = 1), so that row is checked against the specification"""
    rng = np.random.default_rng(n + w)
    for dtype in (np.float32, np.float64):
        x = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(dtype)
        y = rng.normal(size=(n, w)).astype(dtype)
        cub = _spline(x, y, "Natural", False, "auto", rng)
        a, b = cub.strategy.coefficients(cub)
        lin = Interp1DBuilder.new(y).x(x).strategy(Linear.new()).build()
        lo = np.full(n, x[0])
        for ip, ca, cb in ((cub, a, b), (lin, None, None)):
            got = ip.interp_array_integral(lo, x)
            assert _bits_equal(got[:-1], I.table(x, y, ca, cb)[:-1]), (n, w, dtype)
            assert _bits_equal(got, I.integrate(x, y, ca, cb, lo, x, 0)[1]), (n, w, dtype)


# ---- errors: the value call's semantics, per bound -----------------------------------------------------------------
W = 1024
CASES = [(20, None), (20, 7), (1500, None), (1500, 700), (40_000, None), (40_000, 0), (40_000, 35_000)]


@pytest.fixture(scope="module")
def tables():
    from ndarray_interp_b200.interp1d import BoundaryCondition, CubicSpline
    rng = np.random.default_rng(77)
    g = np.cumsum(rng.uniform(0.5, 1.5, 64))
    y = rng.normal(size=(64, W))
    cub = Interp1DBuilder.new(y).x(g).strategy(CubicSpline.new().boundary(BoundaryCondition.Natural)).build()
    return {"linear": Interp1DBuilder.new(y).x(g).strategy(Linear.new()).build(), "cubic": cub,
            "coeffs": cub.strategy.coefficients(cub), "g": g, "y": y}


def _want(tables, kind, lo, hi, mode, out):
    a, b = tables["coeffs"] if kind == "cubic" else (None, None)
    return I.integrate(tables["g"], tables["y"], a, b, lo, hi, mode, out=out)


@pytest.mark.parametrize("nq,bad", CASES)
@pytest.mark.parametrize("out_kind", ["pageable", "pinned", "strided"])
@pytest.mark.parametrize("kind", ["linear", "cubic"])
@pytest.mark.parametrize("where", ["lo", "hi", "both"])
def test_host_batch_errors_and_untouched_rows(tables, kind, out_kind, nq, bad, where):
    rng = np.random.default_rng(nq + (bad or 0))
    g = tables["g"]
    e = np.sort(rng.uniform(g[0], g[-1], nq + 1))
    lo, hi = e[:-1].copy(), e[1:].copy()
    if bad is not None:
        hi[-1] = g[0] - 0.5
        if where in ("lo", "both"):
            lo[bad] = g[-1] + 1.0 + bad
        if where in ("hi", "both"):
            hi[bad] = g[0] - 2.0 - bad
    st, want, want_bad, want_bound = _want(tables, kind, lo, hi, 0, np.full((nq, W), SENTINEL))
    assert want_bad == (-1 if bad is None else bad)
    out = _out_buffer(out_kind, nq)
    if bad is None:
        tables[kind].interp_array_integral_into(lo, hi, out)
    else:
        assert want_bound == (1 if where == "hi" else 0)
        v = hi[bad] if where == "hi" else lo[bad]
        with pytest.raises(InterpolateError.OutOfBounds) as ex:
            tables[kind].interp_array_integral_into(lo, hi, out)
        assert str(ex.value) == f"x = {rust_debug(v)} is not in range"
    assert np.array_equal(out, want)


def test_nan_bound_panics(tables):
    lo = np.array([1.0, 2.0, 2.5, 3.0])
    hi = np.array([1.5, 2.5, np.nan, 3.5])
    ex = Interp1DBuilder.new(tables["y"]).x(tables["g"]).strategy(Linear.new().extrapolate(True)).build()
    with pytest.raises(Panic):
        ex.interp_array_integral(lo, hi)


def test_dev_error_word_is_two_query_plus_bound(tables):
    import torch
    g = tables["g"]
    nq = 5000
    e = np.sort(np.random.default_rng(5).uniform(g[0], g[-1], nq + 1))
    lo, hi = e[:-1].copy(), e[1:].copy()
    hi[1234] = g[-1] + 3.0
    lo[4000] = g[-1] + 3.0
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    lod, hid = torch.from_numpy(lo).cuda(), torch.from_numpy(hi).cuda()
    out = torch.full((nq, W), SENTINEL, dtype=torch.float64, device="cuda")
    err = torch.zeros(1, dtype=torch.int64, device="cuda")
    for kind, fn in (("cubic", "ndi_interp1d_cubic_integral_dev"), ("linear", "ndi_interp1d_linear_integral_dev")):
        tables[kind].prepare_integral()
        L.check(getattr(L.load(), fn)(tables[kind]._handle(), C.c_void_p(lod.data_ptr()), C.c_void_p(hid.data_ptr()), nq, 0,
                                      C.c_void_p(out.data_ptr()), C.c_void_p(err.data_ptr()), s))
        torch.cuda.synchronize()
        assert int(err.item()) == 2 * 1234 + 1, kind
        _, want, _, _ = _want(tables, kind, lo[:1234], hi[:1234], 0, None)
        assert _bits_equal(out[:1234].cpu().numpy(), want), kind


def test_no_integral_until_built_and_after_a_new_spline():
    from ndarray_interp_b200.interp1d import BoundaryCondition, CubicSpline
    rng = np.random.default_rng(3)
    g = np.cumsum(rng.uniform(0.5, 1.5, 50))
    y = rng.normal(size=(50, 6))
    ip = Interp1DBuilder.new(y).x(g).strategy(CubicSpline.new().boundary(BoundaryCondition.Natural)).build()
    lib, h = L.load(), ip._handle()
    lo, hi = np.array([g[1], g[2] + 0.1]), np.array([g[5], g[40]])
    out = np.zeros((2, 6))
    bad, bound = C.c_int64(-1), C.c_int32(-1)
    call = lambda: lib.ndi_interp1d_cubic_integral(h, L.ptr(lo), L.ptr(hi), 2, 0, L.ptr(out), C.byref(bad), C.byref(bound))
    assert call() == L.NO_INTEGRAL
    assert lib.ndi_interp1d_linear_integral(h, L.ptr(lo), L.ptr(hi), 2, 0, L.ptr(out), C.byref(bad), C.byref(bound)) == L.NO_INTEGRAL
    L.check(lib.ndi_interp1d_integral_build(h, L.INTEGRAL_CUBIC))
    assert call() == L.OK
    a, b = ip.strategy.coefficients(ip)
    assert _bits_equal(out, I.integrate(g, y, a, b, lo, hi, 0)[1])
    # new coefficients: the table is dropped until it is built again, then follows them
    for change in ("set_coeffs", "spline_build"):
        if change == "set_coeffs":
            a2, b2 = np.ascontiguousarray(a * 0.5), np.ascontiguousarray(b + 0.25)
            L.check(lib.ndi_interp1d_spline_set_coeffs(h, L.ptr(a2), L.ptr(b2), 0))
        else:
            L.check(lib.ndi_interp1d_spline_build(h, 2, None, None, None, None, C.byref(bad)))     # Clamped
            a2, b2 = ip.strategy.coefficients(ip)
        assert call() == L.NO_INTEGRAL, change
        L.check(lib.ndi_interp1d_integral_build(h, L.INTEGRAL_CUBIC))
        assert call() == L.OK
        assert _bits_equal(out, I.integrate(g, y, a2, b2, lo, hi, 0)[1]), change


def test_rejections(tables):
    lib = L.load()
    gi = np.arange(10, dtype=np.int64)
    yi = np.arange(20, dtype=np.int64).reshape(10, 2)
    ii = Interp1DBuilder.new(yi).x(gi).build()
    assert lib.ndi_interp1d_integral_build(ii._handle(), L.INTEGRAL_LINEAR) == L.UNSUPPORTED_DTYPE
    with pytest.raises(TypeError):
        ii.integrate(1, 2)
    h = tables["cubic"]._handle()
    for kind in (-1, 2, 7):
        assert lib.ndi_interp1d_integral_build(h, kind) == L.INVALID_ARGUMENT
    assert lib.ndi_interp1d_integral_build(tables["linear"]._handle(), L.INTEGRAL_CUBIC) == L.NO_SPLINE

    class Mine(Interp1DStrategy):
        def interp_into(self, interpolator, target, x):
            target[...] = 0

    with pytest.raises(TypeError):
        Interp1D(tables["g"], tables["y"], Mine()).integrate(1.0, 2.0)


def test_broadcasting_and_shapes(tables):
    ip = tables["cubic"]
    g = tables["g"]
    b = np.random.default_rng(9).uniform(g[0], g[-1], (3, 5))
    anti = ip.interp_array_integral(g[0], b)                       # scalar lo: the antiderivative at every b
    assert anti.shape == (3, 5, W)
    assert _bits_equal(anti, ip.interp_array_integral(np.full((3, 5), g[0]), b))
    assert ip.integrate(float(b[1, 2]), float(b[0, 0])).shape == (W,)
    assert _bits_equal(ip.integrate(float(b[1, 2]), float(b[0, 0])), ip.interp_array_integral(b[1, 2], b[0, 0]))
    rows = ip.interp_array_integral(b[:, :1], b[0])                # (3, 1) with (5,) -> (3, 5)
    assert rows.shape == (3, 5, W)
    with pytest.raises(Panic):
        ip.interp_array_integral_into(b, b, np.zeros((3, 4, W)))
    fort = np.asfortranarray(np.zeros((3, 5, W)))
    ip.interp_array_integral_into(g[0], b, fort)
    assert np.array_equal(fort, anti)
    scalar = Interp1DBuilder.new(tables["y"][:, 0].copy()).x(g).strategy(Linear.new()).build()
    assert scalar.integrate(float(g[3]), float(g[9])).shape == ()


def test_properties(tables):
    """additivity within the bars, and a periodic integral over any full period equals C[n-1]"""
    from ndarray_interp_b200.interp1d import BoundaryCondition, CubicSpline
    g, y = tables["g"], tables["y"].copy()
    rng = np.random.default_rng(4)
    pts = np.sort(rng.uniform(g[0], g[-1], (300, 3)), axis=1)
    ip = tables["cubic"]
    ab, bc, ac = (ip.interp_array_integral(pts[:, i], pts[:, j]) for i, j in ((0, 1), (1, 2), (0, 2)))
    scale = (g[-1] - g[0]) * np.abs(y).max(axis=0)
    assert np.max(np.abs(ab + bc - ac) / scale) <= 1e-12
    y[-1] = y[0]
    per = Interp1DBuilder.new(y).x(g).strategy(CubicSpline.new().boundary(BoundaryCondition.Periodic).extrapolate(True)).build()
    a, b = per.strategy.coefficients(per)
    P = g[-1] - g[0]
    lo = np.concatenate([rng.uniform(g[0] - 3 * P, g[-1] + 3 * P, 50), g[:5]])
    full = per.interp_array_integral(lo, lo + P)
    cn = I.table(g, y, a, b)[-1]
    assert np.max(np.abs(full - cn[None, :]) / scale) <= 1e-12


def test_clone_to_device_carries_the_tables(tables):
    ip = tables["linear"]
    ip.prepare_integral()
    clone = C.c_void_p()
    L.check(L.load().ndi_interp1d_clone_to_device(ip._handle(), 0, C.byref(clone)))
    try:
        g = tables["g"]
        lo, hi = np.array([g[0], g[3] + 0.2]), np.array([g[10], g[50]])
        out = np.zeros((2, W))
        bad, bound = C.c_int64(-1), C.c_int32(-1)
        assert L.load().ndi_interp1d_linear_integral(clone, L.ptr(lo), L.ptr(hi), 2, 0, L.ptr(out), C.byref(bad), C.byref(bound)) == 0
        assert _bits_equal(out, ip.interp_array_integral(lo, hi))
    finally:
        L.load().ndi_interp1d_destroy(clone)


def test_c2_size_sampled_rows_bits_equal():
    """4096 x 1024 f64 with 2^20 sorted consecutive bins (the C2 shape), sampled rows against the specification"""
    rng = np.random.default_rng(2)
    n, w, nq = 4096, 1024, 1 << 20
    x = np.cumsum(rng.uniform(0.5, 1.5, n))
    y = rng.normal(size=(n, w))
    ip = _spline(x, y, "Natural", False, "auto", rng)
    a, b = ip.strategy.coefficients(ip)
    e = np.sort(rng.uniform(x[0], x[-1], nq + 1))
    got = ip.interp_array_integral(e[:-1], e[1:])
    rows = np.unique(np.concatenate([rng.integers(0, nq, 512), [0, nq - 1]]))
    cum = I.table(x, y, a, b)
    _, want, _, _ = I.integrate(x, y, a, b, e[:-1][rows], e[1:][rows], 0, cum=cum)
    assert _bits_equal(got[rows], want)


@pytest.mark.skipif(_ndev() < 2, reason="needs two GPUs")
def test_group_calls_first_failure_and_untouched_rows(tables):
    nq = 100_000
    rng = np.random.default_rng(8)
    g = tables["g"]
    e = np.sort(rng.uniform(g[0], g[-1], nq + 1))
    lo, hi = e[:-1].copy(), e[1:].copy()
    hi[[90_000, 99_000]] = g[-1] + 2.0                     # in the second device's block
    for kind in ("linear", "cubic"):
        tables[kind].prepare_integral()
        grp = tables[kind].replicate([0, 1])
        _, want, _, _ = _want(tables, kind, lo, hi, 0, np.full((nq, W), SENTINEL))
        out = np.full((nq, W), SENTINEL)
        with pytest.raises(InterpolateError.OutOfBounds):
            grp.interp_array_integral_into(lo, hi, out)
        assert np.array_equal(out, want), kind
        ok_hi = np.clip(hi, g[0], g[-1])
        assert np.array_equal(grp.interp_array_integral(lo, ok_hi), tables[kind].interp_array_integral(lo, ok_hi))


def test_replicating_before_the_table_is_built_raises():
    rng = np.random.default_rng(1)
    g = np.cumsum(rng.uniform(0.5, 1.5, 20))
    ip = Interp1DBuilder.new(rng.normal(size=(20, 3))).x(g).strategy(Linear.new()).build()
    grp = ip.replicate([0])
    with pytest.raises(L.NdiLibraryError, match="prepare_integral"):
        grp.integrate(g[1], g[5])
