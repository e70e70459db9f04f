"""Derivatives on the GPU (NOT in the reference): ndi_interp1d_cubic_deriv / ndi_interp1d_linear_deriv and their _dev and
group forms, through the Python mirror, compared bit for bit with the specification in tests/deriv_oracle.cpp applied to
the coefficients the handle itself holds (whichever build mode made them).  Query handling and errors must be those of
the value calls: the first failing query, rows at and after it untouched on the host API."""
import ctypes as C

import numpy as np
import pytest

import deriv_oracle as D
from ndarray_interp_b200 import InterpolateError
from ndarray_interp_b200 import _lib as L
from ndarray_interp_b200.errors import Panic
from ndarray_interp_b200.interp1d import (BoundaryCondition, CubicSpline, Interp1D, Interp1DBuilder, Interp1DStrategy,
                                          Linear, RowBoundary, SingleBoundary)

pytestmark = pytest.mark.gpu

SENTINEL = -12345.5


def _bits_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _boundary(kind, w, dtype, rng):
    if kind == "Individual":
        rows = [RowBoundary.Mixed(SingleBoundary.FirstDeriv(float(rng.normal())), SingleBoundary.SecondDeriv(float(rng.normal())))
                for _ in range(w)]
        return BoundaryCondition.Individual([rows])
    return getattr(BoundaryCondition, kind)


def _spline(x, y, kind, extrapolate, solver, rng):
    strat = CubicSpline.new().boundary(_boundary(kind, y.shape[1], y.dtype, rng)).extrapolate(extrapolate).solver(solver)
    return Interp1DBuilder.new(y).x(x).strategy(strat).build()


def _queries(kind, x, nq, rng, dtype):
    lo, hi = x[0], x[-1]
    if kind == "sorted":
        q = np.sort(rng.uniform(lo, hi, nq))
    elif kind == "dense":                                   # many queries per interval: one-interval tiles
        q = np.sort(rng.uniform(x[3], x[4], nq))
    else:
        q = rng.uniform(lo, hi, nq)
    q = q.astype(dtype)
    q[: len(x)] = x[: min(len(x), nq)]                      # exactly on the knots, both ends included
    return q


BOUNDARIES = ["Natural", "Clamped", "Periodic", "Individual", "NotAKnot"]
SOLVERS = ["sequential", "rowsplit", "partition"]
# thin rows of every LPQ, f32 with V = 4 / 2 / 1 (w % 4 == 0 / 2 / odd) and f64 with V = 2 / 1, V remainders, wide slices
WIDTHS = [1, 3, 4, 6, 8, 32, 33, 48, 100, 1024, 1025]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("w", WIDTHS)
def test_cubic_deriv_bits_equal_the_oracle_on_the_handles_coefficients(dtype, w):
    rng = np.random.default_rng(w + (dtype == np.float32))
    n = 300
    nq = 2000 if w < 1000 else 1200                       # the first n queries are the knots, the rest of the given kind
    x = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(dtype)
    y = rng.normal(size=(n, w)).astype(dtype)
    y[-1] = y[0]                                            # periodic data for every case
    for i, kind in enumerate(BOUNDARIES):
        solver = SOLVERS[(i + w) % 3]
        ip = _spline(x, y, kind, True, solver, rng)
        a, b = ip.strategy.coefficients(ip)
        mode = 2 if kind == "Periodic" else 1
        qkind = ["sorted", "dense", "random"][(i + w) % 3]
        q = _queries(qkind, x, nq, rng, dtype)
        q[-3:] = np.array([x[0] - 1.5, x[-1] + 2.25, x[-1] + 40.0], dtype)      # extrapolated / wrapped
        for order in (1, 2):
            st, want, _ = D.cubic_deriv(x, y, a, b, q, mode, order)
            assert st == 0
            got = ip.interp_array_deriv(q, order)
            assert _bits_equal(got, want), (kind, solver, qkind, order)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_cubic_deriv_every_search_mode_and_extrapolation_mode(dtype):
    rng = np.random.default_rng(11)
    n, w, nq = 200, 16, 5000
    x = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(dtype)
    y = rng.normal(size=(n, w)).astype(dtype)
    y[-1] = y[0]
    for kind, extrapolate, mode in (("Natural", False, 0), ("Natural", True, 1), ("Periodic", True, 2)):
        ip = _spline(x, y, kind, extrapolate, "auto", rng)
        a, b = ip.strategy.coefficients(ip)
        q = np.sort(rng.uniform(x[0], x[-1], nq)).astype(dtype)
        if mode:
            q[::97] = rng.uniform(x[0] - 50, x[-1] + 50, q[::97].size).astype(dtype)
        for order in (1, 2):
            _, want, _ = D.cubic_deriv(x, y, a, b, q, mode, order)
            for sm in range(6):
                L.check(L.load().ndi_interp1d_set_search_mode(ip._handle(), sm))
                assert _bits_equal(ip.interp_array_deriv(q, order), want), (kind, order, sm)


LINEAR_DTYPES = [np.float32, np.float64, np.int32, np.int64, np.uint32, np.uint64]


@pytest.mark.parametrize("dtype", LINEAR_DTYPES)
@pytest.mark.parametrize("w", [1, 3, 4, 6, 8, 16, 33, 48, 100, 1025])
def test_linear_slope_bits_equal_the_oracle(dtype, w):
    rng = np.random.default_rng(w * 13 + np.dtype(dtype).itemsize)
    n, nq = 120, 3000
    if np.issubdtype(dtype, np.floating):
        x = np.cumsum(rng.uniform(0.25, 2.0, n)).astype(dtype)
        y = rng.normal(size=(n, w)).astype(dtype)
        y[10, 0], y[11, 0] = dtype(0.0), -dtype(0.0)      # the quotient of -0 keeps its sign
    else:
        info = np.iinfo(dtype)
        x = np.cumsum(rng.integers(1, 40, n)).astype(dtype)
        lo = 0 if info.min == 0 else info.min // 2
        y = rng.integers(lo, info.max, size=(n, w), dtype=dtype)   # unsigned: the upper half included
    for extrapolate in (False, True):
        ip = Interp1DBuilder.new(y).x(x).strategy(Linear.new().extrapolate(extrapolate)).build()
        q = np.concatenate([rng.uniform(float(x[0]), float(x[-1]), nq - n), x.astype(np.float64)]).astype(dtype)
        if extrapolate and np.issubdtype(dtype, np.floating):
            q[::50] = (q[::50] * 3 - float(x[-1])).astype(dtype)
        st, want, _ = D.linear_deriv(x, y, q, extrapolate)
        assert st == 0
        got = ip.interp_array_deriv(q)
        assert _bits_equal(got, want), (dtype, w, extrapolate)
        if np.issubdtype(dtype, np.floating) and not extrapolate:
            k = int(np.nonzero(q == x[10])[0][0])
            assert got[k, 0] == 0 and np.signbit(got[k, 0])


# ---- errors: the value call's semantics ------------------------------------------------------------------------------
W = 1024
CASES = [(20, None), (20, 7), (1500, None), (1500, 700), (40_000, None), (40_000, 0), (40_000, 35_000)]


@pytest.fixture(scope="module")
def tables():
    rng = np.random.default_rng(77)
    g = np.cumsum(rng.uniform(0.5, 1.5, 64))
    y = rng.normal(size=(64, W))
    cub = Interp1DBuilder.new(y).x(g).strategy(CubicSpline.new().boundary(BoundaryCondition.Natural)).build()
    return {"linear": Interp1DBuilder.new(y).x(g).strategy(Linear.new()).build(), "cubic": cub,
            "coeffs": cub.strategy.coefficients(cub), "g": g, "y": y}


def _out_buffer(kind, nq):
    if kind == "pageable":
        return np.full((nq, W), SENTINEL)
    if kind == "pinned":
        import torch
        pinned = torch.empty((nq, W), dtype=torch.float64, pin_memory=True)
        out = pinned.numpy()
        out[...] = SENTINEL
        return out
    return np.full((nq, 2 * W), SENTINEL)[:, ::2]


@pytest.mark.parametrize("nq,bad", CASES)
@pytest.mark.parametrize("out_kind", ["pageable", "pinned", "strided"])
@pytest.mark.parametrize("kind,order", [("linear", 1), ("cubic", 1), ("cubic", 2)])
def test_host_batch_errors_and_untouched_rows(tables, kind, order, out_kind, nq, bad):
    rng = np.random.default_rng(nq + (bad or 0))
    g = tables["g"]
    q = rng.uniform(g[0], g[-1], nq)
    if bad is not None:
        q[-1] = g[0] - 0.5
        q[bad] = g[-1] + 1.0 + bad
    want = np.full((nq, W), SENTINEL)
    if kind == "linear":
        st, want, want_bad = D.linear_deriv(g, tables["y"], q, False, out=want)
    else:
        a, b = tables["coeffs"]
        st, want, want_bad = D.cubic_deriv(g, tables["y"], a, b, q, 0, order, out=want)
    assert want_bad == (-1 if bad is None else bad)
    out = _out_buffer(out_kind, nq)
    if bad is None:
        tables[kind].interp_array_deriv_into(q, out, order)
    else:
        from ndarray_interp_b200.errors import rust_debug
        with pytest.raises(InterpolateError.OutOfBounds) as e:
            tables[kind].interp_array_deriv_into(q, out, order)
        assert str(e.value) == f"x = {rust_debug(q[bad])} is not in range"
    assert np.array_equal(out, want)


def test_nan_query_panics_like_the_value_call(tables):
    q = np.array([1.0, 2.0, np.nan, 3.0])
    ex = Interp1DBuilder.new(tables["y"]).x(tables["g"]).strategy(Linear.new().extrapolate(True)).build()
    with pytest.raises(Panic):
        ex.interp_array_deriv(q)
    with pytest.raises(Panic):
        ex.interp_array(q)


@pytest.mark.parametrize("order", [1, 2])
def test_dev_error_word_is_the_first_failing_query(tables, order):
    import torch
    a, b = tables["coeffs"]
    g = tables["g"]
    nq = 5000
    q = np.random.default_rng(5).uniform(g[0], g[-1], nq)
    q[[1234, 4000]] = g[-1] + 3.0
    qd = torch.from_numpy(q).cuda()
    out = torch.full((nq, W), SENTINEL, dtype=torch.float64, device="cuda")
    err = torch.zeros(1, dtype=torch.int64, device="cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    h = tables["cubic"]._handle()
    L.check(L.load().ndi_interp1d_cubic_deriv_dev(h, C.c_void_p(qd.data_ptr()), nq, 0, order, C.c_void_p(out.data_ptr()),
                                                  C.c_void_p(err.data_ptr()), s))
    torch.cuda.synchronize()
    assert int(err.item()) == 1234
    _, want, _ = D.cubic_deriv(g, tables["y"], a, b, q[:1234], 0, order)
    assert _bits_equal(out[:1234].cpu().numpy(), want)
    lin = tables["linear"]._handle()
    L.check(L.load().ndi_interp1d_linear_deriv_dev(lin, C.c_void_p(qd.data_ptr()), nq, 0, C.c_void_p(out.data_ptr()),
                                                   C.c_void_p(err.data_ptr()), s))
    torch.cuda.synchronize()
    assert int(err.item()) == 1234
    _, want, _ = D.linear_deriv(g, tables["y"], q[:1234], False)
    assert _bits_equal(out[:1234].cpu().numpy(), want)


def test_rejections(tables):
    lib = L.load()
    q = np.array([1.0, 2.0])
    out = np.zeros((2, W))
    bad = C.c_int64(-1)
    h = tables["cubic"]._handle()
    for order in (0, 3, -1):
        assert lib.ndi_interp1d_cubic_deriv(h, L.ptr(q), 2, 0, order, L.ptr(out), C.byref(bad)) == L.INVALID_ARGUMENT
        with pytest.raises(ValueError):
            tables["cubic"].interp_array_deriv(q, order)
    with pytest.raises(ValueError):
        tables["linear"].interp_array_deriv(q, 2)
    with pytest.raises(ValueError):
        tables["linear"].interp_deriv(1.5, 2)
    # no spline on the handle: the linear interpolator's handle has no coefficients
    assert lib.ndi_interp1d_cubic_deriv(tables["linear"]._handle(), L.ptr(q), 2, 0, 1, L.ptr(out), C.byref(bad)) == L.NO_SPLINE

    class Mine(Interp1DStrategy):
        def interp_into(self, interpolator, target, x):
            target[...] = 0

    user = Interp1D(tables["g"], tables["y"], Mine())
    with pytest.raises(TypeError):
        user.interp_array_deriv(q)


def test_shapes_follow_the_value_methods(tables):
    ip = tables["cubic"]
    q2 = np.random.default_rng(9).uniform(tables["g"][0], tables["g"][-1], (3, 5))
    assert ip.interp_array_deriv(q2).shape == ip.interp_array(q2).shape == (3, 5, W)
    d = ip.interp_deriv(float(q2[1, 2]), 2)
    assert d.shape == (W,) and _bits_equal(d, ip.interp_array_deriv(q2, 2)[1, 2])
    with pytest.raises(Panic):
        ip.interp_array_deriv_into(q2, np.zeros((3, 4, W)))
    scalar = Interp1DBuilder.new(tables["y"][:, 0].copy()).x(tables["g"]).strategy(Linear.new()).build()
    assert scalar.interp_deriv(float(tables["g"][3])).shape == ()


def test_c2_size_sampled_rows_bits_equal():
    """4096 x 1024 f64 with 2^20 sorted queries (the C2 evaluation shape), sampled rows against the oracle"""
    rng = np.random.default_rng(2)
    n, w, nq = 4096, 1024, 1 << 20
    x = np.cumsum(rng.uniform(0.5, 1.5, n))
    y = rng.normal(size=(n, w))
    ip = _spline(x, y, "Natural", False, "auto", rng)
    a, b = ip.strategy.coefficients(ip)
    q = np.sort(rng.uniform(x[0], x[-1], nq))
    rows = np.unique(np.concatenate([rng.integers(0, nq, 512), [0, nq - 1]]))
    for order in (1, 2):
        got = ip.interp_array_deriv(q, order)
        _, want, _ = D.cubic_deriv(x, y, a, b, q[rows], 0, order)
        assert _bits_equal(got[rows], want), order


def _ndev():
    n = C.c_int32(0)
    L.load().ndi_device_count(C.byref(n))
    return n.value


@pytest.mark.skipif(_ndev() < 2, reason="needs two GPUs")
def test_group_calls_first_failure_and_untouched_rows(tables):
    nq = 100_000
    rng = np.random.default_rng(8)
    g = tables["g"]
    q = rng.uniform(g[0], g[-1], nq)
    q[[90_000, 99_000]] = g[-1] + 2.0                     # in the second device's block
    for kind, order in (("linear", 1), ("cubic", 1), ("cubic", 2)):
        grp = tables[kind].replicate([0, 1])
        want = np.full((nq, W), SENTINEL)
        if kind == "linear":
            D.linear_deriv(g, tables["y"], q, False, out=want)
        else:
            a, b = tables["coeffs"]
            D.cubic_deriv(g, tables["y"], a, b, q, 0, order, out=want)
        out = np.full((nq, W), SENTINEL)
        with pytest.raises(InterpolateError.OutOfBounds):
            grp.interp_array_deriv_into(q, out, order)
        assert np.array_equal(out, want), (kind, order)
        ok = np.clip(q, g[0], g[-1])
        assert np.array_equal(grp.interp_array_deriv(ok, order), tables[kind].interp_array_deriv(ok, order))
