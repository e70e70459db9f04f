"""Host-side mirror of src/interp1d (Interp1DBuilder, Interp1D, Linear, CubicSpline) over numpy
arrays.  Same names, argument meaning, validation order and error behaviour as the reference;
every numeric result comes from the CUDA path behind include/ndi_b200.h.

The reference's plugin boundary -- the Interp1DStrategyBuilder / Interp1DStrategy traits
(src/interp1d/strategies/mod.rs:12-65) -- is kept: a user strategy implements the per-query
`interp_into` exactly as in examples/custom_strategy.rs and runs as host code.  The batch loop
that the reference runs around it (interp1d/mod.rs:300-343) is the method `interp_batch_into`,
whose default is that loop; the built-in strategies override it with one kernel launch.
"""
import ctypes as C
import threading

import numpy as np

from . import _lib as L
from .errors import BuilderError, InterpolateError, Panic, rust_debug
from .vector_extensions import Monotonic, get_lower_index, monotonic_prop

__all__ = ["Interp1D", "Interp1DBuilder", "Interp1DStrategy", "Interp1DStrategyBuilder", "Linear", "CubicSpline",
           "CubicSplineStrategy", "BoundaryCondition", "RowBoundary", "SingleBoundary", "Pchip", "Akima", "CubicHermite",
           "HermiteStrategy"]


# ---- plugin boundary ---------------------------------------------------------------------------------
class Interp1DStrategyBuilder:
    """trait Interp1DStrategyBuilder (strategies/mod.rs:12-40)"""
    MINIMUM_DATA_LENGHT = 2     # (sic) the reference's spelling

    def build(self, x, data):
        """validate data / compute coefficients; returns the finished Interp1DStrategy"""
        raise NotImplementedError


class Interp1DStrategy:
    """trait Interp1DStrategy (strategies/mod.rs:42-65)"""

    def interp_into(self, interpolator, target, x):
        """interpolate at position x into `target` (shape = data.shape[1:]); raise InterpolateError"""
        raise NotImplementedError

    def interp_batch_into(self, interpolator, xs_flat, out_rows):
        """the reference's batch loop (interp1d/mod.rs:334-342): stop at the first error.
        xs_flat: (Q,), out_rows: (Q, ...data.shape[1:]) C-contiguous."""
        for i in range(xs_flat.shape[0]):
            self.interp_into(interpolator, out_rows[i, ...], xs_flat[i])      # [i, ...]: a view even when 0-d

    def _bind(self, interpolator):
        """called once by Interp1D; built-in strategies grab the device handle here"""


# ---- Linear ----------------------------------------------------------------------------------------------
class Linear(Interp1DStrategyBuilder, Interp1DStrategy):
    """Linear Interpolation Strategy (strategies/linear.rs)"""
    MINIMUM_DATA_LENGHT = 2

    def __init__(self):
        self._extrapolate = False

    @classmethod
    def new(cls):
        return cls()

    def extrapolate(self, extrapolate):
        """does the strategy extrapolate? Default is `false`"""
        self._extrapolate = bool(extrapolate)
        return self

    def build(self, x, data):                              # linear.rs:54-63
        return self

    def interp_batch_into(self, interpolator, xs_flat, out_rows):
        bad = C.c_int64(-1)
        fn, h = ((L.load().ndi_interp1d_group_linear, interpolator._group.ptr) if getattr(interpolator, "_group", None)
                 else (L.load().ndi_interp1d_linear, interpolator._handle()))
        st = L.check(fn(h, L.ptr(xs_flat), xs_flat.size, int(self._extrapolate), L.ptr(out_rows), C.byref(bad)))
        _raise_eval(st, xs_flat, bad.value, "x")

    def interp_into(self, interpolator, target, x):        # linear.rs:73-98
        _single_into(self, interpolator, target, x)

    def deriv_batch_into(self, interpolator, xs_flat, out_rows, order=1):
        """NOT in the reference: slope (y[i+1] - y[i]) / (x[i+1] - x[i]) of the interval each query falls into, with
        interp_batch_into's query handling and errors (include/ndi_b200.h: ndi_interp1d_linear_deriv).  A piecewise
        linear interpolant has no second derivative: order must be 1."""
        if order != 1:
            raise ValueError(f"Linear has only a first derivative, got order {order}")
        bad = C.c_int64(-1)
        fn, h = ((L.load().ndi_interp1d_group_linear_deriv, interpolator._group.ptr) if getattr(interpolator, "_group", None)
                 else (L.load().ndi_interp1d_linear_deriv, interpolator._handle()))
        st = L.check(fn(h, L.ptr(xs_flat), xs_flat.size, int(self._extrapolate), L.ptr(out_rows), C.byref(bad)))
        _raise_eval(st, xs_flat, bad.value, "x")

    def integral_batch_into(self, interpolator, lo_flat, hi_flat, out_rows):
        """NOT in the reference: integral from lo_flat[i] to hi_flat[i] of the piecewise linear interpolant, with
        interp_batch_into's handling of each bound (include/ndi_b200.h: ndi_interp1d_linear_integral)"""
        _integral_batch(interpolator, L.INTEGRAL_LINEAR, int(self._extrapolate), lo_flat, hi_flat, out_rows)


# ---- CubicSpline -------------------------------------------------------------------------------------------
class SingleBoundary:
    """enum SingleBoundary (cubic_spline.rs:203-217)"""

    def __init__(self, kind, value=0.0):
        self.kind, self.value = kind, value

    @classmethod
    def FirstDeriv(cls, v):
        return cls("FirstDeriv", v)

    @classmethod
    def SecondDeriv(cls, v):
        return cls("SecondDeriv", v)

    def __eq__(self, o):
        return isinstance(o, SingleBoundary) and (self.kind, self.value) == (o.kind, o.value)

    def __repr__(self):
        return self.kind if self.kind in ("NotAKnot", "Natural", "Clamped") else f"{self.kind}({self.value})"


SingleBoundary.NotAKnot = SingleBoundary("NotAKnot")
SingleBoundary.Natural = SingleBoundary("Natural")
SingleBoundary.Clamped = SingleBoundary("Clamped")


class RowBoundary:
    """enum RowBoundary (cubic_spline.rs:170-184)"""

    def __init__(self, kind, left=None, right=None):
        self.kind, self.left, self.right = kind, left, right

    @classmethod
    def Mixed(cls, left, right):
        return cls("Mixed", left, right)

    def __eq__(self, o):
        return isinstance(o, RowBoundary) and (self.kind, self.left, self.right) == (o.kind, o.left, o.right)

    def __repr__(self):
        return self.kind if self.kind != "Mixed" else f"Mixed {{ left: {self.left}, right: {self.right} }}"


RowBoundary.NotAKnot = RowBoundary("NotAKnot")
RowBoundary.Natural = RowBoundary("Natural")
RowBoundary.Clamped = RowBoundary("Clamped")


class BoundaryCondition:
    """enum BoundaryCondition (cubic_spline.rs:153-168)"""

    def __init__(self, kind, rows=None):
        self.kind, self.rows = kind, rows

    @classmethod
    def Individual(cls, rows):
        """rows: array-like of RowBoundary with the data's shape, axis 0 of length 1"""
        arr = np.empty(np.shape(_as_object_array(rows)), dtype=object)
        arr[...] = _as_object_array(rows)
        return cls("Individual", arr)

    def __repr__(self):
        return self.kind


def _as_object_array(rows):
    if isinstance(rows, np.ndarray) and rows.dtype == object:
        return rows
    # nested lists of RowBoundary -> object array without numpy trying to iterate the elements
    def shape_of(r):
        return (len(r),) + shape_of(r[0]) if isinstance(r, (list, tuple)) else ()
    shp = shape_of(rows)
    arr = np.empty(shp, dtype=object)
    flat = arr.reshape(-1)

    def walk(r, out):
        if isinstance(r, (list, tuple)):
            for e in r:
                walk(e, out)
        else:
            out.append(r)
    items = []
    walk(rows, items)
    for i, it in enumerate(items):
        flat[i] = it
    return arr


BoundaryCondition.NotAKnot = BoundaryCondition("NotAKnot")
BoundaryCondition.Natural = BoundaryCondition("Natural")
BoundaryCondition.Clamped = BoundaryCondition("Clamped")
BoundaryCondition.Periodic = BoundaryCondition("Periodic")

_BC = {"NotAKnot": 0, "Natural": 1, "Clamped": 2, "Periodic": 3, "Individual": 4}
_SB = {"NotAKnot": 0, "Natural": 1, "Clamped": 2, "FirstDeriv": 3, "SecondDeriv": 4}


class CubicSpline(Interp1DStrategyBuilder):
    """The CubicSpline 1d interpolation Strategy (Builder) (cubic_spline.rs:84-88, :723-772)"""
    MINIMUM_DATA_LENGHT = 3

    def __init__(self):
        self._extrapolate = False
        self._boundary = BoundaryCondition.NotAKnot
        self._solver = (L.BUILD_AUTO, 0)

    @classmethod
    def new(cls):
        return cls()

    def solver(self, mode, levels=0):
        """NOT in the reference (device-side knob, include/ndi_b200.h: ndi_interp1d_set_build_mode): "auto",
        "sequential" -- the reference's elimination order, coefficients bit-identical to its arithmetic -- or
        "rowsplit" -- parallel cyclic reduction + Thomas, `levels` reduction steps (0: the library's choice) -- or
        "partition" -- blocks of `levels` rows (0: 32) solved in registers, the separator rows' system recursively."""
        self._solver = ({"auto": L.BUILD_AUTO, "sequential": L.BUILD_SEQUENTIAL, "rowsplit": L.BUILD_ROWSPLIT,
                         "partition": L.BUILD_PARTITION}[mode], int(levels))
        return self

    def extrapolate(self, extrapolate):
        self._extrapolate = bool(extrapolate)
        return self

    def boundary(self, boundary):
        self._boundary = boundary
        return self

    def build(self, x, data):                              # cubic_spline.rs:754-771
        if not np.issubdtype(data.dtype, np.floating):
            raise TypeError("CubicSpline needs a float element type (SplineNum, cubic_spline.rs:34-49)")
        bc = self._boundary
        lk = lv = rk = rv = None
        if bc.kind == "Individual":                        # calc_coefficients :332-347
            expect = [1] + list(data.shape[1:])
            if list(bc.rows.shape) != expect:
                raise BuilderError.ShapeError(
                    f"Boundary conditions array has wrong shape. Expected: {expect}, got: {list(bc.rows.shape)}")
            rows = bc.rows.reshape(-1)
            w = rows.size
            lk, rk = np.zeros(w, np.int32), np.zeros(w, np.int32)
            lv, rv = np.zeros(w, data.dtype), np.zeros(w, data.dtype)
            for i, r in enumerate(rows):
                if r.kind == "Mixed":
                    lk[i], rk[i] = _SB[r.left.kind], _SB[r.right.kind]
                    lv[i], rv[i] = r.left.value, r.right.value
                else:
                    lk[i] = rk[i] = _SB[r.kind]
        if not self._extrapolate:
            mode = L.EXTRAP_NO
        elif bc.kind == "Periodic":
            mode = L.EXTRAP_PERIODIC
        else:
            mode = L.EXTRAP_YES
        return CubicSplineStrategy(_BC[bc.kind], (lk, lv, rk, rv), mode, self._solver)


class CubicSplineStrategy(Interp1DStrategy):
    """The CubicSpline 1d interpolation Strategy (Implementation) (cubic_spline.rs:94-102).
    The coefficient arrays a, b live on the device inside the interpolator's handle."""

    def __init__(self, bc_kind, individual, mode, solver=(0, 0)):
        self._bc_kind, self._individual, self._mode, self._solver = bc_kind, individual, mode, solver

    def _bind(self, interpolator):
        # CubicSpline::calc_coefficients (cubic_spline.rs:310-368) on the device
        h = interpolator._handle()
        lk, lv, rk, rv = self._individual
        bad = C.c_int64(-1)
        L.check(L.load().ndi_interp1d_set_build_mode(h, *self._solver))
        st = L.check(L.load().ndi_interp1d_spline_build(h, self._bc_kind, L.ptr(lk), L.ptr(lv), L.ptr(rk), L.ptr(rv),
                                                        C.byref(bad)))
        if st == L.PERIODIC_MISMATCH:                      # cubic_spline.rs:483-507
            d = interpolator.data
            first, last = d[0], d[-1]
            if d.ndim == 1:
                msg = f"First: {rust_debug(first)}, last: {rust_debug(last)}"
            else:
                msg = f"First: {_ndarray_debug(first)}, last: {_ndarray_debug(last)}"
            raise BuilderError.ValueError(
                "for periodic boundary condition the first and last value must be equal. " + msg)

    def rowsplit_levels(self, interpolator):
        """how the coefficients were built (ndi_interp1d_build_info): 0 the reference's elimination order, L > 0
        row-split with L levels, -m < 0 partition with blocks of m rows"""
        lv = C.c_int32(-1)
        L.check(L.load().ndi_interp1d_build_info(interpolator._handle(), C.byref(lv)))
        return lv.value

    build_info = rowsplit_levels          # the name says what it returns since the partition build exists

    def coefficients(self, interpolator):
        """(a, b) copied back from the device: shape (n-1, ...data.shape[1:])"""
        d = interpolator.data
        a = np.zeros((d.shape[0] - 1,) + d.shape[1:], dtype=d.dtype)
        b = np.zeros_like(a)
        L.check(L.load().ndi_interp1d_spline_coeffs(interpolator._handle(), L.ptr(a), L.ptr(b)))
        return a, b

    def interp_batch_into(self, interpolator, xs_flat, out_rows):
        bad = C.c_int64(-1)
        fn, h = ((L.load().ndi_interp1d_group_cubic, interpolator._group.ptr) if getattr(interpolator, "_group", None)
                 else (L.load().ndi_interp1d_cubic, interpolator._handle()))
        st = L.check(fn(h, L.ptr(xs_flat), xs_flat.size, self._mode, L.ptr(out_rows), C.byref(bad)))
        _raise_eval(st, xs_flat, bad.value, "x")

    def interp_into(self, interpolator, target, x):        # cubic_spline.rs:791-830
        _single_into(self, interpolator, target, x)

    def deriv_batch_into(self, interpolator, xs_flat, out_rows, order=1):
        """NOT in the reference: first (order 1) or second (order 2) derivative of the spline, as scipy's
        CubicSpline(x, nu), with interp_batch_into's query handling and errors (include/ndi_b200.h:
        ndi_interp1d_cubic_deriv)"""
        if order not in (1, 2):
            raise ValueError(f"CubicSpline derivative order must be 1 or 2, got {order}")
        bad = C.c_int64(-1)
        fn, h = ((L.load().ndi_interp1d_group_cubic_deriv, interpolator._group.ptr) if getattr(interpolator, "_group", None)
                 else (L.load().ndi_interp1d_cubic_deriv, interpolator._handle()))
        st = L.check(fn(h, L.ptr(xs_flat), xs_flat.size, self._mode, int(order), L.ptr(out_rows), C.byref(bad)))
        _raise_eval(st, xs_flat, bad.value, "x")

    def integral_batch_into(self, interpolator, lo_flat, hi_flat, out_rows):
        """NOT in the reference: integral from lo_flat[i] to hi_flat[i] of the spline, as scipy's
        CubicSpline.integrate(a, b, extrapolate), with interp_batch_into's handling of each bound (include/ndi_b200.h:
        ndi_interp1d_cubic_integral)"""
        _integral_batch(interpolator, L.INTEGRAL_CUBIC, self._mode, lo_flat, hi_flat, out_rows)


# ---- shape-preserving cubics: NOT in the reference ---------------------------------------------------------------
class _HermiteBuilder(Interp1DStrategyBuilder):
    """common part of Pchip, Akima and CubicHermite: a C1 piecewise cubic from knot slopes computed on the device
    (include/ndi_b200.h: ndi_interp1d_hermite_build), evaluated exactly like a CubicSpline"""
    MINIMUM_DATA_LENGHT = 2

    def __init__(self):
        self._extrapolate = False

    @classmethod
    def new(cls):
        return cls()

    def extrapolate(self, extrapolate):
        """does the strategy extrapolate (the edge intervals' polynomials)? Default is `false`"""
        self._extrapolate = bool(extrapolate)
        return self

    def _kind(self):
        raise NotImplementedError

    def build(self, x, data):
        if not np.issubdtype(data.dtype, np.floating):
            raise TypeError(f"{type(self).__name__} needs a float element type")
        return HermiteStrategy(self._kind(), None, L.EXTRAP_YES if self._extrapolate else L.EXTRAP_NO)


class Pchip(_HermiteBuilder):
    """NOT in the reference: the monotonicity-preserving cubic of scipy's PchipInterpolator"""

    def _kind(self):
        return L.HERMITE_PCHIP


class Akima(_HermiteBuilder):
    """NOT in the reference: scipy's Akima1DInterpolator, method "akima" (default) or "makima" """

    def __init__(self):
        super().__init__()
        self._method = "akima"

    def method(self, method):
        if method not in ("akima", "makima"):
            raise ValueError(f'Akima method must be "akima" or "makima", got {method!r}')
        self._method = method
        return self

    def _kind(self):
        return L.HERMITE_AKIMA if self._method == "akima" else L.HERMITE_MAKIMA


class CubicHermite(_HermiteBuilder):
    """NOT in the reference: scipy's CubicHermiteSpline(x, y, dydx) -- the slopes at the knots are given, shaped like
    the data"""

    def __init__(self, dydx):
        super().__init__()
        self._dydx = np.asarray(dydx)

    @classmethod
    def new(cls, dydx):
        return cls(dydx)

    def _kind(self):
        return L.HERMITE_GIVEN

    def build(self, x, data):
        if self._dydx.shape != data.shape:
            raise BuilderError.ShapeError(
                f"dydx has wrong shape. Expected: {list(data.shape)}, got: {list(self._dydx.shape)}")
        strat = super().build(x, data)
        strat._dydx = np.ascontiguousarray(self._dydx, dtype=data.dtype)
        return strat


class HermiteStrategy(CubicSplineStrategy):
    """the strategy Pchip, Akima and CubicHermite build: a CubicSplineStrategy whose coefficients come from knot slopes
    instead of the spline's solve; every evaluation (values, derivatives, integrals, replication) is the spline's"""

    def __init__(self, kind, dydx, mode):
        super().__init__(None, None, mode)
        self._kind, self._dydx = kind, dydx

    def _bind(self, interpolator):
        # the slopes stay with the strategy: like a CubicSplineStrategy it may be bound to several interpolators
        L.check(L.load().ndi_interp1d_hermite_build(interpolator._handle(), self._kind, L.ptr(self._dydx), 0))


def _ndarray_debug(a):
    """`{:?}` of a 1-D C-contiguous ndarray view, as pinned by tests/cubic_spline_strat.rs:441-443"""
    a = np.asarray(a)
    if a.ndim == 1:
        body = "[" + ", ".join(rust_debug(v) for v in a) + "]"
        return f"{body}, shape=[{a.shape[0]}], strides=[1], layout=CFcf (0xf), const ndim=1"
    return np.array2string(a, separator=", ") + f", shape={list(a.shape)}, const ndim={a.ndim}"


def _raise_eval(st, xs_flat, first_bad, name):
    if st == L.OUT_OF_BOUNDS:                              # linear.rs:80-84, cubic_spline.rs:798-802
        raise InterpolateError.OutOfBounds(f"{name} = {rust_debug(xs_flat[first_bad])} is not in range")
    if st == L.NAN_QUERY:                                  # vector_extensions.rs:83-84
        raise Panic("not implemented: failed to convert NaN to usize")


def _integral_batch(interpolator, kind, mode, lo_flat, hi_flat, out_rows):
    interpolator.prepare_integral()
    group = getattr(interpolator, "_group", None)
    if group is not None:
        fn, h = (L.load().ndi_interp1d_group_cubic_integral if kind == L.INTEGRAL_CUBIC
                 else L.load().ndi_interp1d_group_linear_integral), group.ptr
    else:
        fn, h = (L.load().ndi_interp1d_cubic_integral if kind == L.INTEGRAL_CUBIC
                 else L.load().ndi_interp1d_linear_integral), interpolator._handle()
    bad, bound = C.c_int64(-1), C.c_int32(-1)
    st = L.check(fn(h, L.ptr(lo_flat), L.ptr(hi_flat), lo_flat.size, mode, L.ptr(out_rows), C.byref(bad), C.byref(bound)))
    _raise_eval(st, hi_flat if bound.value == 1 else lo_flat, bad.value, "x")


def _single_into(strategy, interpolator, target, x):
    """per-query trait method of a built-in strategy: one query through the batched launch"""
    q = np.array([x], dtype=interpolator.data.dtype)
    tgt = np.asarray(target)
    if tgt.flags.c_contiguous and tgt.dtype == interpolator.data.dtype:
        strategy.interp_batch_into(interpolator, q, tgt.reshape((1,) + tgt.shape))
    else:
        tmp = np.zeros((1,) + tgt.shape, dtype=interpolator.data.dtype)
        strategy.interp_batch_into(interpolator, q, tmp)
        tgt[...] = tmp[0]


# ---- Interp1D -------------------------------------------------------------------------------------------------
class _Handle1D:
    """owner of the opaque device handle (freed on drop)"""

    def __init__(self, x, data, flags=0):
        lib = L.require_device()
        self.ptr = C.c_void_p()
        w = int(np.prod(data.shape[1:], dtype=np.int64))
        if L.is_dense(x) and L.is_dense(data):
            self.status = L.check(lib.ndi_interp1d_create(L.dtype_code(data.dtype), L.ptr(x), len(x), L.ptr(data), w, flags,
                                                          C.byref(self.ptr)))
        else:
            # views (any strides, negative included -- tests/interp1d.rs:143-155) go up as they lie in memory
            # and are made dense on the device
            xk, xp, _, xs = L.view_args(x)
            dk, dp, shape, strides = L.view_args(data)
            self.status = L.check(lib.ndi_interp1d_create_strided(L.dtype_code(data.dtype), xp, len(x), xs[0], dp, dk.ndim,
                                                                  shape, strides, flags, C.byref(self.ptr)))

    def __del__(self):
        try:
            if self.ptr:
                L.load().ndi_interp1d_destroy(self.ptr)
                self.ptr = C.c_void_p()
        except Exception:
            pass


class _Group:
    """owner of a ndi_interp{1,2}d_group (the handle it was made from is kept alive)"""

    def __init__(self, create, destroy, handle, devices, keep):
        dev = (C.c_int32 * len(devices))(*[int(d) for d in devices])
        self.ptr, self._destroy, self._keep = C.c_void_p(), destroy, keep
        L.check(create(handle, dev, len(devices), C.byref(self.ptr)))

    def __del__(self):
        try:
            if self.ptr:
                self._destroy(self.ptr)
                self.ptr = C.c_void_p()
        except Exception:
            pass


class Interp1D:
    """One dimensional interpolator (interp1d/mod.rs:38-51)"""

    def __init__(self, x, data, strategy, _handle=None):
        self.x, self.data, self.strategy = x, data, strategy
        self._h = _handle
        self._integral_lock = threading.Lock()
        self._integral_tables = set()          # kinds of cumulative table built on the handle (ndi_interp1d_integral_build)
        if isinstance(strategy, Interp1DStrategy):
            strategy._bind(self)

    # -- construction ----------------------------------------------------------------------------------------
    @staticmethod
    def builder(data):
        """Get the Interp1DBuilder (interp1d/mod.rs:79-81)"""
        return Interp1DBuilder(data)

    @classmethod
    def new_unchecked(cls, x, data, strategy):
        """Create a interpolator without any data validation (interp1d/mod.rs:363-365)"""
        x, data = _prepare(x, data)
        h = _Handle1D(x, data, L.ASSUME_VALID) if _is_builtin(strategy) else None
        return cls(x, data, strategy, h)

    def replicate(self, devices):
        """NOT in the reference: fan this interpolator out over several GPUs of this process (include/ndi_b200.h:
        ndi_interp1d_replicate).  Returns an interpolator with the same methods whose batch calls cut the queries into
        contiguous blocks, one per device, evaluated concurrently; errors and untouched rows as on one device."""
        if not _is_builtin(self.strategy):
            raise TypeError("only the built-in strategies run on the device")
        other = Interp1D.__new__(Interp1D)
        other.x, other.data, other.strategy, other._h = self.x, self.data, self.strategy, self._h
        other._integral_lock = threading.Lock()
        other._integral_tables = frozenset(self._integral_tables)    # the tables the devices received
        other._group = _Group(L.load().ndi_interp1d_replicate, L.load().ndi_interp1d_group_destroy, self._handle(), devices, self)
        return other

    def _handle(self):
        if self._h is None:              # user strategy calling back into the accessors
            self._h = _Handle1D(self.x, self.data, L.ASSUME_VALID)
        return self._h.ptr

    # -- evaluation ----------------------------------------------------------------------------------------------
    def interp_scalar(self, x):
        """interpolation at one point when the data dimension is Ix1 (interp1d/mod.rs:108-114)"""
        if self.data.ndim != 1:
            raise TypeError("interp_scalar needs 1-D data (Ix1)")
        buf = np.zeros((), dtype=self.data.dtype)
        self.strategy.interp_into(self, buf, self.data.dtype.type(x))
        return buf[()]

    def interp(self, x):
        """interpolated values at `x`, one dimension smaller than the data (interp1d/mod.rs:150-156)"""
        target = np.zeros(self.data.shape[1:], dtype=self.data.dtype)
        self.strategy.interp_into(self, target, self.data.dtype.type(x))
        return target

    def interp_into(self, x, buffer):
        """like `interp`, into the provided buffer (interp1d/mod.rs:169-175)"""
        expect = list(self.data.shape[1:])
        if list(np.shape(buffer)) != expect:
            raise Panic(f"Zip: Producer dimension mismatch, expected: {expect}, got: {list(np.shape(buffer))}")
        self.strategy.interp_into(self, buffer, self.data.dtype.type(x))

    def interp_array(self, xs):
        """interpolated values at all points in `xs` (interp1d/mod.rs:197-211)"""
        xs = np.asarray(xs)
        ys = np.zeros(self._buffer_shape(xs.shape), dtype=self.data.dtype)
        self.interp_array_into(xs, ys)
        return ys

    def interp_array_into(self, xs, buffer):
        """like `interp_array`, into the provided buffer of shape xs.shape ++ data.shape[1:]
        (interp1d/mod.rs:272-324).  One launch for the whole batch, whatever the query rank."""
        self._array_into(xs, buffer, self.strategy.interp_batch_into)

    # -- derivatives: NOT in the reference ----------------------------------------------------------------------------
    def interp_deriv(self, x, order=1):
        """NOT in the reference: derivative of order `order` at `x`, shaped like `interp(x)` (the built-in strategies:
        Linear order 1, CubicSpline order 1 or 2; scipy's CubicSpline(x, nu))"""
        target = np.zeros(self.data.shape[1:], dtype=self.data.dtype)
        self.interp_array_deriv_into(np.array([x], dtype=self.data.dtype), target.reshape((1,) + target.shape), order)
        return target

    def interp_array_deriv(self, xs, order=1):
        """NOT in the reference: derivatives at all points in `xs`, shaped like `interp_array(xs)`"""
        xs = np.asarray(xs)
        ys = np.zeros(self._buffer_shape(xs.shape), dtype=self.data.dtype)
        self.interp_array_deriv_into(xs, ys, order)
        return ys

    def interp_array_deriv_into(self, xs, buffer, order=1):
        """NOT in the reference: like `interp_array_deriv`, into the provided buffer; buffer shape, query rank, errors
        and untouched rows after a failing query as `interp_array_into`"""
        if not _is_builtin(self.strategy):
            raise TypeError("derivatives are computed by the built-in strategies (Linear, CubicSpline) only")
        if order not in ((1,) if isinstance(self.strategy, Linear) else (1, 2)):   # before any shape check
            raise ValueError(f"{type(self.strategy).__name__} has no derivative of order {order}")
        self._array_into(xs, buffer, lambda i, q, rows: self.strategy.deriv_batch_into(i, q, rows, order))

    # -- definite integrals: NOT in the reference ------------------------------------------------------------------------
    def integrate(self, a, b):
        """NOT in the reference: the integral from `a` to `b` of the interpolant (scipy's CubicSpline.integrate); `a` and
        `b` broadcast, so a scalar `a` and an array `b` give the antiderivative from `a` at every point of `b`"""
        return self.interp_array_integral(a, b)

    def interp_array_integral(self, a, b):
        """NOT in the reference: integrals over all pairs of the broadcast of `a` and `b`, shaped
        broadcast_shape ++ data.shape[1:]"""
        shape = np.broadcast_shapes(np.shape(a), np.shape(b))
        ys = np.zeros(self._buffer_shape(shape), dtype=self.data.dtype)
        self.interp_array_integral_into(a, b, ys)
        return ys

    def interp_array_integral_into(self, a, b, buffer):
        """NOT in the reference: like `interp_array_integral`, into the provided buffer; buffer layouts, errors and
        untouched rows after a failing pair as `interp_array_into` (the failing bound's value is reported)"""
        self._check_integral()
        shape = np.broadcast_shapes(np.shape(a), np.shape(b))
        lo = np.broadcast_to(np.asarray(a, dtype=self.data.dtype), shape)
        hi = np.ascontiguousarray(np.broadcast_to(np.asarray(b, dtype=self.data.dtype), shape)).reshape(-1)
        self._array_into(lo, buffer, lambda i, q, rows: self.strategy.integral_batch_into(i, q, hi, rows))

    def prepare_integral(self):
        """NOT in the reference: build the cumulative table the integral calls evaluate over (otherwise built on first
        use).  On a replicated interpolator the table must have been built before `replicate`."""
        self._check_integral()
        kind = L.INTEGRAL_CUBIC if isinstance(self.strategy, CubicSplineStrategy) else L.INTEGRAL_LINEAR
        with self._integral_lock:
            if kind in self._integral_tables:
                return
            if getattr(self, "_group", None) is not None:
                raise L.NdiLibraryError("this interpolator was replicated before its integral table was built: call "
                                        "prepare_integral() on the source interpolator before replicate()")
            L.check(L.load().ndi_interp1d_integral_build(self._handle(), kind))
            self._integral_tables.add(kind)

    def _check_integral(self):
        if not _is_builtin(self.strategy):
            raise TypeError("integrals are computed by the built-in strategies (Linear, CubicSpline) only")
        if self.data.dtype.kind not in "f":
            raise TypeError(f"integrals need float data (the integral of {self.data.dtype} data is not an integer)")

    def _array_into(self, xs, buffer, batch):
        xs = np.asarray(xs)
        expect = self._buffer_shape(xs.shape)
        got = tuple(np.shape(buffer))
        if got != expect:
            _panic_buffer_shape(xs.shape, self.data.shape[1:], expect, got)
        q = np.ascontiguousarray(xs, dtype=self.data.dtype).reshape(-1)
        rows_shape = (q.size,) + self.data.shape[1:]
        direct = isinstance(buffer, np.ndarray) and buffer.flags.c_contiguous and buffer.dtype == self.data.dtype
        # a strided / foreign-dtype buffer is evaluated through a dense copy that STARTS from the caller's values:
        # rows at and after a failing query must come back untouched (interp1d/mod.rs:321, :336-340)
        rows = buffer.reshape(rows_shape) if direct else np.array(buffer, dtype=self.data.dtype).reshape(rows_shape)
        try:
            batch(self, q, rows)
        finally:
            if not direct:
                buffer[...] = rows.reshape(expect)

    def _buffer_shape(self, query_shape):                  # get_buffer_shape (interp1d/mod.rs:346-354)
        return tuple(query_shape) + tuple(self.data.shape[1:])

    # -- accessors strategies may call back (interp1d/mod.rs:371-386) -------------------------------------------------
    def index_point(self, index):
        """get `(x, data)` coordinate at given index"""
        return self.x[index], self.data[index]

    def get_index_left_of(self, x):
        """The index of a known value left of, or at x (device search, vector_extensions.rs:55-111)"""
        return get_lower_index(self.x, x)

    def is_in_range(self, x):
        return bool(self.x[0] <= x <= self.x[-1])


def _panic_buffer_shape(qshape, trailing, expect, got):
    """the reference's panics for a wrong output buffer (messages pinned by interp1d/mod.rs:550-607)"""
    if len(qshape) == 1:
        # Ix1 path: Zip over (xs, buffer.axis_iter_mut(0)), then the strategy's Zip over the row
        if len(got) < 1 or got[0] != qshape[0]:
            raise Panic(f"Zip: Producer dimension mismatch, expected: [{qshape[0]}], got: [{got[0] if got else 0}]")
        raise Panic(f"Zip: Producer dimension mismatch, expected: {list(trailing)}, got: {list(got[1:])}")
    # generic path: into_shape_with_order fails (interp1d/mod.rs:312-318); `{:?}` of the Pattern tuples
    fmt = lambda t: f"({', '.join(str(v) for v in t)})" if len(t) != 1 else f"{t[0]}"
    raise Panic(f"ShapeError/IncompatibleShape: incompatible shapes expected: {fmt(expect)}, got: {fmt(got)}")


def _is_builtin(strategy):
    return isinstance(strategy, (Linear, CubicSplineStrategy))


def _prepare(x, data):
    data = np.asarray(data)                                # views / negative strides stay views (_Handle1D)
    L.dtype_code(data.dtype)
    x = np.asarray(x)
    if x.dtype != data.dtype:
        x = x.astype(data.dtype)
    return x, data


class Interp1DBuilder:
    """Create and configure a Interp1D Interpolator (interp1d/mod.rs:53-70, :389-477).

    Default configuration: Linear{extrapolate: false}, interpolation along axis 0, x = index."""

    def __init__(self, data):                              # Interp1DBuilder::new (:399-410)
        self._data = np.asarray(data)
        n = self._data.shape[0] if self._data.ndim >= 1 else 0
        self._x = np.arange(n).astype(self._data.dtype)
        self._strategy = Linear.new()

    @classmethod
    def new(cls, data):
        return cls(data)

    def x(self, x):
        """custom x axis; must be strict monotonic rising and as long as data axis 0"""
        self._x = np.asarray(x)
        return self

    def strategy(self, strategy):
        self._strategy = strategy
        return self

    def build(self):
        """Validate input data and create the configured Interp1D (interp1d/mod.rs:443-476).
        Check order as in the reference: ndim, MINIMUM_DATA_LENGHT, monotonic, lengths."""
        data, x, strat = self._data, self._x, self._strategy
        if data.ndim < 1:
            raise BuilderError.ShapeError("data dimension is 0, needs to be at least 1")
        if data.shape[0] < strat.MINIMUM_DATA_LENGHT:
            raise BuilderError.NotEnoughData(
                f"The chosen Interpolation strategy needs at least {strat.MINIMUM_DATA_LENGHT} data points")
        L.dtype_code(data.dtype)
        x = np.asarray(x)
        if x.dtype != data.dtype:
            x = x.astype(data.dtype)
        if monotonic_prop(x) != Monotonic.Rising(True):    # K1 on the device
            raise BuilderError.Monotonic("Values in the x axis need to be strictly monotonic rising")
        if len(x) != data.shape[0]:
            raise BuilderError.ShapeError(
                f"Lengths of x and data axis need to match. Got x: {len(x)}, data: {data.shape[0]}")
        x, data = _prepare(x, data)
        finished = strat.build(x, data)
        h = _Handle1D(x, data, L.ASSUME_VALID) if _is_builtin(finished) else None
        return Interp1D(x, data, finished, h)
