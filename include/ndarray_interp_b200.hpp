// ndarray_interp_b200.hpp -- C++17 host-side mirror of the ndarray-interp API over include/ndi_b200.h.
//
// north_star asks for a Rust crate; this image has no Rust toolchain, so the compiled host side
// above the C ABI is this header (the crate source in rust/ is written against the same ABI but
// was not compiled here).  Same names, argument meaning, validation order and error behaviour as
// the reference:
//
//   reference (Rust)                                   here (C++)
//   ------------------------------------------------   -------------------------------------------------
//   ndarray::Array / ArrayView (any rank, any stride)  ndarray_interp::Array<T> (owned, C order) /
//                                                      ArrayView<T>, ArrayViewMut<T> (shape + strides)
//   Interp1D::builder(data).x(x).strategy(s).build()   Interp1D<T>::builder(data).x(x).strategy(s).build()
//     -> Result<Interp1D, BuilderError>                  -> Interp1D<T>, throws BuilderError
//   interp_scalar / interp / interp_into /             same names; Result<_, InterpolateError> becomes
//   interp_array / interp_array_into                   a thrown InterpolateError, a panic a thrown Panic
//   trait Interp1DStrategyBuilder / Interp1DStrategy   abstract classes of the same names
//   (src/interp1d/strategies/mod.rs:12-65)             (per-query interp_into, kept byte for byte; plus
//                                                      interp_batch_into = the reference's batch loop,
//                                                      interp1d/mod.rs:300-343, which the built-in
//                                                      strategies override with ONE kernel launch)
//   Linear, CubicSpline, BoundaryCondition,            same names
//   RowBoundary, SingleBoundary
//   Interp2D, Interp2DBuilder, Bilinear                same names (src/interp2d)
//   VectorExtensions::{monotonic_prop,get_lower_index} monotonic_prop(), get_lower_index()
//
// Every number comes from the CUDA library; there is no CPU fallback (a missing device is an
// exception).  Element types: float, double, int32_t, int64_t, uint32_t, uint64_t (integers: Linear and Bilinear only).
//
// Link with -lndi_b200 (ndarray_interp_b200/libndi_b200.so).
#pragma once

#include <algorithm>
#include <charconv>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <functional>
#include <initializer_list>
#include <memory>
#include <numeric>
#include <stdexcept>
#include <string>
#include <vector>

#include "ndi_b200.h"

namespace ndarray_interp {

// ---- errors (src/lib.rs:127-146) ---------------------------------------------------------------------
struct BuilderError : std::runtime_error {
    enum Kind { NotEnoughData, Monotonic, ShapeError, ValueError } kind;
    BuilderError(Kind k, const std::string& m) : std::runtime_error(m), kind(k) {}
};
struct InterpolateError : std::runtime_error {
    enum Kind { OutOfBounds } kind;
    explicit InterpolateError(const std::string& m) : std::runtime_error(m), kind(OutOfBounds) {}
};
// a panic of the reference (wrong buffer shape, NaN reaching get_lower_index, ...)
struct Panic : std::logic_error { using std::logic_error::logic_error; };
// the library itself failed (no device, CUDA error)
struct LibraryError : std::runtime_error { using std::runtime_error::runtime_error; };

namespace detail {
inline void check(ndi_status st) {
    if (st >= NDI_CUDA_ERROR || st == NDI_INVALID_ARGUMENT || st == NDI_UNSUPPORTED_DTYPE || st == NDI_NO_DEVICE || st == NDI_NO_SPLINE)
        throw LibraryError(std::string("ndi status ") + std::to_string((int)st) + ": " + ndi_last_error_message());
}
template <class T> struct dtype_of;
template <> struct dtype_of<float> { static constexpr ndi_dtype value = NDI_F32; };
template <> struct dtype_of<double> { static constexpr ndi_dtype value = NDI_F64; };
template <> struct dtype_of<int32_t> { static constexpr ndi_dtype value = NDI_I32; };
template <> struct dtype_of<int64_t> { static constexpr ndi_dtype value = NDI_I64; };
template <> struct dtype_of<uint32_t> { static constexpr ndi_dtype value = NDI_U32; };
template <> struct dtype_of<uint64_t> { static constexpr ndi_dtype value = NDI_U64; };

// `{:?}` of a Rust number: shortest round-trip digits, "1.0" for integral floats, "NaN", "inf"
template <class T>
std::string rust_debug(T v) {
    if constexpr (std::is_integral<T>::value) return std::to_string(v);
    else {
        if (std::isnan(v)) return "NaN";
        if (std::isinf(v)) return v < 0 ? "-inf" : "inf";
        char buf[64];
        auto r = std::to_chars(buf, buf + sizeof(buf), v);
        std::string s(buf, r.ptr);
        const auto e = s.find('e');
        if (e != std::string::npos) {                       // 1e+30 -> 1e30, 1e-07 -> 1e-7
            std::string mant = s.substr(0, e), ex = s.substr(e + 1);
            const bool neg = !ex.empty() && ex[0] == '-';
            ex.erase(0, ex.find_first_not_of("+-0"));
            return mant + "e" + (neg ? "-" : "") + (ex.empty() ? "0" : ex);
        }
        if (s.find('.') == std::string::npos) s += ".0";
        return s;
    }
}
inline std::string shape_str(const std::vector<size_t>& s) {
    std::string r = "[";
    for (size_t i = 0; i < s.size(); ++i) r += (i ? ", " : "") + std::to_string(s[i]);
    return r + "]";
}
inline size_t product(const std::vector<size_t>& s, size_t from = 0) {
    size_t p = 1;
    for (size_t i = from; i < s.size(); ++i) p *= s[i];
    return p;
}
}  // namespace detail

// ---- arrays --------------------------------------------------------------------------------------------
// A strided view (strides in elements, negative allowed: tests/interp1d.rs:143-155 uses slice(s![..;-1])).
template <class T>
struct ArrayView {
    const T* ptr = nullptr;
    std::vector<size_t> shape;
    std::vector<std::ptrdiff_t> strides;
    size_t ndim() const { return shape.size(); }
    size_t size() const { return detail::product(shape); }
    bool c_contiguous() const {
        std::ptrdiff_t want = 1;
        for (size_t i = shape.size(); i-- > 0;) {
            if (shape[i] != 1 && strides[i] != want) return false;
            want *= (std::ptrdiff_t)shape[i];
        }
        return true;
    }
    // logical (row-major) copy
    std::vector<T> to_vector() const {
        std::vector<T> out(size());
        if (out.empty()) return out;
        if (c_contiguous()) { std::copy(ptr, ptr + out.size(), out.begin()); return out; }
        std::vector<size_t> idx(shape.size(), 0);
        for (size_t k = 0; k < out.size(); ++k) {
            std::ptrdiff_t off = 0;
            for (size_t d = 0; d < shape.size(); ++d) off += (std::ptrdiff_t)idx[d] * strides[d];
            out[k] = ptr[off];
            for (size_t d = shape.size(); d-- > 0;) { if (++idx[d] < shape[d]) break; idx[d] = 0; }
        }
        return out;
    }
};
template <class T>
struct ArrayViewMut {
    T* ptr = nullptr;
    std::vector<size_t> shape;
    std::vector<std::ptrdiff_t> strides;
    size_t size() const { return detail::product(shape); }
    ArrayView<T> view() const { return ArrayView<T>{ptr, shape, strides}; }
    bool c_contiguous() const { return view().c_contiguous(); }
    void assign_rows(const std::vector<T>& rows) {          // rows: logical order
        if (rows.empty()) return;
        if (c_contiguous()) { std::copy(rows.begin(), rows.end(), ptr); return; }
        std::vector<size_t> idx(shape.size(), 0);
        for (size_t k = 0; k < rows.size(); ++k) {
            std::ptrdiff_t off = 0;
            for (size_t d = 0; d < shape.size(); ++d) off += (std::ptrdiff_t)idx[d] * strides[d];
            ptr[off] = rows[k];
            for (size_t d = shape.size(); d-- > 0;) { if (++idx[d] < shape[d]) break; idx[d] = 0; }
        }
    }
};

// Owned array in C order (ndarray::Array).
template <class T>
class Array {
public:
    Array() = default;
    // Array::zeros(shape) / Array(shape, fill).  (No one-argument shape constructor: `Array({n})` would
    // pick the initializer_list constructor below and build a one-element array holding n.)
    Array(std::vector<size_t> shape, T fill) : shape_(std::move(shape)), data_(detail::product(shape_), fill) {}
    static Array zeros(std::vector<size_t> shape) { return Array(std::move(shape), T()); }
    Array(std::vector<size_t> shape, std::vector<T> data) : shape_(std::move(shape)), data_(std::move(data)) {
        if (data_.size() != detail::product(shape_)) throw std::invalid_argument("Array: shape does not match the data length");
    }
    Array(std::initializer_list<T> v) : shape_{v.size()}, data_(v) {}                       // array![a, b, c]
    Array(std::initializer_list<std::initializer_list<T>> rows) {                             // array![[..], [..]]
        shape_ = {rows.size(), rows.size() ? rows.begin()->size() : 0};
        for (const auto& r : rows) {
            if (r.size() != shape_[1]) throw std::invalid_argument("Array: ragged rows");
            data_.insert(data_.end(), r.begin(), r.end());
        }
    }
    static Array linspace(T start, T end, size_t n) {       // ndarray's: start + step * i (SURVEY.md section 8(c))
        Array a = zeros({n});
        const T step = n > 1 ? (end - start) / (T)(n - 1) : T();
        for (size_t i = 0; i < n; ++i) a.data_[i] = start + step * (T)i;
        return a;
    }
    const std::vector<size_t>& shape() const { return shape_; }
    size_t ndim() const { return shape_.size(); }
    size_t size() const { return data_.size(); }
    T* data() { return data_.data(); }
    const T* data() const { return data_.data(); }
    T& operator[](size_t i) { return data_[i]; }
    const T& operator[](size_t i) const { return data_[i]; }
    const std::vector<T>& values() const { return data_; }
    bool operator==(const Array& o) const { return shape_ == o.shape_ && data_ == o.data_; }
    std::vector<std::ptrdiff_t> c_strides() const {
        std::vector<std::ptrdiff_t> s(shape_.size(), 1);
        for (size_t i = shape_.size(); i-- > 1;) s[i - 1] = s[i] * (std::ptrdiff_t)shape_[i];
        return s;
    }
    ArrayView<T> view() const { return ArrayView<T>{data_.data(), shape_, c_strides()}; }
    ArrayViewMut<T> view_mut() { return ArrayViewMut<T>{data_.data(), shape_, c_strides()}; }
    operator ArrayView<T>() const { return view(); }
    // reversed view along axis 0 (slice(s![..;-1]))
    ArrayView<T> reversed() const {
        auto st = c_strides();
        if (shape_.empty() || shape_[0] == 0) return view();
        const T* p = data_.data() + (std::ptrdiff_t)(shape_[0] - 1) * st[0];
        st[0] = -st[0];
        return ArrayView<T>{p, shape_, st};
    }
private:
    std::vector<size_t> shape_;
    std::vector<T> data_;
};

// ---- vector_extensions (src/vector_extensions.rs) -------------------------------------------------------
struct Monotonic {
    enum Kind { Rising, Falling, NotMonotonic } kind;
    bool strict;
    bool operator==(const Monotonic& o) const { return kind == o.kind && (kind == NotMonotonic || strict == o.strict); }
};
// VectorExtensions::monotonic_prop (:40-53, :115-198), on the device
template <class T>
Monotonic monotonic_prop(const ArrayView<T>& v) {
    if (v.ndim() != 1) throw std::invalid_argument("monotonic_prop: 1-D array expected");
    int32_t prop = NDI_MONO_NOT_MONOTONIC;
    detail::check(ndi_monotonic_prop(detail::dtype_of<T>::value, v.ptr, (int64_t)v.shape[0], (int64_t)v.strides[0], &prop));
    switch (prop) {
    case NDI_MONO_RISING_STRICT: return {Monotonic::Rising, true};
    case NDI_MONO_RISING: return {Monotonic::Rising, false};
    case NDI_MONO_FALLING_STRICT: return {Monotonic::Falling, true};
    case NDI_MONO_FALLING: return {Monotonic::Falling, false};
    default: return {Monotonic::NotMonotonic, false};
    }
}
// VectorExtensions::get_lower_index (:55-111); NaN panics like the reference (:83-84)
template <class T>
size_t get_lower_index(const ArrayView<T>& grid, T x) {
    const std::vector<T> g = grid.to_vector();
    int64_t idx = 0, bad = -1;
    const ndi_status st = ndi_lower_index(detail::dtype_of<T>::value, g.data(), (int64_t)g.size(), &x, 1, &idx, &bad);
    if (st == NDI_NAN_QUERY) throw Panic("not implemented: failed to convert NaN to usize");
    detail::check(st);
    return (size_t)idx;
}

// ---- 1-D ---------------------------------------------------------------------------------------------------
template <class T> class Interp1D;

// trait Interp1DStrategy (src/interp1d/strategies/mod.rs:42-65)
template <class T>
struct Interp1DStrategy {
    virtual ~Interp1DStrategy() = default;
    // interpolate at x into target (shape = data.shape[1..]); throw InterpolateError
    virtual void interp_into(const Interp1D<T>& interpolator, ArrayViewMut<T> target, T x) const = 0;
    // the reference's batch loop (interp1d/mod.rs:334-342): row q of out_rows belongs to xs[q], stop at the
    // first error.  out_rows: (nq, ...data.shape[1..]) C order.
    virtual void interp_batch_into(const Interp1D<T>& interpolator, const T* xs, size_t nq, T* out_rows) const;
    virtual void bind(const Interp1D<T>&) const {}          // built-in strategies finish their device state here
    virtual bool uses_device() const { return false; }
};
// trait Interp1DStrategyBuilder (src/interp1d/strategies/mod.rs:12-40)
template <class T>
struct Interp1DStrategyBuilder {
    virtual ~Interp1DStrategyBuilder() = default;
    virtual size_t MINIMUM_DATA_LENGHT() const = 0;         // (sic) the reference's spelling
    virtual std::shared_ptr<const Interp1DStrategy<T>> build(const ArrayView<T>& x, const ArrayView<T>& data) const = 0;
};

namespace detail {
template <class T>
[[noreturn]] void raise_eval(ndi_status st, const T* qs, int64_t first_bad, const char* name) {
    if (st == NDI_OUT_OF_BOUNDS)                             // linear.rs:80-84, cubic_spline.rs:798-802
        throw InterpolateError(std::string(name) + " = " + rust_debug(qs[first_bad]) + " is not in range");
    throw Panic("not implemented: failed to convert NaN to usize");                           // vector_extensions.rs:83-84
}
}  // namespace detail

// Linear Interpolation Strategy (src/interp1d/strategies/linear.rs)
template <class T>
class Linear : public Interp1DStrategyBuilder<T>, public Interp1DStrategy<T> {
public:
    Linear() = default;
    static Linear new_() { return Linear(); }
    Linear extrapolate(bool e) const { Linear l(*this); l.extrapolate_ = e; return l; }     // "does the strategy extrapolate? Default is false"
    size_t MINIMUM_DATA_LENGHT() const override { return 2; }
    std::shared_ptr<const Interp1DStrategy<T>> build(const ArrayView<T>&, const ArrayView<T>&) const override {
        return std::make_shared<Linear>(*this);              // linear.rs:54-63
    }
    bool uses_device() const override { return true; }
    void interp_batch_into(const Interp1D<T>& ip, const T* xs, size_t nq, T* out_rows) const override;
    void interp_into(const Interp1D<T>& ip, ArrayViewMut<T> target, T x) const override;      // linear.rs:73-98
    // NOT in the reference (ndi_interp1d_linear_deriv): slope of each query's interval, interp_batch_into's query
    // handling and errors; order must be 1 (std::invalid_argument otherwise)
    void deriv_batch_into(const Interp1D<T>& ip, const T* xs, size_t nq, T* out_rows, int order) const;
private:
    bool extrapolate_ = false;
};

// enum SingleBoundary / RowBoundary / BoundaryCondition (cubic_spline.rs:153-217)
template <class T>
struct SingleBoundary {
    int kind; T value;
    static SingleBoundary NotAKnot() { return {NDI_SB_NOT_A_KNOT, T()}; }
    static SingleBoundary Natural() { return {NDI_SB_NATURAL, T()}; }
    static SingleBoundary Clamped() { return {NDI_SB_CLAMPED, T()}; }
    static SingleBoundary FirstDeriv(T v) { return {NDI_SB_FIRST_DERIV, v}; }
    static SingleBoundary SecondDeriv(T v) { return {NDI_SB_SECOND_DERIV, v}; }
};
template <class T>
struct RowBoundary {
    SingleBoundary<T> left, right;
    static RowBoundary NotAKnot() { return {SingleBoundary<T>::NotAKnot(), SingleBoundary<T>::NotAKnot()}; }
    static RowBoundary Natural() { return {SingleBoundary<T>::Natural(), SingleBoundary<T>::Natural()}; }
    static RowBoundary Clamped() { return {SingleBoundary<T>::Clamped(), SingleBoundary<T>::Clamped()}; }
    static RowBoundary Mixed(SingleBoundary<T> l, SingleBoundary<T> r) { return {l, r}; }
};
template <class T>
struct BoundaryCondition {
    int kind = NDI_BC_NOT_A_KNOT;
    std::vector<size_t> rows_shape;                          // Individual: shape of the RowBoundary array
    std::vector<RowBoundary<T>> rows;
    static BoundaryCondition NotAKnot() { return {NDI_BC_NOT_A_KNOT, {}, {}}; }
    static BoundaryCondition Natural() { return {NDI_BC_NATURAL, {}, {}}; }
    static BoundaryCondition Clamped() { return {NDI_BC_CLAMPED, {}, {}}; }
    static BoundaryCondition Periodic() { return {NDI_BC_PERIODIC, {}, {}}; }
    // rows: RowBoundary array with the data's shape, axis 0 of length 1 (cubic_spline.rs:160-167)
    static BoundaryCondition Individual(std::vector<size_t> shape, std::vector<RowBoundary<T>> rows) {
        return {NDI_BC_INDIVIDUAL, std::move(shape), std::move(rows)};
    }
};

// The CubicSpline 1d interpolation Strategy (Implementation) (cubic_spline.rs:94-102): a, b live on the device
template <class T>
class CubicSplineStrategy : public Interp1DStrategy<T> {
public:
    CubicSplineStrategy(BoundaryCondition<T> bc, int mode, int build_mode = NDI_BUILD_AUTO, int build_levels = 0)
        : bc_(std::move(bc)), mode_(mode), build_mode_(build_mode), build_levels_(build_levels) {}
    // how the coefficients were built (ndi_interp1d_build_info): 0 the reference's elimination order, L > 0 row-split
    // with L levels, -m < 0 partition with blocks of m rows
    int rowsplit_levels(const Interp1D<T>& ip) const;
    int build_info(const Interp1D<T>& ip) const { return rowsplit_levels(ip); }
    bool uses_device() const override { return true; }
    void bind(const Interp1D<T>& ip) const override;         // CubicSpline::calc_coefficients (:310-368) on the device
    void interp_batch_into(const Interp1D<T>& ip, const T* xs, size_t nq, T* out_rows) const override;
    void interp_into(const Interp1D<T>& ip, ArrayViewMut<T> target, T x) const override;      // :791-830
    // NOT in the reference (ndi_interp1d_cubic_deriv): derivative of order 1 or 2 (std::invalid_argument otherwise),
    // interp_batch_into's query handling and errors
    void deriv_batch_into(const Interp1D<T>& ip, const T* xs, size_t nq, T* out_rows, int order) const;
    // (a, b) copied back from the device: shape (n-1, ...data.shape[1..])
    std::pair<Array<T>, Array<T>> coefficients(const Interp1D<T>& ip) const;
private:
    BoundaryCondition<T> bc_;
    int mode_, build_mode_, build_levels_;
};
// The CubicSpline 1d interpolation Strategy (Builder) (cubic_spline.rs:84-88, :723-772)
template <class T>
class CubicSpline : public Interp1DStrategyBuilder<T> {
    static_assert(std::is_floating_point<T>::value, "CubicSpline needs a float element type (SplineNum, cubic_spline.rs:34-49)");
public:
    static CubicSpline new_() { return CubicSpline(); }
    CubicSpline extrapolate(bool e) const { CubicSpline c(*this); c.extrapolate_ = e; return c; }
    CubicSpline boundary(BoundaryCondition<T> b) const { CubicSpline c(*this); c.boundary_ = std::move(b); return c; }
    // NOT in the reference (ndi_interp1d_set_build_mode): NDI_BUILD_AUTO, NDI_BUILD_SEQUENTIAL -- the reference's
    // elimination order, coefficients bit-identical to its arithmetic --, NDI_BUILD_ROWSPLIT with `levels` steps of
    // cyclic reduction (0: the library's choice) or NDI_BUILD_PARTITION with blocks of `levels` rows (0: 32)
    CubicSpline solver(int mode, int levels = 0) const { CubicSpline c(*this); c.build_mode_ = mode; c.build_levels_ = levels; return c; }
    size_t MINIMUM_DATA_LENGHT() const override { return 3; }
    std::shared_ptr<const Interp1DStrategy<T>> build(const ArrayView<T>&, const ArrayView<T>& data) const override {
        if (boundary_.kind == NDI_BC_INDIVIDUAL) {           // calc_coefficients :332-347
            std::vector<size_t> expect = data.shape;
            expect[0] = 1;
            if (boundary_.rows_shape != expect)
                throw BuilderError(BuilderError::ShapeError, "Boundary conditions array has wrong shape. Expected: " +
                                   detail::shape_str(expect) + ", got: " + detail::shape_str(boundary_.rows_shape));
        }
        const int mode = !extrapolate_ ? NDI_EXTRAP_NO : (boundary_.kind == NDI_BC_PERIODIC ? NDI_EXTRAP_PERIODIC : NDI_EXTRAP_YES);   // :763-769
        return std::make_shared<CubicSplineStrategy<T>>(boundary_, mode, build_mode_, build_levels_);
    }
private:
    bool extrapolate_ = false;
    int build_mode_ = NDI_BUILD_AUTO, build_levels_ = 0;
    BoundaryCondition<T> boundary_ = BoundaryCondition<T>::NotAKnot();
};

template <class T> class Interp1DBuilder;

// One dimensional interpolator (src/interp1d/mod.rs:38-51)
template <class T>
class Interp1D {
public:
    static Interp1DBuilder<T> builder(Array<T> data) { return Interp1DBuilder<T>(std::move(data)); }   // :79-81
    // Create a interpolator without any data validation (:363-365)
    static Interp1D new_unchecked(const ArrayView<T>& x, const ArrayView<T>& data, std::shared_ptr<const Interp1DStrategy<T>> strategy) {
        return Interp1D(Array<T>(x.shape, x.to_vector()), Array<T>(data.shape, data.to_vector()), std::move(strategy));
    }

    T interp_scalar(T x) const {                              // :108-114 (data dimension Ix1)
        if (data_.ndim() != 1) throw std::invalid_argument("interp_scalar needs 1-D data (Ix1)");
        T out{};
        strategy_->interp_into(*this, ArrayViewMut<T>{&out, {}, {}}, x);
        return out;
    }
    Array<T> interp(T x) const {                              // :150-156
        Array<T> target = Array<T>::zeros(trailing_shape());
        strategy_->interp_into(*this, target.view_mut(), x);
        return target;
    }
    void interp_into(T x, ArrayViewMut<T> buffer) const {     // :169-175
        if (buffer.shape != trailing_shape())
            throw Panic("Zip: Producer dimension mismatch, expected: " + detail::shape_str(trailing_shape()) + ", got: " + detail::shape_str(buffer.shape));
        strategy_->interp_into(*this, buffer, x);
    }
    Array<T> interp_array(const ArrayView<T>& xs) const {     // :197-211
        Array<T> ys = Array<T>::zeros(buffer_shape(xs.shape));
        interp_array_into(xs, ys.view_mut());
        return ys;
    }
    // :272-324; one launch for the whole batch, whatever the query rank
    void interp_array_into(const ArrayView<T>& xs, ArrayViewMut<T> buffer) const {
        array_into(xs, buffer, [&](const T* q, size_t nq, T* rows) { strategy_->interp_batch_into(*this, q, nq, rows); });
    }

    // ---- derivatives: NOT in the reference (built-in strategies: Linear order 1, CubicSpline order 1 or 2) ----------
    Array<T> interp_deriv(T x, int order = 1) const {
        Array<T> target = Array<T>::zeros(trailing_shape());
        std::vector<size_t> one_row = trailing_shape();
        one_row.insert(one_row.begin(), 1);
        std::vector<std::ptrdiff_t> st(one_row.size(), 1);
        for (size_t i = one_row.size(); i-- > 1;) st[i - 1] = st[i] * (std::ptrdiff_t)one_row[i];
        interp_array_deriv_into(ArrayView<T>{&x, {1}, {1}}, ArrayViewMut<T>{target.data(), one_row, st}, order);
        return target;
    }
    Array<T> interp_array_deriv(const ArrayView<T>& xs, int order = 1) const {
        Array<T> ys = Array<T>::zeros(buffer_shape(xs.shape));
        interp_array_deriv_into(xs, ys.view_mut(), order);
        return ys;
    }
    // buffer shape, errors and untouched rows after a failing query as interp_array_into
    void interp_array_deriv_into(const ArrayView<T>& xs, ArrayViewMut<T> buffer, int order = 1) const {
        const auto* lin = dynamic_cast<const Linear<T>*>(strategy_.get());
        const auto* cub = dynamic_cast<const CubicSplineStrategy<T>*>(strategy_.get());
        if (!lin && !cub) throw std::invalid_argument("derivatives are computed by the built-in strategies (Linear, CubicSpline) only");
        if (order != 1 && (lin || order != 2)) throw std::invalid_argument("no derivative of order " + std::to_string(order) + " for this strategy");
        array_into(xs, buffer, [&](const T* q, size_t nq, T* rows) {
            if (lin) lin->deriv_batch_into(*this, q, nq, rows, order);
            else cub->deriv_batch_into(*this, q, nq, rows, order);
        });
    }

    // accessors strategies may call back (:371-386)
    std::pair<T, ArrayView<T>> index_point(size_t index) const {
        auto sh = trailing_shape();
        std::vector<std::ptrdiff_t> st(sh.size(), 1);
        for (size_t i = sh.size(); i-- > 1;) st[i - 1] = st[i] * (std::ptrdiff_t)sh[i];
        return {x_[index], ArrayView<T>{data_.data() + index * row_len(), sh, st}};
    }
    size_t get_index_left_of(T x) const { return get_lower_index<T>(x_.view(), x); }
    bool is_in_range(T x) const { return x_[0] <= x && x <= x_[x_.size() - 1]; }

    const Array<T>& x() const { return x_; }
    const Array<T>& data() const { return data_; }
    const Interp1DStrategy<T>& strategy() const { return *strategy_; }
    size_t row_len() const { return detail::product(data_.shape(), 1); }
    std::vector<size_t> trailing_shape() const { return std::vector<size_t>(data_.shape().begin() + 1, data_.shape().end()); }
    // opaque device handle (created on first use; freed with the last copy of the interpolator)
    ndi_interp1d* handle() const {
        if (!handle_) {
            ndi_interp1d* h = nullptr;
            detail::check(ndi_interp1d_create(detail::dtype_of<T>::value, x_.data(), (int64_t)x_.size(), data_.data(), (int64_t)row_len(),
                                              NDI_ASSUME_VALID, &h));
            handle_ = std::shared_ptr<ndi_interp1d>(h, [](ndi_interp1d* p) { ndi_interp1d_destroy(p); });
        }
        return handle_.get();
    }

private:
    friend class Interp1DBuilder<T>;
    template <class Batch>
    void array_into(const ArrayView<T>& xs, ArrayViewMut<T> buffer, Batch&& batch) const {
        const std::vector<size_t> expect = buffer_shape(xs.shape);
        if (buffer.shape != expect)
            throw Panic("ShapeError/IncompatibleShape: incompatible shapes expected: " + detail::shape_str(expect) + ", got: " + detail::shape_str(buffer.shape));
        const std::vector<T> q = xs.to_vector();
        if (buffer.c_contiguous()) { batch(q.data(), q.size(), buffer.ptr); return; }
        std::vector<T> rows = buffer.view().to_vector();       // rows the reference would leave untouched stay as they are
        try { batch(q.data(), q.size(), rows.data()); }
        catch (...) { buffer.assign_rows(rows); throw; }
        buffer.assign_rows(rows);
    }
    Interp1D(Array<T> x, Array<T> data, std::shared_ptr<const Interp1DStrategy<T>> s) : x_(std::move(x)), data_(std::move(data)), strategy_(std::move(s)) {
        strategy_->bind(*this);
    }
    std::vector<size_t> buffer_shape(const std::vector<size_t>& query_shape) const {           // get_buffer_shape :346-354
        std::vector<size_t> s = query_shape;
        s.insert(s.end(), data_.shape().begin() + 1, data_.shape().end());
        return s;
    }
    Array<T> x_, data_;
    std::shared_ptr<const Interp1DStrategy<T>> strategy_;
    mutable std::shared_ptr<ndi_interp1d> handle_;
};

// Create and configure a Interp1D Interpolator (src/interp1d/mod.rs:53-70, :389-477).
// Default configuration: Linear{extrapolate: false}, x = index.
template <class T>
class Interp1DBuilder {
public:
    explicit Interp1DBuilder(Array<T> data) : data_(std::move(data)), strategy_(std::make_shared<Linear<T>>()) {   // :399-410
        const size_t n = data_.ndim() ? data_.shape()[0] : 0;
        x_ = Array<T>::zeros({n});
        for (size_t i = 0; i < n; ++i) x_[i] = (T)i;
    }
    static Interp1DBuilder new_(Array<T> data) { return Interp1DBuilder(std::move(data)); }
    Interp1DBuilder& x(Array<T> x) { x_ = std::move(x); return *this; }                       // must be strict monotonic rising
    template <class S> Interp1DBuilder& strategy(S s) { strategy_ = std::make_shared<S>(std::move(s)); return *this; }
    // Validate input data and create the configured Interp1D (:443-476); check order as in the reference
    Interp1D<T> build() const {
        if (data_.ndim() < 1) throw BuilderError(BuilderError::ShapeError, "data dimension is 0, needs to be at least 1");
        if (data_.shape()[0] < strategy_->MINIMUM_DATA_LENGHT())
            throw BuilderError(BuilderError::NotEnoughData, "The chosen Interpolation strategy needs at least " +
                               std::to_string(strategy_->MINIMUM_DATA_LENGHT()) + " data points");
        if (x_.ndim() != 1) throw BuilderError(BuilderError::ShapeError, "x needs to be 1-D");
        if (!(monotonic_prop<T>(x_.view()) == Monotonic{Monotonic::Rising, true}))                // K1 on the device
            throw BuilderError(BuilderError::Monotonic, "Values in the x axis need to be strictly monotonic rising");
        if (x_.size() != data_.shape()[0])
            throw BuilderError(BuilderError::ShapeError, "Lengths of x and data axis need to match. Got x: " + std::to_string(x_.size()) +
                               ", data: " + std::to_string(data_.shape()[0]));
        return Interp1D<T>(x_, data_, strategy_->build(x_.view(), data_.view()));
    }
private:
    Array<T> data_, x_;
    std::shared_ptr<const Interp1DStrategyBuilder<T>> strategy_;
};

// ---- 1-D member definitions ----------------------------------------------------------------------------------
template <class T>
void Interp1DStrategy<T>::interp_batch_into(const Interp1D<T>& ip, const T* xs, size_t nq, T* out_rows) const {
    const std::vector<size_t> sh = ip.trailing_shape();
    std::vector<std::ptrdiff_t> st(sh.size(), 1);
    for (size_t i = sh.size(); i-- > 1;) st[i - 1] = st[i] * (std::ptrdiff_t)sh[i];
    const size_t w = ip.row_len();
    for (size_t q = 0; q < nq; ++q) interp_into(ip, ArrayViewMut<T>{out_rows + q * w, sh, st}, xs[q]);
}
namespace detail {
// per-query trait method of a built-in strategy: one query through the batched launch
template <class T, class S>
void single_into(const S& strat, const Interp1D<T>& ip, ArrayViewMut<T> target, T x) {
    if (target.c_contiguous()) { strat.interp_batch_into(ip, &x, 1, target.ptr); return; }
    std::vector<T> row(ip.row_len());
    strat.interp_batch_into(ip, &x, 1, row.data());
    target.assign_rows(row);
}
}  // namespace detail
template <class T>
void Linear<T>::interp_batch_into(const Interp1D<T>& ip, const T* xs, size_t nq, T* out_rows) const {
    int64_t bad = -1;
    const ndi_status st = ndi_interp1d_linear(ip.handle(), xs, (int64_t)nq, extrapolate_, out_rows, &bad);
    detail::check(st);
    if (st != NDI_OK) detail::raise_eval<T>(st, xs, bad, "x");
}
template <class T>
void Linear<T>::interp_into(const Interp1D<T>& ip, ArrayViewMut<T> target, T x) const { detail::single_into<T>(*this, ip, target, x); }
template <class T>
void Linear<T>::deriv_batch_into(const Interp1D<T>& ip, const T* xs, size_t nq, T* out_rows, int order) const {
    if (order != 1) throw std::invalid_argument("Linear has only a first derivative, got order " + std::to_string(order));
    int64_t bad = -1;
    const ndi_status st = ndi_interp1d_linear_deriv(ip.handle(), xs, (int64_t)nq, extrapolate_, out_rows, &bad);
    detail::check(st);
    if (st != NDI_OK) detail::raise_eval<T>(st, xs, bad, "x");
}

template <class T>
void CubicSplineStrategy<T>::bind(const Interp1D<T>& ip) const {
    std::vector<int32_t> lk, rk; std::vector<T> lv, rv;
    for (const auto& r : bc_.rows) { lk.push_back(r.left.kind); lv.push_back(r.left.value); rk.push_back(r.right.kind); rv.push_back(r.right.value); }
    int64_t bad = -1;
    const bool ind = bc_.kind == NDI_BC_INDIVIDUAL;
    detail::check(ndi_interp1d_set_build_mode(ip.handle(), build_mode_, build_levels_));
    const ndi_status st = ndi_interp1d_spline_build(ip.handle(), bc_.kind, ind ? lk.data() : nullptr, ind ? lv.data() : nullptr,
                                                    ind ? rk.data() : nullptr, ind ? rv.data() : nullptr, &bad);
    detail::check(st);
    if (st == NDI_PERIODIC_MISMATCH)                          // cubic_spline.rs:483-507
        throw BuilderError(BuilderError::ValueError, "for periodic boundary condition the first and last value must be equal.");
}
template <class T>
void CubicSplineStrategy<T>::interp_batch_into(const Interp1D<T>& ip, const T* xs, size_t nq, T* out_rows) const {
    int64_t bad = -1;
    const ndi_status st = ndi_interp1d_cubic(ip.handle(), xs, (int64_t)nq, mode_, out_rows, &bad);
    detail::check(st);
    if (st != NDI_OK) detail::raise_eval<T>(st, xs, bad, "x");
}
template <class T>
void CubicSplineStrategy<T>::interp_into(const Interp1D<T>& ip, ArrayViewMut<T> target, T x) const { detail::single_into<T>(*this, ip, target, x); }
template <class T>
void CubicSplineStrategy<T>::deriv_batch_into(const Interp1D<T>& ip, const T* xs, size_t nq, T* out_rows, int order) const {
    if (order != 1 && order != 2) throw std::invalid_argument("CubicSpline derivative order must be 1 or 2, got " + std::to_string(order));
    int64_t bad = -1;
    const ndi_status st = ndi_interp1d_cubic_deriv(ip.handle(), xs, (int64_t)nq, mode_, order, out_rows, &bad);
    detail::check(st);
    if (st != NDI_OK) detail::raise_eval<T>(st, xs, bad, "x");
}
template <class T>
int CubicSplineStrategy<T>::rowsplit_levels(const Interp1D<T>& ip) const {
    int32_t lv = -1;
    detail::check(ndi_interp1d_build_info(ip.handle(), &lv));
    return lv;
}
template <class T>
std::pair<Array<T>, Array<T>> CubicSplineStrategy<T>::coefficients(const Interp1D<T>& ip) const {
    std::vector<size_t> sh = ip.data().shape();
    sh[0] -= 1;
    Array<T> a = Array<T>::zeros(sh), b = Array<T>::zeros(sh);
    detail::check(ndi_interp1d_spline_coeffs(ip.handle(), a.data(), b.data()));
    return {std::move(a), std::move(b)};
}

// ---- 2-D (src/interp2d) ----------------------------------------------------------------------------------------
template <class T> class Interp2D;
template <class T>
struct Interp2DStrategy {                                     // strategies/mod.rs:46-73
    virtual ~Interp2DStrategy() = default;
    virtual void interp_into(const Interp2D<T>& interpolator, ArrayViewMut<T> target, T x, T y) const = 0;
    virtual void interp_batch_into(const Interp2D<T>& interpolator, const T* xs, const T* ys, size_t nq, T* out_rows) const;
};
template <class T>
struct Interp2DStrategyBuilder {                              // strategies/mod.rs:14-44
    virtual ~Interp2DStrategyBuilder() = default;
    virtual size_t MINIMUM_DATA_LENGHT() const = 0;
    virtual std::shared_ptr<const Interp2DStrategy<T>> build(const ArrayView<T>& x, const ArrayView<T>& y, const ArrayView<T>& data) const = 0;
};
template <class T>
class Bilinear : public Interp2DStrategyBuilder<T>, public Interp2DStrategy<T> {             // strategies/bilinear.rs
public:
    static Bilinear new_() { return Bilinear(); }
    Bilinear extrapolate(bool e) const { Bilinear b(*this); b.extrapolate_ = e; return b; }
    size_t MINIMUM_DATA_LENGHT() const override { return 2; }
    std::shared_ptr<const Interp2DStrategy<T>> build(const ArrayView<T>&, const ArrayView<T>&, const ArrayView<T>&) const override {
        return std::make_shared<Bilinear>(*this);
    }
    void interp_batch_into(const Interp2D<T>& ip, const T* xs, const T* ys, size_t nq, T* out_rows) const override;
    void interp_into(const Interp2D<T>& ip, ArrayViewMut<T> target, T x, T y) const override;  // bilinear.rs:64-99
private:
    bool extrapolate_ = false;
};
template <class T> class Interp2DBuilder;

template <class T>
class Interp2D {                                              // interp2d/mod.rs:34-48
public:
    static Interp2DBuilder<T> builder(Array<T> data) { return Interp2DBuilder<T>(std::move(data)); }
    static Interp2D new_unchecked(const ArrayView<T>& x, const ArrayView<T>& y, const ArrayView<T>& data,
                                  std::shared_ptr<const Interp2DStrategy<T>> s) {            // :330-342
        return Interp2D(Array<T>(x.shape, x.to_vector()), Array<T>(y.shape, y.to_vector()), Array<T>(data.shape, data.to_vector()), std::move(s));
    }
    T interp_scalar(T x, T y) const {                         // :107-113
        if (data_.ndim() != 2) throw std::invalid_argument("interp_scalar needs 2-D data (Ix2)");
        T out{};
        strategy_->interp_into(*this, ArrayViewMut<T>{&out, {}, {}}, x, y);
        return out;
    }
    Array<T> interp(T x, T y) const {                         // :132-146
        Array<T> target = Array<T>::zeros(trailing_shape());
        strategy_->interp_into(*this, target.view_mut(), x, y);
        return target;
    }
    void interp_into(T x, T y, ArrayViewMut<T> buffer) const {   // :160-167
        if (buffer.shape != trailing_shape())
            throw Panic("Zip: Producer dimension mismatch, expected: " + detail::shape_str(trailing_shape()) + ", got: " + detail::shape_str(buffer.shape));
        strategy_->interp_into(*this, buffer, x, y);
    }
    Array<T> interp_array(const ArrayView<T>& xs, const ArrayView<T>& ys) const {              // :175-196
        if (xs.shape != ys.shape) throw Panic("`xs.shape()` and `ys.shape()` do not match");   // :189-192
        std::vector<size_t> sh = xs.shape;
        sh.insert(sh.end(), data_.shape().begin() + 2, data_.shape().end());
        Array<T> out = Array<T>::zeros(sh);
        interp_array_into(xs, ys, out.view_mut());
        return out;
    }
    void interp_array_into(const ArrayView<T>& xs, const ArrayView<T>& ys, ArrayViewMut<T> buffer) const {   // :215-307
        if (xs.shape != ys.shape) throw Panic("`xs.shape()` and `ys.shape()` do not match");
        std::vector<size_t> expect = xs.shape;
        expect.insert(expect.end(), data_.shape().begin() + 2, data_.shape().end());
        if (buffer.shape != expect)
            throw Panic("ShapeError/IncompatibleShape: incompatible shapes expected: " + detail::shape_str(expect) + ", got: " + detail::shape_str(buffer.shape));
        const std::vector<T> qx = xs.to_vector(), qy = ys.to_vector();
        if (buffer.c_contiguous()) { strategy_->interp_batch_into(*this, qx.data(), qy.data(), qx.size(), buffer.ptr); return; }
        std::vector<T> rows = buffer.view().to_vector();
        try { strategy_->interp_batch_into(*this, qx.data(), qy.data(), qx.size(), rows.data()); }
        catch (...) { buffer.assign_rows(rows); throw; }
        buffer.assign_rows(rows);
    }
    // :348-379
    std::tuple<T, T, ArrayView<T>> index_point(size_t ix, size_t iy) const {
        auto sh = trailing_shape();
        std::vector<std::ptrdiff_t> st(sh.size(), 1);
        for (size_t i = sh.size(); i-- > 1;) st[i - 1] = st[i] * (std::ptrdiff_t)sh[i];
        return {x_[ix], y_[iy], ArrayView<T>{data_.data() + (ix * y_.size() + iy) * row_len(), sh, st}};
    }
    std::pair<size_t, size_t> get_index_left_of(T x, T y) const { return {get_lower_index<T>(x_.view(), x), get_lower_index<T>(y_.view(), y)}; }
    bool is_in_x_range(T x) const { return x_[0] <= x && x <= x_[x_.size() - 1]; }
    bool is_in_y_range(T y) const { return y_[0] <= y && y <= y_[y_.size() - 1]; }
    size_t row_len() const { return detail::product(data_.shape(), 2); }
    std::vector<size_t> trailing_shape() const { return std::vector<size_t>(data_.shape().begin() + 2, data_.shape().end()); }
    const Array<T>& data() const { return data_; }
    ndi_interp2d* handle() const {
        if (!handle_) {
            ndi_interp2d* h = nullptr;
            detail::check(ndi_interp2d_create(detail::dtype_of<T>::value, x_.data(), (int64_t)x_.size(), y_.data(), (int64_t)y_.size(), data_.data(),
                                              (int64_t)row_len(), NDI_ASSUME_VALID, &h));
            handle_ = std::shared_ptr<ndi_interp2d>(h, [](ndi_interp2d* p) { ndi_interp2d_destroy(p); });
        }
        return handle_.get();
    }
private:
    friend class Interp2DBuilder<T>;
    Interp2D(Array<T> x, Array<T> y, Array<T> data, std::shared_ptr<const Interp2DStrategy<T>> s)
        : x_(std::move(x)), y_(std::move(y)), data_(std::move(data)), strategy_(std::move(s)) {}
    Array<T> x_, y_, data_;
    std::shared_ptr<const Interp2DStrategy<T>> strategy_;
    mutable std::shared_ptr<ndi_interp2d> handle_;
};

template <class T>
class Interp2DBuilder {                                       // interp2d/mod.rs:50-68, :381-518
public:
    explicit Interp2DBuilder(Array<T> data) : data_(std::move(data)), strategy_(std::make_shared<Bilinear<T>>()) {
        const size_t n = data_.ndim() > 0 ? data_.shape()[0] : 0, m = data_.ndim() > 1 ? data_.shape()[1] : 0;
        x_ = Array<T>::zeros({n}); y_ = Array<T>::zeros({m});
        for (size_t i = 0; i < n; ++i) x_[i] = (T)i;
        for (size_t i = 0; i < m; ++i) y_[i] = (T)i;
    }
    Interp2DBuilder& x(Array<T> x) { x_ = std::move(x); return *this; }
    Interp2DBuilder& y(Array<T> y) { y_ = std::move(y); return *this; }
    template <class S> Interp2DBuilder& strategy(S s) { strategy_ = std::make_shared<S>(std::move(s)); return *this; }
    Interp2D<T> build() const {                               // :468-518, same check order
        if (data_.ndim() < 2) throw BuilderError(BuilderError::ShapeError, "data dimension needs to be at least 2");
        const size_t need = strategy_->MINIMUM_DATA_LENGHT();
        if (data_.shape()[0] < need)
            throw BuilderError(BuilderError::NotEnoughData, "The 0-dimension has not enough data for the chosen interpolation strategy. Provided: " +
                               std::to_string(data_.shape()[0]) + ", required: " + std::to_string(need));
        if (data_.shape()[1] < need)
            throw BuilderError(BuilderError::NotEnoughData, "The 1-dimension has not enough data for the chosen interpolation strategy. Provided: " +
                               std::to_string(data_.shape()[1]) + ", required: " + std::to_string(need));
        if (!(monotonic_prop<T>(x_.view()) == Monotonic{Monotonic::Rising, true}))
            throw BuilderError(BuilderError::Monotonic, "The x-axis needs to be strictly monotonic rising");
        if (!(monotonic_prop<T>(y_.view()) == Monotonic{Monotonic::Rising, true}))
            throw BuilderError(BuilderError::Monotonic, "The y-axis needs to be strictly monotonic rising");
        if (x_.size() != data_.shape()[0])
            throw BuilderError(BuilderError::ShapeError, "Lengths of x-axis and data-0-axis need to match. Got x: " + std::to_string(x_.size()) +
                               ", data-0: " + std::to_string(data_.shape()[0]));
        if (y_.size() != data_.shape()[1])
            throw BuilderError(BuilderError::ShapeError, "Lengths of y-axis and data-1-axis need to match. Got y: " + std::to_string(y_.size()) +
                               ", data-1: " + std::to_string(data_.shape()[1]));
        return Interp2D<T>(x_, y_, data_, strategy_->build(x_.view(), y_.view(), data_.view()));
    }
private:
    Array<T> data_, x_, y_;
    std::shared_ptr<const Interp2DStrategyBuilder<T>> strategy_;
};

template <class T>
void Interp2DStrategy<T>::interp_batch_into(const Interp2D<T>& ip, const T* xs, const T* ys, size_t nq, T* out_rows) const {
    const std::vector<size_t> sh = ip.trailing_shape();
    std::vector<std::ptrdiff_t> st(sh.size(), 1);
    for (size_t i = sh.size(); i-- > 1;) st[i - 1] = st[i] * (std::ptrdiff_t)sh[i];
    const size_t w = ip.row_len();
    for (size_t q = 0; q < nq; ++q) interp_into(ip, ArrayViewMut<T>{out_rows + q * w, sh, st}, xs[q], ys[q]);
}
template <class T>
void Bilinear<T>::interp_batch_into(const Interp2D<T>& ip, const T* xs, const T* ys, size_t nq, T* out_rows) const {
    int64_t bad = -1; int32_t axis = -1;
    const ndi_status st = ndi_interp2d_bilinear(ip.handle(), xs, ys, (int64_t)nq, extrapolate_, out_rows, &bad, &axis);
    detail::check(st);
    if (st != NDI_OK) detail::raise_eval<T>(st, axis == 0 ? xs : ys, bad, axis == 0 ? "x" : "y");   // x before y: bilinear.rs:71-80
}
template <class T>
void Bilinear<T>::interp_into(const Interp2D<T>& ip, ArrayViewMut<T> target, T x, T y) const {
    if (target.c_contiguous()) { interp_batch_into(ip, &x, &y, 1, target.ptr); return; }
    std::vector<T> row(ip.row_len());
    interp_batch_into(ip, &x, &y, 1, row.data());
    target.assign_rows(row);
}

}  // namespace ndarray_interp
