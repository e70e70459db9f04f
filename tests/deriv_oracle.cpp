// deriv_oracle.cpp -- CPU specification of the derivative calls (ndi_interp1d_cubic_deriv, ndi_interp1d_linear_deriv).
//
// TEST INFRASTRUCTURE, NOT PRODUCT CODE (loaded by tests/deriv_oracle.py and scripts/bench_deriv.py only).  The
// derivatives are NOT part of the reference, so there is nothing to restate: this file states the operation order the
// kernels promise (include/ndi_b200.h, DESIGN.md section 1) on top of the reference restatement in oracle/ndi_oracle.cpp,
// whose query handling -- range check, periodic wrap, NaN, get_lower_index -- it uses unchanged.  Build with the same
// flags as the oracle (-ffp-contract=off, no -ffast-math): one rounding per operation, true division.
#include "../oracle/ndi_oracle.cpp"

namespace {

// The exact derivatives of the value form (1-t) yl + t yr + t (1-t) (a (1-t) + b t) (cubic_spline.rs:825-827), with
// t = (x - xl) / h (:818), h = xr - xl, operations in this order:
//     cur = a (1-t) + b t,  ba = b - a
//     order 1:  d1 = (((yr - yl) + ((1-t) - t) cur) + (t (1-t)) ba) / h
//     order 2:  d2 = ((2 (((1-t) - t) ba - cur)) / h) / h
template <class T>
int32_t interp1d_cubic_deriv(const T* g, int64_t n, const T* data, const T* a, const T* b, int64_t w, const T* q,
                             int64_t nq, int32_t extrap_mode, int32_t order, T* out, int64_t* first_bad) {
    if (order != 1 && order != 2) return ST_INVALID_ARGUMENT;
    const T one = (T)1.0, two = (T)2.0;
    for (int64_t i = 0; i < nq; ++i) {
        T x = q[i];
        bool inr = in_range(g, n, x);                             // as interp1d_cubic (cubic_spline.rs:797-811)
        if (extrap_mode == 0 && !inr) { *first_bad = i; return ST_OUT_OF_BOUNDS; }
        if (extrap_mode == 2 && !inr) {
            T x0 = g[0], xn = g[n - 1];
            x = rem_euclid<T>(x - x0, xn - x0) + x0;
        }
        int32_t st = ST_OK;
        int64_t idx = get_lower_index(g, n, x, &st);
        if (st != ST_OK) { *first_bad = i; return st; }
        const T xl = g[idx], xr = g[idx + 1];
        const T* yl = data + idx * w;
        const T* yr = data + (idx + 1) * w;
        const T* al = a + idx * w;
        const T* bl = b + idx * w;
        const T h = xr - xl;
        const T t = (x - xl) / h;
        const T omt = one - t, dmt = omt - t, tt = t * omt;
        T* y = out + i * w;
        for (int64_t c = 0; c < w; ++c) {
            const T cur = al[c] * omt + bl[c] * t;
            const T ba = bl[c] - al[c];
            if (order == 1) y[c] = (((yr[c] - yl[c]) + dmt * cur) + tt * ba) / h;
            else y[c] = ((two * (dmt * ba - cur)) / h) / h;
        }
    }
    return ST_OK;
}

// slope of Linear: m = (y2 - y1) / (x2 - x1), the first term of calc_frac (linear.rs:29-36); query handling of
// interp1d_linear (linear.rs:80-91), integer arithmetic wrapping / truncating like it
template <class T>
int32_t interp1d_linear_deriv(const T* g, int64_t n, const T* data, int64_t w, const T* q, int64_t nq,
                              int32_t extrapolate, T* out, int64_t* first_bad) {
    for (int64_t i = 0; i < nq; ++i) {
        T x = q[i];
        if (!extrapolate && !in_range(g, n, x)) { *first_bad = i; return ST_OUT_OF_BOUNDS; }
        int32_t st = ST_OK;
        int64_t idx = get_lower_index(g, n, x, &st);
        if (st != ST_OK) { *first_bad = i; return st; }
        const T d = t_sub(g[idx + 1], g[idx]);
        const T* y1 = data + idx * w;
        const T* y2 = data + (idx + 1) * w;
        T* t = out + i * w;
        for (int64_t c = 0; c < w; ++c) t[c] = t_div(t_sub(y2[c], y1[c]), d);
    }
    return ST_OK;
}

}  // namespace

#define ORA_DERIV_LINEAR(SFX, T)                                                                                     \
    extern "C" int32_t ora_interp1d_linear_deriv_##SFX(const T* g, int64_t n, const T* data, int64_t w, const T* q, \
                                                       int64_t nq, int32_t extrapolate, T* out, int64_t* first_bad) { \
        return interp1d_linear_deriv<T>(g, n, data, w, q, nq, extrapolate, out, first_bad);                          \
    }
#define ORA_DERIV_CUBIC(SFX, T)                                                                                      \
    extern "C" int32_t ora_interp1d_cubic_deriv_##SFX(const T* g, int64_t n, const T* data, const T* a, const T* b, \
                                                      int64_t w, const T* q, int64_t nq, int32_t extrap_mode,        \
                                                      int32_t order, T* out, int64_t* first_bad) {                   \
        return interp1d_cubic_deriv<T>(g, n, data, a, b, w, q, nq, extrap_mode, order, out, first_bad);              \
    }

ORA_DERIV_LINEAR(f32, float)
ORA_DERIV_LINEAR(f64, double)
ORA_DERIV_LINEAR(i32, int32_t)
ORA_DERIV_LINEAR(i64, int64_t)
ORA_DERIV_LINEAR(u32, uint32_t)
ORA_DERIV_LINEAR(u64, uint64_t)
ORA_DERIV_CUBIC(f32, float)
ORA_DERIV_CUBIC(f64, double)
