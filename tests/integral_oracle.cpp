// integral_oracle.cpp -- CPU specification of the integral calls (ndi_interp1d_integral_build, ndi_interp1d_cubic_integral,
// ndi_interp1d_linear_integral).
//
// TEST INFRASTRUCTURE, NOT PRODUCT CODE (loaded by tests/integral_oracle.py and scripts/bench_integral.py only).  The
// integrals are NOT part of the reference: this file states the operation order the kernels promise (include/ndi_b200.h,
// DESIGN.md section 1) on top of the reference restatement in oracle/ndi_oracle.cpp, whose query handling -- range check,
// periodic wrap, NaN, get_lower_index -- it uses unchanged for each bound.  Build with the same flags as the oracle
// (-ffp-contract=off, no -ffast-math): one rounding per operation, true division.
#include "../oracle/ndi_oracle.cpp"

namespace {

constexpr int64_t kIntBlock = 32;

// e[i] = h ((y[i] + y[i+1]) * 0.5 + (a[i] + b[i]) / 12) in double (Linear: a == nullptr, no second term)
template <class T>
double interval_integral(const T* x, const T* data, const T* a, const T* b, int64_t w, int64_t i, int64_t c) {
    const double h = (double)(T)(x[i + 1] - x[i]);
    double s = ((double)data[i * w + c] + (double)data[(i + 1) * w + c]) * 0.5;
    if (a) s = s + ((double)a[i * w + c] + (double)b[i * w + c]) / 12.0;
    return h * s;
}

// C[32k + j] = off(k) + local(k, j): running sums inside blocks of 32 intervals, a sequential sum over block totals
template <class T>
void integral_table(const T* x, int64_t n, const T* data, const T* a, const T* b, int64_t w, T* cum) {
    for (int64_t c = 0; c < w; ++c) {
        double off = 0.0;
        for (int64_t k = 0; k * kIntBlock <= n - 1; ++k) {
            double s = 0.0;
            const int64_t i1 = std::min((k + 1) * kIntBlock, n - 1);
            int64_t i = k * kIntBlock;
            for (; i < i1; ++i) {
                cum[i * w + c] = (T)(off + s);
                s = s + interval_integral<T>(x, data, a, b, w, i, c);
            }
            if (i == n - 1) cum[i * w + c] = (T)(off + s);
            off = off + s;
        }
    }
}

// the value call's handling of one bound: ST_OK, ST_OUT_OF_BOUNDS or ST_NAN_QUERY
template <class T>
int32_t bound_status(const T* g, int64_t n, T x, int32_t mode, bool cubic) {
    const bool inr = in_range(g, n, x);
    if (mode == 0 && !inr) return ST_OUT_OF_BOUNDS;
    if (cubic && mode == 2 && !inr) x = rem_euclid<T>(x - g[0], g[n - 1] - g[0]) + g[0];
    int32_t st = ST_OK;
    get_lower_index(g, n, x, &st);
    return st;
}

// W0..W3 of a point (include/ndi_b200.h), i its lower index
template <class T>
int64_t integral_weights(const T* g, int64_t n, T x, T W[4]) {
    int32_t st = ST_OK;
    const int64_t i = get_lower_index(g, n, x, &st);
    const T h = g[i + 1] - g[i];
    const T t = (x - g[i]) / h;
    const T tt = t * t;
    const T c2 = tt * (T)0.5;
    const T c3 = (tt * t) / (T)3;
    const T c4 = (tt * tt) * (T)0.25;
    W[0] = h * (t - c2);
    W[1] = h * c2;
    W[2] = h * ((c2 - (c3 + c3)) + c4);
    W[3] = h * (c3 - c4);
    return i;
}

template <class T>
T integral_f(const T* data, const T* a, const T* b, int64_t w, int64_t i, int64_t c, const T W[4]) {
    T s = W[0] * data[i * w + c] + W[1] * data[(i + 1) * w + c];
    if (a) s = (s + W[2] * a[i * w + c]) + W[3] * b[i * w + c];
    return s;
}

// a == nullptr: Linear (mode = extrapolate, no periodic branch)
template <class T>
int32_t integrate(const T* g, int64_t n, const T* data, const T* a, const T* b, const T* cum, int64_t w, const T* qlo,
                  const T* qhi, int64_t nq, int32_t mode, T* out, int64_t* first_bad, int32_t* bad_bound) {
    const bool cubic = a != nullptr;
    const T g0 = g[0], gl = g[n - 1];
    for (int64_t q = 0; q < nq; ++q) {
        T lo = qlo[q], hi = qhi[q];
        for (int32_t bound = 0; bound < 2; ++bound) {                // lo before hi
            const int32_t st = bound_status<T>(g, n, bound ? hi : lo, mode, cubic);
            if (st != ST_OK) { *first_bad = q; *bad_bound = bound; return st; }
        }
        bool neg = false, seam = false;
        if (hi < lo) { std::swap(lo, hi); neg = true; }
        T u = lo, v = hi, k = (T)0;
        if (cubic && mode == 2) {                                    // scipy's PPoly.integrate, periodic branch
            const T P = gl - g0;
            const T d = hi - lo;
            const T left = rem_euclid<T>(d, P);
            k = std::nearbyint((d - left) / P);
            if (!in_range(g, n, u)) u = rem_euclid<T>(u - g0, P) + g0;
            const T e = u + left;
            if (e <= gl) v = e;
            else { v = g0 + (e - gl); seam = true; }
        }
        T WL[4], WH[4];
        const int64_t i = integral_weights<T>(g, n, u, WL), j = integral_weights<T>(g, n, v, WH);
        for (int64_t c = 0; c < w; ++c) {
            const T cn = cum[(n - 1) * w + c];
            const T ch = seam ? cum[j * w + c] + cn : cum[j * w + c];
            T r = ((ch - cum[i * w + c]) + integral_f<T>(data, a, b, w, j, c, WH)) - integral_f<T>(data, a, b, w, i, c, WL);
            if (cubic && mode == 2) r = k * cn + r;
            out[q * w + c] = neg ? -r : r;
        }
    }
    return ST_OK;
}

}  // namespace

#define ORA_INTEGRAL(SFX, T)                                                                                          \
    extern "C" void ora_integral_table_##SFX(const T* x, int64_t n, const T* data, const T* a, const T* b, int64_t w,  \
                                             T* cum) {                                                                \
        integral_table<T>(x, n, data, a, b, w, cum);                                                                  \
    }                                                                                                                 \
    extern "C" int32_t ora_integrate_##SFX(const T* g, int64_t n, const T* data, const T* a, const T* b, const T* cum, \
                                           int64_t w, const T* lo, const T* hi, int64_t nq, int32_t mode, T* out,     \
                                           int64_t* first_bad, int32_t* bad_bound) {                                  \
        return integrate<T>(g, n, data, a, b, cum, w, lo, hi, nq, mode, out, first_bad, bad_bound);                   \
    }

ORA_INTEGRAL(f32, float)
ORA_INTEGRAL(f64, double)
