// hermite_oracle.cpp -- CPU specification of ndi_interp1d_hermite_build (PCHIP, Akima, makima, given slopes).
//
// TEST INFRASTRUCTURE, NOT PRODUCT CODE (loaded by tests/hermite_oracle.py and scripts/bench_hermite.py only).  It
// states the operation order the build promises (include/ndi_b200.h): scipy's (scipy/interpolate/_cubic.py,
// PchipInterpolator._find_derivatives / _edge_case and Akima1DInterpolator.__init__), every operation rounded on its
// own in the table's dtype, so that in f64 the knot slopes are scipy's bit for bit.  Built with the oracle's flags
// (-ffp-contract=off, no -ffast-math): one rounding per operation, true division.
#include <cmath>
#include <cstdint>
#include <vector>

namespace {

enum { PCHIP = 0, AKIMA = 1, MAKIMA = 2, GIVEN = 3 };

// numpy's sign: sign(+-0) = 0, sign(NaN) = NaN (unequal to everything)
template <class T>
T sgn(T v) { return v > (T)0 ? (T)1 : (v < (T)0 ? (T)-1 : (v == (T)0 ? (T)0 : v)); }

// PchipInterpolator._edge_case
template <class T>
T pchip_edge(T h0, T h1, T m0, T m1) {
    const T e = (((T)2 * h0 + h1) * m0 - h0 * m1) / (h0 + h1);
    if (sgn(e) != sgn(m0)) return (T)0;
    if (sgn(m0) != sgn(m1) && std::fabs(e) > (T)3 * std::fabs(m0)) return (T)3 * m0;
    return e;
}

// d (n, w) for kind; dydx is only read for GIVEN
template <class T>
int32_t slopes(const T* x, int64_t n, const T* y, int64_t w, int32_t kind, const T* dydx, T* d) {
    if (n < 2 || kind < PCHIP || kind > GIVEN || (kind == GIVEN) != (dydx != nullptr)) return 2;
    if (kind == GIVEN) {
        for (int64_t i = 0; i < n * w; ++i) d[i] = dydx[i];
        return 0;
    }
    std::vector<T> h((size_t)(n - 1)), m((size_t)(n - 1) * w);
    for (int64_t k = 0; k + 1 < n; ++k) {
        h[k] = x[k + 1] - x[k];
        for (int64_t c = 0; c < w; ++c) m[k * w + c] = (y[(k + 1) * w + c] - y[k * w + c]) / h[k];
    }
    if (n == 2) {                                                     // both kinds: the straight line
        for (int64_t c = 0; c < w; ++c) d[c] = d[w + c] = m[c];
        return 0;
    }
    if (kind == PCHIP) {
        for (int64_t c = 0; c < w; ++c) {
            for (int64_t k = 1; k + 1 < n; ++k) {
                const T ml = m[(k - 1) * w + c], mr = m[k * w + c];
                if (sgn(ml) != sgn(mr) || mr == (T)0 || ml == (T)0) { d[k * w + c] = (T)0; continue; }
                const T w1 = (T)2 * h[k] + h[k - 1], w2 = h[k] + (T)2 * h[k - 1];
                const T whmean = (w1 / ml + w2 / mr) / (w1 + w2);
                d[k * w + c] = (T)1 / whmean;
            }
            d[c] = pchip_edge<T>(h[0], h[1], m[c], m[w + c]);
            d[(n - 1) * w + c] = pchip_edge<T>(h[n - 2], h[n - 3], m[(n - 2) * w + c], m[(n - 3) * w + c]);
        }
        return 0;
    }
    // Akima / makima: segment slopes extended by two on each side, mp[j + 2] = m[j] for j = -2 .. n
    const int64_t np = n + 3;
    std::vector<T> mp((size_t)np * w), f1((size_t)n * w), f2((size_t)n * w), f12((size_t)n * w);
    for (int64_t c = 0; c < w; ++c) {
        for (int64_t j = 0; j + 1 < n; ++j) mp[(j + 2) * w + c] = m[j * w + c];
        mp[1 * w + c] = (T)2 * mp[2 * w + c] - mp[3 * w + c];
        mp[0 * w + c] = (T)2 * mp[1 * w + c] - mp[2 * w + c];
        mp[(np - 2) * w + c] = (T)2 * mp[(np - 3) * w + c] - mp[(np - 4) * w + c];
        mp[(np - 1) * w + c] = (T)2 * mp[(np - 2) * w + c] - mp[(np - 3) * w + c];
    }
    // M: the maximum of f12 over the whole table; NaN as soon as one f12 is NaN (numpy's max)
    bool nan = false;
    T mmax = (T)0;
    for (int64_t i = 0; i < n; ++i)
        for (int64_t c = 0; c < w; ++c) {
            const T a3 = mp[(i + 3) * w + c], a2 = mp[(i + 2) * w + c], a1 = mp[(i + 1) * w + c], a0 = mp[i * w + c];
            T g1 = std::fabs(a3 - a2), g2 = std::fabs(a1 - a0);
            if (kind == MAKIMA) { g1 = g1 + (T)0.5 * std::fabs(a3 + a2); g2 = g2 + (T)0.5 * std::fabs(a1 + a0); }
            const T s = g1 + g2;
            f1[i * w + c] = g1; f2[i * w + c] = g2; f12[i * w + c] = s;
            if (s != s) nan = true;
            else if (s > mmax) mmax = s;
        }
    const T thr = (T)1e-9 * (nan ? (T)NAN : mmax);
    for (int64_t i = 0; i < n; ++i)
        for (int64_t c = 0; c < w; ++c) {
            const T a3 = mp[(i + 3) * w + c], a2 = mp[(i + 2) * w + c], a1 = mp[(i + 1) * w + c], a0 = mp[i * w + c];
            const T s = f12[i * w + c];
            d[i * w + c] = s > thr ? a1 + (f2[i * w + c] / s) * (a2 - a1) : (T)0.5 * (a3 + a0);
        }
    return 0;
}

// coefficients of the handle's cubic form from knot slopes: a[i] = d[i] h - dy, b[i] = dy - d[i+1] h
template <class T>
void coeffs(const T* x, int64_t n, const T* y, int64_t w, const T* d, T* a, T* b) {
    for (int64_t i = 0; i + 1 < n; ++i) {
        const T h = x[i + 1] - x[i];
        for (int64_t c = 0; c < w; ++c) {
            const T dy = y[(i + 1) * w + c] - y[i * w + c];
            a[i * w + c] = d[i * w + c] * h - dy;
            b[i * w + c] = dy - d[(i + 1) * w + c] * h;
        }
    }
}

}  // namespace

#define ORA_HERMITE(SFX, T)                                                                                          \
    extern "C" int32_t ora_hermite_##SFX(const T* x, int64_t n, const T* y, int64_t w, int32_t kind, const T* dydx, \
                                         T* d, T* a, T* b) {                                                         \
        const int32_t st = slopes<T>(x, n, y, w, kind, dydx, d);                                                     \
        if (st == 0) coeffs<T>(x, n, y, w, d, a, b);                                                                 \
        return st;                                                                                                   \
    }

ORA_HERMITE(f32, float)
ORA_HERMITE(f64, double)
