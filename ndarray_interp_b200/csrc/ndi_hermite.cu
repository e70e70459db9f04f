// ndi_hermite.cu -- K10: knot slopes and coefficients of the shape-preserving cubics (NOT in the reference; built by
// ndi_interp1d_hermite_build, include/ndi_b200.h).  PCHIP, Akima, makima, or slopes the caller gives; the slopes k
// become the handle's cubic form a[i] = k[i] h - dy, b[i] = dy - k[i+1] h, which every cubic kernel reads unchanged.
//
// One thread owns V consecutive columns (one 16-byte vector, or a single column when rows are narrower than 16 bytes
// or w is not a multiple of the vector) and a run of R consecutive intervals.  It walks the run with a window of four
// segments j = k-2 .. k+1 (spacing h, difference dy, slope m) held in registers, so each knot's slope is computed once
// per column and each segment slope once, apart from the window's set-up at the start of a run.  All arithmetic is
// in the table's dtype with one rounding per operation, in scipy's order (tests/hermite_oracle.cpp states it).  The
// divisors shared by a row -- h and PCHIP's w1 + w2 -- have their reciprocal formed once (Hoisted<T>: the quotient
// keeps the bits of an IEEE division); the divisions by per-column values are IEEE divisions.
//
// Akima / makima first need M, the maximum of f12 over the whole table: a first pass reduces it per block and
// combines the blocks with an atomicMax on the bit pattern (f12 >= 0, so the integer order is the value order and the
// result does not depend on the order of the blocks), with a separate flag for a NaN f12.
#include "ndi_device.cuh"
#include "ndi_internal.h"

namespace ndi {

enum { HERMITE_PCHIP = 0, HERMITE_AKIMA = 1, HERMITE_MAKIMA = 2, HERMITE_GIVEN = 3 };   // NDI_HERMITE_*
constexpr int kHermiteThinRun = 4;      // intervals per thread on rows narrower than a vector: a warp reads 128 rows
constexpr int kHermiteMaxRun = 64;

// numpy's sign: sign(+-0) = 0, sign(NaN) = NaN (unequal to everything)
template <class T>
__device__ __forceinline__ T sgn(T v) { return v > (T)0 ? (T)1 : (v < (T)0 ? (T)-1 : (v == (T)0 ? (T)0 : v)); }

template <class T, int V>
struct Seg { T h; Vec<T, V> dy, m; };

// segment j (0 <= j <= n-2): h = x[j+1] - x[j], dy = y[j+1] - y[j], m = dy / h (GIVEN needs no m)
template <class T, int V, int KIND>
__device__ __forceinline__ Seg<T, V> load_seg(const T* __restrict__ x, const T* __restrict__ y, long long w, long long j,
                                               long long c0) {
    Seg<T, V> s;
    s.h = Ar<T>::sub(x[j + 1], x[j]);
    const Vec<T, V> yl = ld_table<T, V>(y + j * w + c0), yr = ld_table<T, V>(y + (j + 1) * w + c0);
    const T r = KIND == HERMITE_GIVEN ? (T)0 : Hoisted<T>::rcp(s.h);
#pragma unroll
    for (int e = 0; e < V; ++e) {
        s.dy.v[e] = Ar<T>::sub(yr.v[e], yl.v[e]);
        s.m.v[e] = KIND == HERMITE_GIVEN ? (T)0 : Hoisted<T>::div(s.dy.v[e], s.h, r);
    }
    return s;
}

// Akima's extended slope beyond an end: 2 m1 - m2
template <class T, int V>
__device__ __forceinline__ void extend(Vec<T, V>& m, const Vec<T, V>& m1, const Vec<T, V>& m2) {
#pragma unroll
    for (int e = 0; e < V; ++e) m.v[e] = Ar<T>::sub(Ar<T>::mul((T)2, m1.v[e]), m2.v[e]);
}

// the window of segments k0-2 .. k0+1 at the first knot k0 of a run (n >= 3 for the extensions)
template <class T, int V, int KIND>
__device__ __forceinline__ void window_init(const T* x, long long n, const T* y, long long w, long long k0, long long c0,
                                            Seg<T, V> (&win)[4]) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const long long j = k0 - 2 + q;
        if (j >= 0 && j <= n - 2) win[q] = load_seg<T, V, KIND>(x, y, w, j, c0);
        else { win[q].h = (T)0; for (int e = 0; e < V; ++e) win[q].dy.v[e] = win[q].m.v[e] = (T)0; }
    }
    if constexpr (KIND == HERMITE_AKIMA || KIND == HERMITE_MAKIMA) {
        if (n >= 3) {
            // m[-1] = 2 m[0] - m[1], then m[-2] = 2 m[-1] - m[0]; m[n-1] = 2 m[n-2] - m[n-3], then m[n] = 2 m[n-1] - m[n-2]
            if (k0 == 0) extend<T, V>(win[1].m, win[2].m, win[3].m);
            if (k0 <= 1) extend<T, V>(win[0].m, win[1].m, win[2].m);
#pragma unroll
            for (int q = 2; q < 4; ++q)
                if (k0 - 2 + q > n - 2) extend<T, V>(win[q].m, win[q - 1].m, win[q - 2].m);
        }
    }
}

// advance the window from knot k to k+1: segment k+2 enters
template <class T, int V, int KIND>
__device__ __forceinline__ void window_shift(const T* x, long long n, const T* y, long long w, long long k, long long c0,
                                             Seg<T, V> (&win)[4]) {
    win[0] = win[1]; win[1] = win[2]; win[2] = win[3];
    const long long j = k + 2;
    if (j <= n - 2) win[3] = load_seg<T, V, KIND>(x, y, w, j, c0);
    else if constexpr (KIND == HERMITE_AKIMA || KIND == HERMITE_MAKIMA) extend<T, V>(win[3].m, win[2].m, win[1].m);
}

// PchipInterpolator._edge_case
template <class T>
__device__ __forceinline__ T pchip_edge(T h0, T h1, T m0, T m1, T rs) {
    const T num = Ar<T>::sub(Ar<T>::mul(Ar<T>::add(Ar<T>::mul((T)2, h0), h1), m0), Ar<T>::mul(h0, m1));
    const T e = Hoisted<T>::div(num, Ar<T>::add(h0, h1), rs);
    if (sgn(e) != sgn(m0)) return (T)0;
    if (sgn(m0) != sgn(m1) && fabs(e) > Ar<T>::mul((T)3, fabs(m0))) return Ar<T>::mul((T)3, m0);
    return e;
}

// Akima's f1, f2 at knot k from the window (m[k-2] .. m[k+1])
template <class T, int KIND>
__device__ __forceinline__ void akima_weights(T m0, T m1, T m2, T m3, T& f1, T& f2) {
    f1 = fabs(Ar<T>::sub(m3, m2));
    f2 = fabs(Ar<T>::sub(m1, m0));
    if constexpr (KIND == HERMITE_MAKIMA) {
        f1 = Ar<T>::add(f1, Ar<T>::mul((T)0.5, fabs(Ar<T>::add(m3, m2))));
        f2 = Ar<T>::add(f2, Ar<T>::mul((T)0.5, fabs(Ar<T>::add(m1, m0))));
    }
}

// slope at knot k from the window; thr = 1e-9 M (Akima), dydx (GIVEN)
template <class T, int V, int KIND>
__device__ __forceinline__ Vec<T, V> knot_slope(const Seg<T, V> (&win)[4], long long k, long long n, T thr,
                                                const T* __restrict__ dydx, long long w, long long c0) {
    Vec<T, V> d;
    if constexpr (KIND == HERMITE_GIVEN) {
        d = ld_table<T, V>(dydx + k * w + c0);
    } else if (n == 2) {
        d = k == 0 ? win[2].m : win[1].m;
    } else if constexpr (KIND == HERMITE_PCHIP) {
        if (k == 0 || k == n - 1) {
            const bool left = k == 0;
            const T h0 = left ? win[2].h : win[1].h, h1 = left ? win[3].h : win[0].h;
            const T rs = Hoisted<T>::rcp(Ar<T>::add(h0, h1));
#pragma unroll
            for (int e = 0; e < V; ++e)
                d.v[e] = left ? pchip_edge<T>(h0, h1, win[2].m.v[e], win[3].m.v[e], rs)
                              : pchip_edge<T>(h0, h1, win[1].m.v[e], win[0].m.v[e], rs);
        } else {
            const T hl = win[1].h, hr = win[2].h;
            const T w1 = Ar<T>::add(Ar<T>::mul((T)2, hr), hl), w2 = Ar<T>::add(hr, Ar<T>::mul((T)2, hl));
            const T s = Ar<T>::add(w1, w2), rs = Hoisted<T>::rcp(s);
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const T ml = win[1].m.v[e], mr = win[2].m.v[e];
                if (sgn(ml) != sgn(mr) || mr == (T)0 || ml == (T)0) { d.v[e] = (T)0; continue; }
                const T whmean = Hoisted<T>::div(Ar<T>::add(Ar<T>::div(w1, ml), Ar<T>::div(w2, mr)), s, rs);
                d.v[e] = Ar<T>::div((T)1, whmean);
            }
        }
    } else {
#pragma unroll
        for (int e = 0; e < V; ++e) {
            const T m0 = win[0].m.v[e], m1 = win[1].m.v[e], m2 = win[2].m.v[e], m3 = win[3].m.v[e];
            T f1, f2;
            akima_weights<T, KIND>(m0, m1, m2, m3, f1, f2);
            const T f12 = Ar<T>::add(f1, f2);
            d.v[e] = f12 > thr ? Ar<T>::add(m1, Ar<T>::mul(Ar<T>::div(f2, f12), Ar<T>::sub(m2, m1)))
                               : Ar<T>::mul((T)0.5, Ar<T>::add(m3, m0));
        }
    }
    return d;
}

template <class T> struct Bits;
template <> struct Bits<float> {
    static __device__ __forceinline__ unsigned long long of(float v) { return __float_as_uint(v); }
    static __device__ __forceinline__ float val(unsigned long long b) { return __uint_as_float((unsigned)b); }
};
template <> struct Bits<double> {
    static __device__ __forceinline__ unsigned long long of(double v) { return (unsigned long long)__double_as_longlong(v); }
    static __device__ __forceinline__ double val(unsigned long long b) { return __longlong_as_double((long long)b); }
};

// Akima pass 1: mx[0] = bits of max f12 over the table, mx[1] = 1 if some f12 is NaN (both zeroed before the launch)
template <class T, int V, int KIND>
__global__ void __launch_bounds__(256) hermite_f12_max_kernel(const T* __restrict__ x, long long n, const T* __restrict__ y,
                                                              long long w, long long R, long long groups, long long total,
                                                              unsigned long long* __restrict__ mx) {
    unsigned long long best = 0;
    int nan = 0;
    const long long step = (long long)gridDim.x * blockDim.x;
    for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += step) {
        const long long g = o % groups, r = o / groups, c0 = g * V;
        const long long k0 = r * R, k1 = min(k0 + R, n - 1), kend = k1 == n - 1 ? n : k1;   // the last run takes knot n-1
        Seg<T, V> win[4];
        window_init<T, V, KIND>(x, n, y, w, k0, c0, win);
        for (long long k = k0; k < kend; ++k) {
#pragma unroll
            for (int e = 0; e < V; ++e) {
                T f1, f2;
                akima_weights<T, KIND>(win[0].m.v[e], win[1].m.v[e], win[2].m.v[e], win[3].m.v[e], f1, f2);
                const T f12 = Ar<T>::add(f1, f2);
                if (f12 != f12) nan = 1;
                else best = max(best, Bits<T>::of(f12));
            }
            if (k + 1 < kend) window_shift<T, V, KIND>(x, n, y, w, k, c0, win);
        }
    }
    for (int off = 16; off; off >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, off));
    __shared__ unsigned long long warp_best[8];
    if ((threadIdx.x & 31) == 0) warp_best[threadIdx.x >> 5] = best;
    nan = __syncthreads_or(nan);
    if (threadIdx.x == 0) {
        for (int i = 1; i < (int)(blockDim.x >> 5); ++i) best = max(best, warp_best[i]);
        if (best) atomicMax(mx, best);
        if (nan) atomicOr(mx + 1, 1ull);
    }
}

// pass 2 (the only pass of PCHIP and GIVEN): the knot slopes of a run, and a, b of its intervals
template <class T, int V, int KIND>
__global__ void __launch_bounds__(256) hermite_coeffs_kernel(const T* __restrict__ x, long long n, const T* __restrict__ y,
                                                             long long w, const T* __restrict__ dydx, long long R,
                                                             long long groups, long long total,
                                                             const unsigned long long* __restrict__ mx, T* __restrict__ a,
                                                             T* __restrict__ b) {
    T thr = (T)0;
    if constexpr (KIND == HERMITE_AKIMA || KIND == HERMITE_MAKIMA)
        thr = Ar<T>::mul((T)1e-9, mx[1] ? (T)NAN : Bits<T>::val(mx[0]));
    const long long step = (long long)gridDim.x * blockDim.x;
    for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += step) {
        const long long g = o % groups, r = o / groups, c0 = g * V;
        const long long k0 = r * R, k1 = min(k0 + R, n - 1);
        Seg<T, V> win[4];
        window_init<T, V, KIND>(x, n, y, w, k0, c0, win);
        Vec<T, V> dl = knot_slope<T, V, KIND>(win, k0, n, thr, dydx, w, c0);
        for (long long k = k0; k < k1; ++k) {
            window_shift<T, V, KIND>(x, n, y, w, k, c0, win);
            const Vec<T, V> dr = knot_slope<T, V, KIND>(win, k + 1, n, thr, dydx, w, c0);
            // interval k is segment k + 1 - 1 of the shifted window: win[1]
            const T h = win[1].h;
            Vec<T, V> va, vb;
#pragma unroll
            for (int e = 0; e < V; ++e) {
                va.v[e] = Ar<T>::sub(Ar<T>::mul(dl.v[e], h), win[1].dy.v[e]);
                vb.v[e] = Ar<T>::sub(win[1].dy.v[e], Ar<T>::mul(dr.v[e], h));
            }
            st_stream<T, V>(a + k * w + c0, va);
            st_stream<T, V>(b + k * w + c0, vb);
            dl = dr;
        }
    }
}

template <class T, int V, int KIND>
static cudaError_t launch_kind(const T* x, int64_t n, const T* y, int64_t w, const T* dydx, long long R,
                               unsigned long long* mx, T* a, T* b, cudaStream_t st) {
    const long long groups = w / V, runs = (n - 1 + R - 1) / R, total = groups * runs;
    const long long want = (total + 255) / 256, cap = (long long)device_info().sm_count * 64;
    const unsigned grid = (unsigned)(want < cap ? (want ? want : 1) : cap);
    if constexpr (KIND == HERMITE_AKIMA || KIND == HERMITE_MAKIMA) {
        cudaError_t e = cudaMemsetAsync(mx, 0, 2 * sizeof(unsigned long long), st);
        if (e != cudaSuccess) return e;
        hermite_f12_max_kernel<T, V, KIND><<<grid, 256, 0, st>>>(x, (long long)n, y, (long long)w, R, groups, total, mx);
        count_launch();
    }
    hermite_coeffs_kernel<T, V, KIND><<<grid, 256, 0, st>>>(x, (long long)n, y, (long long)w, dydx, R, groups, total, mx, a, b);
    count_launch();
    return cudaGetLastError();
}

template <class T, int V>
static cudaError_t launch_vec(int kind, const T* x, int64_t n, const T* y, int64_t w, const T* dydx, long long R,
                              unsigned long long* mx, T* a, T* b, cudaStream_t st) {
    switch (kind) {
    case HERMITE_PCHIP: return launch_kind<T, V, HERMITE_PCHIP>(x, n, y, w, dydx, R, mx, a, b, st);
    case HERMITE_AKIMA: return launch_kind<T, V, HERMITE_AKIMA>(x, n, y, w, dydx, R, mx, a, b, st);
    case HERMITE_MAKIMA: return launch_kind<T, V, HERMITE_MAKIMA>(x, n, y, w, dydx, R, mx, a, b, st);
    case HERMITE_GIVEN: return launch_kind<T, V, HERMITE_GIVEN>(x, n, y, w, dydx, R, mx, a, b, st);
    default: return cudaErrorInvalidValue;
    }
}

template <class T>
cudaError_t launch_hermite_build(int kind, const T* x, int64_t n, const T* data, int64_t w, const T* dydx,
                                 unsigned long long* mx, T* a, T* b, cudaStream_t st) {
    constexpr int VW = 16 / sizeof(T);
    auto aligned = [](const void* p) { return ((uintptr_t)p & 15) == 0; };
    const bool vec = w % VW == 0 && aligned(data) && aligned(a) && aligned(b) && (!dydx || aligned(dydx));
    // runs long enough to leave about 1024 threads per SM, at most kHermiteMaxRun intervals; rows narrower than a vector
    // take short runs so that a warp's loads stay within a few cache lines
    const long long groups = vec ? w / VW : w, sms = device_info().sm_count;
    long long R = ((n - 1) * groups + sms * 1024 - 1) / (sms * 1024);
    R = R < 1 ? 1 : (R > kHermiteMaxRun ? kHermiteMaxRun : R);
    if ((size_t)w * sizeof(T) < 16 && R > kHermiteThinRun) R = kHermiteThinRun;
    return vec ? launch_vec<T, VW>(kind, x, n, data, w, dydx, R, mx, a, b, st)
               : launch_vec<T, 1>(kind, x, n, data, w, dydx, R, mx, a, b, st);
}

template cudaError_t launch_hermite_build<float>(int, const float*, int64_t, const float*, int64_t, const float*,
                                                 unsigned long long*, float*, float*, cudaStream_t);
template cudaError_t launch_hermite_build<double>(int, const double*, int64_t, const double*, int64_t, const double*,
                                                  unsigned long long*, double*, double*, cudaStream_t);

}  // namespace ndi
