// ndi_integral.cu -- K9b: the cumulative table C of a 1-D interpolant (NOT in the reference; the integral calls of
// include/ndi_b200.h evaluate over it, K9c / K9l in ndi_eval.cu).
//
// C[0] = 0, C[i] = the integral from x[0] to x[i], accumulated in double (for f32 tables too: the error of the sum then
// does not grow with n) and rounded once when stored.  The summation order is fixed so that it is parallel and the
// same on every run: blocks of 32 intervals, a running sum inside each block, a sequential sum over the block totals.
//     pass 1  one thread per (block, column): the block's total                         -> scratch[k][c]
//     pass 2  one thread per column: the totals become offsets (exclusive, in order)    -> scratch[k][c]
//     pass 3  one thread per (block, column): C[32k + j] = off(k) + local(k, j), local formed again from the table
// Pass 2 is a chain of n / 32 additions per column (2048 for n = 65536); its loads are issued ahead of the chain.
#include "ndi_device.cuh"
#include "ndi_internal.h"

namespace ndi {

constexpr int kIntBlock = 32;                 // intervals per block of the summation order

// e[i] = h ((y[i] + y[i+1]) * 0.5 + (a[i] + b[i]) / 12), Linear without the second term; in double
template <class T>
__device__ __forceinline__ double interval_integral(const T* x, const T* data, const T* a, const T* b, long long w,
                                                    long long i, long long c) {
    const double h = (double)Ar<T>::sub(x[i + 1], x[i]);
    double s = Ar<double>::mul(Ar<double>::add((double)data[i * w + c], (double)data[(i + 1) * w + c]), 0.5);
    if (a) s = Ar<double>::add(s, Ar<double>::div(Ar<double>::add((double)a[i * w + c], (double)b[i * w + c]), 12.0));
    return Ar<double>::mul(h, s);
}

template <class T>
__global__ void __launch_bounds__(256) integral_block_totals_kernel(const T* __restrict__ x, long long n, const T* __restrict__ data,
                                                                    const T* __restrict__ a, const T* __restrict__ b, long long w,
                                                                    long long nblk, double* __restrict__ tot) {
    const long long total = nblk * w, step = (long long)gridDim.x * blockDim.x;
    for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += step) {
        const long long k = o / w, c = o - k * w;
        const long long i1 = min((k + 1) * kIntBlock, n - 1);
        double s = 0.0;
#pragma unroll 8
        for (long long i = k * kIntBlock; i < i1; ++i) s = Ar<double>::add(s, interval_integral<T>(x, data, a, b, w, i, c));
        tot[o] = s;
    }
}

__global__ void __launch_bounds__(256) integral_offsets_kernel(double* __restrict__ tot, long long nblk, long long w) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= w) return;
    double off = 0.0;
    long long k = 0;
    constexpr int kAhead = 8;
    for (; k + kAhead <= nblk; k += kAhead) {
        double t[kAhead];
#pragma unroll
        for (int u = 0; u < kAhead; ++u) t[u] = tot[(k + u) * w + c];
#pragma unroll
        for (int u = 0; u < kAhead; ++u) { tot[(k + u) * w + c] = off; off = Ar<double>::add(off, t[u]); }
    }
    for (; k < nblk; ++k) { const double t = tot[k * w + c]; tot[k * w + c] = off; off = Ar<double>::add(off, t); }
}

template <class T>
__global__ void __launch_bounds__(256) integral_fill_kernel(const T* __restrict__ x, long long n, const T* __restrict__ data,
                                                            const T* __restrict__ a, const T* __restrict__ b, long long w,
                                                            long long nblk, const double* __restrict__ off, T* __restrict__ cum) {
    const long long total = nblk * w, step = (long long)gridDim.x * blockDim.x;
    for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += step) {
        const long long k = o / w, c = o - k * w;
        const double base = off[o];
        const long long i1 = min((k + 1) * kIntBlock, n - 1);
        double s = 0.0;
        long long i = k * kIntBlock;
#pragma unroll 8
        for (; i < i1; ++i) {
            cum[i * w + c] = (T)Ar<double>::add(base, s);
            s = Ar<double>::add(s, interval_integral<T>(x, data, a, b, w, i, c));
        }
        if (i == n - 1) cum[i * w + c] = (T)Ar<double>::add(base, s);    // the last row closes the last block
    }
}

// blocks of C: C[n-1] belongs to block (n-1) / 32, which is empty when 32 divides n - 1
static long long offset_blocks(int64_t n) { return (n - 1) / kIntBlock + 1; }

size_t integral_build_scratch(int64_t n, int64_t w) { return (size_t)offset_blocks(n) * (size_t)w; }

template <class T>
cudaError_t launch_integral_build(const T* x, int64_t n, const T* data, const T* a, const T* b, int64_t w, T* cum,
                                  double* scratch, cudaStream_t st) {
    const long long nblk = offset_blocks(n);
    const long long total = nblk * w;
    const long long want = (total + 255) / 256, cap = (long long)device_info().sm_count * 16;
    const unsigned grid = (unsigned)(want < cap ? (want ? want : 1) : cap);
    integral_block_totals_kernel<T><<<grid, 256, 0, st>>>(x, (long long)n, data, a, b, (long long)w, nblk, scratch);
    count_launch();
    integral_offsets_kernel<<<(unsigned)((w + 255) / 256), 256, 0, st>>>(scratch, nblk, (long long)w);
    count_launch();
    integral_fill_kernel<T><<<grid, 256, 0, st>>>(x, (long long)n, data, a, b, (long long)w, nblk, scratch, cum);
    count_launch();
    return cudaGetLastError();
}

template cudaError_t launch_integral_build<float>(const float*, int64_t, const float*, const float*, const float*, int64_t,
                                                  float*, double*, cudaStream_t);
template cudaError_t launch_integral_build<double>(const double*, int64_t, const double*, const double*, const double*,
                                                   int64_t, double*, double*, cudaStream_t);

}  // namespace ndi
