// ndi_eval.cu -- K2 lower_index, K3 interp1d_linear, K4 interp2d_bilinear, K5 interp1d_cubic,
// with K7 (first-error reduction) fused in, plus the query validation pre-pass.
//
// One launch replaces the reference's per-query loop (interp1d/mod.rs:300-343,
// interp2d/mod.rs:255-307).  All three evaluation kernels share one work decomposition:
//
//   * a TILE is 32 consecutive queries.  Each lane of a warp loads one query of the tile
//     (coalesced), does the bounds check and the lower-index search for it, and keeps the
//     per-query scalars (interval index, x - x1, x2 - x1, t ...) in registers.
//   * the per-query scalars are then handed round the warp with shuffles and the trailing axis
//     is processed by LPQ lanes per query with V-element (16-byte when possible) vector loads
//     and stores, so that a warp's stores cover whole contiguous output rows:
//       - thin rows (w <= 32*V):  LPQ = pow2ceil(w / V) lanes per query, 32/LPQ queries per
//         round, LPQ rounds per tile -- one thread per query when w == 1.  A warp takes TPW
//         tiles per iteration and searches them in lock step (search_multi), so the
//         dependent-probe latency of the bisection is paid once per TPW*32 queries; the row
//         gathers of a few rounds are issued together before any of them is consumed.
//       - wide rows (w > 32*V):   LPQ = 32, the row is cut into SLICES of 32*V columns and a
//         (tile, slice) pair is one warp task; consecutive warps take consecutive slices of the
//         same tile, so a block writes whole rows.  Within a task the table rows stay in
//         registers while consecutive queries fall into the same interval (sorted batches).
//   * a persistent grid (SM count x resident blocks) strides over the tasks.
//
// HBM traffic per query is the compulsory s*c (query) + s*w (output); table rows come out of
// L1/L2 unless the table exceeds L2.  Output uses streaming stores so it does not evict the table.
#include <initializer_list>

#include "ndi_device.cuh"
#include "ndi_internal.h"

namespace ndi {

constexpr int kBlock = 256;          // 8 warps
constexpr int kWarpsPerBlock = kBlock / 32;

template <class T>
struct Eval1 {                       // 1-D kernels
    const T* grid; int n; SearchCfg sc;
    const T* data; const T* a; const T* b; long long w;
    const T* q; long long nq; int mode;
    T* out; unsigned long long* err;
    long long ntasks; int nslices;
    int fast_tables;                 // every table value is 0 or in [2^-56, 2^30]: hoisted-reciprocal division allowed
};
template <class T>
struct Eval2 {                       // bilinear
    const T* gx; int n; SearchCfg scx;
    const T* gy; int m; SearchCfg scy;
    const T* data; long long w;
    const T* qx; const T* qy; long long nq; int extrapolate;
    T* out; unsigned long long* err;
    long long ntasks; int nslices;
    const unsigned* perm;            // binned batch (ndi_bin.cu): output row of query i is perm[i]
    int fast_tables;
    unsigned long long* next_task;   // binned batch: tiles are handed out in order through this counter (zeroed by the binning pass)
};

// first-error report for a binned batch: lanes are not in query order, every failing lane reports
__device__ __forceinline__ void report_bad_unordered(unsigned long long* err, bool bad, unsigned long long word) {
    if (bad && err != nullptr) atomicMin(err, word);
}

__device__ __forceinline__ bool shfl_b(bool v, int src) { return __shfl_sync(0xffffffffu, (int)v, src) != 0; }
template <class T> __device__ __forceinline__ T shfl_t(T v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// thin rows: tiles searched in lock step by one warp (TPW), tunable at build time for measurement.
// Measured on B200 (profiles/r01): with the bucket-table search the chains are short, and one tile
// per warp with one round of gathers in flight wins on every thin workload because the registers
// saved buy occupancy (C3 0.37 vs 0.41 ms at 2 tiles / 4 rounds batched, C5a 3.7 vs 5.2 ms).
#ifndef NDI_TPW_LINEAR
#define NDI_TPW_LINEAR 1
#endif
#ifndef NDI_TPW_CUBIC
#define NDI_TPW_CUBIC 1
#endif
#ifndef NDI_TPW_BILINEAR
#define NDI_TPW_BILINEAR 1
#endif
constexpr int kTilesLinear = NDI_TPW_LINEAR, kTilesCubic = NDI_TPW_CUBIC, kTilesBilinear = NDI_TPW_BILINEAR;

// Handing a query's scalars to the lanes that work on its row.  Every warp shuffle is a wavefront on the L1TEX
// data pipe, the unit that binds the thin-row kernels (profiles/r01/l1_wavefronts.md: a sixth of C3's wavefronts,
// nine shuffles per round in the bilinear kernel).  With NDI_BCAST_SMEM each lane writes its query's record to a
// per-warp slab of shared memory once per tile and every round reads the records of its queries with ONE 16-byte
// (f32) load per 16 bytes of record -- lanes of one query read the same address (broadcast), the queries of a round
// lie next to each other -- so a round costs 1 (linear) / 3 (bilinear) wavefronts instead of 4 / 9.  Used when a
// query has at least four lanes (with two or fewer the records of a round span as many wavefronts as the shuffles).
#ifndef NDI_BCAST_SMEM
#define NDI_BCAST_SMEM 1
#endif
template <class T> struct alignas(16) LinRec { T dq; Slope<T> sl; int is; };                 // f32: 16 bytes
template <class T> struct alignas(16) BilRec { long long cs; T bx, by; Slope<T> sx, sy; unsigned orow; };   // f32: 48 bytes

// ------------------------------------------------------------------------------------------------
// K3: Linear::interp_into x batch (linear.rs:73-98)
// ------------------------------------------------------------------------------------------------
#ifndef NDI_THIN_MINBLOCKS
#define NDI_THIN_MINBLOCKS 0          // 0: leave the register budget to ptxas
#endif
// (Measured and dropped: issuing the NEXT tile's bucket-table probe before this tile's gathers -- C3 0.3110 ->
// 0.3090 ms, C3d 0.634 -> 0.627: these kernels are bound by L1TEX / L2 throughput, not by the length of the
// dependent chain; profiles/r01/gather_ceiling.md.)
template <class T, int V, int LPQ>
__global__ void __launch_bounds__(kBlock, (sizeof(T) == 4 && LPQ < 32) ? NDI_THIN_MINBLOCKS : 0) interp1d_linear_kernel(const Eval1<T> p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    constexpr bool kBcast = NDI_BCAST_SMEM && LPQ >= 4 && LPQ < 32 && kTilesLinear == 1;
    __shared__ LinRec<T> recs[kBcast ? kWarpsPerBlock : 1][kBcast ? 32 : 1];
    const GridView<T> g = make_grid_view<T>(p.grid, p.n, p.sc, smem_raw, &bar);
    const T g0 = g.g0, gl = g.gl;
    const int lane = threadIdx.x & 31;
    const long long nwarps = (long long)gridDim.x * kWarpsPerBlock;
    const long long task0 = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    // thin rows: the query of the NEXT tile is loaded while this one is processed, so a tile does not start
    // with a DRAM round trip (with ~40 resident warps per SM the kernel is bound by per-tile latency)
    T x_ahead = g0;
    if (LPQ < 32 && kTilesLinear == 1 && task0 < p.ntasks && task0 * 32 + lane < p.nq) x_ahead = ld_query(p.q + task0 * 32 + lane);
    for (long long task = task0; task < p.ntasks; task += nwarps) {
        if constexpr (LPQ < 32) {
            constexpr int TPW = kTilesLinear, QPR = 32 / LPQ;
            const long long qbase0 = task * (32 * TPW);
            T x[TPW]; int idx[TPW]; T dx21[TPW], dxq[TPW]; bool skip[TPW]; Slope<T> slope[TPW];   // dx21/dxq: x1, x2 from the search
            if constexpr (TPW == 1) {
                x[0] = x_ahead;
                const long long qn = (task + nwarps) * 32 + lane;
                x_ahead = (task + nwarps < p.ntasks && qn < p.nq) ? ld_query(p.q + qn) : g0;
            } else {
#pragma unroll
                for (int t = 0; t < TPW; ++t) {
                    const long long qi = qbase0 + t * 32 + lane;
                    x[t] = qi < p.nq ? ld_query(p.q + qi) : g0;
                }
            }
            search_multi<T, TPW>(g, x, idx, dx21, dxq);                               // linear.rs:87, :90-91 (x1, x2)
#pragma unroll
            for (int t = 0; t < TPW; ++t) {
                const long long qi = qbase0 + t * 32 + lane;
                const bool live = qi < p.nq;
                // linear.rs:80-84: out of range (or NaN) without extrapolation is an error;
                // with extrapolation only NaN fails (vector_extensions.rs:83-84)
                const bool bad = live && (p.mode ? Ar<T>::is_nan(x[t]) : !in_range(g0, gl, x[t]));
                const T x1 = dx21[t], x2 = dxq[t];
                dxq[t] = Ar<T>::sub(x[t], x1);
                slope[t] = Slope<T>::make(Ar<T>::sub(x2, x1), dxq[t], p.fast_tables != 0);
                if (qbase0 + t * 32 < p.nq) report_first_bad(p.err, bad, (unsigned long long)qi);
                skip[t] = bad || !live;
            }
            const int sub = lane % LPQ, qsel = lane / LPQ;
            const long long col = (long long)sub * V;
            const bool colok = col < p.w;
#pragma unroll
            for (int t = 0; t < TPW; ++t) {
                const long long qbase = qbase0 + t * 32;
                if (qbase >= p.nq) break;
                // A tile whose queries all fall into one interval (dense sorted batches) gathers its two
                // table rows once instead of once per round.
                const int idx0 = __shfl_sync(0xffffffffu, idx[t], __ffs(__ballot_sync(0xffffffffu, !skip[t]) | 0x80000000u) - 1);
                const bool one_interval = LPQ > 1 && __all_sync(0xffffffffu, skip[t] || idx[t] == idx0);
                Vec<T, V> y1, y2;
                if (one_interval && colok) {
                    const T* row = p.data + (long long)idx0 * p.w + col;
                    y1 = ld_table<T, V>(row);
                    y2 = ld_table<T, V>(row + p.w);
                }
                if constexpr (kBcast) {
                    recs[threadIdx.x >> 5][lane] = LinRec<T>{dxq[t], slope[t], skip[t] ? -1 : idx[t]};
                    __syncwarp();
                }
#pragma unroll
                for (int r = 0; r < LPQ; ++r) {
                    const int src = r * QPR + qsel;
                    int is; bool live_s; T dq; Slope<T> sl;
                    if constexpr (kBcast) {
                        const LinRec<T> rc = recs[threadIdx.x >> 5][src];
                        is = rc.is; live_s = is >= 0; dq = rc.dq; sl = rc.sl;
                    } else {
#if NDI_PACK_SHFL >= 1
                        is = __shfl_sync(0xffffffffu, skip[t] ? -1 : idx[t], src);
                        live_s = is >= 0;
#else
                        is = __shfl_sync(0xffffffffu, idx[t], src);
                        live_s = !shfl_b(skip[t], src);
#endif
                        dq = shfl_t(dxq[t], src);
                        sl = slope[t].from_lane(src, dq, p.fast_tables != 0);
                    }
                    if (live_s && colok) {
                        if (!one_interval) {
                            const T* row = p.data + (long long)is * p.w + col;
                            y1 = ld_table<T, V>(row);
                            y2 = ld_table<T, V>(row + p.w);
                        }
                        st_stream<T, V>(p.out + (qbase + src) * p.w + col, lerp_vec<T, V>(y1, y2, sl, dq));   // linear.rs:94-96
                    }
                }
                if constexpr (kBcast) __syncwarp();                    // the slab is rewritten by the next tile
            }
        } else {
            const long long tile = task / p.nslices;
            const int slice = (int)(task - tile * p.nslices);
            const long long qbase = tile * 32;
            const long long qi = qbase + lane;
            const bool live = qi < p.nq;
            T x[1] = {live ? ld_query(p.q + qi) : g0};
            int idx[1]; T xl[1], xr[1];
            search_multi<T, 1>(g, x, idx, xl, xr);
            const bool bad = live && (p.mode ? Ar<T>::is_nan(x[0]) : !in_range(g0, gl, x[0]));
            const T x1 = xl[0], x2 = xr[0];
            const T dxq = Ar<T>::sub(x[0], x1);
            const Slope<T> slope = Slope<T>::make(Ar<T>::sub(x2, x1), dxq, p.fast_tables != 0);
            if (slice == 0) report_first_bad(p.err, bad, (unsigned long long)qi);
            const bool skip = bad || !live;
            const long long col = ((long long)slice * 32 + lane) * V;
            const bool colok = col < p.w;
            int cur = -1;
            Vec<T, V> y1, y2;
            const int nlive = (int)min((long long)32, p.nq - qbase);
            for (int s = 0; s < nlive; ++s) {
                const int is = __shfl_sync(0xffffffffu, idx[0], s);
                const Slope<T> sl = slope.from_lane(s);
                const T dq = shfl_t(dxq, s);
                const bool sk = shfl_b(skip, s);
                if (sk || !colok) continue;
                if (is != cur) {
                    const T* row = p.data + (long long)is * p.w + col;
                    y1 = ld_table<T, V>(row);
                    y2 = ld_table<T, V>(row + p.w);
                    cur = is;
                }
                const Vec<T, V> res = lerp_vec<T, V>(y1, y2, sl, dq);
                st_stream<T, V>(p.out + (qbase + s) * p.w + col, res);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K3 on a PAIR TABLE (rows of 16 - 64 bytes: an interval's two rows fit one cache line)
// ------------------------------------------------------------------------------------------------
// Linear::interp_into gathers rows i and i+1.  For rows of 16 - 64 bytes the two row gathers are two L1TEX
// wavefronts per query (one per row: the lanes of a load instruction touch one row each), and on C3 those 64
// wavefronts per 32-query tile are half of what binds the kernel (profiles/r01/l1_wavefronts.md).  A handle
// with such rows therefore also keeps P, the table with every interval's two rows interleaved in granules of
// two columns:
//     P[i] = { y[i][0], y[i][1], y[i+1][0], y[i+1][1],  y[i][2], y[i][3], y[i+1][2], y[i+1][3], ... }   (2 w elements)
// A query's whole gather is then ONE aligned segment of 2 w elements (at most 128 bytes: one wavefront), and a
// lane's 32-byte load holds exactly the y1 / y2 values of the columns it produces -- already paired up for the
// two-column arithmetic of lerp_vec.  Twice the table memory, so only built while P stays L2-resident
// (ndi_api.cu: want_pair_table).  Same arithmetic, same bits.
template <class T> struct alignas(32) Pair32 { T v[32 / sizeof(T)]; };
template <class T>
__device__ __forceinline__ Pair32<T> ld_pair(const T* p) {          // one 256-bit load (LDG.E.256), read-only path
    unsigned long long a, b, c, d;
    asm("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
    unsigned long long t[4] = {a, b, c, d};
    return *reinterpret_cast<const Pair32<T>*>(t);
}
template <class T, int V>
__device__ __forceinline__ void unpair(const Pair32<T>& pr, Vec<T, V>& y1, Vec<T, V>& y2) {
#pragma unroll
    for (int e = 0; e < V; e += 2) {
        y1.v[e] = pr.v[2 * e]; y1.v[e + 1] = pr.v[2 * e + 1];
        y2.v[e] = pr.v[2 * e + 2]; y2.v[e + 1] = pr.v[2 * e + 3];
    }
}

template <class T, int LPQ>
__global__ void __launch_bounds__(kBlock) interp1d_linear_pair_kernel(const Eval1<T> p) {
    constexpr int V = 16 / (int)sizeof(T), QPR = 32 / LPQ;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    constexpr bool kBcast = NDI_BCAST_SMEM && LPQ >= 4;
    __shared__ LinRec<T> recs[kBcast ? kWarpsPerBlock : 1][kBcast ? 32 : 1];
    const GridView<T> g = make_grid_view<T>(p.grid, p.n, p.sc, smem_raw, &bar);
    const T g0 = g.g0, gl = g.gl;
    const int lane = threadIdx.x & 31;
    const long long nwarps = (long long)gridDim.x * kWarpsPerBlock;
    const long long task0 = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const long long pw = 2 * p.w;                                  // elements per row of P (p.data is P here)
    T x_ahead = g0;
    if (task0 < p.ntasks && task0 * 32 + lane < p.nq) x_ahead = ld_query(p.q + task0 * 32 + lane);
    const int sub = lane % LPQ, qsel = lane / LPQ;
    const long long col = (long long)sub * V;
    for (long long task = task0; task < p.ntasks; task += nwarps) {
        const long long qbase = task * 32, qi = qbase + lane;
        T x[1] = {x_ahead};
        const long long qn = (task + nwarps) * 32 + lane;
        x_ahead = (task + nwarps < p.ntasks && qn < p.nq) ? ld_query(p.q + qn) : g0;
        int idx[1]; T x1s[1], x2s[1];
        search_multi<T, 1>(g, x, idx, x1s, x2s);                                       // linear.rs:87, :90-91
        const bool live = qi < p.nq;
        const bool bad = live && (p.mode ? Ar<T>::is_nan(x[0]) : !in_range(g0, gl, x[0]));   // linear.rs:80-84
        const T dxq = Ar<T>::sub(x[0], x1s[0]);
        const Slope<T> slope = Slope<T>::make(Ar<T>::sub(x2s[0], x1s[0]), dxq, p.fast_tables != 0);
        report_first_bad(p.err, bad, (unsigned long long)qi);
        const bool skip = bad || !live;
        const int idx0 = __shfl_sync(0xffffffffu, idx[0], __ffs(__ballot_sync(0xffffffffu, !skip) | 0x80000000u) - 1);
        const bool one_interval = __all_sync(0xffffffffu, skip || idx[0] == idx0);
        Vec<T, V> y1, y2;
        if (one_interval) unpair<T, V>(ld_pair<T>(p.data + (long long)idx0 * pw + 2 * col), y1, y2);
        if constexpr (kBcast) {
            recs[threadIdx.x >> 5][lane] = LinRec<T>{dxq, slope, skip ? -1 : idx[0]};
            __syncwarp();
        }
#pragma unroll
        for (int r = 0; r < LPQ; ++r) {
            const int src = r * QPR + qsel;
            int is; T dq; Slope<T> sl;
            if constexpr (kBcast) {
                const LinRec<T> rc = recs[threadIdx.x >> 5][src];
                is = rc.is; dq = rc.dq; sl = rc.sl;
            } else if constexpr (LPQ == 1) {                                   // one lane per query: nothing to hand round
                is = skip ? -1 : idx[0]; dq = dxq; sl = slope;
            } else {
                is = __shfl_sync(0xffffffffu, skip ? -1 : idx[0], src);
                dq = shfl_t(dxq, src);
                sl = slope.from_lane(src, dq, p.fast_tables != 0);
            }
            if (is >= 0) {
                if (!one_interval) unpair<T, V>(ld_pair<T>(p.data + (long long)is * pw + 2 * col), y1, y2);
                st_stream<T, V>(p.out + (qbase + src) * p.w + col, lerp_vec<T, V>(y1, y2, sl, dq));   // linear.rs:94-96
            }
        }
        if constexpr (kBcast) __syncwarp();
    }
}

// P from the dense table (once per handle)
template <class T>
__global__ void __launch_bounds__(256) pack_pairs_kernel(const T* __restrict__ y, long long n, long long w, T* __restrict__ P) {
    const long long total = (n - 1) * 2 * w, step = (long long)gridDim.x * blockDim.x;
    for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += step) {
        const long long i = o / (2 * w), e = o - i * 2 * w;
        const long long granule = e >> 2, within = e & 3;          // {y[i][2g], y[i][2g+1], y[i+1][2g], y[i+1][2g+1]}
        P[o] = y[(i + (within >> 1)) * w + 2 * granule + (within & 1)];
    }
}
template <class T>
cudaError_t launch_pack_pairs(const T* y, int64_t n, int64_t w, T* P, cudaStream_t st) {
    const long long total = (n - 1) * 2 * w;
    const long long want = (total + 255) / 256, cap = (long long)device_info().sm_count * 16;
    pack_pairs_kernel<T><<<(unsigned)(want < cap ? (want ? want : 1) : cap), 256, 0, st>>>(y, (long long)n, (long long)w, P);
    count_launch();
    return cudaGetLastError();
}
bool pair_table_shape_ok(int64_t w, size_t elem) {
    const int64_t v = 16 / (int64_t)elem;                             // columns per lane
    const int64_t lanes = w / v;
    return w % v == 0 && (lanes == 1 || lanes == 2 || lanes == 4);    // rows of 16, 32 or 64 bytes: P rows of 32 - 128 bytes
}

// ------------------------------------------------------------------------------------------------
// K5: CubicSplineStrategy::interp_into x batch (cubic_spline.rs:791-830)
// ------------------------------------------------------------------------------------------------
template <class T>
__device__ __forceinline__ T rem_euclid(T a, T b) {            // num_traits::Euclid for floats
    T r = fmod(a, b);
    return r < (T)0 ? Ar<T>::add(r, fabs(b)) : r;
}

template <class T>
__device__ __forceinline__ T cubic_point(T yl, T yr, T al, T bl, T t, T omt, T tt) {
    // (1 - t) * yl + t * yr + t * (1 - t) * (a * (1 - t) + b * t)        cubic_spline.rs:825-827
    const T lin = Ar<T>::add(Ar<T>::mul(omt, yl), Ar<T>::mul(t, yr));
    const T cur = Ar<T>::add(Ar<T>::mul(al, omt), Ar<T>::mul(bl, t));
    return Ar<T>::add(lin, Ar<T>::mul(tt, cur));
}

// the V columns one lane holds of one query; f32: two columns per instruction (ndi_device.cuh, F2)
template <class T, int V>
__device__ __forceinline__ Vec<T, V> cubic_vec(const Vec<T, V>& yl, const Vec<T, V>& yr, const Vec<T, V>& al, const Vec<T, V>& bl,
                                               T t, T omt, T tt) {
    Vec<T, V> res;
    if constexpr (std::is_same<T, float>::value && NDI_F32X2 && V % 2 == 0) {
        const F2 t2 = F2::both(t), o2 = F2::both(omt), tt2 = F2::both(tt);
#pragma unroll
        for (int e = 0; e < V; e += 2) {
            const F2 l{yl.v[e], yl.v[e + 1]}, r{yr.v[e], yr.v[e + 1]}, a{al.v[e], al.v[e + 1]}, b{bl.v[e], bl.v[e + 1]};
            const F2 lin = add_halves(mul2(o2, l), mul2(t2, r));       // sums of products: per half (ndi_device.cuh)
            const F2 cur = add_halves(mul2(a, o2), mul2(b, t2));
            const F2 o = add_halves(lin, mul2(tt2, cur));
            res.v[e] = o.lo; res.v[e + 1] = o.hi;
        }
        return res;
    }
#pragma unroll
    for (int e = 0; e < V; ++e) res.v[e] = cubic_point<T>(yl.v[e], yr.v[e], al.v[e], bl.v[e], t, omt, tt);
    return res;
}

// range check, periodic wrap and NaN test of one query (cubic_spline.rs:797-809); returns `bad`
template <class T>
__device__ __forceinline__ bool cubic_prepare(T& x, T g0, T gl, int mode) {
    const bool inr = in_range(g0, gl, x);                                              // :797
    if (mode == 0) return !inr;                                                        // :798-802
    if (mode == 2 && !inr) x = Ar<T>::add(rem_euclid<T>(Ar<T>::sub(x, g0), Ar<T>::sub(gl, g0)), g0);  // :805-809
    return Ar<T>::is_nan(x);                                                           // NaN reaches get_lower_index
}

template <class T, int V, int LPQ>
__global__ void __launch_bounds__(kBlock, (sizeof(T) == 4 && LPQ < 32) ? NDI_THIN_MINBLOCKS : 0) interp1d_cubic_kernel(const Eval1<T> p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    const GridView<T> g = make_grid_view<T>(p.grid, p.n, p.sc, smem_raw, &bar);
    const T g0 = g.g0, gl = g.gl;
    const T one = (T)1;
    const int lane = threadIdx.x & 31;
    const long long nwarps = (long long)gridDim.x * kWarpsPerBlock;
    const long long task0 = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    T x_ahead = g0;                                           // thin rows: the next tile's query, loaded one tile ahead
    if (LPQ < 32 && kTilesCubic == 1 && task0 < p.ntasks && task0 * 32 + lane < p.nq) x_ahead = ld_query(p.q + task0 * 32 + lane);
    for (long long task = task0; task < p.ntasks; task += nwarps) {
        if constexpr (LPQ < 32) {
            constexpr int TPW = kTilesCubic, QPR = 32 / LPQ;
            const long long qbase0 = task * (32 * TPW);
            T x[TPW]; int idx[TPW]; T tq[TPW], omt[TPW], tt[TPW]; bool skip[TPW], bad[TPW];
            if constexpr (TPW == 1) {
                x[0] = x_ahead;
                const long long qn = (task + nwarps) * 32 + lane;
                x_ahead = (task + nwarps < p.ntasks && qn < p.nq) ? ld_query(p.q + qn) : g0;
                bad[0] = cubic_prepare<T>(x[0], g0, gl, p.mode) && qbase0 + lane < p.nq;
            } else {
#pragma unroll
                for (int t = 0; t < TPW; ++t) {
                    const long long qi = qbase0 + t * 32 + lane;
                    const bool live = qi < p.nq;
                    x[t] = live ? ld_query(p.q + qi) : g0;
                    bad[t] = cubic_prepare<T>(x[t], g0, gl, p.mode) && live;
                }
            }
            search_multi<T, TPW>(g, x, idx, tq, omt);                                 // :811 (+ x_left, x_right)
#pragma unroll
            for (int t = 0; t < TPW; ++t) {
                const long long qi = qbase0 + t * 32 + lane;
                const T xl = tq[t], xr = omt[t];
                tq[t] = Ar<T>::div(Ar<T>::sub(x[t], xl), Ar<T>::sub(xr, xl));          // :818
                omt[t] = Ar<T>::sub(one, tq[t]);
                tt[t] = Ar<T>::mul(tq[t], omt[t]);
                if (qbase0 + t * 32 < p.nq) report_first_bad(p.err, bad[t], (unsigned long long)qi);
                skip[t] = bad[t] || !(qi < p.nq);
            }
            const int sub = lane % LPQ, qsel = lane / LPQ;
            const long long col = (long long)sub * V;
            const bool colok = col < p.w;
#pragma unroll
            for (int t = 0; t < TPW; ++t) {
                const long long qbase = qbase0 + t * 32;
                if (qbase >= p.nq) break;
                // A tile whose queries all fall into one interval (dense sorted batches: C5b has 8192 queries
                // per interval) gathers its four table rows once instead of once per round.
                const int idx0 = __shfl_sync(0xffffffffu, idx[t], __ffs(__ballot_sync(0xffffffffu, !skip[t]) | 0x80000000u) - 1);
                const bool one_interval = LPQ > 1 && __all_sync(0xffffffffu, skip[t] || idx[t] == idx0);
                Vec<T, V> yl, yr, al, bl;
                if (one_interval && colok) {
                    const long long ro = (long long)idx0 * p.w + col;
                    yl = ld_table<T, V>(p.data + ro);
                    yr = ld_table<T, V>(p.data + ro + p.w);
                    al = ld_table<T, V>(p.a + ro);
                    bl = ld_table<T, V>(p.b + ro);
                }
#pragma unroll
                for (int r = 0; r < LPQ; ++r) {
                    const int src = r * QPR + qsel;
#if NDI_PACK_SHFL >= 1
                    const int is = __shfl_sync(0xffffffffu, skip[t] ? -1 : idx[t], src);
                    const bool live_s = is >= 0;
#else
                    const int is = __shfl_sync(0xffffffffu, idx[t], src);
                    const bool live_s = !shfl_b(skip[t], src);
#endif
#if NDI_PACK_CUBIC >= 2
                    const T ts = shfl_t(tq[t], src);
                    const T os = Ar<T>::sub(one, ts), tts = Ar<T>::mul(ts, os);       // the operations of :818-827 again
#else
                    const T ts = shfl_t(tq[t], src), os = shfl_t(omt[t], src), tts = shfl_t(tt[t], src);
#endif
                    if (live_s && colok) {
                        if (!one_interval) {
                            const long long ro = (long long)is * p.w + col;
                            yl = ld_table<T, V>(p.data + ro);
                            yr = ld_table<T, V>(p.data + ro + p.w);
                            al = ld_table<T, V>(p.a + ro);
                            bl = ld_table<T, V>(p.b + ro);
                        }
                        st_stream<T, V>(p.out + (qbase + src) * p.w + col, cubic_vec<T, V>(yl, yr, al, bl, ts, os, tts));
                    }
                }
            }
        } else {
            const long long tile = task / p.nslices;
            const int slice = (int)(task - tile * p.nslices);
            const long long qbase = tile * 32;
            const long long qi = qbase + lane;
            const bool live = qi < p.nq;
            T x[1] = {live ? ld_query(p.q + qi) : g0};
            const bool bad = cubic_prepare<T>(x[0], g0, gl, p.mode) && live;
            int idx[1]; T xls[1], xrs[1];
            search_multi<T, 1>(g, x, idx, xls, xrs);
            const T xl = xls[0], xr = xrs[0];
            const T t = Ar<T>::div(Ar<T>::sub(x[0], xl), Ar<T>::sub(xr, xl));
            const T omt = Ar<T>::sub(one, t);
            const T tt = Ar<T>::mul(t, omt);
            if (slice == 0) report_first_bad(p.err, bad, (unsigned long long)qi);
            const bool skip = bad || !live;
            const long long col = ((long long)slice * 32 + lane) * V;
            const bool colok = col < p.w;
            int cur = -1;
            Vec<T, V> yl, yr, al, bl;
            const int nlive = (int)min((long long)32, p.nq - qbase);
            for (int s = 0; s < nlive; ++s) {
                const int is = __shfl_sync(0xffffffffu, idx[0], s);
                const T ts = shfl_t(t, s), os = shfl_t(omt, s), tts = shfl_t(tt, s);
                const bool sk = shfl_b(skip, s);
                if (sk || !colok) continue;
                if (is != cur) {
                    const long long ro = (long long)is * p.w + col;
                    yl = ld_table<T, V>(p.data + ro);
                    yr = ld_table<T, V>(p.data + ro + p.w);
                    al = ld_table<T, V>(p.a + ro);
                    bl = ld_table<T, V>(p.b + ro);
                    cur = is;
                }
                st_stream<T, V>(p.out + (qbase + s) * p.w + col, cubic_vec<T, V>(yl, yr, al, bl, ts, os, tts));
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K5d: first / second derivative of the cubic spline (NOT in the reference; scipy's CubicSpline(x, nu))
// ------------------------------------------------------------------------------------------------
// The exact derivatives of the value form (1-t) yl + t yr + t (1-t) (a (1-t) + b t) with t = (x - xl) / h, h = xr - xl:
//     cur = a (1-t) + b t,  ba = b - a
//     d1  = (((yr - yl) + ((1-t) - t) cur) + (t (1-t)) ba) / h
//     d2  = ((2 (((1-t) - t) ba - cur)) / h) / h
// every operation rounded on its own.  Query handling (range check, periodic wrap, NaN, lower index, t) is K5's.
// The divisor h is the same for every column of a query: its reciprocal is formed once per query (Hoisted<T>::rcp)
// and every quotient is finished with the hoisted sequence, which falls back to the IEEE division wherever it could
// differ from it -- bit-identical to a true division per element.
__device__ __forceinline__ F2 sub_halves(F2 p, F2 z) { return F2{__fsub_rn(p.lo, z.lo), __fsub_rn(p.hi, z.hi)}; }

template <class T, int ORDER>
__device__ __forceinline__ T cubic_deriv_point(T num, T h, T r) {
    if constexpr (ORDER == 1) return Hoisted<T>::div(num, h, r);
    else return Hoisted<T>::div(Hoisted<T>::div(num, h, r), h, r);
}

template <class T, int V, int ORDER>
__device__ __forceinline__ Vec<T, V> cubic_deriv_vec(const Vec<T, V>& yl, const Vec<T, V>& yr, const Vec<T, V>& al,
                                                     const Vec<T, V>& bl, T t, T omt, T h, T r) {
    const T dmt = Ar<T>::sub(omt, t), tt = Ar<T>::mul(t, omt);
    const T two = (T)2;
    Vec<T, V> res;
    if constexpr (std::is_same<T, float>::value && NDI_F32X2 && V % 2 == 0) {
        const F2 t2 = F2::both(t), o2 = F2::both(omt), d2 = F2::both(dmt), tt2 = F2::both(tt), two2 = F2::both(two);
#pragma unroll
        for (int e = 0; e < V; e += 2) {
            const F2 l{yl.v[e], yl.v[e + 1]}, rr{yr.v[e], yr.v[e + 1]}, a{al.v[e], al.v[e + 1]}, b{bl.v[e], bl.v[e + 1]};
            const F2 cur = add_halves(mul2(a, o2), mul2(b, t2));       // sums and differences of products: per half
            const F2 ba = sub2(b, a);
            F2 num;
            if constexpr (ORDER == 1) num = add_halves(mul2(tt2, ba), add_halves(mul2(d2, cur), sub2(rr, l)));
            else num = mul2(two2, sub_halves(mul2(d2, ba), cur));
            res.v[e] = cubic_deriv_point<T, ORDER>(num.lo, h, r);
            res.v[e + 1] = cubic_deriv_point<T, ORDER>(num.hi, h, r);
        }
        return res;
    }
#pragma unroll
    for (int e = 0; e < V; ++e) {
        const T cur = Ar<T>::add(Ar<T>::mul(al.v[e], omt), Ar<T>::mul(bl.v[e], t));
        const T ba = Ar<T>::sub(bl.v[e], al.v[e]);
        T num;
        if constexpr (ORDER == 1)
            num = Ar<T>::add(Ar<T>::add(Ar<T>::sub(yr.v[e], yl.v[e]), Ar<T>::mul(dmt, cur)), Ar<T>::mul(tt, ba));
        else num = Ar<T>::mul(two, Ar<T>::sub(Ar<T>::mul(dmt, ba), cur));
        res.v[e] = cubic_deriv_point<T, ORDER>(num, h, r);
    }
    return res;
}

// K5's work decomposition (one tile per warp on thin rows, next tile's query loaded ahead, one-interval tiles, wide
// rows in slices with the rows kept in registers while the interval does not change); each lane of a query gets t, h
// and the hoisted reciprocal of h.
template <class T, int V, int LPQ, int ORDER>
__global__ void __launch_bounds__(kBlock) interp1d_cubic_deriv_kernel(const Eval1<T> p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    const GridView<T> g = make_grid_view<T>(p.grid, p.n, p.sc, smem_raw, &bar);
    const T g0 = g.g0, gl = g.gl;
    const T one = (T)1;
    const int lane = threadIdx.x & 31;
    const long long nwarps = (long long)gridDim.x * kWarpsPerBlock;
    const long long task0 = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    T x_ahead = g0;
    if (LPQ < 32 && task0 < p.ntasks && task0 * 32 + lane < p.nq) x_ahead = ld_query(p.q + task0 * 32 + lane);
    for (long long task = task0; task < p.ntasks; task += nwarps) {
        if constexpr (LPQ < 32) {
            constexpr int QPR = 32 / LPQ;
            const long long qbase = task * 32, qi = qbase + lane;
            T x[1] = {x_ahead};
            const long long qn = (task + nwarps) * 32 + lane;
            x_ahead = (task + nwarps < p.ntasks && qn < p.nq) ? ld_query(p.q + qn) : g0;
            const bool bad = cubic_prepare<T>(x[0], g0, gl, p.mode) && qi < p.nq;
            int idx[1]; T xls[1], xrs[1];
            search_multi<T, 1>(g, x, idx, xls, xrs);
            const T h = Ar<T>::sub(xrs[0], xls[0]);
            const T t = Ar<T>::div(Ar<T>::sub(x[0], xls[0]), h);
            const T r = Hoisted<T>::rcp(h);
            report_first_bad(p.err, bad, (unsigned long long)qi);
            const bool skip = bad || !(qi < p.nq);
            const int sub = lane % LPQ, qsel = lane / LPQ;
            const long long col = (long long)sub * V;
            const bool colok = col < p.w;
            const int idx0 = __shfl_sync(0xffffffffu, idx[0], __ffs(__ballot_sync(0xffffffffu, !skip) | 0x80000000u) - 1);
            const bool one_interval = LPQ > 1 && __all_sync(0xffffffffu, skip || idx[0] == idx0);
            Vec<T, V> yl, yr, al, bl;
            if (one_interval && colok) {
                const long long ro = (long long)idx0 * p.w + col;
                yl = ld_table<T, V>(p.data + ro);
                yr = ld_table<T, V>(p.data + ro + p.w);
                al = ld_table<T, V>(p.a + ro);
                bl = ld_table<T, V>(p.b + ro);
            }
#pragma unroll
            for (int rd = 0; rd < LPQ; ++rd) {
                const int src = rd * QPR + qsel;
                const int is = __shfl_sync(0xffffffffu, skip ? -1 : idx[0], src);
                const T ts = shfl_t(t, src), hs = shfl_t(h, src), rs = shfl_t(r, src);
                if (is >= 0 && colok) {
                    if (!one_interval) {
                        const long long ro = (long long)is * p.w + col;
                        yl = ld_table<T, V>(p.data + ro);
                        yr = ld_table<T, V>(p.data + ro + p.w);
                        al = ld_table<T, V>(p.a + ro);
                        bl = ld_table<T, V>(p.b + ro);
                    }
                    st_stream<T, V>(p.out + (qbase + src) * p.w + col,
                                    cubic_deriv_vec<T, V, ORDER>(yl, yr, al, bl, ts, Ar<T>::sub(one, ts), hs, rs));
                }
            }
        } else {
            const long long tile = task / p.nslices;
            const int slice = (int)(task - tile * p.nslices);
            const long long qbase = tile * 32;
            const long long qi = qbase + lane;
            const bool live = qi < p.nq;
            T x[1] = {live ? ld_query(p.q + qi) : g0};
            const bool bad = cubic_prepare<T>(x[0], g0, gl, p.mode) && live;
            int idx[1]; T xls[1], xrs[1];
            search_multi<T, 1>(g, x, idx, xls, xrs);
            const T h = Ar<T>::sub(xrs[0], xls[0]);
            const T t = Ar<T>::div(Ar<T>::sub(x[0], xls[0]), h);
            const T omt = Ar<T>::sub(one, t);
            const T r = Hoisted<T>::rcp(h);
            if (slice == 0) report_first_bad(p.err, bad, (unsigned long long)qi);
            const bool skip = bad || !live;
            const long long col = ((long long)slice * 32 + lane) * V;
            const bool colok = col < p.w;
            int cur = -1;
            Vec<T, V> yl, yr, al, bl;
            const int nlive = (int)min((long long)32, p.nq - qbase);
            for (int s = 0; s < nlive; ++s) {
                const int is = __shfl_sync(0xffffffffu, skip ? -1 : idx[0], s);
                const T ts = shfl_t(t, s), os = shfl_t(omt, s), hs = shfl_t(h, s), rs = shfl_t(r, s);
                if (is < 0 || !colok) continue;
                if (is != cur) {
                    const long long ro = (long long)is * p.w + col;
                    yl = ld_table<T, V>(p.data + ro);
                    yr = ld_table<T, V>(p.data + ro + p.w);
                    al = ld_table<T, V>(p.a + ro);
                    bl = ld_table<T, V>(p.b + ro);
                    cur = is;
                }
                st_stream<T, V>(p.out + (qbase + s) * p.w + col, cubic_deriv_vec<T, V, ORDER>(yl, yr, al, bl, ts, os, hs, rs));
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K3d: slope of Linear (NOT in the reference): m = (y2 - y1) / (x2 - x1), the first term of calc_frac (linear.rs:29-36)
// ------------------------------------------------------------------------------------------------
// K3's query handling and work decomposition; per element one division, nothing of x - x1.  The quotient IS the
// output here, so the sign of a zero numerator must survive (y2 = -0, y1 = +0 gives -0): floats divide through
// Hoisted<T>, which sends zero numerators to the IEEE division; integers wrap and truncate like K3's m.
template <class T>
__device__ __forceinline__ T slope_div(T num, T d, T r) {
    if constexpr (std::is_floating_point<T>::value) return Hoisted<T>::div(num, d, r);
    else return Ar<T>::div(num, d);
}
template <class T>
__device__ __forceinline__ T slope_rcp(T d) {
    if constexpr (std::is_floating_point<T>::value) return Hoisted<T>::rcp(d);
    else return (T)0;
}
template <class T, int V>
__device__ __forceinline__ Vec<T, V> slope_vec(const Vec<T, V>& y1, const Vec<T, V>& y2, T d, T r) {
    Vec<T, V> res;
#pragma unroll
    for (int e = 0; e < V; ++e) res.v[e] = slope_div<T>(Ar<T>::sub(y2.v[e], y1.v[e]), d, r);
    return res;
}

template <class T, int V, int LPQ>
__global__ void __launch_bounds__(kBlock) interp1d_linear_slope_kernel(const Eval1<T> p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    const GridView<T> g = make_grid_view<T>(p.grid, p.n, p.sc, smem_raw, &bar);
    const T g0 = g.g0, gl = g.gl;
    const int lane = threadIdx.x & 31;
    const long long nwarps = (long long)gridDim.x * kWarpsPerBlock;
    const long long task0 = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    T x_ahead = g0;
    if (LPQ < 32 && task0 < p.ntasks && task0 * 32 + lane < p.nq) x_ahead = ld_query(p.q + task0 * 32 + lane);
    for (long long task = task0; task < p.ntasks; task += nwarps) {
        if constexpr (LPQ < 32) {
            constexpr int QPR = 32 / LPQ;
            const long long qbase = task * 32, qi = qbase + lane;
            T x[1] = {x_ahead};
            const long long qn = (task + nwarps) * 32 + lane;
            x_ahead = (task + nwarps < p.ntasks && qn < p.nq) ? ld_query(p.q + qn) : g0;
            int idx[1]; T x1s[1], x2s[1];
            search_multi<T, 1>(g, x, idx, x1s, x2s);                                    // linear.rs:87, :90-91
            const bool live = qi < p.nq;
            const bool bad = live && (p.mode ? Ar<T>::is_nan(x[0]) : !in_range(g0, gl, x[0]));   // linear.rs:80-84
            const T d = Ar<T>::sub(x2s[0], x1s[0]);
            const T r = slope_rcp<T>(d);
            report_first_bad(p.err, bad, (unsigned long long)qi);
            const bool skip = bad || !live;
            const int sub = lane % LPQ, qsel = lane / LPQ;
            const long long col = (long long)sub * V;
            const bool colok = col < p.w;
            const int idx0 = __shfl_sync(0xffffffffu, idx[0], __ffs(__ballot_sync(0xffffffffu, !skip) | 0x80000000u) - 1);
            const bool one_interval = LPQ > 1 && __all_sync(0xffffffffu, skip || idx[0] == idx0);
            Vec<T, V> y1, y2;
            if (one_interval && colok) {
                const T* row = p.data + (long long)idx0 * p.w + col;
                y1 = ld_table<T, V>(row);
                y2 = ld_table<T, V>(row + p.w);
            }
#pragma unroll
            for (int rd = 0; rd < LPQ; ++rd) {
                const int src = rd * QPR + qsel;
                const int is = __shfl_sync(0xffffffffu, skip ? -1 : idx[0], src);
                const T ds = shfl_t(d, src), rs = shfl_t(r, src);
                if (is >= 0 && colok) {
                    if (!one_interval) {
                        const T* row = p.data + (long long)is * p.w + col;
                        y1 = ld_table<T, V>(row);
                        y2 = ld_table<T, V>(row + p.w);
                    }
                    st_stream<T, V>(p.out + (qbase + src) * p.w + col, slope_vec<T, V>(y1, y2, ds, rs));
                }
            }
        } else {
            const long long tile = task / p.nslices;
            const int slice = (int)(task - tile * p.nslices);
            const long long qbase = tile * 32;
            const long long qi = qbase + lane;
            const bool live = qi < p.nq;
            T x[1] = {live ? ld_query(p.q + qi) : g0};
            int idx[1]; T x1s[1], x2s[1];
            search_multi<T, 1>(g, x, idx, x1s, x2s);
            const bool bad = live && (p.mode ? Ar<T>::is_nan(x[0]) : !in_range(g0, gl, x[0]));
            const T d = Ar<T>::sub(x2s[0], x1s[0]);
            const T r = slope_rcp<T>(d);
            if (slice == 0) report_first_bad(p.err, bad, (unsigned long long)qi);
            const bool skip = bad || !live;
            const long long col = ((long long)slice * 32 + lane) * V;
            const bool colok = col < p.w;
            int cur = -1;
            Vec<T, V> y1, y2;
            const int nlive = (int)min((long long)32, p.nq - qbase);
            for (int s = 0; s < nlive; ++s) {
                const int is = __shfl_sync(0xffffffffu, skip ? -1 : idx[0], s);
                const T ds = shfl_t(d, s), rs = shfl_t(r, s);
                if (is < 0 || !colok) continue;
                if (is != cur) {
                    const T* row = p.data + (long long)is * p.w + col;
                    y1 = ld_table<T, V>(row);
                    y2 = ld_table<T, V>(row + p.w);
                    cur = is;
                }
                st_stream<T, V>(p.out + (qbase + s) * p.w + col, slope_vec<T, V>(y1, y2, ds, rs));
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K4: Bilinear::interp_into x batch (bilinear.rs:64-99)
// ------------------------------------------------------------------------------------------------
// Very thin rows (LPQ <= 2, e.g. C4: 8 f32 columns) are bound by gather latency: five resident blocks
// (48 registers, a few spilled bytes) beat four (C4 0.589 -> 0.543 ms).  Wider rows are bound by
// instruction issue and lose from the spills (C5a 2.28 -> 2.75 ms): four blocks (64 registers, no spills).
// (Asking for one block only lets ptxas take 95 registers: two resident blocks, 3.36 ms.)
template <class T, int V, int LPQ, bool PERM>
__global__ void __launch_bounds__(kBlock, sizeof(T) == 4 ? (LPQ <= 2 ? 5 : 4) : 3) interp2d_bilinear_kernel(const Eval2<T> p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint64_t bar[2];
    constexpr bool kBcast = NDI_BCAST_SMEM && LPQ >= 4 && LPQ < 32 && kTilesBilinear == 1;
    __shared__ BilRec<T> recs[kBcast ? kWarpsPerBlock : 1][kBcast ? 32 : 1];
    const GridView<T> gx = make_grid_view<T>(p.gx, p.n, p.scx, smem_raw, &bar[0]);
    const GridView<T> gy = make_grid_view<T>(p.gy, p.m, p.scy, smem_raw + stage_bytes(p.scx, sizeof(T)), &bar[1]);
    const T gx0 = gx.g0, gxl = gx.gl, gy0 = gy.g0, gyl = gy.gl;
    const int lane = threadIdx.x & 31;
    const long long rowx = (long long)p.m * p.w;      // elements between x-rows
    const long long nwarps = (long long)gridDim.x * kWarpsPerBlock;
    const long long task0 = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    // A binned batch is only as good as the L2 residency of the band it walks through.  With tiles assigned by a
    // fixed stride the warps of a long launch drift apart (a 2^28-query batch runs for 20 ms; SMs a few per cent
    // slower end up many bands behind, the set of bands in flight outgrows L2 and every gather goes to DRAM:
    // 74 GB read for a 2.1 GB table, profiles/r02).  So the tiles of a binned batch are handed out IN ORDER through
    // an atomic counter: whatever the speed of an SM, all warps work within a few thousand tiles of each other.
    const bool dyn = PERM && LPQ < 32 && kTilesBilinear == 1 && p.next_task != nullptr;
    auto fetch_task = [&]() -> long long {
        unsigned long long t = 0;
        if (lane == 0) t = atomicAdd(p.next_task, 1ull);
        return (long long)__shfl_sync(0xffffffffu, t, 0);
    };
    const long long first = dyn ? fetch_task() : task0;
    T x_ahead = gx0, y_ahead = gy0; unsigned row_ahead = 0;   // thin rows: the next tile's query, loaded one tile ahead
    if (LPQ < 32 && kTilesBilinear == 1 && first < p.ntasks && first * 32 + lane < p.nq) {
        x_ahead = ld_query(p.qx + first * 32 + lane); y_ahead = ld_query(p.qy + first * 32 + lane);
        if constexpr (PERM) row_ahead = __ldcs(p.perm + first * 32 + lane);
    }
    long long next = 0;
    for (long long task = first; task < p.ntasks; task = next) {
        next = dyn ? fetch_task() : task + nwarps;
        if constexpr (LPQ < 32) {
            constexpr int TPW = kTilesBilinear, QPR = 32 / LPQ;
            const long long qbase0 = task * (32 * TPW);
            T x[TPW], y[TPW]; int ix[TPW], iy[TPW];
            long long cell[TPW]; T ax[TPW], bx[TPW], ay[TPW], by[TPW]; bool skip[TPW];   // ax..by: x1, x2, y1, y2 from the search
            Slope<T> slx[TPW], sly[TPW];
            unsigned orow[TPW];                                                        // output row (PERM only)
            if constexpr (TPW == 1) {
                x[0] = x_ahead; y[0] = y_ahead; orow[0] = row_ahead;
                const long long qn = next * 32 + lane;
                const bool more = next < p.ntasks && qn < p.nq;
                x_ahead = more ? ld_query(p.qx + qn) : gx0;
                y_ahead = more ? ld_query(p.qy + qn) : gy0;
                if constexpr (PERM) row_ahead = more ? __ldcs(p.perm + qn) : 0u;
            } else {
#pragma unroll
                for (int t = 0; t < TPW; ++t) {
                    const long long qi = qbase0 + t * 32 + lane;
                    const bool live = qi < p.nq;
                    x[t] = live ? ld_query(p.qx + qi) : gx0;
                    y[t] = live ? ld_query(p.qy + qi) : gy0;
                    if constexpr (PERM) orow[t] = live ? __ldcs(p.perm + qi) : 0u;
                }
            }
            search_multi<T, TPW>(gx, x, ix, ax, bx);                                  // bilinear.rs:82 (+ x1, x2)
            search_multi<T, TPW>(gy, y, iy, ay, by);
#pragma unroll
            for (int t = 0; t < TPW; ++t) {
                const long long qi = qbase0 + t * 32 + lane;
                const bool live = qi < p.nq;
                bool badx, bady;                                                       // :71-80: x is checked before y
                if (p.extrapolate) { badx = Ar<T>::is_nan(x[t]); bady = Ar<T>::is_nan(y[t]); }
                else { badx = !in_range(gx0, gxl, x[t]); bady = !in_range(gy0, gyl, y[t]); }
                const bool bad = live && (badx || bady);
                const T x1 = ax[t], x2 = bx[t], y1 = ay[t], y2 = by[t];
                bx[t] = Ar<T>::sub(x[t], x1); by[t] = Ar<T>::sub(y[t], y1);
                slx[t] = Slope<T>::make(Ar<T>::sub(x2, x1), bx[t], p.fast_tables != 0);
                sly[t] = Slope<T>::make(Ar<T>::sub(y2, y1), by[t], p.fast_tables != 0);
                cell[t] = ((long long)ix[t] * p.m + iy[t]) * p.w;                     // z11 (:83)
                if constexpr (PERM) report_bad_unordered(p.err, bad, 2ull * orow[t] + (badx ? 0ull : 1ull));
                else if (qbase0 + t * 32 < p.nq)
                    report_first_bad(p.err, bad, 2ull * (unsigned long long)qi + (badx ? 0ull : 1ull));
                skip[t] = bad || !live;
            }
            const int sub = lane % LPQ, qsel = lane / LPQ;
            const long long col = (long long)sub * V;
            const bool colok = col < p.w;
#pragma unroll
            for (int t = 0; t < TPW; ++t) {
                const long long qbase = qbase0 + t * 32;
                if (qbase >= p.nq) break;
                if constexpr (kBcast) {
                    recs[threadIdx.x >> 5][lane] = BilRec<T>{skip[t] ? -1ll : cell[t], bx[t], by[t], slx[t], sly[t], orow[t]};
                    __syncwarp();
                }
#pragma unroll
                for (int r = 0; r < LPQ; ++r) {
                    const int src = r * QPR + qsel;
                    long long cs, srow = qbase + src; bool live_s; T sbx, sby; Slope<T> ssx, ssy;
                    if constexpr (kBcast) {
                        const BilRec<T> rc = recs[threadIdx.x >> 5][src];
                        cs = rc.cs; live_s = cs >= 0; sbx = rc.bx; sby = rc.by; ssx = rc.sx; ssy = rc.sy;
                        if constexpr (PERM) srow = rc.orow;
                    } else {
#if NDI_PACK_SHFL >= 1
                        cs = __shfl_sync(0xffffffffu, skip[t] ? -1ll : cell[t], src);
                        live_s = cs >= 0;
#else
                        cs = __shfl_sync(0xffffffffu, cell[t], src);
                        live_s = !shfl_b(skip[t], src);
#endif
                        sbx = shfl_t(bx[t], src); sby = shfl_t(by[t], src);
                        ssx = slx[t].from_lane(src, sbx, p.fast_tables != 0); ssy = sly[t].from_lane(src, sby, p.fast_tables != 0);
                        if constexpr (PERM) srow = __shfl_sync(0xffffffffu, orow[t], src);
                    }
                    if (live_s && colok) {
                        const T* c0 = p.data + cs + col;
                        const Vec<T, V> z11 = ld_table<T, V>(c0), z12 = ld_table<T, V>(c0 + p.w);
                        const Vec<T, V> z21 = ld_table<T, V>(c0 + rowx), z22 = ld_table<T, V>(c0 + rowx + p.w);
                        st_stream<T, V>(p.out + srow * p.w + col, bilerp_vec<T, V, (LPQ > 2)>(z11, z12, z21, z22, ssx, sbx, ssy, sby));
                    }
                }
                if constexpr (kBcast) __syncwarp();                    // the slab is rewritten by the next tile
            }
        } else {
            const long long tile = task / p.nslices;
            const int slice = (int)(task - tile * p.nslices);
            const long long qbase = tile * 32;
            const long long qi = qbase + lane;
            const bool live = qi < p.nq;
            T x[1] = {live ? ld_query(p.qx + qi) : gx0};
            T y[1] = {live ? ld_query(p.qy + qi) : gy0};
            bool badx, bady;
            if (p.extrapolate) { badx = Ar<T>::is_nan(x[0]); bady = Ar<T>::is_nan(y[0]); }
            else { badx = !in_range(gx0, gxl, x[0]); bady = !in_range(gy0, gyl, y[0]); }
            const bool bad = live && (badx || bady);
            int ix[1], iy[1]; T x1s[1], x2s[1], y1s[1], y2s[1];
            search_multi<T, 1>(gx, x, ix, x1s, x2s);
            search_multi<T, 1>(gy, y, iy, y1s, y2s);
            const T x1 = x1s[0], x2 = x2s[0], y1 = y1s[0], y2 = y2s[0];
            const T dxq = Ar<T>::sub(x[0], x1), dyq = Ar<T>::sub(y[0], y1);
            const Slope<T> slx = Slope<T>::make(Ar<T>::sub(x2, x1), dxq, p.fast_tables != 0);
            const Slope<T> sly = Slope<T>::make(Ar<T>::sub(y2, y1), dyq, p.fast_tables != 0);
            const long long cell = ((long long)ix[0] * p.m + iy[0]) * p.w;
            unsigned orow = 0;
            if constexpr (PERM) {
                orow = live ? __ldcs(p.perm + qi) : 0u;
                if (slice == 0) report_bad_unordered(p.err, bad, 2ull * orow + (badx ? 0ull : 1ull));
            } else if (slice == 0) report_first_bad(p.err, bad, 2ull * (unsigned long long)qi + (badx ? 0ull : 1ull));
            const bool skip = bad || !live;
            const long long col = ((long long)slice * 32 + lane) * V;
            const bool colok = col < p.w;
            long long cur = -1;
            Vec<T, V> z11, z12, z21, z22;
            const int nlive = (int)min((long long)32, p.nq - qbase);
            for (int s = 0; s < nlive; ++s) {
                const long long cs = __shfl_sync(0xffffffffu, cell, s);
                const Slope<T> ssx = slx.from_lane(s), ssy = sly.from_lane(s);
                const T bx = shfl_t(dxq, s), by = shfl_t(dyq, s);
                const bool sk = shfl_b(skip, s);
                long long srow = qbase + s;
                if constexpr (PERM) srow = __shfl_sync(0xffffffffu, orow, s);
                if (sk || !colok) continue;
                if (cs != cur) {
                    const T* c0 = p.data + cs + col;
                    z11 = ld_table<T, V>(c0);
                    z12 = ld_table<T, V>(c0 + p.w);
                    z21 = ld_table<T, V>(c0 + rowx);
                    z22 = ld_table<T, V>(c0 + rowx + p.w);
                    cur = cs;
                }
                const Vec<T, V> res = bilerp_vec<T, V>(z11, z12, z21, z22, ssx, bx, ssy, by);
                st_stream<T, V>(p.out + srow * p.w + col, res);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K2 standalone: get_lower_index for a batch (vector_extensions.rs:55-111)
// ------------------------------------------------------------------------------------------------
template <class T>
__global__ void __launch_bounds__(kBlock) lower_index_kernel(const T* __restrict__ grid, int n, SearchCfg sc,
                                                            const T* __restrict__ q, long long nq,
                                                            long long* __restrict__ idx, unsigned long long* err) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    constexpr int K = 4;
    const GridView<T> g = make_grid_view<T>(grid, n, sc, smem_raw, &bar);
    const T g0 = g.g0;
    const long long span = (long long)blockDim.x * K;
    const long long nspans = (nq + span - 1) / span;
    for (long long sp = blockIdx.x; sp < nspans; sp += gridDim.x) {
        T x[K]; int r[K]; T vlo[K], vhi[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const long long i = sp * span + (long long)k * blockDim.x + threadIdx.x;
            x[k] = i < nq ? ld_query(q + i) : g0;
        }
        search_multi<T, K>(g, x, r, vlo, vhi);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const long long i = sp * span + (long long)k * blockDim.x + threadIdx.x;
            const bool live = i < nq;
            const bool bad = live && Ar<T>::is_nan(x[k]);
            report_first_bad(err, bad, (unsigned long long)i);
            if (live && !bad) idx[i] = r[k];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K7 pre-pass for the host entry points: first failing query, reading only the queries.
// ------------------------------------------------------------------------------------------------
template <class T>
__global__ void __launch_bounds__(kBlock) validate_queries_kernel(const T* __restrict__ gx, int n, const T* __restrict__ gy,
                                                                 int m, const T* __restrict__ qx,
                                                                 const T* __restrict__ qy, long long nq, int check,
                                                                 unsigned long long* err) {
    const T gx0 = gx[0], gxl = gx[n - 1];
    const T gy0 = gy ? gy[0] : (T)0, gyl = gy ? gy[m - 1] : (T)0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long nq_pad = (nq + 31) & ~31ll;
    unsigned long long first = ~0ull;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nq_pad; i += stride) {
        if (i >= nq) continue;
        const T x = ld_query(qx + i);
        bool badx, bady = false;
        if (check == CHECK_IN_RANGE) badx = !in_range(gx0, gxl, x);
        else if (check == CHECK_NOT_NAN) badx = Ar<T>::is_nan(x);
        else badx = !in_range(gx0, gxl, x) && !Ar<T>::is_finite(x);   // periodic wrap of +-inf / NaN gives NaN
        if (qy) {
            const T y = ld_query(qy + i);
            bady = (check == CHECK_IN_RANGE) ? !in_range(gy0, gyl, y) : Ar<T>::is_nan(y);
        }
        if (badx || bady) {
            unsigned long long word = qy ? 2ull * (unsigned long long)i + (badx ? 0ull : 1ull) : (unsigned long long)i;
            first = min(first, word);
        }
    }
    // warp min, then one atomic per warp that saw a failure
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
    if ((threadIdx.x & 31) == 0 && first != ~0ull) atomicMin(err, first);
}

// ------------------------------------------------------------------------------------------------
// host-side dispatch
// ------------------------------------------------------------------------------------------------
static int pow2ceil(long long v) { int p = 1; while (p < v && p < 32) p <<= 1; return p; }

static bool aligned(const void* p, size_t a) { return ((uintptr_t)p % a) == 0; }

template <class T>
static int pick_vec(long long w, std::initializer_list<const void*> ptrs) {
    constexpr int vmax = 16 / (int)sizeof(T);
    for (int v = vmax; v > 1; v >>= 1) {
        bool ok = (w % v) == 0;
        for (const void* p : ptrs) ok = ok && aligned(p, sizeof(T) * v);
        if (ok) return v;
    }
    return 1;
}

struct Shape { int v; int lpq; int nslices; long long ntasks; };

static Shape pick_shape(long long w, long long nq, int v, int tiles_per_warp) {
    Shape s;
    s.v = v;
    long long groups = (w + v - 1) / v;
    s.lpq = pow2ceil(groups);
    long long tiles = (nq + 31) / 32;
    if (s.lpq == 32) {
        s.nslices = (int)((groups + 31) / 32);
        s.ntasks = tiles * s.nslices;
    } else {
        s.nslices = 1;
        s.ntasks = (tiles + tiles_per_warp - 1) / tiles_per_warp;
    }
    return s;
}

template <class K>
static cudaError_t prep_smem(K kernel, size_t bytes) {
    // static shared memory (barriers, up to 16 KB of per-warp record slabs) counts against the 48 KB default as well
    if (bytes > 30 * 1024) return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    return cudaSuccess;
}

template <class K>
static int persistent_grid(K kernel, size_t smem, long long ntasks) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kBlock, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    long long want = (ntasks + kWarpsPerBlock - 1) / kWarpsPerBlock;
    long long cap = (long long)device_info().sm_count * per_sm;
    return (int)(want < cap ? (want < 1 ? 1 : want) : cap);
}

template <class P, class K>
static cudaError_t launch_eval(K kernel, const P& p, size_t smem, cudaStream_t st) {
    cudaError_t e = prep_smem(kernel, smem);
    if (e != cudaSuccess) return e;
    int grid = persistent_grid(kernel, smem, p.ntasks);
    kernel<<<grid, kBlock, smem, st>>>(p);
    count_launch();
    return cudaGetLastError();
}

#define NDI_LPQ_SWITCH(KERNEL, T, V, LPQ, P, SMEM, ST)                                   \
    switch (LPQ) {                                                                        \
    case 1:  return launch_eval(KERNEL<T, V, 1>, P, SMEM, ST);                            \
    case 2:  return launch_eval(KERNEL<T, V, 2>, P, SMEM, ST);                            \
    case 4:  return launch_eval(KERNEL<T, V, 4>, P, SMEM, ST);                            \
    case 8:  return launch_eval(KERNEL<T, V, 8>, P, SMEM, ST);                            \
    case 16: return launch_eval(KERNEL<T, V, 16>, P, SMEM, ST);                           \
    default: return launch_eval(KERNEL<T, V, 32>, P, SMEM, ST);                           \
    }

#define NDI_VEC_SWITCH(KERNEL, T, SH, P, SMEM, ST)                                        \
    if constexpr (sizeof(T) == 4) {                                                       \
        if (SH.v == 4) { NDI_LPQ_SWITCH(KERNEL, T, 4, SH.lpq, P, SMEM, ST) }              \
        if (SH.v == 2) { NDI_LPQ_SWITCH(KERNEL, T, 2, SH.lpq, P, SMEM, ST) }              \
        NDI_LPQ_SWITCH(KERNEL, T, 1, SH.lpq, P, SMEM, ST)                                 \
    } else {                                                                              \
        if (SH.v == 2) { NDI_LPQ_SWITCH(KERNEL, T, 2, SH.lpq, P, SMEM, ST) }              \
        NDI_LPQ_SWITCH(KERNEL, T, 1, SH.lpq, P, SMEM, ST)                                 \
    }

template <class T, int V, int LPQ> constexpr auto bilinear_direct = interp2d_bilinear_kernel<T, V, LPQ, false>;
template <class T, int V, int LPQ> constexpr auto bilinear_binned = interp2d_bilinear_kernel<T, V, LPQ, true>;

template <class T>
cudaError_t launch_interp1d_linear(const T* grid, int64_t n, SearchCfg sc, const T* data, int64_t w, const T* q,
                                   int64_t nq, int extrapolate, T* out, unsigned long long* err, int fast_tables,
                                   const T* pair, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    if (pair && pair_table_shape_ok(w, sizeof(T)) && aligned(out, 16)) {
        const long long tiles = (nq + 31) / 32;
        Eval1<T> p{grid, (int)n, sc, pair, nullptr, nullptr, (long long)w, q, (long long)nq, extrapolate, out, err, tiles, 1, fast_tables};
        const size_t smem = stage_bytes(sc, sizeof(T));
        switch ((int)(w / (16 / (int64_t)sizeof(T)))) {
        case 1: return launch_eval(interp1d_linear_pair_kernel<T, 1>, p, smem, st);
        case 2: return launch_eval(interp1d_linear_pair_kernel<T, 2>, p, smem, st);
        default: return launch_eval(interp1d_linear_pair_kernel<T, 4>, p, smem, st);
        }
    }
    Shape sh = pick_shape(w, nq, pick_vec<T>(w, {data, out}), kTilesLinear);
    Eval1<T> p{grid, (int)n, sc, data, nullptr, nullptr, (long long)w, q, (long long)nq, extrapolate, out, err, sh.ntasks, sh.nslices, fast_tables};
    size_t smem = stage_bytes(sc, sizeof(T));
    NDI_VEC_SWITCH(interp1d_linear_kernel, T, sh, p, smem, st)
}

template <class T>
cudaError_t launch_interp1d_cubic(const T* grid, int64_t n, SearchCfg sc, const T* data, const T* a, const T* b,
                                  int64_t w, const T* q, int64_t nq, int extrap_mode, T* out,
                                  unsigned long long* err, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    Shape sh = pick_shape(w, nq, pick_vec<T>(w, {data, a, b, out}), kTilesCubic);
    Eval1<T> p{grid, (int)n, sc, data, a, b, (long long)w, q, (long long)nq, extrap_mode, out, err, sh.ntasks, sh.nslices, 0};
    size_t smem = stage_bytes(sc, sizeof(T));
    NDI_VEC_SWITCH(interp1d_cubic_kernel, T, sh, p, smem, st)
}

template <class T, int V, int LPQ> constexpr auto cubic_deriv1 = interp1d_cubic_deriv_kernel<T, V, LPQ, 1>;
template <class T, int V, int LPQ> constexpr auto cubic_deriv2 = interp1d_cubic_deriv_kernel<T, V, LPQ, 2>;

template <class T>
cudaError_t launch_interp1d_cubic_deriv(const T* grid, int64_t n, SearchCfg sc, const T* data, const T* a, const T* b,
                                        int64_t w, const T* q, int64_t nq, int extrap_mode, int order, T* out,
                                        unsigned long long* err, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    Shape sh = pick_shape(w, nq, pick_vec<T>(w, {data, a, b, out}), 1);
    Eval1<T> p{grid, (int)n, sc, data, a, b, (long long)w, q, (long long)nq, extrap_mode, out, err, sh.ntasks, sh.nslices, 0};
    size_t smem = stage_bytes(sc, sizeof(T));
    if (order == 1) { NDI_VEC_SWITCH(cubic_deriv1, T, sh, p, smem, st) }
    NDI_VEC_SWITCH(cubic_deriv2, T, sh, p, smem, st)
}

template <class T>
cudaError_t launch_interp1d_linear_slope(const T* grid, int64_t n, SearchCfg sc, const T* data, int64_t w, const T* q,
                                         int64_t nq, int extrapolate, T* out, unsigned long long* err, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    Shape sh = pick_shape(w, nq, pick_vec<T>(w, {data, out}), 1);
    Eval1<T> p{grid, (int)n, sc, data, nullptr, nullptr, (long long)w, q, (long long)nq, extrapolate, out, err, sh.ntasks, sh.nslices, 0};
    size_t smem = stage_bytes(sc, sizeof(T));
    NDI_VEC_SWITCH(interp1d_linear_slope_kernel, T, sh, p, smem, st)
}

template <class T>
cudaError_t launch_interp2d_bilinear(const T* gx, int64_t n, SearchCfg scx, const T* gy, int64_t m, SearchCfg scy,
                                     const T* data, int64_t w, const T* qx, const T* qy, int64_t nq, int extrapolate,
                                     T* out, unsigned long long* err, const unsigned* perm, int fast_tables,
                                     unsigned long long* next_task, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    Shape sh = pick_shape(w, nq, pick_vec<T>(w, {data, out}), kTilesBilinear);
    Eval2<T> p{gx, (int)n, scx, gy, (int)m, scy, data, (long long)w, qx, qy, (long long)nq, extrapolate, out, err, sh.ntasks, sh.nslices, perm, fast_tables, perm ? next_task : nullptr};
    size_t smem = stage_bytes(scx, sizeof(T)) + stage_bytes(scy, sizeof(T));
    if (perm) { NDI_VEC_SWITCH(bilinear_binned, T, sh, p, smem, st) }
    NDI_VEC_SWITCH(bilinear_direct, T, sh, p, smem, st)
}

template <class T>
cudaError_t launch_lower_index(const T* grid, int64_t n, SearchCfg sc, const T* q, int64_t nq, int64_t* idx,
                               unsigned long long* err, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    size_t smem = stage_bytes(sc, sizeof(T));
    cudaError_t e = prep_smem(lower_index_kernel<T>, smem);
    if (e != cudaSuccess) return e;
    long long blocks = (nq + (long long)kBlock * 4 - 1) / ((long long)kBlock * 4);
    long long cap = (long long)device_info().sm_count * 8;
    lower_index_kernel<T><<<(int)(blocks < cap ? blocks : cap), kBlock, smem, st>>>(grid, (int)n, sc, q, (long long)nq,
                                                                                   (long long*)idx, err);
    count_launch();
    return cudaGetLastError();
}

template <class T>
cudaError_t launch_validate_queries(const T* gx, int64_t n, const T* gy, int64_t m, const T* qx, const T* qy,
                                    int64_t nq, int check, unsigned long long* err, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    long long blocks = (nq + kBlock - 1) / kBlock;
    long long cap = (long long)device_info().sm_count * 8;
    validate_queries_kernel<T><<<(int)(blocks < cap ? blocks : cap), kBlock, 0, st>>>(gx, (int)n, gy, (int)m, qx, qy,
                                                                                     (long long)nq, check, err);
    count_launch();
    return cudaGetLastError();
}

#define NDI_INST_COMMON(T)                                                                                             \
    template cudaError_t launch_interp1d_linear<T>(const T*, int64_t, SearchCfg, const T*, int64_t, const T*, int64_t, \
                                                   int, T*, unsigned long long*, int, const T*, cudaStream_t);         \
    template cudaError_t launch_pack_pairs<T>(const T*, int64_t, int64_t, T*, cudaStream_t);                           \
    template cudaError_t launch_interp2d_bilinear<T>(const T*, int64_t, SearchCfg, const T*, int64_t, SearchCfg,       \
                                                     const T*, int64_t, const T*, const T*, int64_t, int, T*,          \
                                                     unsigned long long*, const unsigned*, int, unsigned long long*,   \
                                                     cudaStream_t);                                                    \
    template cudaError_t launch_lower_index<T>(const T*, int64_t, SearchCfg, const T*, int64_t, int64_t*,              \
                                               unsigned long long*, cudaStream_t);                                     \
    template cudaError_t launch_validate_queries<T>(const T*, int64_t, const T*, int64_t, const T*, const T*, int64_t, \
                                                    int, unsigned long long*, cudaStream_t);                           \
    template cudaError_t launch_interp1d_linear_slope<T>(const T*, int64_t, SearchCfg, const T*, int64_t, const T*,    \
                                                         int64_t, int, T*, unsigned long long*, cudaStream_t);
NDI_INST_COMMON(float)
NDI_INST_COMMON(double)
NDI_INST_COMMON(int32_t)
NDI_INST_COMMON(int64_t)
NDI_INST_COMMON(uint32_t)
NDI_INST_COMMON(uint64_t)
template cudaError_t launch_interp1d_cubic<float>(const float*, int64_t, SearchCfg, const float*, const float*,
                                                  const float*, int64_t, const float*, int64_t, int, float*,
                                                  unsigned long long*, cudaStream_t);
template cudaError_t launch_interp1d_cubic<double>(const double*, int64_t, SearchCfg, const double*, const double*,
                                                   const double*, int64_t, const double*, int64_t, int, double*,
                                                   unsigned long long*, cudaStream_t);
template cudaError_t launch_interp1d_cubic_deriv<float>(const float*, int64_t, SearchCfg, const float*, const float*,
                                                        const float*, int64_t, const float*, int64_t, int, int, float*,
                                                        unsigned long long*, cudaStream_t);
template cudaError_t launch_interp1d_cubic_deriv<double>(const double*, int64_t, SearchCfg, const double*, const double*,
                                                         const double*, int64_t, const double*, int64_t, int, int, double*,
                                                         unsigned long long*, cudaStream_t);

}  // namespace ndi
