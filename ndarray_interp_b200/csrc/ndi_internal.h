// ndi_internal.h -- launcher prototypes shared between the kernel translation units and the
// C ABI (ndi_api.cu).  Nothing here is exported.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace ndi {

// how the lower-index search reads one grid
struct SearchCfg {
    int top_step;           // largest power of two <= n-2 (bisect_top_step)
    int guess;              // 1: try the O(1) even-spacing guess first (uniform grids)
    int smem;               // 1: stage `stage_n` elements from `stage_src` into shared memory (bulk copy)
    int coarse_shift;       // log2 of the stride of the staged table (0: it is the whole grid)
    int stage_n;
    const void* stage_src;  // the grid itself, or the handle's coarse table grid[0], grid[S], grid[2S], ...
    const void* lut;        // non-null: bucket-table search (LutEntry per bucket, see ndi_device.cuh)
    int lut_n;              // number of buckets
    double g0d, scale;      // bucket(x) = (x - g0d) * scale
    int merge;              // 1: warp-level merge search for sorted batches (bracket from the warp's min / max query)
};

// largest power of two <= n-2 (0 when n == 2): the first probe distance of the bisection
inline int bisect_top_step(int64_t n) {
    int s = 0;
    if (n - 2 >= 1) { s = 1; while ((int64_t)s * 2 <= n - 2) s *= 2; }
    return s;
}

struct DeviceInfo {
    int device;
    int sm_count;
    size_t smem_optin;   // max dynamic shared memory per block
    size_t l2_bytes;
};
const DeviceInfo& device_info();          // of the current device
void count_launch();                      // bumps ndi_kernel_launch_count()

// ---- evaluation (ndi_eval.cu) -----------------------------------------------------------
template <class T>
cudaError_t launch_lower_index(const T* grid, int64_t n, SearchCfg sc, const T* q, int64_t nq, int64_t* idx,
                               unsigned long long* err, cudaStream_t st);

// mode for validate_queries / the fused checks: which queries make the reference fail
enum QueryCheck { CHECK_IN_RANGE = 0, CHECK_NOT_NAN = 1, CHECK_FINITE_IF_OUTSIDE = 2 };
// K7 pre-pass used by the host entry points: first query (row-major) the reference would fail on
template <class T>
cudaError_t launch_validate_queries(const T* g0_gl_x /* grid x */, int64_t n, const T* gy, int64_t m,
                                    const T* qx, const T* qy, int64_t nq, int check, unsigned long long* err,
                                    cudaStream_t st);

// pair: the handle's pair table (rows i, i+1 interleaved; launch_pack_pairs) or nullptr
template <class T>
cudaError_t launch_interp1d_linear(const T* grid, int64_t n, SearchCfg sc, const T* data, int64_t w, const T* q,
                                   int64_t nq, int extrapolate, T* out, unsigned long long* err, int fast_tables,
                                   const T* pair, cudaStream_t st);
// thin rows (32 - 64 bytes, a whole number of 16-byte lanes): may the linear kernel use a pair table?
bool pair_table_shape_ok(int64_t w, size_t elem);
template <class T>
cudaError_t launch_pack_pairs(const T* y, int64_t n, int64_t w, T* P, cudaStream_t st);
template <class T>
cudaError_t launch_interp1d_cubic(const T* grid, int64_t n, SearchCfg sc, const T* data, const T* a, const T* b,
                                  int64_t w, const T* q, int64_t nq, int extrap_mode, T* out,
                                  unsigned long long* err, cudaStream_t st);
// derivative of order 1 or 2 of the cubic spline (K5d), slope of Linear (K3d): query handling as the value launchers
template <class T>
cudaError_t launch_interp1d_cubic_deriv(const T* grid, int64_t n, SearchCfg sc, const T* data, const T* a, const T* b,
                                        int64_t w, const T* q, int64_t nq, int extrap_mode, int order, T* out,
                                        unsigned long long* err, cudaStream_t st);
template <class T>
cudaError_t launch_interp1d_linear_slope(const T* grid, int64_t n, SearchCfg sc, const T* data, int64_t w, const T* q,
                                         int64_t nq, int extrapolate, T* out, unsigned long long* err, cudaStream_t st);
// definite integrals (K9c / K9l) over the cumulative table C (ndi_integral.cu: K9b builds it); a == nullptr: Linear
template <class T>
cudaError_t launch_interp1d_integral(const T* grid, int64_t n, SearchCfg sc, const T* data, const T* a, const T* b,
                                     const T* cum, int64_t w, const T* lo, const T* hi, int64_t nq, int mode, T* out,
                                     unsigned long long* err, cudaStream_t st);
// pre-pass of the integral calls: the value call's check on each bound, error word 2 * query + bound
template <class T>
cudaError_t launch_validate_bounds(const T* grid, int64_t n, const T* lo, const T* hi, int64_t nq, int check,
                                   unsigned long long* err, cudaStream_t st);
// scratch: integral_build_scratch(n, w) doubles
size_t integral_build_scratch(int64_t n, int64_t w);
template <class T>
cudaError_t launch_integral_build(const T* x, int64_t n, const T* data, const T* a, const T* b, int64_t w, T* cum,
                                  double* scratch, cudaStream_t st);
// knot slopes and cubic coefficients of a shape-preserving cubic (K10, ndi_hermite.cu); kind: NDI_HERMITE_*,
// dydx: device slopes (n, w) for NDI_HERMITE_GIVEN, else nullptr; mx: two zeroable device words (Akima's maximum)
template <class T>
cudaError_t launch_hermite_build(int kind, const T* x, int64_t n, const T* data, int64_t w, const T* dydx,
                                 unsigned long long* mx, T* a, T* b, cudaStream_t st);
template <class T>
cudaError_t launch_interp2d_bilinear(const T* gx, int64_t n, SearchCfg scx, const T* gy, int64_t m, SearchCfg scy,
                                     const T* data, int64_t w, const T* qx, const T* qy, int64_t nq, int extrapolate,
                                     T* out, unsigned long long* err, const unsigned* perm, int fast_tables,
                                     unsigned long long* next_task, cudaStream_t st);

// ---- locality binning of 2-D query batches (ndi_bin.cu) --------------------------------------
// The x-axis is cut into nbands bands of 2^band_shift intervals; launch_bin_queries groups the
// queries by band.  perm != nullptr in launch_interp2d_bilinear: qx/qy are the binned copies and
// the result of binned query i goes to output row perm[i].
constexpr int kMaxBands = 256;
struct BandPlan { int band_shift; int nbands; };
// band_rows > 0 fixes the band height (tests); else bands of about band_bytes of table
BandPlan plan_bands(int64_t n, int64_t m, int64_t w, size_t elem, size_t band_bytes, int band_rows);
size_t bin_scratch_bytes(int64_t nq, size_t elem);
template <class T>
cudaError_t launch_bin_queries(const T* gx, int64_t n, SearchCfg scx, const T* qx, const T* qy, int64_t nq,
                               BandPlan bp, void* scratch, const unsigned** perm, const T** bqx, const T** bqy,
                               unsigned long long** next_task, cudaStream_t st);

// ---- bilinear in band sweeps (ndi_sweep.cu) ----------------------------------------------------
// The launch walks the batch nsweeps times; sweep b evaluates the queries whose x-interval lies in
// [b * band_rows, (b + 1) * band_rows), compacted into full tiles, so that the band's table rows stay in L2.
// Rows of 16 / 32 / 64 / 128 bytes only (sweep_shape_ok).  next_task: a zeroed 8-byte device word.
constexpr int kMaxSweeps = 16;
struct SweepPlan { int band_rows; int nsweeps; };
SweepPlan plan_sweeps(int64_t n, int64_t m, int64_t w, size_t elem, size_t band_bytes, int band_rows);
bool sweep_shape_ok(int64_t n, int64_t m, int64_t w, size_t elem, const void* data, const void* out, int64_t nq);
template <class T>
cudaError_t launch_interp2d_bilinear_sweep(const T* gx, int64_t n, SearchCfg scx, const T* gy, int64_t m, SearchCfg scy,
                                           const T* data, int64_t w, const T* qx, const T* qy, int64_t nq, int extrapolate,
                                           T* out, unsigned long long* err, int fast_tables, SweepPlan sp,
                                           unsigned long long* next_task, cudaStream_t st);

// fast_tables (linear, bilinear; f32 only): 1 when launch_table_fast_div found every table value to
// be 0 or in [2^-56, 2^30], which lets the kernels divide with a per-query reciprocal (ndi_device.cuh)
cudaError_t launch_table_fast_div(const float* data, size_t count, int32_t* flag_dev, cudaStream_t st);
// all-pairs check of div_by() against __fdiv_rn (ndi_selftest_fdiv)
cudaError_t launch_selftest_fdiv(uint32_t a_mant_begin, uint32_t a_mant_count, int a_exp, int b_exp,
                                 unsigned long long* mismatches_dev, cudaStream_t st);

cudaError_t launch_selftest_ddiv(uint64_t seed, int blocks, int per_thread, unsigned long long* mismatches_dev, cudaStream_t st);

cudaError_t launch_publish(unsigned long long* d_err, void* h_err, void* h_flag, unsigned long long seq, cudaStream_t st);

// ---- grid checks (ndi_grid.cu) -----------------------------------------------------------
// result[0] = Monotonic enum, result[1] = 1 when the even-spacing guess hits on every cell
template <class T>
cudaError_t launch_grid_classify(const T* x, int64_t n, int32_t* result_dev, uint32_t* scratch_dev,
                                 cudaStream_t st);
size_t grid_classify_scratch_words();
// bucket table of a strictly rising grid (entry format: LutEntry in ndi_device.cuh)
size_t lut_entry_bytes(size_t elem);
template <class T>
cudaError_t launch_build_lut(const T* x, int64_t n, double g0d, double scale, int nb, void* lut_dev, cudaStream_t st);

// ---- strided views -> dense tables (ndi_grid.cu) ----------------------------------------------
// dst[row-major index] = src[origin + sum(idx[d] * stride[d])], elements of `elem` bytes (4 or 8);
// strides are in elements and may be negative or zero (ndarray views, interp1d/aliases.rs).
constexpr int kMaxDims = 8;
struct StridedDesc { int ndim; long long shape[kMaxDims]; long long stride[kMaxDims]; };
cudaError_t launch_pack_strided(const void* src_dev, long long origin, const StridedDesc& d, size_t elem,
                                long long count, void* dst_dev, cudaStream_t st);

// ---- spline construction (ndi_spline.cu, ndi_rowsplit.cu) ----------------------------------------
// Builds a, b ((n-1) x w each) on the device.  For bc_kind == INDIVIDUAL the four boundary arrays are
// device arrays of w entries; pos (device, w entries) gives every column its position when the
// columns are grouped by (left kind, right kind) after specialisation, group_count (host, 9
// entries, group = 3 * variant(left) + variant(right), variant: NotAKnot 0, FirstDeriv 1,
// SecondDeriv 2) the size of each group.  scratch: spline_scratch_elems() elements.
// levels == 0: the reference's elimination order (bit-identical coefficients); levels > 0: the row-split
// build, `levels` steps of parallel cyclic reduction followed by 2^levels interleaved Thomas solves per
// column (see rowsplit_levels_for).  err: device word, set to the first column with a periodic mismatch.
template <class T>
cudaError_t launch_spline_build(const T* x, int64_t n, const T* data, int64_t w, int bc_kind, const int32_t* lk,
                                const T* lv, const int32_t* rk, const T* rv, const int32_t* pos, const int64_t* group_count,
                                int levels, T* a, T* b, T* scratch, unsigned long long* err, cudaStream_t st);
template <class T>
size_t spline_scratch_elems(int64_t n, int64_t w, int bc_kind, int levels);
// row-split depth for a system of `rows` rows: `requested` > 0 is honoured up to the deepest split that keeps
// two rows per system and fits the reduce kernel's shared-memory tile; requested == 0 picks the depth that
// leaves chains of about 256 rows -- unless the system is shorter than kRowsplitAutoRows and `force` is
// not set, where the reference's order is kept (0); 0 also when the system is too short to split at all
constexpr int kMaxRowsplitLevels = 6;
constexpr int64_t kRowsplitAutoRows = 2048;         // depth chosen for an unforced request: systems below this keep the reference order
constexpr int64_t kPartitionAutoRows = 1024;        // NDI_BUILD_AUTO: partition build from this many rows on
int rowsplit_levels_for(int64_t rows, int requested, bool force);
// partition build (ndi_partition.cu): rows per block for a request (0: the default), passed on as levels = -block
int partition_block_for(int requested);

}  // namespace ndi
