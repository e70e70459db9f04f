/*
 * ndi_b200.h -- C ABI of the B200-native batched interpolation path.
 *
 * This is the drop-in boundary for the hot path of jonasBoss/ndarray-interp v0.6.0:
 * grid validation -> lower-index search -> gather + linear / bilinear / cubic-spline
 * evaluation, plus cubic-spline coefficient construction.  Everything behind these entry
 * points runs as hand-written CUDA for sm_100a; there is no CPU fallback.  Plain pointers
 * and sizes only -- no torch / ndarray types cross this boundary.
 *
 * Each entry point names the reference interface it replaces (paths relative to the
 * reference repository).  INTEGRATION.md shows the Rust FFI binding a maintainer would add.
 *
 * Conventions
 *   - Arrays are C-contiguous.  `w` is the product of the trailing data dimensions
 *     (data.shape[1..] for 1-D, data.shape[2..] for 2-D); `nq` is the flattened query count.
 *     Output row q holds the `w` values for query q: shape = query.shape ++ data.shape[1..]
 *     (src/interp1d/mod.rs:346-354, src/interp2d/mod.rs:310-321).
 *   - `dtype` selects the element type of every `void*` argument of the call.
 *   - Every function returns an ndi_status and never unwinds.
 *   - Functions without a `_dev` suffix take HOST pointers, are synchronous and may be called
 *     concurrently from many host threads on the same handle (the reference's `&self` methods
 *     are called from rayon workers, benches/bench_interp1d.rs:49-79).  `_dev` functions take
 *     DEVICE pointers and a cudaStream_t (passed as void*), enqueue one fused launch and return
 *     without synchronising.
 *   - Errors follow the reference: evaluation stops at the FIRST failing query in row-major
 *     order (src/interp1d/mod.rs:321,336-340).  The host functions leave output rows at and
 *     after `*first_bad` untouched, like the reference.  The `_dev` functions report the first
 *     failing query through a device error word and skip only the failing rows.
 */
#ifndef NDI_B200_H
#define NDI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NDI_VERSION_MAJOR 0
#define NDI_VERSION_MINOR 1

typedef int32_t ndi_status;
#define NDI_OK 0
/* InterpolateError::OutOfBounds (src/lib.rs:142-146; raised at linear.rs:80-84,
 * bilinear.rs:71-80, cubic_spline.rs:797-802) */
#define NDI_OUT_OF_BOUNDS 1
/* the reference panics with "not implemented: failed to convert NaN to usize"
 * (src/vector_extensions.rs:83-84) when a NaN query reaches get_lower_index */
#define NDI_NAN_QUERY 2
/* BuilderError::ValueError: periodic spline with data[0] != data[n-1] (cubic_spline.rs:483-507) */
#define NDI_PERIODIC_MISMATCH 3
#define NDI_INVALID_ARGUMENT 4
/* BuilderError::Monotonic (src/interp1d/mod.rs:460-464, src/interp2d/mod.rs:500-509) */
#define NDI_NOT_MONOTONIC 5
/* cubic evaluation requested before ndi_interp1d_spline_build */
#define NDI_NO_SPLINE 6
#define NDI_UNSUPPORTED_DTYPE 7
#define NDI_NO_DEVICE 8
/* 100 + cudaError_t; text via ndi_last_error_message() */
#define NDI_CUDA_ERROR 100

typedef int32_t ndi_dtype;
#define NDI_F32 0
#define NDI_F64 1
#define NDI_I32 2 /* everything except splines (SplineNum is float-only, cubic_spline.rs:34-49) */
#define NDI_I64 3 /* as NDI_I32: wrapping arithmetic, truncating division (Linear / Bilinear are generic over Num) */
#define NDI_U32 4 /* unsigned: the reference's generic bound admits them (linear.rs:29-36, T: Num); arithmetic modulo 2^32 as in */
#define NDI_U64 5 /* a release build of the reference (a debug build panics where a difference would be negative), unsigned / and < */

/* enum Monotonic (src/vector_extensions.rs:24-29) */
#define NDI_MONO_NOT_MONOTONIC 0
#define NDI_MONO_RISING_STRICT 1
#define NDI_MONO_RISING 2
#define NDI_MONO_FALLING_STRICT 3
#define NDI_MONO_FALLING 4

/* enum BoundaryCondition (cubic_spline.rs:153-168) */
#define NDI_BC_NOT_A_KNOT 0
#define NDI_BC_NATURAL 1
#define NDI_BC_CLAMPED 2
#define NDI_BC_PERIODIC 3
#define NDI_BC_INDIVIDUAL 4
/* enum SingleBoundary (cubic_spline.rs:203-217); RowBoundary::{NotAKnot,Natural,Clamped} is
 * the same kind on both sides (InternalBoundary::specialize, cubic_spline.rs:255-274) */
#define NDI_SB_NOT_A_KNOT 0
#define NDI_SB_NATURAL 1
#define NDI_SB_CLAMPED 2
#define NDI_SB_FIRST_DERIV 3
#define NDI_SB_SECOND_DERIV 4

/* enum Extrapolate (cubic_spline.rs:219-224) */
#define NDI_EXTRAP_NO 0
#define NDI_EXTRAP_YES 1
#define NDI_EXTRAP_PERIODIC 2

/* create flags */
#define NDI_ASSUME_VALID 1u    /* skip the strict-rising check: Interp1D::new_unchecked (interp1d/mod.rs:363) */
#define NDI_DEVICE_POINTERS 2u /* x / y / data are device pointers on the current device (copied D2D) */
#define NDI_BORROW 4u          /* with NDI_DEVICE_POINTERS: keep the caller's buffers instead of copying
                                  (the Interp1DView / ViewRepr case, interp1d/aliases.rs); caller keeps them alive
                                  AND unchanged: create() derives search tables from the grid and classifies the
                                  value range of the data (which division sequence the kernels may use) */

/* lower-index search strategy, for measurement; NDI_SEARCH_AUTO is what production uses */
#define NDI_SEARCH_AUTO 0
#define NDI_SEARCH_BINARY_GLOBAL 1 /* branch-free binary search, grid read through L1/L2 */
#define NDI_SEARCH_BINARY_SMEM 2   /* grid staged into shared memory by a bulk (TMA) copy */
#define NDI_SEARCH_UNIFORM_GUESS 3 /* O(1) even-spacing guess (vector_extensions.rs:68-90) + verify, binary fallback */
#define NDI_SEARCH_BUCKET_LUT 4    /* O(1) expected on any grid: per-handle bucket table + exact finish on the grid */
#define NDI_SEARCH_MERGE 5         /* sorted batches: a warp searches its smallest and largest query, the rest bisect inside that bracket */

/* value of the device error word when no query failed */
#define NDI_ERR_WORD_NONE UINT64_MAX

typedef struct ndi_interp1d ndi_interp1d;
typedef struct ndi_interp2d ndi_interp2d;

/* ---- runtime ---------------------------------------------------------------------------- */
const char* ndi_version_string(void);
/* message of the last failing call on this thread (CUDA error text or argument complaint) */
const char* ndi_last_error_message(void);
ndi_status ndi_device_count(int32_t* count);
ndi_status ndi_set_device(int32_t device); /* one process per GPU: call once with LOCAL_RANK */
ndi_status ndi_get_device(int32_t* device);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t ndi_kernel_launch_count(void);

/* ---- src/vector_extensions.rs ------------------------------------------------------------ */
/* VectorExtensions::monotonic_prop (vector_extensions.rs:40-53, :115-198).  `stride` is in
 * elements and may be negative (x then points at the FIRST logical element); n <= 1 gives
 * NDI_MONO_NOT_MONOTONIC.  The classification itself runs on the device. */
ndi_status ndi_monotonic_prop(ndi_dtype dtype, const void* x, int64_t n, int64_t stride, int32_t* prop);

/* VectorExtensions::get_lower_index for a batch (vector_extensions.rs:55-111): idx[i] is the
 * unique i in [0, n-2] with grid[i] <= q < grid[i+1], clamped at both ends.  A NaN query gives
 * NDI_NAN_QUERY with *first_bad = its index (the reference panics there). */
ndi_status ndi_lower_index(ndi_dtype dtype, const void* grid, int64_t n, const void* q, int64_t nq,
                           int64_t* idx, int64_t* first_bad);
ndi_status ndi_lower_index_dev(ndi_dtype dtype, const void* grid_dev, int64_t n, const void* q_dev, int64_t nq,
                               int64_t* idx_dev, uint64_t* err_word_dev, int32_t search_mode, void* stream);

/* ---- src/interp1d ------------------------------------------------------------------------ */
/* Interp1DBuilder::build data upload (interp1d/mod.rs:443-476).  x: n grid values, data: (n, w).
 * Runs the strict-rising check on the device unless NDI_ASSUME_VALID; n >= 2 required.  Shape
 * checks and their order (ndim, MINIMUM_DATA_LENGHT, monotonic, x.len == data.shape[0]) are
 * host logic of the caller (see the host mirrors), not data-parallel work. */
ndi_status ndi_interp1d_create(ndi_dtype dtype, const void* x, int64_t n, const void* data, int64_t w,
                               uint32_t flags, ndi_interp1d** out);
/* The same for ndarray VIEWS (interp1d/aliases.rs: Interp1DView; any strides, negative included --
 * tests/interp1d.rs:143-155): x is n elements `x_stride` apart, data has `ndim` (1..8) dimensions
 * with shape[0] == n and `strides` per dimension, all strides in ELEMENTS as ndarray reports them;
 * both pointers address the view's first logical element.  The view's memory is uploaded as it lies
 * and made dense on the device (a view that touches less than half of its span is gathered by the
 * library on the host instead); the handle owns the dense copy.  NDI_BORROW is rejected. */
ndi_status ndi_interp1d_create_strided(ndi_dtype dtype, const void* x, int64_t n, int64_t x_stride, const void* data,
                                       int32_t ndim, const int64_t* shape, const int64_t* strides, uint32_t flags,
                                       ndi_interp1d** out);
ndi_status ndi_interp1d_destroy(ndi_interp1d* h);
ndi_status ndi_interp1d_info(const ndi_interp1d* h, ndi_dtype* dtype, int64_t* n, int64_t* w, int32_t* has_spline,
                             int32_t* device);
ndi_status ndi_interp1d_set_search_mode(ndi_interp1d* h, int32_t search_mode);
/* device addresses of the tables the handle holds (x: n, data: n*w, a/b: (n-1)*w or NULL) */
ndi_status ndi_interp1d_device_ptrs(const ndi_interp1d* h, const void** x_dev, const void** data_dev,
                                    const void** a_dev, const void** b_dev);
/* copy of the handle's tables on another device of this process (peer copy over NVLink) */
ndi_status ndi_interp1d_clone_to_device(const ndi_interp1d* h, int32_t device, ndi_interp1d** out);

/* Linear::interp_into over a query batch (linear.rs:73-98 x interp1d/mod.rs:272-343).
 * out: (nq, w).  extrapolate == 0: a query outside [x[0], x[n-1]] (or NaN) stops the batch with
 * NDI_OUT_OF_BOUNDS.  extrapolate != 0: only a NaN query fails, with NDI_NAN_QUERY. */
ndi_status ndi_interp1d_linear(const ndi_interp1d* h, const void* q, int64_t nq, int32_t extrapolate, void* out,
                               int64_t* first_bad);
ndi_status ndi_interp1d_linear_dev(const ndi_interp1d* h, const void* q_dev, int64_t nq, int32_t extrapolate,
                                   void* out_dev, uint64_t* err_word_dev, void* stream);

/* CubicSpline::calc_coefficients (cubic_spline.rs:310-368) = solve_for_k + thomas + a/b.
 * For NDI_BC_INDIVIDUAL the four arrays have one entry per trailing column (w entries, values in
 * the handle's dtype; cubic_spline.rs:332-347, :370-403); otherwise pass NULL.  n >= 3 required.
 * NDI_PERIODIC_MISMATCH sets *bad_column to the first column with data[0] != data[n-1]. */
ndi_status ndi_interp1d_spline_build(ndi_interp1d* h, int32_t bc_kind, const int32_t* left_kind,
                                     const void* left_val, const int32_t* right_kind, const void* right_val,
                                     int64_t* bad_column);
/* How ndi_interp1d_spline_build solves the tridiagonal system (cubic_spline.rs:409-721).
 *   NDI_BUILD_SEQUENTIAL  the reference's elimination order, one serial Thomas sweep per column: coefficients
 *                         bit-identical to the reference arithmetic; chain-latency-bound on long columns.
 *   NDI_BUILD_ROWSPLIT    `levels` steps of parallel cyclic reduction, then 2^levels interleaved Thomas solves per
 *                         column (csrc/ndi_rowsplit.cu); different rounding, inside north_star's 1e-12 (f64) /
 *                         1e-5 (f32) bars, bit-identical to the oracle's specification of the same scheme.
 *                         levels == 0 lets the library choose; a request is capped so every system keeps two rows.
 *   NDI_BUILD_PARTITION   rows cut into blocks of `levels` rows (0: 32; 3 .. 32) by single separator rows: every
 *                         (block, column) pair is solved in registers, the separators' equations form a system
 *                         `levels` times shorter that is treated the same way (csrc/ndi_partition.cu); different
 *                         rounding (fused multiply-adds), inside the same bars, bit-identical to the oracle's
 *                         specification of the same scheme.
 *   NDI_BUILD_AUTO        partition (blocks of 32 rows) for tables of 1024 rows or more, the reference's order
 *                         otherwise (default) -- and also where a NotAKnot row on the right meets a grid whose last
 *                         step is about 0.55 of the one before it: the reference's system (cubic_spline.rs:635) is
 *                         then nearly singular and only its own order of operations reproduces its result.
 * ndi_interp1d_build_info reports how the current coefficients were built: 0 reference order, L > 0 row-split with L
 * levels, -m < 0 partition with blocks of m rows. */
#define NDI_BUILD_AUTO 0
#define NDI_BUILD_SEQUENTIAL 1
#define NDI_BUILD_ROWSPLIT 2
#define NDI_BUILD_PARTITION 3
ndi_status ndi_interp1d_set_build_mode(ndi_interp1d* h, int32_t mode, int32_t levels);
ndi_status ndi_interp1d_build_info(const ndi_interp1d* h, int32_t* rowsplit_levels);
/* spline coefficient arrays a, b: (n-1, w) each, copied to host (CubicSplineStrategy, cubic_spline.rs:94-102) */
ndi_status ndi_interp1d_spline_coeffs(const ndi_interp1d* h, void* a, void* b);
/* install externally computed coefficients (device or host pointers per NDI_DEVICE_POINTERS) */
ndi_status ndi_interp1d_spline_set_coeffs(ndi_interp1d* h, const void* a, const void* b, uint32_t flags);

/* CubicSplineStrategy::interp_into over a query batch (cubic_spline.rs:791-830). */
ndi_status ndi_interp1d_cubic(const ndi_interp1d* h, const void* q, int64_t nq, int32_t extrap_mode, void* out,
                              int64_t* first_bad);
ndi_status ndi_interp1d_cubic_dev(const ndi_interp1d* h, const void* q_dev, int64_t nq, int32_t extrap_mode,
                                  void* out_dev, uint64_t* err_word_dev, void* stream);

/* ---- derivatives (NOT in the reference; scipy.interpolate.CubicSpline.__call__(x, nu)) ------------ */
/* Query handling is exactly that of the value call for the same handle and mode: the same range check, periodic
 * wrap (NDI_EXTRAP_PERIODIC), NaN handling, lower-index search, error statuses and untouched rows.  So a query on
 * an interior knot x[i] gets the derivative of interval i (the right-hand one, as scipy), a query at x[n-1] that of
 * interval n-2 at t = 1, and an extrapolated query that of the edge interval's polynomial.
 * Cubic spline, order 1 or 2 (any other order: NDI_INVALID_ARGUMENT; order 0 is ndi_interp1d_cubic), with i, t, a, b
 * as in the value call, h = x[i+1] - x[i], every operation rounded on its own:
 *     cur = a (1-t) + b t,  ba = b - a
 *     order 1:  (((y[i+1] - y[i]) + ((1-t) - t) cur) + (t (1-t)) ba) / h
 *     order 2:  ((2 (((1-t) - t) ba - cur)) / h) / h
 * Linear, order 1 only: (y[i+1] - y[i]) / (x[i+1] - x[i]), the slope term of linear.rs:29-36 in the handle's dtype
 * (integers wrap and truncate like the value call; a zero quotient keeps IEEE's sign). */
ndi_status ndi_interp1d_cubic_deriv(const ndi_interp1d* h, const void* q, int64_t nq, int32_t extrap_mode,
                                    int32_t order, void* out, int64_t* first_bad);
ndi_status ndi_interp1d_cubic_deriv_dev(const ndi_interp1d* h, const void* q_dev, int64_t nq, int32_t extrap_mode,
                                        int32_t order, void* out_dev, uint64_t* err_word_dev, void* stream);
ndi_status ndi_interp1d_linear_deriv(const ndi_interp1d* h, const void* q, int64_t nq, int32_t extrapolate,
                                     void* out, int64_t* first_bad);
ndi_status ndi_interp1d_linear_deriv_dev(const ndi_interp1d* h, const void* q_dev, int64_t nq, int32_t extrapolate,
                                         void* out_dev, uint64_t* err_word_dev, void* stream);

/* ---- src/interp2d ------------------------------------------------------------------------ */
/* Interp2DBuilder::build data upload (interp2d/mod.rs:468-518).  x: n, y: m, data: (n, m, w).
 * NDI_NOT_MONOTONIC reports the failing axis in the message ("x-axis" before "y-axis"). */
ndi_status ndi_interp2d_create(ndi_dtype dtype, const void* x, int64_t n, const void* y, int64_t m, const void* data,
                               int64_t w, uint32_t flags, ndi_interp2d** out);
/* strided views, as ndi_interp1d_create_strided: shape[0] == n, shape[1] == m, ndim in 2..8 */
ndi_status ndi_interp2d_create_strided(ndi_dtype dtype, const void* x, int64_t n, int64_t x_stride, const void* y,
                                       int64_t m, int64_t y_stride, const void* data, int32_t ndim, const int64_t* shape,
                                       const int64_t* strides, uint32_t flags, ndi_interp2d** out);
ndi_status ndi_interp2d_destroy(ndi_interp2d* h);
ndi_status ndi_interp2d_info(const ndi_interp2d* h, ndi_dtype* dtype, int64_t* n, int64_t* m, int64_t* w,
                             int32_t* device);
ndi_status ndi_interp2d_set_search_mode(ndi_interp2d* h, int32_t search_mode);
ndi_status ndi_interp2d_device_ptrs(const ndi_interp2d* h, const void** x_dev, const void** y_dev,
                                    const void** data_dev);
ndi_status ndi_interp2d_clone_to_device(const ndi_interp2d* h, int32_t device, ndi_interp2d** out);
/* Locality binning of query batches: the batch loop of interp2d/mod.rs:255-307 is order-independent,
 * so a launch may group the queries by table band before evaluating them (csrc/ndi_bin.cu); results
 * and error reporting are unchanged.  AUTO bins when the table exceeds L2 and the batch is large.
 * band_rows > 0 fixes the band height in grid intervals (0: sized from L2).
 * NDI_BIN_SWEEP: the batch is not reordered; the launch walks it once per band of band_rows intervals (at most 16
 * bands, coarsened otherwise) and each sweep evaluates only that band's queries, compacted into full tiles
 * (csrc/ndi_sweep.cu; rows of 16 / 32 / 64 / 128 bytes, else the direct kernel).  Less DRAM traffic, not less time on
 * B200 (C4: 1.36 GB instead of 3.14 GB, 0.58 ms instead of 0.54 ms), so AUTO never picks it. */
enum { NDI_BIN_AUTO = 0, NDI_BIN_OFF = 1, NDI_BIN_ON = 2, NDI_BIN_SWEEP = 3 };
ndi_status ndi_interp2d_set_binning(ndi_interp2d* h, int32_t mode, int32_t band_rows);

/* Bilinear::interp_into over a query batch (bilinear.rs:64-99 x interp2d/mod.rs:215-307).
 * *bad_axis: 0 = x failed, 1 = y failed (x is checked first, bilinear.rs:71-80). */
ndi_status ndi_interp2d_bilinear(const ndi_interp2d* h, const void* qx, const void* qy, int64_t nq,
                                 int32_t extrapolate, void* out, int64_t* first_bad, int32_t* bad_axis);
/* error word = 2 * query_index + axis */
ndi_status ndi_interp2d_bilinear_dev(const ndi_interp2d* h, const void* qx_dev, const void* qy_dev, int64_t nq,
                                     int32_t extrapolate, void* out_dev, uint64_t* err_word_dev, void* stream);

/* ---- one interpolator on several devices of one process ------------------------------------------- */
/* SURVEY.md section 8(b) `ndi_replicate`: the handle's tables (grid, data, spline coefficients, search aids) are
 * peer-copied to every listed device of this process (the handle's own device may be in the list and is then used
 * as it is).  A group call takes HOST pointers like the single-device entry point it replaces -- the batch loops of
 * interp1d/mod.rs:272-343 and interp2d/mod.rs:215-307 -- cuts the batch into contiguous blocks of queries, one per
 * device, and evaluates the blocks concurrently (one worker thread, two streams and one set of pinned staging
 * buffers per device; no collective).  Error semantics are those of the single-device call for the WHOLE batch:
 * *first_bad is the first failing query in row-major order whichever block holds it, and rows at and after it stay
 * untouched in every block (a query-only pre-pass runs on all blocks before any row is written).  Batches below
 * 32768 queries stay on the first device.  Build the spline BEFORE replicating.  The handle must outlive the group. */
typedef struct ndi_interp1d_group ndi_interp1d_group;
typedef struct ndi_interp2d_group ndi_interp2d_group;
ndi_status ndi_interp1d_replicate(const ndi_interp1d* h, const int32_t* devices, int32_t ndev, ndi_interp1d_group** out);
ndi_status ndi_interp1d_group_destroy(ndi_interp1d_group* g);
ndi_status ndi_interp1d_group_size(const ndi_interp1d_group* g, int32_t* ndev);
ndi_status ndi_interp1d_group_linear(ndi_interp1d_group* g, const void* q, int64_t nq, int32_t extrapolate, void* out,
                                     int64_t* first_bad);
ndi_status ndi_interp1d_group_cubic(ndi_interp1d_group* g, const void* q, int64_t nq, int32_t extrap_mode, void* out,
                                    int64_t* first_bad);
/* the derivative calls above, on a group */
ndi_status ndi_interp1d_group_linear_deriv(ndi_interp1d_group* g, const void* q, int64_t nq, int32_t extrapolate,
                                           void* out, int64_t* first_bad);
ndi_status ndi_interp1d_group_cubic_deriv(ndi_interp1d_group* g, const void* q, int64_t nq, int32_t extrap_mode,
                                          int32_t order, void* out, int64_t* first_bad);
ndi_status ndi_interp2d_replicate(const ndi_interp2d* h, const int32_t* devices, int32_t ndev, ndi_interp2d_group** out);
ndi_status ndi_interp2d_group_destroy(ndi_interp2d_group* g);
ndi_status ndi_interp2d_group_bilinear(ndi_interp2d_group* g, const void* qx, const void* qy, int64_t nq,
                                       int32_t extrapolate, void* out, int64_t* first_bad, int32_t* bad_axis);

/* ---- self-test ------------------------------------------------------------------------------ */
/* The Linear / Bilinear kernels form the reciprocal of a query's divisor once and finish every
 * quotient with two fused multiply-adds (csrc/ndi_device.cuh: rcp_refined, div_by) instead of a full
 * IEEE division per element (linear.rs:32).  This entry point counts the operand pairs for which that
 * differs from the correctly rounded quotient: a = 1.m_a * 2^a_exp for m_a in [a_mant_begin,
 * a_mant_begin + a_mant_count), b = 1.m_b * 2^b_exp for every 23-bit m_b.  Must report 0. */
ndi_status ndi_selftest_fdiv(uint32_t a_mant_begin, uint32_t a_mant_count, int32_t a_exp, int32_t b_exp,
                             uint64_t* mismatches);

/* f64 counterpart for the spline sweeps (cubic_spline.rs:716 divides by a matrix entry shared by all
 * columns; csrc/ndi_device.cuh: Hoisted<double>): counts mismatches against the correctly rounded
 * quotient over about `pairs` pseudo-random operand pairs covering every exponent.  Must report 0. */
ndi_status ndi_selftest_ddiv(uint64_t seed, uint64_t pairs, uint64_t* mismatches);

#ifdef __cplusplus
}
#endif
#endif /* NDI_B200_H */
