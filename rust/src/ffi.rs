//! Raw bindings of `include/ndi_b200.h`.  One declaration per C entry point, nothing else.
#![allow(non_camel_case_types)]
use std::ffi::{c_char, c_void};

pub type ndi_status = i32;
pub const NDI_OK: ndi_status = 0;
pub const NDI_OUT_OF_BOUNDS: ndi_status = 1;
pub const NDI_NAN_QUERY: ndi_status = 2;
pub const NDI_PERIODIC_MISMATCH: ndi_status = 3;
pub const NDI_NOT_MONOTONIC: ndi_status = 5;
pub const NDI_NO_INTEGRAL: ndi_status = 9;

pub const NDI_INTEGRAL_LINEAR: i32 = 0;
pub const NDI_INTEGRAL_CUBIC: i32 = 1;

pub const NDI_HERMITE_PCHIP: i32 = 0;
pub const NDI_HERMITE_AKIMA: i32 = 1;
pub const NDI_HERMITE_MAKIMA: i32 = 2;
pub const NDI_HERMITE_GIVEN: i32 = 3;

pub const NDI_F32: i32 = 0;
pub const NDI_F64: i32 = 1;
pub const NDI_I32: i32 = 2;
pub const NDI_I64: i32 = 3;
pub const NDI_U32: i32 = 4;
pub const NDI_U64: i32 = 5;

pub const NDI_ASSUME_VALID: u32 = 1;

#[repr(C)]
pub struct ndi_interp1d {
    _private: [u8; 0],
}
#[repr(C)]
pub struct ndi_interp2d {
    _private: [u8; 0],
}

extern "C" {
    pub fn ndi_last_error_message() -> *const c_char;
    pub fn ndi_set_device(device: i32) -> ndi_status;
    pub fn ndi_monotonic_prop(dtype: i32, x: *const c_void, n: i64, stride: i64, prop: *mut i32) -> ndi_status;
    pub fn ndi_lower_index(dtype: i32, grid: *const c_void, n: i64, q: *const c_void, nq: i64, idx: *mut i64, first_bad: *mut i64) -> ndi_status;

    pub fn ndi_interp1d_create(dtype: i32, x: *const c_void, n: i64, data: *const c_void, w: i64, flags: u32, out: *mut *mut ndi_interp1d) -> ndi_status;
    pub fn ndi_interp1d_destroy(h: *mut ndi_interp1d) -> ndi_status;
    pub fn ndi_interp1d_linear(h: *const ndi_interp1d, q: *const c_void, nq: i64, extrapolate: i32, out: *mut c_void, first_bad: *mut i64) -> ndi_status;
    pub fn ndi_interp1d_spline_build(h: *mut ndi_interp1d, bc_kind: i32, left_kind: *const i32, left_val: *const c_void, right_kind: *const i32, right_val: *const c_void, bad_column: *mut i64) -> ndi_status;
    /// spline solve: 0 auto, 1 the reference's elimination order, 2 row-split (PCR + Thomas) with `levels` reduction steps
    pub fn ndi_interp1d_set_build_mode(h: *mut ndi_interp1d, mode: i32, levels: i32) -> ndi_status;
    pub fn ndi_interp1d_build_info(h: *const ndi_interp1d, rowsplit_levels: *mut i32) -> ndi_status;
    pub fn ndi_interp1d_spline_coeffs(h: *const ndi_interp1d, a: *mut c_void, b: *mut c_void) -> ndi_status;
    pub fn ndi_interp1d_cubic(h: *const ndi_interp1d, q: *const c_void, nq: i64, extrap_mode: i32, out: *mut c_void, first_bad: *mut i64) -> ndi_status;
    /// derivatives (not in the reference): order 1 or 2 of the spline, the slope of Linear
    pub fn ndi_interp1d_cubic_deriv(h: *const ndi_interp1d, q: *const c_void, nq: i64, extrap_mode: i32, order: i32, out: *mut c_void, first_bad: *mut i64) -> ndi_status;
    pub fn ndi_interp1d_linear_deriv(h: *const ndi_interp1d, q: *const c_void, nq: i64, extrapolate: i32, out: *mut c_void, first_bad: *mut i64) -> ndi_status;
    /// definite integrals (not in the reference): the cumulative table of one kind, then integrals over (lo, hi) pairs
    pub fn ndi_interp1d_integral_build(h: *mut ndi_interp1d, kind: i32) -> ndi_status;
    pub fn ndi_interp1d_cubic_integral(h: *const ndi_interp1d, lo: *const c_void, hi: *const c_void, nq: i64, extrap_mode: i32, out: *mut c_void, first_bad: *mut i64, bad_bound: *mut i32) -> ndi_status;
    pub fn ndi_interp1d_linear_integral(h: *const ndi_interp1d, lo: *const c_void, hi: *const c_void, nq: i64, extrapolate: i32, out: *mut c_void, first_bad: *mut i64, bad_bound: *mut i32) -> ndi_status;
    /// shape-preserving cubics (not in the reference): PCHIP, Akima, makima or given slopes (`dydx`, host memory)
    pub fn ndi_interp1d_hermite_build(h: *mut ndi_interp1d, kind: i32, dydx: *const c_void, flags: u32) -> ndi_status;

    pub fn ndi_interp1d_create_strided(dtype: i32, x: *const c_void, n: i64, x_stride: i64, data: *const c_void, ndim: i32, shape: *const i64, strides: *const i64, flags: u32, out: *mut *mut ndi_interp1d) -> ndi_status;
    pub fn ndi_interp2d_create_strided(dtype: i32, x: *const c_void, n: i64, x_stride: i64, y: *const c_void, m: i64, y_stride: i64, data: *const c_void, ndim: i32, shape: *const i64, strides: *const i64, flags: u32, out: *mut *mut ndi_interp2d) -> ndi_status;
    pub fn ndi_interp2d_create(dtype: i32, x: *const c_void, n: i64, y: *const c_void, m: i64, data: *const c_void, w: i64, flags: u32, out: *mut *mut ndi_interp2d) -> ndi_status;
    pub fn ndi_interp2d_destroy(h: *mut ndi_interp2d) -> ndi_status;
    /// locality binning of query batches by table band: 0 auto, 1 off, 2 on (csrc/ndi_bin.cu), 3 band sweeps (csrc/ndi_sweep.cu)
    pub fn ndi_interp2d_set_binning(h: *mut ndi_interp2d, mode: i32, band_rows: i32) -> ndi_status;
    pub fn ndi_interp2d_bilinear(h: *const ndi_interp2d, qx: *const c_void, qy: *const c_void, nq: i64, extrapolate: i32, out: *mut c_void, first_bad: *mut i64, bad_axis: *mut i32) -> ndi_status;
}

/// text of the last failing call on this thread
pub fn last_error() -> String {
    unsafe { std::ffi::CStr::from_ptr(ndi_last_error_message()).to_string_lossy().into_owned() }
}
