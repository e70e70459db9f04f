"""ctypes binding of include/ndi_b200.h (the C ABI of the CUDA path).

There is no CPU fallback: importing this module without the built library, or calling into it
without a CUDA device, fails loudly.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# NDI_B200_LIB: A/B-test another in-tree build of the same sources (see build.py --out / --define)
SO_PATH = os.environ.get("NDI_B200_LIB") or os.path.join(_HERE, "libndi_b200.so")

OK, OUT_OF_BOUNDS, NAN_QUERY, PERIODIC_MISMATCH, INVALID_ARGUMENT, NOT_MONOTONIC, NO_SPLINE, UNSUPPORTED_DTYPE, \
    NO_DEVICE = range(9)
CUDA_ERROR = 100
F32, F64, I32, I64, U32, U64 = 0, 1, 2, 3, 4, 5
ASSUME_VALID, DEVICE_POINTERS, BORROW = 1, 2, 4
SEARCH_AUTO, SEARCH_BINARY_GLOBAL, SEARCH_BINARY_SMEM, SEARCH_UNIFORM_GUESS, SEARCH_BUCKET_LUT, SEARCH_MERGE = 0, 1, 2, 3, 4, 5
EXTRAP_NO, EXTRAP_YES, EXTRAP_PERIODIC = 0, 1, 2
BIN_AUTO, BIN_OFF, BIN_ON, BIN_SWEEP = 0, 1, 2, 3
BUILD_AUTO, BUILD_SEQUENTIAL, BUILD_ROWSPLIT, BUILD_PARTITION = 0, 1, 2, 3
ERR_WORD_NONE = 2 ** 64 - 1

DTYPES = {np.dtype(np.float32): F32, np.dtype(np.float64): F64, np.dtype(np.int32): I32,
          np.dtype(np.int64): I64, np.dtype(np.uint32): U32, np.dtype(np.uint64): U64}

_vp, _i64, _i32, _u32, _u64 = C.c_void_p, C.c_int64, C.c_int32, C.c_uint32, C.c_uint64
_pi64, _pi32 = C.POINTER(C.c_int64), C.POINTER(C.c_int32)

# every symbol include/ndi_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "ndi_version_string": (C.c_char_p, []),
    "ndi_last_error_message": (C.c_char_p, []),
    "ndi_device_count": (_i32, [_pi32]),
    "ndi_set_device": (_i32, [_i32]),
    "ndi_get_device": (_i32, [_pi32]),
    "ndi_kernel_launch_count": (_u64, []),
    "ndi_monotonic_prop": (_i32, [_i32, _vp, _i64, _i64, _pi32]),
    "ndi_lower_index": (_i32, [_i32, _vp, _i64, _vp, _i64, _vp, _pi64]),
    "ndi_lower_index_dev": (_i32, [_i32, _vp, _i64, _vp, _i64, _vp, _vp, _i32, _vp]),
    "ndi_interp1d_create": (_i32, [_i32, _vp, _i64, _vp, _i64, _u32, C.POINTER(_vp)]),
    "ndi_interp1d_create_strided": (_i32, [_i32, _vp, _i64, _i64, _vp, _i32, _vp, _vp, _u32, C.POINTER(_vp)]),
    "ndi_interp1d_destroy": (_i32, [_vp]),
    "ndi_interp1d_info": (_i32, [_vp, _pi32, _pi64, _pi64, _pi32, _pi32]),
    "ndi_interp1d_set_search_mode": (_i32, [_vp, _i32]),
    "ndi_interp1d_device_ptrs": (_i32, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "ndi_interp1d_clone_to_device": (_i32, [_vp, _i32, C.POINTER(_vp)]),
    "ndi_interp1d_linear": (_i32, [_vp, _vp, _i64, _i32, _vp, _pi64]),
    "ndi_interp1d_linear_dev": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "ndi_interp1d_spline_build": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _pi64]),
    "ndi_interp1d_set_build_mode": (_i32, [_vp, _i32, _i32]),
    "ndi_interp1d_build_info": (_i32, [_vp, _pi32]),
    "ndi_interp1d_spline_coeffs": (_i32, [_vp, _vp, _vp]),
    "ndi_interp1d_spline_set_coeffs": (_i32, [_vp, _vp, _vp, _u32]),
    "ndi_interp1d_cubic": (_i32, [_vp, _vp, _i64, _i32, _vp, _pi64]),
    "ndi_interp1d_cubic_dev": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "ndi_interp1d_cubic_deriv": (_i32, [_vp, _vp, _i64, _i32, _i32, _vp, _pi64]),
    "ndi_interp1d_cubic_deriv_dev": (_i32, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp]),
    "ndi_interp1d_linear_deriv": (_i32, [_vp, _vp, _i64, _i32, _vp, _pi64]),
    "ndi_interp1d_linear_deriv_dev": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "ndi_interp2d_create": (_i32, [_i32, _vp, _i64, _vp, _i64, _vp, _i64, _u32, C.POINTER(_vp)]),
    "ndi_interp2d_create_strided": (_i32, [_i32, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i32, _vp, _vp, _u32,
                                           C.POINTER(_vp)]),
    "ndi_interp2d_destroy": (_i32, [_vp]),
    "ndi_interp2d_info": (_i32, [_vp, _pi32, _pi64, _pi64, _pi64, _pi32]),
    "ndi_interp2d_set_search_mode": (_i32, [_vp, _i32]),
    "ndi_interp2d_device_ptrs": (_i32, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "ndi_interp2d_clone_to_device": (_i32, [_vp, _i32, C.POINTER(_vp)]),
    "ndi_selftest_fdiv": (_i32, [_u32, _u32, _i32, _i32, C.POINTER(_u64)]),
    "ndi_selftest_ddiv": (_i32, [_u64, _u64, C.POINTER(_u64)]),
    "ndi_interp2d_set_binning": (_i32, [_vp, _i32, _i32]),
    "ndi_interp2d_bilinear": (_i32, [_vp, _vp, _vp, _i64, _i32, _vp, _pi64, _pi32]),
    "ndi_interp2d_bilinear_dev": (_i32, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "ndi_interp1d_replicate": (_i32, [_vp, _pi32, _i32, C.POINTER(_vp)]),
    "ndi_interp1d_group_destroy": (_i32, [_vp]),
    "ndi_interp1d_group_size": (_i32, [_vp, _pi32]),
    "ndi_interp1d_group_linear": (_i32, [_vp, _vp, _i64, _i32, _vp, _pi64]),
    "ndi_interp1d_group_cubic": (_i32, [_vp, _vp, _i64, _i32, _vp, _pi64]),
    "ndi_interp1d_group_linear_deriv": (_i32, [_vp, _vp, _i64, _i32, _vp, _pi64]),
    "ndi_interp1d_group_cubic_deriv": (_i32, [_vp, _vp, _i64, _i32, _i32, _vp, _pi64]),
    "ndi_interp2d_replicate": (_i32, [_vp, _pi32, _i32, C.POINTER(_vp)]),
    "ndi_interp2d_group_destroy": (_i32, [_vp]),
    "ndi_interp2d_group_bilinear": (_i32, [_vp, _vp, _vp, _i64, _i32, _vp, _pi64, _pi32]),
}

_lib = None


class NdiLibraryError(RuntimeError):
    """the CUDA library is missing, has no device, or a CUDA call failed"""


def load():
    """dlopen the in-tree library and type every entry point (no GPU needed for this)"""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise NdiLibraryError(
            f"{SO_PATH} is missing: build it with `python -m ndarray_interp_b200.build` "
            "(there is no CPU fallback)")
    lib = C.CDLL(SO_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library disagree
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


_device_checked = False


def require_device():
    global _device_checked
    lib = load()
    if not _device_checked:
        n = C.c_int32(0)
        st = lib.ndi_device_count(C.byref(n))
        if st != OK or n.value < 1:
            raise NdiLibraryError("no CUDA device visible: ndarray_interp_b200 runs on B200 only, "
                                  "there is no CPU fallback (" + last_error() + ")")
        _device_checked = True
    return lib


def last_error():
    return load().ndi_last_error_message().decode("utf-8", "replace")


def check(st):
    """turn a non-domain status into an exception"""
    if st >= CUDA_ERROR or st in (INVALID_ARGUMENT, UNSUPPORTED_DTYPE, NO_DEVICE, NO_SPLINE):
        raise NdiLibraryError(f"ndi status {st}: {last_error()}")
    return st


def ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def view_args(a):
    """an ndarray view as the C ABI takes it: (array kept alive, pointer to the first logical element, shape,
    strides in elements).  numpy reports strides in bytes; a view whose byte strides are not multiples of the
    item size (never produced by slicing) is copied."""
    a = np.asarray(a)
    if any(s % a.itemsize for s in a.strides):
        a = np.ascontiguousarray(a)
    shape = (C.c_int64 * max(a.ndim, 1))(*a.shape)
    strides = (C.c_int64 * max(a.ndim, 1))(*(s // a.itemsize for s in a.strides))
    return a, C.c_void_p(a.ctypes.data), shape, strides


def is_dense(a):
    return a.flags.c_contiguous


def dtype_code(dt):
    try:
        return DTYPES[np.dtype(dt)]
    except KeyError:
        raise TypeError(f"element type {np.dtype(dt)} is not supported on the device path "
                        "(f32, f64, i32, i64, u32 and u64 are)") from None
