"""ctypes loader for tests/deriv_oracle.cpp, the CPU specification of the derivative calls.

TEST INFRASTRUCTURE ONLY (tests and scripts/bench_deriv.py).  The library is compiled with the oracle's flags into a
directory under the system temporary directory, keyed by the sources' hash, so the repository tree stays untouched.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SOURCES = [os.path.join(_HERE, "deriv_oracle.cpp"), os.path.join(_ROOT, "oracle", "ndi_oracle.cpp")]


def _oracle_cxxflags():
    """the compiler flags of oracle/Makefile (one rounding per operation, no contraction into FMA), read from it so the
    specification is always built exactly like the oracle it includes"""
    for line in open(os.path.join(_ROOT, "oracle", "Makefile")):
        if line.startswith("CXXFLAGS"):
            return line.split("=", 1)[1].split()
    raise RuntimeError("oracle/Makefile has no CXXFLAGS line")


CXXFLAGS = _oracle_cxxflags() + ["-shared"]

_SFX = {np.dtype(np.float32): "f32", np.dtype(np.float64): "f64", np.dtype(np.int32): "i32",
        np.dtype(np.int64): "i64", np.dtype(np.uint32): "u32", np.dtype(np.uint64): "u64"}

_lib = None


def build():
    h = hashlib.sha256()
    for s in _SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(CXXFLAGS).encode())
    d = os.path.join(tempfile.gettempdir(), f"ndi_deriv_oracle_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    so = os.path.join(d, f"libndi_deriv_oracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CXX", "g++")] + CXXFLAGS + ["-o", tmp, _SOURCES[0]])
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def cubic_deriv(x, data, a, b, q, extrap_mode, order, out=None):
    """(status, out, first_bad) of ndi_interp1d_cubic_deriv's specification on the given coefficients"""
    x = np.ascontiguousarray(x)
    data = np.ascontiguousarray(data, dtype=x.dtype)
    a = np.ascontiguousarray(a, dtype=x.dtype)
    b = np.ascontiguousarray(b, dtype=x.dtype)
    q = np.ascontiguousarray(q, dtype=x.dtype)
    w = int(np.prod(data.shape[1:], dtype=np.int64))
    if out is None:
        out = np.zeros(q.shape + data.shape[1:], dtype=x.dtype)
    bad = C.c_int64(-1)
    st = getattr(lib(), f"ora_interp1d_cubic_deriv_{_SFX[x.dtype]}")(
        _p(x), C.c_int64(len(x)), _p(data), _p(a), _p(b), C.c_int64(w), _p(q), C.c_int64(q.size),
        C.c_int32(extrap_mode), C.c_int32(order), _p(out), C.byref(bad))
    return st, out, bad.value


def linear_deriv(x, data, q, extrapolate, out=None):
    """(status, out, first_bad) of ndi_interp1d_linear_deriv's specification"""
    x = np.ascontiguousarray(x)
    data = np.ascontiguousarray(data, dtype=x.dtype)
    q = np.ascontiguousarray(q, dtype=x.dtype)
    w = int(np.prod(data.shape[1:], dtype=np.int64))
    if out is None:
        out = np.zeros(q.shape + data.shape[1:], dtype=x.dtype)
    bad = C.c_int64(-1)
    st = getattr(lib(), f"ora_interp1d_linear_deriv_{_SFX[x.dtype]}")(
        _p(x), C.c_int64(len(x)), _p(data), C.c_int64(w), _p(q), C.c_int64(q.size), C.c_int32(int(extrapolate)),
        _p(out), C.byref(bad))
    return st, out, bad.value
