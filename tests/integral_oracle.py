"""ctypes loader for tests/integral_oracle.cpp, the CPU specification of the integral calls.

TEST INFRASTRUCTURE ONLY (tests and scripts/bench_integral.py).  Built like tests/deriv_oracle.cpp, with the compiler
flags deriv_oracle.py reads from oracle/Makefile, into a directory under the system temporary directory keyed by the
sources' hash, so the repository tree stays untouched.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import deriv_oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = [os.path.join(_HERE, "integral_oracle.cpp"), os.path.join(os.path.dirname(_HERE), "oracle", "ndi_oracle.cpp")]
_SFX = {np.dtype(np.float32): "f32", np.dtype(np.float64): "f64"}

_lib = None


def build():
    h = hashlib.sha256()
    for s in _SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(deriv_oracle.CXXFLAGS).encode())
    d = os.path.join(tempfile.gettempdir(), f"ndi_integral_oracle_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    so = os.path.join(d, f"libndi_integral_oracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CXX", "g++")] + deriv_oracle.CXXFLAGS + ["-o", tmp, _SOURCES[0]])
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


_p = deriv_oracle._p


def table(x, data, a=None, b=None):
    """the cumulative table C (n, ...data.shape[1:]) of ndi_interp1d_integral_build (a, b None: Linear)"""
    x = np.ascontiguousarray(x)
    data = np.ascontiguousarray(data, dtype=x.dtype)
    a = None if a is None else np.ascontiguousarray(a, dtype=x.dtype)
    b = None if b is None else np.ascontiguousarray(b, dtype=x.dtype)
    w = int(np.prod(data.shape[1:], dtype=np.int64))
    cum = np.zeros(data.shape, dtype=x.dtype)
    getattr(lib(), f"ora_integral_table_{_SFX[x.dtype]}")(_p(x), C.c_int64(len(x)), _p(data), _p(a), _p(b), C.c_int64(w),
                                                          _p(cum))
    return cum


def integrate(x, data, a, b, lo, hi, mode, out=None, cum=None):
    """(status, out, first_bad, bad_bound) of the integral calls' specification (a, b None: Linear, mode = extrapolate)"""
    x = np.ascontiguousarray(x)
    data = np.ascontiguousarray(data, dtype=x.dtype)
    if cum is None:
        cum = table(x, data, a, b)
    a = None if a is None else np.ascontiguousarray(a, dtype=x.dtype)
    b = None if b is None else np.ascontiguousarray(b, dtype=x.dtype)
    lo = np.ascontiguousarray(lo, dtype=x.dtype)
    hi = np.ascontiguousarray(hi, dtype=x.dtype)
    w = int(np.prod(data.shape[1:], dtype=np.int64))
    if out is None:
        out = np.zeros(lo.shape + data.shape[1:], dtype=x.dtype)
    bad, bound = C.c_int64(-1), C.c_int32(-1)
    st = getattr(lib(), f"ora_integrate_{_SFX[x.dtype]}")(
        _p(x), C.c_int64(len(x)), _p(data), _p(a), _p(b), _p(np.ascontiguousarray(cum)), C.c_int64(w), _p(lo), _p(hi),
        C.c_int64(lo.size), C.c_int32(int(mode)), _p(out), C.byref(bad), C.byref(bound))
    return st, out, bad.value, bound.value
