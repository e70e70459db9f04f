"""ctypes loader for tests/hermite_oracle.cpp, the CPU specification of ndi_interp1d_hermite_build.

TEST INFRASTRUCTURE ONLY (tests and scripts/bench_hermite.py).  Built like tests/deriv_oracle.cpp, with the compiler
flags deriv_oracle.py reads from oracle/Makefile, into a directory under the system temporary directory keyed by the
source's hash, so the repository tree stays untouched.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import deriv_oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCE = os.path.join(_HERE, "hermite_oracle.cpp")
_SFX = {np.dtype(np.float32): "f32", np.dtype(np.float64): "f64"}

PCHIP, AKIMA, MAKIMA, GIVEN = 0, 1, 2, 3

_lib = None


def build():
    h = hashlib.sha256()
    h.update(open(_SOURCE, "rb").read())
    h.update(" ".join(deriv_oracle.CXXFLAGS).encode())
    d = os.path.join(tempfile.gettempdir(), f"ndi_hermite_oracle_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    so = os.path.join(d, f"libndi_hermite_oracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CXX", "g++")] + deriv_oracle.CXXFLAGS + ["-o", tmp, _SOURCE])
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


_p = deriv_oracle._p


def hermite(x, data, kind, dydx=None):
    """(d, a, b) of the specification: knot slopes d (n, ...) and coefficients a, b (n-1, ...) in x's dtype"""
    x = np.ascontiguousarray(x)
    data = np.ascontiguousarray(data, dtype=x.dtype)
    if dydx is not None:
        dydx = np.ascontiguousarray(dydx, dtype=x.dtype)
    n = len(x)
    w = int(np.prod(data.shape[1:], dtype=np.int64))
    d = np.zeros(data.shape, dtype=x.dtype)
    a = np.zeros((n - 1,) + data.shape[1:], dtype=x.dtype)
    b = np.zeros_like(a)
    st = getattr(lib(), f"ora_hermite_{_SFX[x.dtype]}")(_p(x), C.c_int64(n), _p(data), C.c_int64(w), C.c_int32(kind),
                                                        _p(dydx), _p(d), _p(a), _p(b))
    if st != 0:
        raise ValueError(f"hermite specification: bad arguments (status {st})")
    return d, a, b
