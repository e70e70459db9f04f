"""Build the CUDA extension in-tree: ndarray_interp_b200/libndi_b200.so (sm_100a only).

    python -m ndarray_interp_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  Flags that matter for parity (SURVEY.md section 0, fact 4):
  -fmad=false   no FMA contraction (the kernels also use explicit round-to-nearest intrinsics)
  defaults kept: -prec-div=true -prec-sqrt=true -ftz=false  (IEEE division, denormals kept)
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libndi_b200.so")
SOURCES = ["ndi_api.cu", "ndi_eval.cu", "ndi_bin.cu", "ndi_sweep.cu", "ndi_grid.cu", "ndi_spline.cu", "ndi_rowsplit.cu", "ndi_partition.cu", "ndi_integral.cu", "ndi_hermite.cu"]
HEADERS = ["ndi_device.cuh", "ndi_spline.cuh", "ndi_internal.h", os.path.join("..", "..", "include", "ndi_b200.h")]

NVCC_FLAGS = [
    "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-fmad=false", "-Xcompiler", "-fPIC",
    "-Xcompiler", "-pthread", "--expt-relaxed-constexpr",
]


def nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def stale():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), out=None):
    """defines / out: build a variant (-DNAME=VALUE ...) into another .so for A/B measurements"""
    so = os.path.join(HERE, out) if out else SO
    if not out and not force and not stale():
        return SO
    objs = []
    procs = []
    tag = ("_" + os.path.splitext(os.path.basename(out))[0]) if out else ""
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for s in SOURCES:
        o = os.path.join(HERE, "build", s.replace(".cu", tag + ".o"))
        cmd = ([nvcc()] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else [])
               + ["-c", os.path.join(CSRC, s), "-o", o])
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {s} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    link = [nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-o", so] + objs
    subprocess.check_call(link)
    return so


if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--define", action="append", default=[], help="NAME=VALUE, e.g. NDI_TPW_LINEAR=1")
    ap.add_argument("--out", default=None, help="variant library name, e.g. libndi_b200_v1.so")
    a = ap.parse_args()
    print(build(force=a.force, verbose=a.verbose, defines=a.define, out=a.out))
