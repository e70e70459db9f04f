#!/usr/bin/env python3
"""Shape-preserving cubic builds (ndi_interp1d_hermite_build) next to the spline build on the same handle, one GPU.

    python scripts/bench_hermite.py [--steps 20] [--warmup 3] [--out FILE.json] [--profile DIR]

Shapes: the three build shapes of scripts/bench_integral.py -- C2 (4096 x 1024 f64), (65536 x 64) f64 and
(4096 x 131072) f32 -- and a tall single column (2^22 x 1) f64.  At each shape every kind (PCHIP, Akima, makima, given
slopes from device memory) alternates call by call with ndi_interp1d_spline_build (NotAKnot, NDI_BUILD_AUTO) on the
same handle; each call is timed with the host clock around it (the build ends in a device synchronise), after warm-up
calls of both.  Reported: median / min ms, algorithmic bytes s (n w + 2 (n-1) w) -- y read once, a and b written --
plus n w s for the slopes (given) or for the first pass over y (Akima's maximum), and their fraction of the measured
6 443 GB/s copy peak.  y (32 MB at C2, at (65536 x 64) and at the tall shape) can stay in the 126 MB L2 between the
passes of a call; at the wide shape (2 GB) it cannot ("y_fits_l2").  The coefficients of the last call are
checked bit for bit against tests/hermite_oracle.cpp on sampled columns (all rows); for Akima the sampled columns' own
maximum of f12 stands in for the table's, which decides nothing differently unless an f12 lies between the two
thresholds (reported as a mismatch, not hidden).  The card's name and power limit are read in the same run.
--profile DIR: instead, three calls of every kind and of the spline build per shape under torch.profiler (CUDA
activities); the kernel table goes to DIR/hermite_profile.txt.  Read per-call kernel times from its "CUDA time avg"
column: the profiler can drop a record, so a total divided by 3 can be wrong.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import hermite_oracle as H  # noqa: E402
from ndarray_interp_b200 import _lib as L  # noqa: E402
from ndarray_interp_b200.interp1d import Interp1D, Pchip  # noqa: E402

PEAK_GBPS = 6443.0          # measured device copy peak (DESIGN.md section 4)
L2_BYTES = 126 * 2 ** 20
SHAPES = [("c2", np.float64, 4096, 1024), ("long", np.float64, 65536, 64), ("wide", np.float32, 4096, 131072),
          ("tall", np.float64, 1 << 22, 1)]
KINDS = {"pchip": L.HERMITE_PCHIP, "akima": L.HERMITE_AKIMA, "makima": L.HERMITE_MAKIMA, "given": L.HERMITE_GIVEN}


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def _table(dt, n, w):
    rng = np.random.default_rng(n + w)
    g = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(dt)
    y = rng.standard_normal((n, w), dtype=np.float32).astype(dt)
    d = rng.standard_normal((n, w), dtype=np.float32).astype(dt)
    return g, y, d


def _calls(ip, dydx_dev):
    lib, h = L.load(), ip._handle()
    calls = {k: (lambda k=k, v=v: lib.ndi_interp1d_hermite_build(
        h, v, C.c_void_p(dydx_dev.data_ptr()) if v == L.HERMITE_GIVEN else None,
        L.DEVICE_POINTERS if v == L.HERMITE_GIVEN else 0)) for k, v in KINDS.items()}
    calls["spline"] = lambda: lib.ndi_interp1d_spline_build(h, 0, None, None, None, None, None)
    return calls


def run_shape(name, dt, n, w, steps, warmup):
    g, y, d = _table(dt, n, w)
    s_ = np.dtype(dt).itemsize
    ip = Interp1D.new_unchecked(g, y, Pchip.new().build(g, y))
    dydx_dev = torch.from_numpy(d).cuda()
    torch.cuda.synchronize()
    calls = _calls(ip, dydx_dev)
    base_bytes = s_ * (n * w + 2 * (n - 1) * w)
    res = {"shape": name, "dtype": np.dtype(dt).name, "n": n, "w": w, "y_fits_l2": y.nbytes < L2_BYTES,
           "steps": steps, "warmup": warmup, "kinds": {}}
    rng = np.random.default_rng(7)
    cols = np.sort(rng.choice(w, min(w, 16), replace=False))
    for k, fn in calls.items():
        if k == "spline":
            continue
        for _ in range(warmup):
            L.check(fn())
            L.check(calls["spline"]())
        ts, tsp = [], []
        for _ in range(steps):               # alternate with the spline build on the same handle
            for lst, f in ((ts, fn), (tsp, calls["spline"])):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                L.check(f())
                lst.append((time.perf_counter() - t0) * 1e3)
        L.check(fn())
        a, b = ip.strategy.coefficients(ip)
        a, b = a.reshape(n - 1, w), b.reshape(n - 1, w)
        ys = np.ascontiguousarray(y.reshape(n, w)[:, cols])
        ds = np.ascontiguousarray(d.reshape(n, w)[:, cols]) if k == "given" else None
        _, wa, wb = H.hermite(g, ys, KINDS[k], ds)
        same = bool(np.array_equal(np.ascontiguousarray(a[:, cols]).view(np.uint8), wa.view(np.uint8)) and
                    np.array_equal(np.ascontiguousarray(b[:, cols]).view(np.uint8), wb.view(np.uint8)))
        nbytes = base_bytes + (s_ * n * w if k != "pchip" else 0)
        med = float(np.median(ts))
        res["kinds"][k] = {"ms_median": round(med, 4), "ms_min": round(float(np.min(ts)), 4),
                           "algorithmic_bytes": nbytes, "GBps": round(nbytes / (med * 1e-3) / 1e9, 1),
                           "fraction_of_copy_peak": round(nbytes / (med * 1e-3) / 1e9 / PEAK_GBPS, 3),
                           "spline_build_ms_median": round(float(np.median(tsp)), 4),
                           "spline_build_ms_min": round(float(np.min(tsp)), 4),
                           "oracle_bits_equal_on_sampled_columns": same}
    del dydx_dev
    torch.cuda.empty_cache()
    return res


def profile(out_dir):
    from torch.profiler import ProfilerActivity, profile as prof
    os.makedirs(out_dir, exist_ok=True)
    lines = []
    for name, dt, n, w in SHAPES:
        g, y, d = _table(dt, n, w)
        ip = Interp1D.new_unchecked(g, y, Pchip.new().build(g, y))
        dydx_dev = torch.from_numpy(d).cuda()
        calls = _calls(ip, dydx_dev)
        for fn in calls.values():
            L.check(fn())
        torch.cuda.synchronize()
        with prof(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as p:
            for _ in range(3):
                for fn in calls.values():
                    L.check(fn())
            torch.cuda.synchronize()
        # the profiler may drop a kernel record: per-call kernel time is "CUDA time avg" (total / "# of Calls")
        lines.append(f"==== {name} {np.dtype(dt).name} n={n} w={w} (3 calls of each requested; the table's '# of Calls' "
                     "counts the kernel records kept, 'CUDA time avg' is the time per record)\n")
        lines.append(p.key_averages().table(sort_by="self_device_time_total", row_limit=25, max_name_column_width=90))
        del dydx_dev
        torch.cuda.empty_cache()
    with open(os.path.join(out_dir, "hermite_profile.txt"), "w") as f:
        f.write("\n".join(lines))
    print("\n".join(lines))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    ap.add_argument("--profile", default=None, help="directory for a torch.profiler kernel table (no timing run)")
    a = ap.parse_args()
    L.require_device()
    L.check(L.load().ndi_set_device(0))
    torch.cuda.set_device(0)
    if a.profile:
        profile(a.profile)
        return
    result = {"card": card(), "copy_peak_GBps": PEAK_GBPS, "shapes": []}
    for name, dt, n, w in SHAPES:
        if name in a.shapes.split(","):
            r = run_shape(name, dt, n, w, a.steps, a.warmup)
            print(json.dumps(r), flush=True)
            result["shapes"].append(r)
    ok = all(v["oracle_bits_equal_on_sampled_columns"] for r in result["shapes"] for v in r["kinds"].values())
    result["all_sampled_columns_bits_equal"] = ok
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({"card": result["card"], "all_sampled_columns_bits_equal": ok}))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
