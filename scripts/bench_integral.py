#!/usr/bin/env python3
"""Integral kernels against the value kernels of the same table, and the cumulative-table build, in one run on one GPU.

    python scripts/bench_integral.py [--steps 20] [--warmup 3] [--out FILE.json]

Evaluation shapes: C2's table (cubic, 4096 x 1024 f64) with 2^20 sorted consecutive bins (lo = e[:-1], hi = e[1:]),
C5b's evaluation table (cubic, 4096 x 32 f32) with 2^25 random pairs, and C3 (linear, grid 65 536, 16 f32 columns)
with 2^24 random pairs, extrapolation on.  Within a shape the value call (on the lo bounds) and the integral call
alternate step by step through the _dev entry points on device-resident bounds, each call between its own CUDA events.
Reported per call: median / min ms, algorithmic bytes -- s (2 + W) Q plus the tables once (y, a, b and C for the
spline; y and C for Linear; the value call: s (1 + W) Q plus its own tables) -- and their fraction of the measured
6 443 GB/s copy peak; the integral's time over the value call's.  Every integral output is checked bit for bit against
tests/integral_oracle.cpp on a sample of rows.  ndi_interp1d_integral_build is timed (host clock around the call,
which ends in a device synchronise) at C2's shape, at (65536, 64) f64 and at (4096, 131072) f32; its bytes are the
tables read plus C written.  The card's name and power limit are read in the same run.
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
import integral_oracle as I  # noqa: E402
from ndarray_interp_b200 import _lib as L  # noqa: E402
from ndarray_interp_b200.interp1d import BoundaryCondition, CubicSpline, Interp1D, Linear  # noqa: E402

PEAK_GBPS = 6443.0          # measured device copy peak (DESIGN.md section 4)
SHAPES = {
    "c2": dict(kind="cubic", dtype=np.float64, n=4096, w=1024, q=1 << 20, bins=True, extrap=0),
    "c5b_eval": dict(kind="cubic", dtype=np.float32, n=4096, w=32, q=1 << 25, bins=False, extrap=0),
    "c3": dict(kind="linear", dtype=np.float32, n=65536, w=16, q=1 << 24, bins=False, extrap=1),
}
BUILDS = [("c2", np.float64, 4096, 1024), ("long", np.float64, 65536, 64), ("wide", np.float32, 4096, 131072)]


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def _interp(cfg, g, y):
    if cfg["kind"] == "cubic":
        return Interp1D.new_unchecked(g, y, CubicSpline.new().boundary(BoundaryCondition.Natural).build(g, y))
    return Interp1D.new_unchecked(g, y, Linear.new().extrapolate(bool(cfg["extrap"])))


def run_shape(name, cfg, steps, warmup):
    rng = np.random.default_rng(0)
    dt, n, w, nq = cfg["dtype"], cfg["n"], cfg["w"], cfg["q"]
    s_ = np.dtype(dt).itemsize
    g = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(dt)
    y = rng.standard_normal((n, w)).astype(dt)
    if cfg["bins"]:
        e = np.sort(rng.uniform(g[0], g[-1], nq + 1)).astype(dt)
        lo, hi = e[:-1].copy(), e[1:].copy()
    else:
        lo, hi = rng.uniform(g[0], g[-1], nq).astype(dt), rng.uniform(g[0], g[-1], nq).astype(dt)
    ip = _interp(cfg, g, y)
    ip.prepare_integral()
    cubic = cfg["kind"] == "cubic"
    a, b = ip.strategy.coefficients(ip) if cubic else (None, None)
    lib, h = L.load(), ip._handle()
    lod, hid = torch.from_numpy(lo).cuda(), torch.from_numpy(hi).cuda()
    out = torch.empty((nq, w), dtype=lod.dtype, device="cuda")
    err = torch.empty(1, dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream()
    s = C.c_void_p(stream.cuda_stream)
    lp, hp, op, ep = (C.c_void_p(t.data_ptr()) for t in (lod, hid, out, err))
    if cubic:
        calls = {"value": lambda: lib.ndi_interp1d_cubic_dev(h, lp, nq, cfg["extrap"], op, ep, s),
                 "integral": lambda: lib.ndi_interp1d_cubic_integral_dev(h, lp, hp, nq, cfg["extrap"], op, ep, s)}
    else:
        calls = {"value": lambda: lib.ndi_interp1d_linear_dev(h, lp, nq, cfg["extrap"], op, ep, s),
                 "integral": lambda: lib.ndi_interp1d_linear_integral_dev(h, lp, hp, nq, cfg["extrap"], op, ep, s)}
    for _ in range(warmup):
        for fn in calls.values():
            L.check(fn())
    torch.cuda.synchronize()
    times = {k: [] for k in calls}
    for _ in range(steps):                   # alternate the calls within every step
        for k, fn in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            L.check(fn())
            e1.record(stream)
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
    L.check(calls["integral"]())
    torch.cuda.synchronize()
    assert int(err.item()) == -1, (name, int(err.item()))
    rows = np.unique(np.concatenate([rng.integers(0, nq, 4096), [0, nq - 1]]))
    got = out.index_select(0, torch.from_numpy(rows).cuda()).cpu().numpy()
    st, want, _, _ = I.integrate(g, y, a, b, lo[rows], hi[rows], cfg["extrap"])
    bits_equal = bool(st == 0 and np.array_equal(got.view(np.uint8), want.view(np.uint8)))
    table = (4 if cubic else 2) * y.nbytes
    nbytes = {"value": s_ * (1 + w) * nq + (3 if cubic else 1) * y.nbytes, "integral": s_ * (2 + w) * nq + table}
    res = {"shape": name, **{k: (v if not isinstance(v, type) else np.dtype(v).name) for k, v in cfg.items()},
           "steps": steps, "warmup": warmup, "calls": {}}
    base = float(np.median(times["value"]))
    for k, ts in times.items():
        med = float(np.median(ts))
        res["calls"][k] = {"ms_median": round(med, 4), "ms_min": round(float(np.min(ts)), 4),
                           "algorithmic_bytes": nbytes[k], "GBps": round(nbytes[k] / (med * 1e-3) / 1e9, 1),
                           "fraction_of_copy_peak": round(nbytes[k] / (med * 1e-3) / 1e9 / PEAK_GBPS, 3),
                           "vs_value": round(med / base, 3)}
    res["calls"]["integral"]["oracle_bits_equal_on_sample"] = bits_equal
    del out, lod, hid
    torch.cuda.empty_cache()
    return res


def run_build(name, dt, n, w, steps):
    rng = np.random.default_rng(1)
    g = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(dt)
    y = rng.standard_normal((n, w)).astype(dt)
    ip = _interp({"kind": "cubic"}, g, y)
    lib, h = L.load(), ip._handle()
    L.check(lib.ndi_interp1d_integral_build(h, L.INTEGRAL_CUBIC))          # warm-up: allocations, module load
    ts = []
    for _ in range(steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        L.check(lib.ndi_interp1d_integral_build(h, L.INTEGRAL_CUBIC))
        ts.append((time.perf_counter() - t0) * 1e3)
    nbytes = 3 * y.nbytes + y.nbytes                  # y, a, b read (a, b: n-1 rows), C written
    med = float(np.median(ts))
    return {"build": name, "dtype": np.dtype(dt).name, "n": n, "w": w, "ms_median": round(med, 4),
            "ms_min": round(float(np.min(ts)), 4), "algorithmic_bytes": nbytes,
            "fraction_of_copy_peak": round(nbytes / (med * 1e-3) / 1e9 / PEAK_GBPS, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--builds", default=",".join(b[0] for b in BUILDS))
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    a = ap.parse_args()
    L.require_device()
    L.check(L.load().ndi_set_device(0))
    torch.cuda.set_device(0)
    result = {"card": card(), "copy_peak_GBps": PEAK_GBPS, "shapes": [], "builds": []}
    for name in filter(None, a.shapes.split(",")):
        r = run_shape(name, SHAPES[name], a.steps, a.warmup)
        print(json.dumps(r), flush=True)
        result["shapes"].append(r)
    for name, dt, n, w in BUILDS:
        if name in a.builds.split(","):
            r = run_build(name, dt, n, w, a.steps)
            print(json.dumps(r), flush=True)
            result["builds"].append(r)
    ok = all(r["calls"]["integral"]["oracle_bits_equal_on_sample"] for r in result["shapes"])
    result["all_sampled_rows_bits_equal"] = ok
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({"card": result["card"], "all_sampled_rows_bits_equal": ok}))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
