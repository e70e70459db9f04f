#!/usr/bin/env python3
"""Derivative kernels against the value kernels of the same shape, in one run on one GPU.

    python scripts/bench_deriv.py [--steps 20] [--warmup 3] [--out FILE.json]

Shapes: C2 (cubic, 4096 x 1024 f64, 2^20 sorted queries), C5b's evaluation table (cubic, 4096 x 32 f32, 2^25 sorted
queries) and C3 (linear, grid 65 536, 16 f32 columns, 2^24 random queries, extrapolation on).  Within a shape the value
call and the derivative calls (cubic: order 1 and 2; linear: the slope) alternate step by step through the _dev entry
points on device-resident queries, each call between its own CUDA events.  Reported per call: median / min ms over the
steps, algorithmic GB/s -- s (c + W) Q plus the table (data, and a, b for the spline), as DESIGN.md section 4 -- and its
fraction of the measured 6 443 GB/s copy peak; the derivative's time over the value kernel's.  Every derivative output
is checked bit for bit against tests/deriv_oracle.cpp on a sample of rows, with the coefficients the handle holds.
The card's name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import deriv_oracle as D  # noqa: E402
from ndarray_interp_b200 import _lib as L  # noqa: E402
from ndarray_interp_b200.interp1d import BoundaryCondition, CubicSpline, Interp1D, Linear  # noqa: E402

PEAK_GBPS = 6443.0          # measured device copy peak (DESIGN.md section 4)
SHAPES = {
    "c2": dict(kind="cubic", dtype=np.float64, n=4096, w=1024, q=1 << 20, sorted=True, extrap=0),
    "c5b_eval": dict(kind="cubic", dtype=np.float32, n=4096, w=32, q=1 << 25, sorted=True, extrap=0),
    "c3": dict(kind="linear", dtype=np.float32, n=65536, w=16, q=1 << 24, sorted=False, extrap=1),
}


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def run_shape(name, cfg, steps, warmup):
    rng = np.random.default_rng(0)
    dt, n, w, nq = cfg["dtype"], cfg["n"], cfg["w"], cfg["q"]
    g = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(dt)
    y = rng.standard_normal((n, w)).astype(dt)
    q = rng.uniform(g[0], g[-1], nq).astype(dt)
    if cfg["sorted"]:
        q.sort()
    if cfg["kind"] == "cubic":
        ip = Interp1D.new_unchecked(g, y, CubicSpline.new().boundary(BoundaryCondition.Natural).build(g, y))
        a, b = ip.strategy.coefficients(ip)
        table = 3 * y.nbytes
    else:
        ip = Interp1D.new_unchecked(g, y, Linear.new().extrapolate(bool(cfg["extrap"])))
        table = y.nbytes
    lib, h = L.load(), ip._handle()
    qd = torch.from_numpy(q).cuda()
    out = torch.empty((nq, w), dtype=qd.dtype, device="cuda")
    err = torch.empty(1, dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream()
    s = C.c_void_p(stream.cuda_stream)
    qp, op, ep = C.c_void_p(qd.data_ptr()), C.c_void_p(out.data_ptr()), C.c_void_p(err.data_ptr())
    if cfg["kind"] == "cubic":
        calls = {"value": lambda: lib.ndi_interp1d_cubic_dev(h, qp, nq, cfg["extrap"], op, ep, s),
                 "deriv1": lambda: lib.ndi_interp1d_cubic_deriv_dev(h, qp, nq, cfg["extrap"], 1, op, ep, s),
                 "deriv2": lambda: lib.ndi_interp1d_cubic_deriv_dev(h, qp, nq, cfg["extrap"], 2, op, ep, s)}
    else:
        calls = {"value": lambda: lib.ndi_interp1d_linear_dev(h, qp, nq, cfg["extrap"], op, ep, s),
                 "slope": lambda: lib.ndi_interp1d_linear_deriv_dev(h, qp, nq, cfg["extrap"], op, ep, s)}
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
    # sampled bit-exact check of every derivative against the specification on the handle's coefficients
    rows = np.unique(np.concatenate([rng.integers(0, nq, 4096), [0, nq - 1]]))
    rows_d = torch.from_numpy(rows).cuda()
    checks = {}
    for k, fn in calls.items():
        if k == "value":
            continue
        L.check(fn())
        torch.cuda.synchronize()
        assert int(err.item()) == -1, (name, k, int(err.item()))
        got = out.index_select(0, rows_d).cpu().numpy()
        if cfg["kind"] == "cubic":
            st, want, _ = D.cubic_deriv(g, y, a, b, q[rows], cfg["extrap"], int(k[-1]))
        else:
            st, want, _ = D.linear_deriv(g, y, q[rows], cfg["extrap"])
        checks[k] = bool(st == 0 and np.array_equal(got.view(np.uint8), want.view(np.uint8)))
    nbytes = dt(0).itemsize * (1 + w) * nq + table
    res = {"shape": name, **{k: (v if not isinstance(v, type) else np.dtype(v).name) for k, v in cfg.items()},
           "algorithmic_bytes": nbytes, "steps": steps, "warmup": warmup, "calls": {}}
    base = float(np.median(times["value"]))
    for k, ts in times.items():
        med = float(np.median(ts))
        res["calls"][k] = {"ms_median": round(med, 4), "ms_min": round(float(np.min(ts)), 4),
                           "GBps": round(nbytes / (med * 1e-3) / 1e9, 1),
                           "fraction_of_copy_peak": round(nbytes / (med * 1e-3) / 1e9 / PEAK_GBPS, 3),
                           "vs_value": round(med / base, 3)}
        if k in checks:
            res["calls"][k]["oracle_bits_equal_on_sample"] = checks[k]
    del out, qd
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    a = ap.parse_args()
    L.require_device()
    L.check(L.load().ndi_set_device(0))
    torch.cuda.set_device(0)
    result = {"card": card(), "copy_peak_GBps": PEAK_GBPS, "shapes": []}
    for name in a.shapes.split(","):
        r = run_shape(name, SHAPES[name], a.steps, a.warmup)
        print(json.dumps(r), flush=True)
        result["shapes"].append(r)
    ok = all(c.get("oracle_bits_equal_on_sample", True) for r in result["shapes"] for c in r["calls"].values())
    result["all_sampled_rows_bits_equal"] = ok
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({"card": result["card"], "all_sampled_rows_bits_equal": ok}))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
