#!/usr/bin/env python3
"""bench.py -- throughput of the batched interpolation hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload c2|c1|c3|c3d|c4|c4x|c5a|c5b|c5b_build]   (one workload only; default: all of BASELINE.json)
                    [--dump-outputs DIR]   (the headline's last timed step, see dump_outputs)

Prints ONE JSON line (rank 0).  A "step" is one pass of the hot path over one query batch (one fused evaluation
launch; three launches when a bilinear batch is binned).  The headline is BASELINE.json configs[1] (C2: Interp1D
CubicSpline natural, x len 4096, data (4096, 1024), 2^20 sorted queries, f64); the `workloads` object carries the
same measurements for every other BASELINE config (C1, C3, C4 with and without extrapolation, C5 bilinear and cubic
at their named scale of 2^28 queries, and the column-sharded (4096, 131072) spline build of C5).  Per workload:

  ms_per_step   K steps, every one bracketed by its own CUDA events on the launch stream, mean = (first start ->
                last end) / K; per_step gives median / best / worst of the same K steps
  value         whole-job queries/s, queries + tables + output resident in HBM
  roofline      HBM roofline of the step: algorithmic bytes per launch (s*c*Q queries + s*W*Q output + unique table
                bytes, SURVEY.md section 8(d)) over ms_per_step, against the measured copy peak (MEASURED_PEAKS.json)
  e2e           the same metric through the host-array API (Interp{1,2}D.interp_array_into -> the C ABI's host entry
                points): pinned host queries H2D and the result rows D2H inside the timed region, every step
  check         sampled rows of the device-resident result compared BIT FOR BIT with the CPU oracle -- on every rank's
                shard (the samples travel to rank 0), also after the column-sharded build + all-gather route
  cpu_baseline  the CPU oracle (restatement of the reference algorithm: the Rust crate cannot be built here) on the
                host cores, on a bounded strided sample of the same queries (N = 1 only)

Multi-GPU (torchrun, one process per GPU): tables generated on rank 0 and replicated by NCCL broadcast; C2 builds its
spline column-sharded and all-gathers the coefficients; every rank evaluates its own query shard with no collective in
the timed region.  C1 - C4 are weak-scaled (the named batch per GPU); C5 is STRONG-scaled: 2^28 queries in total,
2^28 / N per GPU, and 131072 / N spline columns per GPU.
"""
import argparse
import contextlib
import hashlib
import io
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # q: queries per GPU (weak scaling) or, with strong=True, in total
    "c1": dict(kind="linear", dtype="f64", n=1000, w=1, q=10_000, extrap=False, sorted=False,
               desc="Interp1D Linear, sorted x len 1000, data (1000,), 10k random queries, f64"),
    "c2": dict(kind="cubic", dtype="f64", n=4096, w=1024, q=1 << 20, extrap=False, sorted=True,
               desc="Interp1D CubicSpline natural, x len 4096, data (4096,1024), 2^20 sorted queries, f64"),
    "c3": dict(kind="linear", dtype="f32", n=65536, w=16, q=1 << 24, extrap=True, sorted=False,
               desc="Interp1D Linear extrapolate, query (4096,4096) on non-uniform grid len 65536, data (65536,16), f32"),
    "c3d": dict(kind="linear", dtype="f64", n=65536, w=16, q=1 << 24, extrap=True, sorted=False,
                desc="as c3 with f64 tables (the reference's default element type)"),
    "c4": dict(kind="bilinear", dtype="f32", n=2048, m=2048, w=8, q=1 << 24, extrap=False, sorted=False,
               desc="Interp2D Bilinear, 2048x2048 grid, data (2048,2048,8), 16M random queries, f32, no extrapolation"),
    "c4x": dict(kind="bilinear", dtype="f32", n=2048, m=2048, w=8, q=1 << 24, extrap=True, sorted=False,
                desc="Interp2D Bilinear, 2048x2048 grid, data (2048,2048,8), 16M random queries, f32, extrapolation, 5% outside per axis"),
    "c5a": dict(kind="bilinear", dtype="f32", n=4096, m=4096, w=32, q=1 << 28, extrap=False, sorted=False, strong=True,
                desc="Interp2D Bilinear at scale, data (4096,4096,32), 2^28 queries in total (sharded over the GPUs), f32"),
    "c5b": dict(kind="cubic", dtype="f32", n=4096, w=32, q=1 << 28, extrap=False, sorted=True, strong=True,
                desc="Interp1D CubicSpline at scale, data (4096,32), 2^28 queries in total (sharded, sorted per shard), f32"),
    "c5b_build": dict(kind="build", dtype="f32", n=4096, w=131072, q=0, strong=True,
                      desc="CubicSpline coefficient construction at scale: data (4096, 131072) f32, trailing columns sharded over the GPUs, coefficients all-gathered"),
}
DEFAULT_OTHERS = ["c1", "c3", "c4", "c4x", "c5a", "c5b", "c5b_build"]
ESIZE = {"f32": 4, "f64": 8}
BC_NATURAL = 1


def queries_per_gpu(wl, world):
    return wl["q"] // world if wl.get("strong") else wl["q"]


def algorithmic_bytes(wl, q):
    """SURVEY.md section 8(d): s*c*Q + s*W*Q + unique table bytes, per launch (q = queries of one launch)"""
    s, w = ESIZE[wl["dtype"]], wl["w"]
    c = 2 if wl["kind"] == "bilinear" else 1
    if wl["kind"] == "bilinear":
        table = s * (wl["n"] + wl["m"] + wl["n"] * wl["m"] * w)
    elif wl["kind"] == "cubic":
        table = s * (wl["n"] + wl["n"] * w + 2 * (wl["n"] - 1) * w)
    else:
        table = s * (wl["n"] + wl["n"] * w)
    return s * c * q + s * w * q + table


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def l2_note(wl, nq):
    """how the timed steps stand to the 126 MB L2 (the contract wants it said in `config`)"""
    ab = algorithmic_bytes(wl, nq)
    if ab < (512 << 20):
        return "flushed between timed steps (512 MB overwrite); ms_per_step = mean of the K individually timed steps"
    return "working set per step (%.2f GB, output streamed once) exceeds the 126 MB L2; no explicit flush" % (ab / 1e9)


def workload_config(name, wl, world):
    """`config` of the JSON line: names the workload -- the same dictionary in both arms (`--impl reference` measures the
    reference's CPU path on this arm's config); what is specific to a GPU run goes to the line's `run` object"""
    nq = queries_per_gpu(wl, world)
    return {"workload": f"{name}: {wl['desc']}", "queries_per_gpu": nq, "columns": wl["w"],
            "l2": l2_note(wl, nq) if wl["kind"] != "build" else None}


EVAL_SOURCES_1D = ("ndi_device.cuh", "ndi_eval.cu", "ndi_grid.cu", "ndi_internal.h")
EVAL_SOURCES = EVAL_SOURCES_1D + ("ndi_bin.cu", "ndi_sweep.cu")          # bilinear: binning and band sweeps as well
BUILD_SOURCES = ("ndi_device.cuh", "ndi_internal.h", "ndi_partition.cu", "ndi_rowsplit.cu", "ndi_spline.cu", "ndi_spline.cuh")


def kernel_source_hash(files=EVAL_SOURCES):
    """sha256 over kernel sources: ties a recorded ncu capture to the kernels it was taken from.  The DRAM-traffic stamps
    (profiles/roofline_traffic.json) belong to the EVALUATION workloads, so they carry the hash of the sources the
    evaluation kernels of that workload are compiled from (workload_sources); the spline-build sources have a hash of
    their own (`run.build_source_hash`)"""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "ndarray_interp_b200", "csrc")
    for f in sorted(files):
        h.update(f.encode())
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def workload_sources(name):
    return EVAL_SOURCES if WORKLOADS[name]["kind"] == "bilinear" else EVAL_SOURCES_1D


def recorded_traffic(name, nq):
    """dram bytes per step from the committed `ncu --set full` capture of this workload, with the commit and the
    hash of the kernel sources it was taken from; `current` says whether the sources are still those.  A capture
    taken at another batch size than this run's is reported in the stamp only (traffic: null)."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        e = json.load(open(p)).get(name)
    except Exception:
        return None, None
    if not isinstance(e, dict) or e.get("bytes") is None:
        return None, None
    stamp = {k: e.get(k) for k in ("commit", "source_hash", "capture", "per")}
    stamp["current"] = e.get("source_hash") == kernel_source_hash(workload_sources(name))
    if e.get("queries") not in (None, nq):
        stamp["bytes_at_capture_size"] = e["bytes"]
        return None, stamp
    return e["bytes"], stamp


# ---- synthetic inputs (seeded) -------------------------------------------------------------------------------
def make_tables(wl):
    """grids and data on the host (numpy, seed 1234): the same arrays for the GPU arm, its oracle check and the CPU arm"""
    dt = np.float32 if wl["dtype"] == "f32" else np.float64
    rng = np.random.default_rng(1234)
    out = {}
    if wl["kind"] == "bilinear":
        n, m, w = wl["n"], wl["m"], wl["w"]
        out["x"] = np.linspace(0.0, 1.0, n).astype(dt)                            # uniform
        out["y"] = (np.cumsum(rng.uniform(0.5, 1.5, m)) / m).astype(dt)           # non-uniform
        out["data"] = rng.standard_normal((n, m, w), dtype=np.float32).astype(dt, copy=False)
        return out
    n, w = wl["n"], wl["w"]
    if wl["kind"] == "linear" and n >= 65536:
        g = np.cumsum(np.exp(rng.uniform(-2.0, 2.0, n)))                          # log-spaced steps + jitter
    else:
        g = np.cumsum(rng.uniform(0.5, 1.5, n))
    g = g.astype(dt)
    assert len(np.unique(g)) == n
    out["x"] = g
    out["data"] = (rng.standard_normal((n, w), dtype=np.float32).astype(dt, copy=False) if w > 1
                   else rng.standard_normal(n).astype(dt))
    return out


def query_range(wl):
    return (-0.026, 1.026) if wl["extrap"] else (0.0, 1.0)                        # ~5 % outside per axis


def make_queries_host(wl, tables, nq, seed):
    """numpy queries of the workload's distribution (CPU arm; the GPU arm draws on the device)"""
    dt = tables["x"].dtype
    rng = np.random.default_rng(seed)
    lo, hi = query_range(wl)

    def axis(g):
        q = (float(g[0]) + (float(g[-1]) - float(g[0])) * rng.uniform(lo, hi, nq)).astype(dt)
        return q if wl["extrap"] else np.clip(q, g[0], g[-1])
    if wl["kind"] == "bilinear":
        return axis(tables["x"]), axis(tables["y"])
    q = axis(tables["x"])
    return (np.sort(q) if wl["sorted"] else q), None


# ---- clocks during the timed region ------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.window = index, [], False, [None, None]
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max_mhz = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, reasons))
            except Exception:
                pass
            time.sleep(0.005)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        t0, t1 = self.window
        inside = [s for s in self.samples if t0 is not None and t1 is not None and t0 <= s[0] <= t1] or self.samples
        names = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
                 0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
                 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}
        bits = 0
        for s in inside:
            bits |= s[2]
        reasons = [v for k, v in names.items() if bits & k and v != "gpu_idle"]
        return {"sm_mhz": float(np.median([s[1] for s in inside])), "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(inside)}


# ---- CPU leg (the oracle, timed; test infrastructure used as the baseline, never as the product) ------------------
def cpu_eval(wl, tables, coeffs, qx, qy, threads, out):
    from oracle import oracle_py as O
    if wl["kind"] == "bilinear":
        st = O.interp2d_bilinear(tables["x"], tables["y"], tables["data"], qx, qy, wl["extrap"], nthreads=threads, out=out)[0]
    elif wl["kind"] == "cubic":
        st = O.interp1d_cubic(tables["x"], tables["data"], coeffs[0], coeffs[1], qx, 1 if wl["extrap"] else 0,
                              nthreads=threads, out=out)[0]
    else:
        st = O.interp1d_linear(tables["x"], tables["data"], qx, wl["extrap"], nthreads=threads, out=out)[0]
    assert st == 0, st
    return out


def cpu_sample_size(wl, target_elems):
    """bounded sample: about target_elems output elements per pass"""
    return int(min(wl["q"], max(1024, target_elems // wl["w"])))


def time_cpu(wl, tables, coeffs, qx, qy, threads, budget_s, max_reps):
    out = np.zeros((len(qx), wl["w"]), dtype=tables["x"].dtype)
    cpu_eval(wl, tables, coeffs, qx, qy, threads, out)
    reps, t0 = 0, time.perf_counter()
    while reps < 2 or (time.perf_counter() - t0 < budget_s and reps < max_reps):
        cpu_eval(wl, tables, coeffs, qx, qy, threads, out)
        reps += 1
    return len(qx) / ((time.perf_counter() - t0) / reps), reps


def cpu_baseline_for(wl, tables, coeffs, qx, qy, budget_s, how):
    """multi-threaded (queries sharded from outside like the reference's rayon benches) and single-threaded (what
    the reference itself is) oracle throughput on the given sample"""
    from oracle import oracle_py as O
    threads = O.hardware_threads()
    value, reps = time_cpu(wl, tables, coeffs, qx, qy, threads, budget_s, 200)
    n1 = max(1024, len(qx) // 8)
    single, _ = time_cpu(wl, tables, coeffs, qx[:n1], None if qy is None else qy[:n1], 1, budget_s / 3, 50)
    return {"value": value, "unit": "queries/s", "cores": threads, "kind": "port", "value_1_thread": single,
            "sample": f"{len(qx)} of {wl['q']} queries ({how}), all {wl['w']} columns, {reps} passes, {threads} threads "
                      "(query-sharded from outside); oracle = C++ restatement of the reference algorithm"}


def oracle_coeffs(tables, levels):
    """levels: ndi_interp1d_build_info's value (0 reference order, L > 0 row-split levels, -m partition blocks)"""
    from oracle import oracle_py as O
    st, a, b = O.spline_build_as(tables["x"], tables["data"], {"kind": "Natural"}, levels)
    assert st == 0
    return a, b


def build_spec_name(levels):
    if levels > 0:
        return "row-split specification with %d levels" % levels
    return ("partition specification with blocks of %d rows" % -levels) if levels < 0 else "reference order"


# ---- the reference arm: the reference's own CPU implementation of the path (here: its restatement) ---------------
def reference_workload(wl, name, steps, warmup, budget_elems):
    from oracle import oracle_py as O
    if wl["kind"] == "build":
        n, cols = wl["n"], 1024
        rng = np.random.default_rng(7)
        x = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(np.float32)
        y = rng.standard_normal((n, cols), dtype=np.float32)
        O.spline_build(x, y, {"kind": "Natural"})
        t0 = time.perf_counter()
        for _ in range(max(1, steps)):
            O.spline_build(x, y, {"kind": "Natural"})
        dt_s = (time.perf_counter() - t0) / max(1, steps)
        return {"value": cols / dt_s, "unit": "columns/s", "ms_per_step": dt_s * 1e3, "cores": 1,
                "sample": f"{cols} of {wl['w']} columns of {n} rows, one thread (the reference's calc_coefficients is serial)"}
    tables = make_tables(wl)
    nq = cpu_sample_size(wl, budget_elems)
    qx, qy = make_queries_host(wl, tables, nq, 99)
    coeffs = oracle_coeffs(tables, 0) if wl["kind"] == "cubic" else None
    threads = O.hardware_threads()
    out = np.zeros((nq, wl["w"]), dtype=tables["x"].dtype)
    for _ in range(max(1, min(warmup, 3))):
        cpu_eval(wl, tables, coeffs, qx, qy, threads, out)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_eval(wl, tables, coeffs, qx, qy, threads, out)
    dt_s = (time.perf_counter() - t0) / steps
    return {"value": nq / dt_s, "unit": "queries/s", "ms_per_step": dt_s * 1e3, "cores": threads, "kind": "port",
            "sample": f"{nq} queries of the workload's distribution per step (the whole table range"
                      f"{', sorted' if wl['sorted'] else ''}), all {wl['w']} columns, {threads} threads "
                      "(queries sharded from outside, like the reference's rayon benches)"}


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    name = args.workload or "c2"
    wl = WORKLOADS[name]
    head = reference_workload(wl, name, args.steps, args.warmup, 1 << 26)
    others = {}
    if not args.workload:
        for o in DEFAULT_OTHERS:
            try:
                others[o] = reference_workload(WORKLOADS[o], o, max(2, min(args.steps, 5)), 1, 1 << 25)
                others[o]["workload"] = f"{o}: {WORKLOADS[o]['desc']}"
            except Exception as e:                                  # a side measurement must not cost the headline
                others[o] = {"error": repr(e)}
    line = {
        "impl": "reference", "metric": "queries/s", "value": head["value"], "unit": "queries/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": wl["dtype"], "data": "synthetic",
        "config": workload_config(name, wl, max(1, args.gpus)),
        "note": "CPU restatement of the reference algorithm (oracle/ndi_oracle.cpp, g++ -O2 -ffp-contract=off); "
                "the Rust crate itself cannot be built in this image (no cargo/rustc)",
        "cpu_baseline": {"value": head["value"], "unit": "queries/s", "cores": head["cores"], "kind": "port", "sample": head["sample"]},
        "e2e": {"value": head["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "workloads": others,
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def bind_to_gpu_numa_node(index):
    """One process per GPU: run this rank (and so allocate its pinned host buffers, first touch) on the CPU socket
    the GPU hangs off.  Returns the node, or a string saying why nothing was bound."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:                      # nvml prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        path = f"/sys/bus/pci/devices/{bus}/numa_node"
        if not os.path.exists(path):
            return "not exposed (no sysfs entry for the GPU's PCI device in this container)"
        node = int(open(path).read())
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        if node < 0 or len(nodes) < 2:
            return f"single NUMA node (sysfs reports {node}, {len(nodes)} node(s)): nothing to bind"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
        return f"node {node} has no CPU this process may run on"
    except Exception as e:
        return f"lookup failed: {e!r}"


# ---- GPU arm -------------------------------------------------------------------------------------------------
class Ctx:
    pass


def _tensor_from_ptr(torch, ptr, nel, dtype, dev):
    """borrow library-owned device memory as a torch tensor (no copy) via __cuda_array_interface__"""
    typestr = {torch.float32: "<f4", torch.float64: "<f8"}[dtype]

    class _Holder:
        __cuda_array_interface__ = {"shape": (nel,), "typestr": typestr, "data": (int(ptr), False), "version": 3}
    return torch.as_tensor(_Holder(), device=dev)


def device_queries(ctx, wl, tables, nq, seed):
    """this rank's query shard, drawn on the device (2^28 queries would take numpy tens of seconds)"""
    torch = ctx.torch
    tdt = torch.float32 if wl["dtype"] == "f32" else torch.float64
    gen = torch.Generator(device=ctx.dev)
    gen.manual_seed(seed)
    lo, hi = query_range(wl)

    def axis(g):
        g0, gl = float(g[0]), float(g[-1])
        u = torch.rand(nq, dtype=torch.float64 if nq <= (1 << 26) else torch.float32, device=ctx.dev, generator=gen)
        q = (g0 + (gl - g0) * (lo + (hi - lo) * u)).to(tdt)
        del u
        return q if wl["extrap"] else q.clamp_(g0, gl)
    if wl["kind"] == "bilinear":
        return axis(tables["x"]), axis(tables["y"])
    q = axis(tables["x"])
    if wl["sorted"]:
        q = torch.sort(q)[0]
    return q, None


def gather_samples(ctx, tensors):
    """rows sampled on every rank, gathered on all ranks (tiny); returns a list per rank of numpy arrays"""
    torch, dist = ctx.torch, ctx.dist
    if ctx.world == 1:
        return [[t.cpu().numpy() for t in tensors]]
    per_rank = [[] for _ in range(ctx.world)]
    for t in tensors:
        parts = [torch.empty_like(t) for _ in range(ctx.world)]
        dist.all_gather(parts, t.contiguous())
        for r in range(ctx.world):
            per_rank[r].append(parts[r].cpu().numpy())
    return per_rank


DUMP_BYTES = 48 << 20          # --dump-outputs: sampled output bytes of all files together


def dump_outputs(ctx, arrays, axis):
    """--dump-outputs DIR: what the last timed step handed its caller, written by rank 0 as DIR/<name>.npy.
    arrays: {name: device tensor}; an output too large for DUMP_BYTES keeps the slices along `axis` (query rows,
    spline columns) at sorted indices drawn from a fixed seed, on every rank's shard, so that two builds run with
    the same arguments write files that compare element for element."""
    torch = ctx.torch
    budget = DUMP_BYTES // (len(arrays) * ctx.world)
    samples = []
    for t in arrays.values():
        n = t.shape[axis]
        k = min(n, max(1, budget // (t.element_size() * t.numel() // n)))
        idx = np.sort(np.random.default_rng(0).choice(n, k, replace=False))
        samples.append(t.index_select(axis, torch.from_numpy(idx).to(t.device)))
    per_rank = gather_samples(ctx, samples)
    if ctx.rank == 0:
        os.makedirs(ctx.args.dump_outputs, exist_ok=True)
        for i, name in enumerate(arrays):
            a = np.concatenate([parts[i] for parts in per_rank], axis=axis)
            np.save(os.path.join(ctx.args.dump_outputs, name + ".npy"), a)
            print(f"dump-outputs: {name}.npy {a.dtype} {a.shape}", file=sys.stderr)


def timed_steps(ctx, step, steps, flush_l2, sampler=None):
    """K steps, each bracketed by its own CUDA events on the launch stream.  Returns (ms per step from the first
    start to the last end -- or the sum of the steps when L2 is scrubbed in between --, sorted per-step list)."""
    torch = ctx.torch
    scrub = torch.empty(512 << 20, dtype=torch.uint8, device=ctx.dev) if flush_l2 else None
    ctx.barrier()
    if sampler is not None:
        sampler.window[0] = time.perf_counter()
    if flush_l2:
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a_ev, b_ev in evs:
            scrub.fill_(1)                                    # no step finds its queries, tables or output lines in L2
            a_ev.record()
            step()
            b_ev.record()
        ctx.barrier()
        per = [a.elapsed_time(b) for a, b in evs]
        total = sum(per)
    else:
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        evs[0].record()
        for i in range(steps):
            step()
            evs[i + 1].record()
        ctx.barrier()
        per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
        total = evs[0].elapsed_time(evs[steps])
    if sampler is not None:
        sampler.window[1] = time.perf_counter()
    del scrub
    return ctx.max_over_ranks(total / steps), sorted(per)


def link_probes(ctx):
    """what the platform gives a plain pinned device-to-host copy and a plain host-to-host copy, measured with ALL
    ranks copying at the same time (the ceilings of any host-buffer API at this rank count)"""
    torch = ctx.torch
    nbytes = 1 << 28
    dev_buf = torch.empty(nbytes, dtype=torch.uint8, device=ctx.dev)
    pin_a = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    pin_b = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    pin_a.copy_(dev_buf, non_blocking=True)
    pin_b.copy_(pin_a)
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        pin_a.copy_(dev_buf, non_blocking=True)
    torch.cuda.synchronize()
    d2h_s = time.perf_counter() - t0
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(2):
        pin_b.copy_(pin_a)
    h2h_s = time.perf_counter() - t0
    # whole-job figures the way the metric itself is timed: all ranks' bytes over the SLOWEST rank's time
    out = {"d2h_link_GBps": 4 * nbytes / d2h_s / 1e9,
           "d2h_link_GBps_all_ranks": ctx.world * 4 * nbytes / ctx.max_over_ranks(d2h_s) / 1e9,
           "host_sink_GBps": 2 * nbytes / h2h_s / 1e9,
           "host_sink_GBps_all_ranks": ctx.world * 2 * nbytes / ctx.max_over_ranks(h2h_s) / 1e9,
           "how": "256 MB pinned buffers; device-to-host: 4 async copies; host sink: 2 pinned-to-pinned CPU copies "
                  f"(torch copy_, {torch.get_num_threads()} thread(s) per rank); all {ctx.world} rank(s) at the same time, "
                  "all-ranks figures = all ranks' bytes over the slowest rank's time (like the metric)"}
    del dev_buf, pin_a, pin_b
    return out


def measure_eval(ctx, name, wl, steps, warmup, role, sampler=None):
    """one evaluation workload: device-resident timing, oracle check, e2e through the host API, CPU baseline"""
    torch, dist = ctx.torch, ctx.dist
    from ndarray_interp_b200 import _lib as L
    from ndarray_interp_b200 import device as D
    from ndarray_interp_b200.interp1d import CubicSplineStrategy, Interp1D, Linear
    from ndarray_interp_b200.interp2d import Bilinear, Interp2D

    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    tdt = torch.float32 if wl["dtype"] == "f32" else torch.float64
    s = ESIZE[wl["dtype"]]
    nq = queries_per_gpu(wl, world)
    extrap = wl["extrap"]
    res = {"workload": f"{name}: {wl['desc']}", "dtype": wl["dtype"], "scaling": "strong" if wl.get("strong") else "weak",
           "queries_per_gpu": nq, "queries_total": nq * world, "columns": wl["w"]}

    # ---- tables: generated on rank 0, replicated to every GPU over NVLink by NCCL broadcast ----
    tables = make_tables(wl) if (rank == 0 or wl["kind"] != "bilinear" or wl["n"] * wl["m"] * wl["w"] < (1 << 26)) else None
    shapes = {"x": (wl["n"],), "y": (wl.get("m", 0),),
              "data": (wl["n"], wl["m"], wl["w"]) if wl["kind"] == "bilinear" else ((wl["n"], wl["w"]))}

    def replicated(key):
        t = torch.from_numpy(tables[key].reshape(shapes[key])).to(dev) if rank == 0 else torch.empty(shapes[key], dtype=tdt, device=dev)
        if world > 1:
            dist.broadcast(t, 0)
        return t

    levels = 0
    build_info = None
    if wl["kind"] == "bilinear":
        gx, gy, data = replicated("x"), replicated("y"), replicated("data")
        if tables is None:                                      # big table: the other ranks keep only the grids on the host
            tables = {"x": gx.cpu().numpy(), "y": gy.cpu().numpy(), "data": None}
        ip = D.DeviceInterp2D(gx, gy, data)
        ip.set_search_mode(ctx.args.search_mode)
    else:
        g, data = replicated("x"), replicated("data")
        ip = D.DeviceInterp1D(g, data)
        ip.set_search_mode(ctx.args.search_mode)
        if wl["kind"] == "cubic":
            w = wl["w"]
            sharded = world > 1 and w % world == 0 and w // world >= 32
            if sharded:
                # spline construction sharded over the trailing columns, coefficients all-gathered (SURVEY.md 8(e))
                cw = w // world
                shard = data[:, rank * cw:(rank + 1) * cw].contiguous()
                part = D.DeviceInterp1D(g, shard, assume_valid=True)
                st, _ = part.spline_build(BC_NATURAL)
                assert st == 0
                levels = part.build_levels()
                pa, pb = part.coeff_ptrs()
                nel = (wl["n"] - 1) * cw
                a_sh = _tensor_from_ptr(torch, pa, nel, tdt, dev).view(wl["n"] - 1, cw)
                b_sh = _tensor_from_ptr(torch, pb, nel, tdt, dev).view(wl["n"] - 1, cw)
                ga = [torch.empty_like(a_sh) for _ in range(world)]
                gb = [torch.empty_like(b_sh) for _ in range(world)]
                dist.all_gather(ga, a_sh.contiguous())
                dist.all_gather(gb, b_sh.contiguous())
                a_full, b_full = torch.cat(ga, dim=1).contiguous(), torch.cat(gb, dim=1).contiguous()
                torch.cuda.synchronize()
                L.check(ip.lib.ndi_interp1d_spline_set_coeffs(ip.h, D._p(a_full), D._p(b_full), L.DEVICE_POINTERS))
                del part, ga, gb
            else:
                st, _ = ip.spline_build(BC_NATURAL)
                assert st == 0
                levels = ip.build_levels()
            res["spline_route"] = ("column-sharded build (%d columns per GPU) + all_gather + ndi_interp1d_spline_set_coeffs" % (w // world)
                                   if sharded else "built on every GPU")
            if world == 1 and role == "headline":
                build_info = time_builds(ctx, ip, wl)

    # ---- queries and output ----
    qx, qy = device_queries(ctx, wl, tables, nq, 99 + 1000 * rank + sum(name.encode()) % 251)
    out = torch.empty((nq, wl["w"]), dtype=tdt, device=dev)
    err = D.new_err_word(dev)
    if wl["kind"] == "bilinear":
        def step():
            ip.bilinear(qx, qy, extrap, out=out, err=err)
    elif wl["kind"] == "cubic":
        def step():
            ip.cubic(qx, 1 if extrap else 0, out=out, err=err)
    else:
        def step():
            ip.linear(qx, extrap, out=out, err=err)

    # ---- device-resident timing ----
    for _ in range(max(warmup, 3)):
        step()
    abytes = algorithmic_bytes(wl, nq)
    flush_l2 = abytes < (512 << 20)          # a working set the 126 MB L2 could hold: flush it between timed steps
    launches0 = D.kernel_launch_count()
    ms_per_step, per = timed_steps(ctx, step, steps, flush_l2, sampler)
    launches = D.kernel_launch_count() - launches0
    assert D.err_word_value(err) == D.ERR_NONE, "a benchmark query failed"
    if role == "headline" and ctx.args.dump_outputs:
        dump_outputs(ctx, {name + "_out": out}, 0)
    value = world * nq / (ms_per_step * 1e-3)
    peak, peak_src = measured_peak()
    achieved = abytes / (ms_per_step * 1e-3) / 1e9
    traffic, stamp = recorded_traffic(name, nq)
    res.update({
        "value": value, "unit": "queries/s", "ms_per_step": ms_per_step, "steps": steps,
        "per_step": {"median_ms": per[len(per) // 2], "best_ms": per[0], "worst_ms": per[-1], "n": len(per),
                     "note": "the same K steps as ms_per_step, each between its own CUDA events (this rank)"},
        "launches_per_step": int(launches) // max(steps, 1),
        "l2": l2_note(wl, nq),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_capture": stamp, "algorithmic_bytes": abytes, "peak_source": peak_src,
                     "frac_of_nominal_8000": achieved / 8000.0},
    })
    if levels or wl["kind"] == "cubic":
        res["spline_build_info"] = levels                     # 0 reference order, L > 0 row-split levels, -m partition blocks

    # ---- check: sampled rows, bit for bit against the oracle, for every rank's shard (also at world > 1) ----
    nsamp = 256 if wl["w"] >= 256 else 1024
    gen = torch.Generator(device=dev)
    gen.manual_seed(5 + rank)
    idx = torch.randint(0, nq, (nsamp,), device=dev, generator=gen)
    sample = [qx[idx]] + ([qy[idx]] if qy is not None else []) + [out[idx]]
    per_rank = gather_samples(ctx, sample)
    if rank == 0:
        coeffs = oracle_coeffs(tables, levels) if wl["kind"] == "cubic" else None
        ok, rows = True, 0
        for parts in per_rank:
            sq = parts[0]
            sy = parts[1] if qy is not None else None
            ref = cpu_eval(wl, tables, coeffs, sq, sy, 8, np.zeros((len(sq), wl["w"]), dtype=tables["x"].dtype))
            ok = ok and bool(np.array_equal(ref, parts[-1].reshape(ref.shape)))
            rows += len(sq)
        res["check"] = {"bit_exact": ok, "rows": rows, "ranks": len(per_rank),
                        "what": "rows of the device-resident result at random query indices of every rank's shard, against the oracle"}
        if wl["kind"] == "cubic":
            a_dev, b_dev = ip.coeffs_to_host()
            res["check"]["coefficients_bit_exact"] = bool(np.array_equal(a_dev.reshape(coeffs[0].shape), coeffs[0]) and
                                                          np.array_equal(b_dev.reshape(coeffs[1].shape), coeffs[1]))
            res["check"]["coefficients_vs"] = "oracle, " + build_spec_name(levels)

    # ---- end to end through the host-array API (pinned host buffers, H2D + D2H in the timed region) ----
    e2e_q = int(min(nq, max(1 << 14, (1 << 31) // (wl["w"] * s)))) if role != "headline" else nq    # <= 2 GB of result rows
    e2e_steps = max(1, min(steps, ctx.args.e2e_steps))
    del out
    torch.cuda.empty_cache()
    host_x = tables["x"]
    if wl["kind"] == "bilinear":
        host_data = tables["data"] if tables["data"] is not None else data.cpu().numpy()
        hi = Interp2D.new_unchecked(host_x, tables["y"], host_data, Bilinear.new().extrapolate(extrap))
        qx_pin, qy_pin = qx[:e2e_q].cpu().pin_memory(), qy[:e2e_q].cpu().pin_memory()
        out_pin = torch.empty((e2e_q, wl["w"]), dtype=tdt, pin_memory=True)
        out_np = out_pin.numpy()

        def e2e_step():
            hi.interp_array_into(qx_pin.numpy(), qy_pin.numpy(), out_np)
    else:
        host_data = tables["data"]
        if wl["kind"] == "cubic":
            strat = CubicSplineStrategy(BC_NATURAL, (None, None, None, None), L.EXTRAP_YES if extrap else L.EXTRAP_NO)
        else:
            strat = Linear.new().extrapolate(extrap)
        hi = Interp1D.new_unchecked(host_x, host_data, strat)
        q_pin = qx[:e2e_q].cpu().pin_memory()
        out_pin = torch.empty((e2e_q,) + tuple(host_data.shape[1:]), dtype=tdt, pin_memory=True)
        out_np = out_pin.numpy()

        def e2e_step():
            hi.interp_array_into(q_pin.numpy(), out_np)
    e2e_step()                                            # warm-up (workspace allocation)
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    ctx.barrier()
    e2e_s = ctx.max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    c = 2 if wl["kind"] == "bilinear" else 1
    res["e2e"] = {"value": world * e2e_q / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": s * c * e2e_q,
                  "d2h_bytes_per_step": s * wl["w"] * e2e_q, "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
                  "queries_per_gpu": e2e_q,
                  "api": "Interp{1,2}D.interp_array_into -> ndi_interp*_{cubic,linear,bilinear} (host pointers, pinned)",
                  "d2h_achieved_GBps": s * wl["w"] * e2e_q / e2e_s / 1e9,
                  "d2h_achieved_GBps_all_ranks": world * s * wl["w"] * e2e_q / e2e_s / 1e9}
    if e2e_q != nq:
        res["e2e"]["note"] = f"the first {e2e_q} queries of every rank's shard (2 GB of result rows per step and rank)"
    if rank == 0 and res.get("check") is not None:
        # the host-API result on its first rows equals the oracle as well
        k = min(64, e2e_q)
        sq = qx[:k].cpu().numpy()
        sy = qy[:k].cpu().numpy() if qy is not None else None
        coeffs = None
        if wl["kind"] == "cubic":
            ha, hb = hi.strategy.coefficients(hi)
            coeffs = (ha, hb)                                 # the host mirror built its own spline (same mode)
            lv = hi.strategy.rowsplit_levels(hi)
            oa, ob = oracle_coeffs(tables, lv)
            res["check"]["e2e_coefficients_bit_exact"] = bool(np.array_equal(ha.reshape(oa.shape), oa) and np.array_equal(hb.reshape(ob.shape), ob))
        ref = cpu_eval(wl, tables, coeffs, sq, sy, 1, np.zeros((k, wl["w"]), dtype=host_x.dtype))
        res["check"]["e2e_bit_exact"] = bool(np.array_equal(ref, out_np.reshape(e2e_q, -1)[:k]))

    # ---- CPU baseline (rank 0, N = 1 only): strided sample of the SAME queries, so the CPU walks the whole table ----
    if rank == 0 and world == 1 and not ctx.args.no_cpu:
        ns = cpu_sample_size(wl, (1 << 26) if role == "headline" else (1 << 24))
        stride = max(1, nq // ns)
        sq = qx[::stride][:ns].contiguous().cpu().numpy()
        sy = qy[::stride][:ns].contiguous().cpu().numpy() if qy is not None else None
        coeffs = oracle_coeffs(tables, 0) if wl["kind"] == "cubic" else None
        res["cpu_baseline"] = cpu_baseline_for(wl, tables, coeffs, sq, sy, 10.0 if role == "headline" else 2.0,
                                               f"every {stride}-th query of the batch")
    if build_info is not None:
        res["spline_build"] = build_info
    del ip, hi, qx, qy, out_pin, data
    torch.cuda.empty_cache()
    return res


def time_builds(ctx, ip, wl):
    """K6 on its own: CubicSpline::calc_coefficients for this table in the three build modes (host-synchronous calls,
    wall clock per call including allocation and the final synchronisation; kernels alone by CUDA events are in
    profiles/)"""
    from ndarray_interp_b200 import _lib as L
    torch = ctx.torch
    s = ESIZE[wl["dtype"]]
    out = {"columns": wl["w"], "rows": wl["n"], "algorithmic_bytes": s * (3 * wl["n"] - 2) * wl["w"],
           "note": "ndi_interp1d_spline_build, Natural boundary, wall clock per call (allocation + launches + final sync)"}
    peak, _ = measured_peak()
    for label, mode in (("sequential", L.BUILD_SEQUENTIAL), ("rowsplit", L.BUILD_ROWSPLIT), ("partition", L.BUILD_PARTITION)):
        ip.set_build_mode(mode, 0)
        for _ in range(3):
            ip.spline_build(BC_NATURAL)
        torch.cuda.synchronize()
        reps, t0 = 10, time.perf_counter()
        for _ in range(reps):
            st, _ = ip.spline_build(BC_NATURAL)
            assert st == 0
        ms = (time.perf_counter() - t0) / reps * 1e3
        gbs = out["algorithmic_bytes"] / ms / 1e6
        out[label] = {"ms": ms, "levels": ip.build_levels(), "algorithmic_GBps": gbs, "frac_of_hbm_peak": gbs / peak}
    ip.set_build_mode(L.BUILD_AUTO, 0)
    st, _ = ip.spline_build(BC_NATURAL)                       # leave the handle with the AUTO coefficients
    assert st == 0
    out["auto_levels"] = ip.build_levels()
    out["auto"] = "partition" if out["auto_levels"] < 0 else ("rowsplit" if out["auto_levels"] else "sequential")
    out["ms"] = out[out["auto"]]["ms"]
    out["frac_of_hbm_peak"] = out[out["auto"]]["frac_of_hbm_peak"]
    return out


def measure_build(ctx, name, wl, steps, warmup, role):
    """C5's spline construction at scale: (4096, 131072) f32, columns sharded over the GPUs, coefficients all-gathered"""
    torch, dist = ctx.torch, ctx.dist
    from ndarray_interp_b200 import device as D
    from oracle import oracle_py as O
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    n, w = wl["n"], wl["w"]
    cw = w // world
    rng = np.random.default_rng(77)
    x_host = np.cumsum(rng.uniform(0.5, 1.5, n)).astype(np.float32)
    g = torch.from_numpy(x_host).to(dev)

    def shard_data(r):                                         # any rank can regenerate any shard (the check needs that)
        gen = torch.Generator(device=dev)
        gen.manual_seed(4000 + r)
        return torch.randn((n, cw), dtype=torch.float32, device=dev, generator=gen)
    y = shard_data(rank)
    part = D.DeviceInterp1D(g, y, assume_valid=True)
    for _ in range(2):
        st, _ = part.spline_build(BC_NATURAL)
        assert st == 0
    levels = part.build_levels()
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        part.spline_build(BC_NATURAL)                          # host-synchronous: wall clock = launches + final sync
    build_ms = ctx.max_over_ranks((time.perf_counter() - t0) / steps * 1e3)
    pa, pb = part.coeff_ptrs()
    nel = (n - 1) * cw
    a_sh = _tensor_from_ptr(torch, pa, nel, torch.float32, dev).view(n - 1, cw)
    b_sh = _tensor_from_ptr(torch, pb, nel, torch.float32, dev).view(n - 1, cw)
    if role == "headline" and ctx.args.dump_outputs:
        dump_outputs(ctx, {name + "_a": a_sh, name + "_b": b_sh}, 1)
    gather_ms, a_full, b_full = 0.0, a_sh, b_sh
    if world > 1:
        a_full = torch.empty((world, n - 1, cw), dtype=torch.float32, device=dev)
        b_full = torch.empty((world, n - 1, cw), dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(a_full, a_sh.contiguous())     # warm-up (communicator, buffers)
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dist.all_gather_into_tensor(a_full, a_sh.contiguous())
        dist.all_gather_into_tensor(b_full, b_sh.contiguous())
        e1.record()
        ctx.barrier()
        gather_ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    s = 4
    moved = s * (3 * n - 2) * w
    peak, _ = measured_peak()
    res = {"workload": f"{name}: {wl['desc']}", "dtype": "f32", "scaling": "strong", "columns_per_gpu": cw, "rows": n,
           "build_info": levels, "build_ms": build_ms, "value": w / (build_ms * 1e-3), "unit": "columns/s",
           "algorithmic_bytes_per_gpu": moved // world, "algorithmic_GBps_per_gpu": moved / world / build_ms / 1e6,
           "frac_of_hbm_peak": moved / world / build_ms / 1e6 / peak,
           "allgather_ms": gather_ms, "allgather_bytes_received_per_gpu": 2 * (world - 1) * (n - 1) * cw * s,
           "allgather_GBps_per_gpu": (2 * (world - 1) * (n - 1) * cw * s / gather_ms / 1e6) if gather_ms else None,
           "note": "build: wall clock per ndi_interp1d_spline_build call on the slowest rank; all-gather of a and b: CUDA events, slowest rank"}
    if rank == 0:
        # check: columns of EVERY shard of the gathered coefficients, bit for bit against the oracle
        ok, ncols = True, 0
        for r in range(world):
            cols = np.sort(np.random.default_rng(r).choice(cw, 16, replace=False))
            yr = (y if r == rank else shard_data(r))[:, torch.from_numpy(cols).to(dev)].cpu().numpy()
            st, a_ref, b_ref = O.spline_build_as(x_host, np.ascontiguousarray(yr), {"kind": "Natural"}, levels)
            src_a = a_full[r] if world > 1 else a_full
            src_b = b_full[r] if world > 1 else b_full
            ga = src_a[:, torch.from_numpy(cols).to(dev)].cpu().numpy()
            gb = src_b[:, torch.from_numpy(cols).to(dev)].cpu().numpy()
            ok = ok and st == 0 and bool(np.array_equal(ga, a_ref) and np.array_equal(gb, b_ref))
            ncols += len(cols)
        res["check"] = {"bit_exact": ok, "columns": ncols, "ranks": world,
                        "what": "16 columns of every rank's shard of the all-gathered a, b against the oracle "
                                + "(" + build_spec_name(levels) + ")"}
    del part, y, a_full, b_full
    torch.cuda.empty_cache()
    return res


def run_b200(args):
    import torch
    import torch.distributed as dist

    from ndarray_interp_b200 import device as D

    ctx = Ctx()
    ctx.torch, ctx.dist, ctx.args = torch, dist, args
    ctx.rank = int(os.environ.get("RANK", "0"))
    ctx.world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if ctx.world != args.gpus and ctx.world > 1:
        args.gpus = ctx.world
    D.set_device(local)
    ctx.dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local) if ctx.world > 1 else "one process: not bound"
    if ctx.world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=ctx.dev)

    def barrier():
        torch.cuda.synchronize()
        if ctx.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(v, op):
        if ctx.world == 1:
            return float(v)
        t = torch.tensor([v], dtype=torch.float64, device=ctx.dev)
        dist.all_reduce(t, op=op)
        return float(t.item())
    ctx.barrier = barrier
    ctx.max_over_ranks = lambda v: reduce(v, dist.ReduceOp.MAX)
    ctx.sum_over_ranks = lambda v: reduce(v, dist.ReduceOp.SUM)

    name = args.workload or "c2"
    wl = WORKLOADS[name]
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = D.kernel_launch_count()
    if wl["kind"] == "build":
        head = measure_build(ctx, name, wl, args.steps, args.warmup, "headline")
        head.setdefault("ms_per_step", head["build_ms"])
    else:
        head = measure_eval(ctx, name, wl, args.steps, max(args.warmup, 3), "headline", sampler)
    sampler.stop_flag = True
    head_launches = head.get("launches_per_step", 0) * args.steps
    probes = link_probes(ctx)
    if "e2e" in head:
        head["e2e"].update(probes)
        head["e2e"]["frac_of_d2h_link_all_ranks"] = head["e2e"]["d2h_achieved_GBps_all_ranks"] / probes["d2h_link_GBps_all_ranks"]
        head["e2e"]["note2"] = ("bounded by the device-to-host copy of the result rows: compare d2h_achieved_GBps_all_ranks with "
                                "d2h_link_GBps_all_ranks, a plain pinned copy issued by all ranks at the same time")
    others = {}
    if not args.workload:
        for o in DEFAULT_OTHERS:
            try:
                owl = WORKLOADS[o]
                k = max(3, min(args.steps, 10 if owl.get("strong") else 20))
                others[o] = (measure_build(ctx, o, owl, min(k, 5), 2, "side") if owl["kind"] == "build"
                             else measure_eval(ctx, o, owl, k, 3, "side"))
                if "e2e" in others[o]:
                    others[o]["e2e"]["frac_of_d2h_link_all_ranks"] = (others[o]["e2e"]["d2h_achieved_GBps_all_ranks"]
                                                                      / probes["d2h_link_GBps_all_ranks"])
            except Exception as e:                              # a side measurement must not cost the headline
                import traceback
                others[o] = {"error": repr(e), "trace": traceback.format_exc()[-600:]}
                torch.cuda.empty_cache()
    total_launches = D.kernel_launch_count() - launches0

    if ctx.rank == 0:
        line = {
            "metric": "queries/s", "value": head.get("value"), "unit": head.get("unit", "queries/s"), "n_gpus": ctx.world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": head["scaling"], "vs_baseline": None, "dtype": wl["dtype"], "data": "synthetic",
            "config": workload_config(name, wl, ctx.world),
            "run": {"tables": "generated on rank 0, replicated per GPU by NCCL broadcast; queries sharded, no collective in the timed region",
                    "search_mode": args.search_mode, "numa_node": numa,
                    "launches_per_step": head.get("launches_per_step"),
                    "spline_route": head.get("spline_route"), "spline_build_info": head.get("spline_build_info"),
                    "timed": "every step between its own CUDA events on the launch stream; ms_per_step = (first start -> last end) / steps, "
                             "max over ranks; per_step = median / best / worst of the same steps",
                    "kernel_source_hash": kernel_source_hash(), "build_source_hash": kernel_source_hash(BUILD_SOURCES)},
            "roofline": head.get("roofline"),
            "per_step": head.get("per_step"),
            "check": head.get("check"),
            "cpu_baseline": head.get("cpu_baseline"),
            "spline_build": head.get("spline_build"),
            "e2e": head.get("e2e"),
            "workloads": others,
            "gpu_launches": int(head_launches) * ctx.world,
            "gpu_launches_all_workloads": int(total_launches) * ctx.world,
            "clocks": sampler.summary(),
        }
        if wl["kind"] == "build":
            line["metric"] = "columns/s"
            line["build"] = head
        print(json.dumps(line))
    if ctx.world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="timed steps of the headline workload")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="measure this workload only (default: c2 as the headline plus every other BASELINE config under `workloads`)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--search-mode", type=int, default=0,
                    help="lower-index search strategy for measurement (0 auto, 1 global bisect, 2 smem bisect, 3 guess, 4 bucket table, 5 merge)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline's last timed step computed as DIR/<name>.npy (a fixed, seeded sample "
                         "of a large output; at most 48 MB in all) so that two builds can be compared output for output")
    args = ap.parse_args()
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints "NCCL version ..." at the
    # first communicator, seen on the GPU boxes), so everything but the final line goes to stderr: file
    # descriptor 1 points at stderr while the run is in progress and is restored for the JSON line.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    out = io.StringIO()
    try:
        with contextlib.redirect_stdout(out):
            rc = run_reference(args) if args.impl == "reference" else run_b200(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    lines = [ln for ln in out.getvalue().splitlines() if ln.strip()]
    for ln in lines[:-1]:
        print(ln, file=sys.stderr)
    if lines:
        print(lines[-1], flush=True)
    return rc


if __name__ == "__main__":
    sys.exit(main())
