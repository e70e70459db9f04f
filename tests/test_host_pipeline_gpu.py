"""The host-buffer pipeline of the C ABI (ndi_api.cu: run_host_eval) against the CPU oracle, for every way a host
batch can travel: the mapped-memory path for results up to 256 KB, one chunk, and more chunks than the copy-in
stream keeps in flight -- into ordinary (pageable) numpy memory, which goes through pinned staging buffers and
the copy pool, into page-locked memory, which receives the chunks directly, and into a strided buffer.

Rows of 1024 f64 (8 KB): a direct chunk is 8192 rows and a staged chunk 2048, so 40 000 queries make 5 direct and
20 staged chunks.  A failing query stops the batch like the reference's loop: the reported query and axis are the
first failing ones, every row before it equals the oracle bit for bit, and the rows at and after it keep whatever
the caller's buffer held."""
import numpy as np
import pytest

from ndarray_interp_b200 import InterpolateError
from ndarray_interp_b200.errors import rust_debug
from ndarray_interp_b200.interp1d import BoundaryCondition, CubicSpline, Interp1DBuilder, Linear
from ndarray_interp_b200.interp2d import Interp2DBuilder
from oracle import oracle_py as O

pytestmark = pytest.mark.gpu

W = 1024
SENTINEL = -12345.5
# (queries, first failing query or None): mapped path, one chunk, many chunks; a failure in a chunk after the
# third (query 35 000: direct chunk 4, staged chunk 17) is read after the copy-in stream has wrapped around
CASES = [(20, None), (20, 0), (20, 7),
         (1500, None), (1500, 0), (1500, 700),
         (40_000, None), (40_000, 0), (40_000, 1000), (40_000, 35_000)]


@pytest.fixture(scope="module")
def tables():
    rng = np.random.default_rng(2024)
    g = np.cumsum(rng.uniform(0.5, 1.5, 64))
    y = rng.normal(size=(64, W))
    gx, gy = np.cumsum(rng.uniform(0.5, 1.5, 8)), np.cumsum(rng.uniform(0.5, 1.5, 8))
    z = rng.normal(size=(8, 8, W))
    cub = Interp1DBuilder.new(y).x(g).strategy(CubicSpline.new().boundary(BoundaryCondition.Natural)).build()
    return {
        "linear": Interp1DBuilder.new(y).x(g).strategy(Linear.new()).build(),
        "cubic": cub, "cubic_coeffs": cub.strategy.coefficients(cub),
        "bilinear": Interp2DBuilder.new(z).x(gx).y(gy).build(),
        "g": g, "y": y, "gx": gx, "gy": gy, "z": z,
    }


def queries(t, kind, nq, bad):
    """seeded in-range queries; the first failing one at `bad` and a second one on the last query"""
    rng = np.random.default_rng(nq + (bad or 0))
    if kind != "bilinear":
        q = rng.uniform(t["g"][0], t["g"][-1], nq)
        if bad is not None:
            q[-1] = t["g"][0] - 0.5
            q[bad] = t["g"][-1] + 1.0 + bad
        return (q,)
    qx, qy = rng.uniform(t["gx"][0], t["gx"][-1], nq), rng.uniform(t["gy"][0], t["gy"][-1], nq)
    if bad is not None:
        qx[-1] = t["gx"][0] - 0.5
        if bad == 0:
            qx[0] = t["gx"][-1] + 1.0
        else:
            qy[bad] = t["gy"][-1] + 1.0 + bad                # the y axis fails while x is in range
    return qx, qy


def oracle(t, kind, qs):
    """(rows over a sentinel-filled buffer, first failing query, its axis)"""
    out = np.full((qs[0].size, W), SENTINEL)
    if kind == "linear":
        _, out, bad = O.interp1d_linear(t["g"], t["y"], qs[0], False, out=out)
        return out, bad, 0
    if kind == "cubic":
        a, b = t["cubic_coeffs"]
        _, out, bad = O.interp1d_cubic(t["g"], t["y"], a, b, qs[0], 0, out=out)
        return out, bad, 0
    _, out, bad, axis = O.interp2d_bilinear(t["gx"], t["gy"], t["z"], qs[0], qs[1], False, out=out)
    return out, bad, axis


def output_buffer(kind, nq):
    if kind == "pageable":
        return np.full((nq, W), SENTINEL)
    if kind == "pinned":
        import torch
        pinned = torch.empty((nq, W), dtype=torch.float64, pin_memory=True)      # as bench.py's e2e leg
        assert pinned.is_pinned()
        out = pinned.numpy()                               # shares the page-locked memory and keeps it alive
        out[...] = SENTINEL
        return out
    return np.full((nq, 2 * W), SENTINEL)[:, ::2]


@pytest.mark.parametrize("nq,bad", CASES)
@pytest.mark.parametrize("out_kind", ["pageable", "pinned", "strided"])
@pytest.mark.parametrize("kind", ["linear", "cubic", "bilinear"])
def test_host_batch_matches_oracle(tables, kind, out_kind, nq, bad):
    qs = queries(tables, kind, nq, bad)
    want, want_bad, want_axis = oracle(tables, kind, qs)
    assert want_bad == (-1 if bad is None else bad)
    out = output_buffer(out_kind, nq)
    if bad is None:
        tables[kind].interp_array_into(*qs, out)
    else:
        name = "xy"[want_axis]
        msg = f"{name} = {rust_debug(qs[want_axis][bad])} is not in range"
        with pytest.raises(InterpolateError.OutOfBounds) as e:
            tables[kind].interp_array_into(*qs, out)
        assert str(e.value) == msg
    assert np.array_equal(out, want)
