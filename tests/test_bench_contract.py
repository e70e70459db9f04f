"""bench.py's reference arm runs on the host cores only, so its JSON contract can be checked without a GPU:
one line, the keys a reader of the line relies on, rank != 0 silent.  On the GPU: --steps sets the timed steps and
--dump-outputs writes the same values for the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(extra_env=None, *args):
    env = dict(os.environ, **(extra_env or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1",
                           "--steps", "2", "--warmup", "1", *args], capture_output=True, text=True, env=env, timeout=300)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = run()
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "queries/s" and d["unit"] == "queries/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 2 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("c1") and d["gpu_launches"] == 0 and d["vs_baseline"] is None
    # `config` is the dictionary the GPU arm prints for the same workload and GPU count (bench.workload_config)
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config("c1", bench.WORKLOADS["c1"], 1)
    assert set(d["config"]) == {"workload", "queries_per_gpu", "columns", "l2"}


def test_reference_arm_other_ranks_exit_silently():
    r = run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2")
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_steps_and_dump_outputs_on_the_gpu(tmp_path):
    """the headline times exactly --steps steps, and two runs with the same arguments dump the same values"""
    dumps = []
    for i, steps in enumerate((4, 7)):
        d = tmp_path / str(i)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", str(steps),
                            "--warmup", "1", "--no-cpu", "--e2e-steps", "1", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr
        line = json.loads(r.stdout)
        assert line["steps"] == steps and line["per_step"]["n"] == steps and line["check"]["bit_exact"]
        assert sorted(os.listdir(d)) == ["c1_out.npy"]
        dumps.append(np.load(d / "c1_out.npy"))
    assert dumps[0].dtype == np.float64 and dumps[0].shape == (10_000, 1)
    assert np.array_equal(dumps[0], dumps[1])


def test_traffic_stamps_name_committed_captures_of_the_current_kernel_sources():
    """profiles/roofline_traffic.json: every entry points at ncu summaries that are in the tree, carries the commit of
    its capture, and -- as long as nobody has edited the evaluation kernels since -- the hash bench.py compares with"""
    sys.path.insert(0, ROOT)
    import bench
    d = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
    entries = {k: v for k, v in d.items() if k != "_note"}
    assert set(entries) == {"c2", "c3", "c4", "c5a", "c5b"}
    for name, e in entries.items():
        assert e["bytes"] > 0 and e["commit"] and len(e["source_hash"]) == 16
        for cap in e["capture"].split(" + "):
            assert os.path.exists(os.path.join(ROOT, cap.split(" (")[0])), cap
        traffic, stamp = bench.recorded_traffic(name, e["queries"])
        assert traffic == e["bytes"] and stamp["commit"] == e["commit"]
        assert stamp["current"] == (e["source_hash"] == bench.kernel_source_hash(bench.workload_sources(name)))
