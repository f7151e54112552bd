"""bench.py's output contract, as far as it can be checked without a GPU: the reference arm (`--impl reference`) runs the unmodified
reference from oracle/_ref (or the torch port) on a bounded sample and prints ONE JSON line with the contract keys, with
the same `config` the GPU arm would print for those arguments."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--nodes", "60", "--supports", "3", "--obs", "4",
                        "--batch", "2", "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["gpu_launches"] == 0 and d["vs_baseline"] is None
    assert d["unit"] == "OD-cells/s" and d["higher_is_better"] is True and d["dtype"] == "f32" and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and "no size extrapolation" in cb["sample"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "OD-cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # value = credited cells / measured time of the sample: T * N * N / 6 cells per sample
    assert abs(d["value"] - (4 * 60 * 60 / 6.0) / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]
    sys.path.insert(0, ROOT)
    import bench
    a = type("A", (), dict(nodes=60, supports=3, obs=4, batch=2, hidden=32, precision="fp16", shard="batch", row_ranks=0))()
    assert d["config"] == bench.workload_config(a, 1)
    if os.path.isfile(os.path.join(ROOT, "oracle", "_ref", "MPGCN.py")):
        assert cb["kind"] == "reference"


def test_workload_table_matches_baseline_json():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.WORKLOADS["headline"][:3] == (1000, 3, 12) and bench.WORKLOADS["headline"][3] == 8        # SURVEY.md 8(d): headline B = 8
    assert bench.WORKLOADS["cfg2"] == (200, 3, 8, 16) and bench.WORKLOADS["cfg3"] == (500, 3, 12, 32)       # BASELINE.json configs[1], [2]
    assert bench.WORKLOADS["cfg4"][:3] == (1000, 6, 12) and bench.WORKLOADS["cfg5"][:3] == (2000, 3, 8)     # configs[3], [4]
