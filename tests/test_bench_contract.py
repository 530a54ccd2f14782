"""bench.py contract (task prompt / DESIGN.md §d): the reference arm runs here on the CPU; the native arm's line
is checked on the committed round-1 output."""
import json
import os
import subprocess
import sys

from conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def test_reference_arm_runs_on_cpu_and_prints_the_contract_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert BASE_KEYS <= set(line) and line["impl"] == "reference"
    assert line["metric"] == "gp_lml_grad_evals_per_sec" and line["unit"] == "evals/s" and line["dtype"] == "f64"
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["value"] > 0


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_zero_steps_is_rejected():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                       text=True, timeout=120)
    assert p.returncode == 2 and "--steps" in p.stderr


def test_dump_outputs_is_float64_bounded_and_repeatable(tmp_path):
    import importlib.util

    import numpy as np

    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    arrays = {"big": np.arange(9_000_000, dtype=np.float64).reshape(3000, 3000), "small": np.arange(7, dtype=np.int32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    total = sum(f.stat().st_size for f in (tmp_path / "a").iterdir())
    assert total <= 64_000_000
    small = np.load(tmp_path / "a" / "small.npy")
    assert small.dtype == np.float64 and np.array_equal(small, arrays["small"])
    big_a, big_b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert big_a.dtype == np.float64 and 0 < big_a.size < arrays["big"].size
    assert np.array_equal(big_a, big_b) and np.all(np.diff(big_a) > 0)      # same positions, in storage order


def test_committed_native_line_has_every_contract_key():
    line = json.load(open(os.path.join(ROOT, "profiles", "r01c_bench_n1.json")))
    assert BASE_KEYS | {"clocks", "gpu_launches", "roofline"} <= set(line)
    assert line["metric"] == "gp_lml_grad_evals_per_sec" and line["higher_is_better"] is True
    assert line["vs_baseline"] is None and line["data"] == "synthetic" and line["scaling"] == "weak"
    r = line["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "tensor"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and r["traffic"] > 0
    e = line["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] > 0
    assert line["gpu_launches"] > 0 and "workload" in line["config"] and "model" not in line["config"]
    c = line["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(c)
    assert not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(line["clocks"]["reasons"]))
