"""GPU test of bench.py's contract on a small system: ONE JSON line with the keys the driver
reads (metric/value/unit/..., roofline, cpu_baseline, e2e, clocks, gpu_launches), produced by
the CUDA path (gpu_launches > 0) and consistent with itself."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True,
                       text=True, timeout=560)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def test_bench_line_small_system(O, tmp_path):
    dump = tmp_path / "out"
    d = _bench("--size", "4096", "--iters", "50", "--steps", "3", "--warmup", "3", "--cpu-iters", "10",
               "--dump-outputs", str(dump))
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e",
                "gpu_launches", "clocks"):
        assert key in d, key
    assert d["metric"] == "cg_iterations_per_second" and d["unit"] == "iterations/s"
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 3 and d["dtype"] == "f64"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and "workload" in d["config"]
    assert d["value"] > 0 and abs(d["value"] - 3 * 50 / (d["ms_per_step"] * 3e-3)) <= 1e-6 * d["value"]
    # persistent schedule: ONE launch runs the whole loop; + init (2) + finalize (1) per step
    assert "persistent" in d["config"]["schedule"]
    assert d["gpu_launches"] == 3 * (1 + 3)
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and rf["achieved"] > 0
    assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert rf["algorithmic_bytes_per_launch"] == 50 * 8.0 * 4096 * 4096 and rf["launches_timed"] == 3
    assert abs(rf["launch_ms"] - d["ms_per_step"]) < 1e-9 and rf["graph_schedule_it_per_s"] > 0
    ck = d["check"]
    assert ck["ok"] is True and ck["ranks_bitwise_identical"] and ck["k"] == 50
    e = d["e2e"]
    assert 0 < e["value"] <= d["value"] * 1.05            # host copies + DEBUG block inside the timed region
    assert e["h2d_bytes_per_step"] == 16 * 4096 and e["d2h_bytes_per_step"] >= 8 * 4096
    cb = d["cpu_baseline"]
    if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "cgsolver_ref")):
        assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] > 0
    assert "sm_mhz" in d["clocks"] and "reasons" in d["clocks"]
    # --dump-outputs: what the last timed step returned, bit for bit the oracle's 50 iterations
    ref = O.solve(O.generate_lap2d(4096), O.init_source_term(4096), max_iter=50, nranks=1, nblk=148)
    out = {f.stem: np.load(f) for f in dump.glob("*.npy")}
    assert sorted(out) == ["converged", "iterations", "k", "rsnew", "rsold", "x"]
    assert all(a.dtype == np.float64 for a in out.values())
    assert np.array_equal(out["x"], ref.x)
    assert (out["k"], out["iterations"], out["converged"]) == (ref.k, len(ref.hist), ref.converged)
    assert (out["rsold"], out["rsnew"]) == (ref.rsold, ref.rsnew)


def test_bench_line_graph_schedule():
    """--schedule 0: the CUDA graph of four kernels per iteration; the roofline kernel is then the mat-vec."""
    d = _bench("--size", "4096", "--iters", "50", "--steps", "3", "--warmup", "3", "--no-cpu-baseline",
               "--schedule", "0")
    # 4 launches per iteration (mat-vec, p'Ap partials, update_xr, update_p) + init (2) + finalize (1) per step
    assert d["gpu_launches"] == 3 * (4 * 50 + 3) and "graph" in d["config"]["schedule"]
    rf = d["roofline"]
    assert rf["algorithmic_bytes_per_launch"] == 8.0 * 4096 * 4096 and rf["launches_timed"] == 50


def test_reference_arm_line_small_system():
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "cgsolver_ref")):
        pytest.skip("oracle/_ref not built")
    d = _bench("--impl", "reference", "--size", "2048", "--steps", "2", "--warmup", "1")
    assert d["impl"] == "reference" and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["value"] == d["value"]
