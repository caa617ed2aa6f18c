"""bench.py contract pieces: the reference arm (CPU oracle port) prints the required JSON line on rank 0 and stays silent
on the other ranks; the GPU arm refuses to run without CUDA; on a GPU, --dump-outputs writes the last timed step's
outputs and repeats them from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env, *args):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", **extra_env)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=600, env=env)


def test_reference_arm_prints_the_contract_line_on_rank0_only():
    args = ("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--cpu-rays", "2", "--levels", "2")
    r0 = _run({"RANK": "0", "WORLD_SIZE": "2"}, *args)
    assert r0.returncode == 0, r0.stderr[-400:]
    line = json.loads([ln for ln in r0.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "rays/s" and line["higher_is_better"] is True
    assert line["n_gpus"] == 2 and line["steps"] == 1 and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["metric"].startswith("training rays/sec") and "workload" in line["config"]
    r1 = _run({"RANK": "1", "WORLD_SIZE": "2"}, *args)
    assert r1.returncode == 0 and not [ln for ln in r1.stdout.splitlines() if ln.startswith("{")]


def test_gpu_arm_fails_loudly_without_cuda():
    r = _run({"RANK": "0", "WORLD_SIZE": "1"}, "--steps", "1", "--warmup", "1", "--no-cpu-baseline")
    assert r.returncode != 0
    assert "needs a GPU" in (r.stderr + r.stdout)


def test_executed_red_count_of_the_static_scatter():
    """bench.py's RED-rate binding of k_bwd_scatter_static uses the reductions the kernel EXECUTES: 8 per level, and at the
    warp-aggregated levels 8 per run of consecutive samples that share a cell (host-side run statistics of the rays)."""
    sys.path.insert(0, ROOT)
    import bench
    from lidar4d_b200.geometry import FieldConfig
    from lidar4d_b200.rays import synthetic_sweep
    cfg = FieldConfig(**bench.model_kwargs(16))
    assert bench.red_counts(cfg)["k_bwd_scatter_static"] == 128.0
    ro, rd, _ = synthetic_sweep(7)
    r = bench.red_counts(cfg, (ro, rd))
    agg = int((cfg.static_grid().resolution <= bench.STATIC_AGG_RES).sum())
    assert agg == 4 and r["k_bwd_scatter_static_algorithmic"] == 128.0
    assert 128.0 - 8.0 * agg < r["k_bwd_scatter_static"] < 128.0          # runs exist, and no level disappears
    # a ray that stays inside one cell for a whole warp issues 8 reductions per 32 samples at an aggregated level
    still = (np.zeros((4, 3), np.float32), np.zeros((4, 3), np.float32))
    assert abs(bench.red_counts(cfg, still)["k_bwd_scatter_static"] - (128.0 - 8.0 * agg * (1 - 1 / 32))) < 1e-6
    # the macro the count mirrors
    src = open(os.path.join(ROOT, "lidar4d_b200", "csrc", "l4d_split.cuh")).read()
    assert f"#define L4D_STATIC_AGG_RES {bench.STATIC_AGG_RES}" in src


def test_committed_bench_line_carries_the_contract_keys():
    """The last GPU bench line of the round (profiles/r02_v8_bench.json, written by `python bench.py` on a B200) has every key
    the bench contract names and a roofline fraction <= 1 against the unit that binds the dominant kernel."""
    line = json.load(open(os.path.join(ROOT, "profiles", "r02_v8_bench.json")))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in line, k
    assert line["warmup"] >= 3 and line["gpu_launches"] > 0 and "workload" in line["config"] and "l2" in line["config"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["value"] < line["value"] * 1.001
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(line["clocks"]) and not line["clocks"]["reasons"]
    r = line["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and 0 < r["frac"] <= 1.0
    assert {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"])
    ks = r["kernels"]
    assert abs(sum(v["avg_ms"] for k, v in ks.items() if "adam" not in k) * 4 - line["ms_per_step"]) < 0.03 * line["ms_per_step"]
    b = ks["k_bwd_scatter_static"]["binding"]
    assert b["frac"] <= 1.0 and b["red_lane_ops_per_sample_executed"] < b["red_lane_ops_per_sample_algorithmic"]


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs writes what the last timed step computed as float32 / float64 .npy files within 64 MB, and two runs
    with the same arguments start from the same inputs: the first step's forward outputs agree, its gradients agree up to
    the re-ordering of fp32 atomics."""
    args = ("--rays", "2048", "--ray-batch", "1024", "--levels", "8", "--steps", "1", "--warmup", "0", "--eager-rays", "0",
            "--no-cpu-baseline")
    runs = []
    for k in range(2):
        out = tmp_path / f"run{k}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900, env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
        assert r.returncode == 0, r.stderr[-800:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 1 and line["warmup"] == 0
        runs.append({f[:-len(".npy")]: np.load(out / f) for f in os.listdir(out)})
    a, b = runs
    assert set(a) == {"depth", "image", "loss", "grad_sample", "param_sample"}
    assert a["depth"].shape == (2048,) and a["image"].shape == (2048, 2) and a["loss"].shape == (1,)
    assert a["grad_sample"].shape == a["param_sample"].shape
    assert all(v.dtype in (np.float32, np.float64) for v in a.values()) and sum(v.nbytes for v in a.values()) <= 64 << 20
    assert all(np.isfinite(v).all() for v in a.values()) and np.abs(a["grad_sample"]).max() > 0
    for k in ("depth", "image", "loss"):
        assert np.abs(a[k] - b[k]).max() <= 1e-6 * np.abs(b[k]).max(), k
    assert np.abs(a["grad_sample"] - b["grad_sample"]).max() <= 1e-4 * np.abs(b["grad_sample"]).max()
