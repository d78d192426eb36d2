"""The bench lines kept under profiles/ carry every key the measurement contract asks for and are internally
consistent (CPU check of recorded evidence; the driver's own BENCH_rNN.json is produced by the same code)."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
FINAL = ROOT / "profiles" / "r02_bench_b200_v7.json"
FINAL_REF = ROOT / "profiles" / "r02_bench_reference_v7.json"
SCALE = [ROOT / "profiles" / f"r02_bench_b200_{n}.json" for n in ("2gpu", "4gpu", "8gpu")]


def load(path):
    if not path.exists():
        pytest.skip(f"{path.name} is not in this checkout")
    return json.loads(path.read_text())


def check_common(d):
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "cpu_baseline"):
        assert k in d, k
    assert d["unit"] == "views/s" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["warmup"] >= 3 and d["steps"] >= 1
    assert "workload" in d["config"] and "model" not in d["config"]
    # value = views of all ranks per second of the max-over-ranks step time
    assert d["value"] == pytest.approx(d["n_gpus"] * 1000.0 / d["ms_per_step"], rel=1e-6)
    c = d["clocks"]
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert c["sm_mhz"] >= 0.9 * c["sm_max_mhz"]
    baseline_metric = json.loads((ROOT / "BASELINE.json").read_text())["metric"]
    assert d["metric"].split(",")[0] == baseline_metric.split(",")[0] == "fwd+bwd views/sec @1080p"


def test_final_bench_line_meets_the_contract():
    d = load(FINAL)
    check_common(d)
    assert d["impl"] == "b200" and d["n_gpus"] == 1
    e = d["e2e"]
    assert e["unit"] == "views/s" and 0 < e["value"] < d["value"]
    assert e["h2d_bytes_per_step"] >= 1920 * 1080 * 3 * 4 and e["d2h_bytes_per_step"] == 1920 * 1080 * 3 * 4
    assert d["gpu_launches"] == len(d["kernels"]) * d["steps"] > 0
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] == "GB/s" and r["kernel"] == "k_render_bwd"
    assert r["frac"] == pytest.approx(r["achieved"] / r["peak"], rel=1e-6) and 0 < r["frac"] < 1
    assert r["achieved"] == pytest.approx(r["algorithmic_bytes"] / (r["duration_ms"] * 1e-3) / 1e9, rel=1e-6)
    assert r["traffic"] >= r["algorithmic_bytes"]            # ncu DRAM bytes per launch vs the algorithmic figure
    assert (ROOT / r["traffic_source"].split(" ")[0]).exists()
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["unit"] == "views/s" and 1 <= cb["cores"] <= 32 and cb["value"] > 0 and cb["sample"]
    st = d["config"]["stage_ms"]
    assert sum(st.values()) < d["ms_per_step"] * 1.02          # the kernels' stage times fit inside the step


def test_final_reference_line_is_the_unmodified_reference_on_the_same_workload():
    d, r = load(FINAL), load(FINAL_REF)
    check_common(r)
    assert r["impl"] == "reference" and r["metric"] == d["metric"] and r["n_gpus"] == 1
    same = "synthetic 3M Gaussians, 1080p, SH deg 3"
    assert r["config"]["workload"].startswith(same) and d["config"]["workload"].startswith(same)
    assert r["e2e"] == {"value": r["value"], "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert r["cpu_baseline"]["kind"] == "reference" and r["cpu_baseline"]["value"] == r["value"]
    assert d["e2e"]["value"] / r["value"] > 8.0               # the round's target for the end-to-end ratio


@pytest.mark.parametrize("path", SCALE, ids=lambda p: p.stem)
def test_scaling_lines_are_whole_job_aggregates(path):
    d = load(path)
    check_common(d)
    assert d["n_gpus"] in (2, 4, 8) and len(d["per_rank"]["ms_per_step"]) == d["n_gpus"]
    assert max(d["per_rank"]["ms_per_step"]) == pytest.approx(d["ms_per_step"], rel=1e-6)


def test_bench_cli_parses_without_a_gpu():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    text = out.stdout + out.stderr  # bench.py keeps stdout for the one JSON line: everything else goes to stderr
    assert out.returncode == 0 and "--impl" in text and "--gpus" in text


def test_every_arm_names_the_same_workload():
    """config.workload of the b200, reference and reference-cpu lines comes from one constant."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_module", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    src = (ROOT / "bench.py").read_text()
    assert src.count('"workload": WORKLOAD') == 3 and bench.WORKLOAD.startswith("synthetic 3M Gaussians, 1080p, SH deg 3")
    assert bench.METRIC.startswith("fwd+bwd views/sec @1080p, 3M Gaussians")


def test_dumped_outputs_are_finite_float_arrays_within_64_mb(tmp_path):
    """--dump-outputs writes float32 / float64 arrays, all finite (culled gaussians included), at most 64 MB in all
    at the bench's image size and sample size; the sample of gaussians is the same from run to run."""
    import importlib.util

    import numpy as np
    import torch

    from gaussian_splatting_b200 import synth

    spec = importlib.util.spec_from_file_location("bench_module", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    n = bench.DUMP_ROWS + 1000
    g = synth.make_gaussians(n, "tiny", sh_degree=bench.SH_DEGREE, seed=0, requires_grad=True)
    for p in (g.xyz, g.rgb, g.opacity, g.scale, g.quaternion, g.sh):
        p.grad = torch.randn_like(p)
    mask = torch.rand(n, generator=torch.Generator().manual_seed(0)) < 0.3
    uv = torch.randn(int((~mask).sum()), 2)
    image = torch.rand(1080, 1920, 3)
    names = bench.dump_outputs(tmp_path / "a", image, mask, uv, g)
    bench.dump_outputs(tmp_path / "b", image, mask, uv, g)
    total = 0
    for name in names:
        a = np.load(tmp_path / "a" / f"{name}.npy")
        assert a.dtype in (np.float32, np.float64), name
        assert np.isfinite(a).all(), name
        assert np.array_equal(a, np.load(tmp_path / "b" / f"{name}.npy")), name
        total += (tmp_path / "a" / f"{name}.npy").stat().st_size
    assert total <= 64 * 2**20, total
    rows = np.load(tmp_path / "a" / "gaussian_rows.npy").astype(np.int64)
    culled = np.load(tmp_path / "a" / "culling_mask.npy")
    assert culled.tolist() == mask[rows].float().tolist() and culled.any()
    uv_rows = np.load(tmp_path / "a" / "uv.npy")
    assert (uv_rows[culled == 1] == 0).all()
    uv_all = np.zeros((n, 2), np.float32)
    uv_all[~mask.numpy()] = uv.numpy()
    assert np.array_equal(uv_rows, uv_all[rows])
