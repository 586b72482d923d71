"""CPU: the one-JSON-line contract of bench.py.  The B200 arm cannot run here, so its committed output
(profiles/r2_bench_head.json, written by `python bench.py` on a B200) is checked for the keys
and the internal consistency the driver relies on; the reference arm (CPU oracle) is executed for real."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def test_committed_b200_line_has_the_contract_keys():
    d = json.load(open(os.path.join(ROOT, "profiles", "r2_bench_head.json")))
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert BASE_KEYS | {"roofline", "clocks"} <= set(d)
    assert d["metric"] in base["metric"] and d["unit"] == "pairs/s" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and base["published"] == {}  # no published number for this metric
    assert "workload" in d["config"] and "model" not in d["config"] and d["dtype"] == "f32" and d["scaling"] == "weak"
    # value = pairs per step / time per step
    pairs = d["n_gpus"] * d["config"]["pairs_per_gpu_per_step"]
    assert abs(d["value"] - pairs / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
    assert "measured" in r["peak_source"] or "fallback" in r["peak_source"]
    # achieved = algorithmic bytes of the dominant kernel / its measured duration
    k = next(k for k in d["kernels"] if k["kernel"] == r["kernel"])
    assert abs(r["achieved"] - k["algo_bytes"] / (k["ms"] * 1e-3) / 1e9) <= 1e-6 * r["achieved"]
    # DRAM traffic from ncu agrees with the algorithmic bytes: no re-reads
    assert 0.9 < r["traffic"] / k["algo_bytes"] < 1.05
    e = d["e2e"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e)
    assert e["h2d_bytes_per_step"] > 3e9 and e["d2h_bytes_per_step"] > 0 and e["value"] < d["value"]
    assert d["gpu_launches"] >= 3 * d["steps"]
    c = d["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(c) and c["kind"] in ("port", "reference")
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(d["clocks"]["reasons"])
    # round 2: nominal-peak fractions, the non-HBM kernels on their own rooflines, the tensor-core variant
    assert 0 < r["frac_nominal"] < r["frac"] and 0.7 < r["pipeline_frac"] < 1.0
    patch = next(k for k in d["kernels"] if "patch" in k["kernel"])
    assert patch["bound"].startswith("lsu") and 0 < patch["frac"] < 1
    assert d["variant_fused_upsample"]["fused_soft_argmin_kernel"]["bound"] == "mufu"
    vc = d["variant_implicit_volume_conv"]
    assert vc["roofline"]["bound"] == "tensor" and 0 < vc["roofline"]["frac"] < 1 and vc["speedup"] > 1.0
    # the batch-pipelined schedule (patch loss of batch i under the HBM kernels of batch i+1): informational, faster
    bp = d["variant_batch_pipelined"]
    assert "error" not in bp and bp["unit"] == "pairs/s" and bp["ms_per_step"] < d["ms_per_step_eager"]
    assert abs(bp["value"] - pairs / (bp["ms_per_step"] * 1e-3)) <= 1e-6 * bp["value"] and 0.8 < bp["pipeline_frac"] < 1.0


def test_dump_outputs_writes_the_step_outputs_as_float32(tmp_path, monkeypatch):
    import numpy as np
    import torch

    import bench

    # at the bench's shapes: at most 64 MB in all
    assert 4 * (2 * bench.B * bench.H * bench.W + 1 + bench.VOLUME_SAMPLE) <= 64e6
    monkeypatch.setattr(bench, "VOLUME_SAMPLE", 100)
    vol = torch.randn(2, 8, 3, 5, 7)
    disp, vis = torch.rand(2, 1, 20, 28), torch.rand(2, 1, 20, 28)
    loss = torch.tensor(0.25)
    bench.dump_outputs(str(tmp_path / "out"), (vol, disp, loss, vis))
    got = {p.stem: np.load(p) for p in (tmp_path / "out").glob("*.npy")}
    assert sorted(got) == ["cost_volume_sample", "disparity", "fold_image", "loss"]
    assert all(a.dtype == np.float32 for a in got.values())
    assert np.array_equal(got["disparity"], disp.numpy()) and np.array_equal(got["fold_image"], vis.numpy())
    assert got["loss"] == np.float32(0.25)
    # the sample is fixed: the same flat indices on every run
    idx = torch.randint(vol.numel(), (bench.VOLUME_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
    assert np.array_equal(got["cost_volume_sample"], vol.reshape(-1)[idx].numpy())


def test_reference_arm_runs_and_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    ref = json.load(open(os.path.join(ROOT, "profiles", "r2_bench_head.json")))
    assert d["metric"] == ref["metric"] and d["unit"] == ref["unit"] and d["higher_is_better"] is True
    assert d["config"] == ref["config"]  # the driver compares the two arms' config dicts (`same_config`)
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1 and d["value"] > 0
