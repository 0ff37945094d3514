"""The bench line's contract (the driver parses it): checked on the committed output of the final `python bench.py` run of
the round (profiles/round2_bench_final.json), and on the N=4 line for the multi-GPU keys.  CPU-only: no GPU work here."""
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load(name):
    path = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(path):
        pytest.skip(f"{name} not committed")
    return json.loads(open(path).read().strip().splitlines()[-1])


def test_single_gpu_line_carries_every_contract_key():
    d = load("round2_bench_final.json")
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))   # "512² patches/s (50-step TeReDiff) at 1/2/4/8 B200; ..."
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in d, k
    assert "patches/s" in base["metric"] and "50-step" in base["metric"]
    assert d["metric"] == "patches_per_s_50step_512px" and d["unit"] == "patches/s"
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "bf16"
    assert "workload" in d["config"] and "model" not in d["config"]
    e = d["e2e"]
    assert e["unit"] == d["unit"] and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    assert 0.5 * d["value"] < e["value"] <= 1.05 * d["value"] and e["value"] != d["value"]
    assert d["gpu_launches"] > 0
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s")
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-6 and 0 < r["frac"] <= 1 and r["traffic"]
    c = d["cpu_baseline"]
    assert c["kind"] in ("reference", "port") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    ck = d["clocks"]
    assert ck["sm_mhz"] and ck["sm_max_mhz"] and not set(ck["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    # the wider path of the north star, all from the same run
    assert d["full_step"]["unit"] == d["unit"] and d["full_step"]["ms_per_denoise_step"] > d["unet_step_latency_ms"]
    px = d["e2e_pixels"]
    assert px["tiles"] == 25 and px["h2d_bytes_per_image"] == 512 * 512 * 3 and px["d2h_bytes_per_image"] == 3 * 2048 * 2048 * 4
    assert set(d["cfg_sweep"]["tiles_per_gpu"]) == {"1", "4", "16", "32"}
    assert d["norm_families"]["family_ms"] > 0 and d["gpu_eager_baseline"]["value"] < d["value"]


def test_dump_outputs_writes_float_npy_within_the_limit(tmp_path):
    import sys
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    out = tmp_path / "dump"
    lat = np.random.default_rng(0).standard_normal((2, 4, 8, 8)).astype(np.float32)
    bench.dump_outputs(str(out), {"latent": lat, "polys": np.arange(32, dtype=np.int32).reshape(1, 16, 2),
                                  "table": np.linspace(0, 1, 5)})
    assert sorted(p.name for p in out.iterdir()) == ["latent.npy", "polys.npy", "table.npy"]
    assert np.array_equal(np.load(out / "latent.npy"), lat)
    assert np.load(out / "polys.npy").dtype == np.float32 and np.load(out / "table.npy").dtype == np.float64
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_LIMIT_BYTES // 4 + 1, np.float32)})
    assert not (tmp_path / "big").exists()


def _bench_error(*argv):
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True)
    return r.returncode != 0, r.stderr


def test_bench_rejects_zero_timed_steps():
    failed, err = _bench_error("--steps", "0")
    assert failed and "--steps" in err


def test_bench_reference_arm_rejects_dump_outputs():
    failed, err = _bench_error("--impl", "reference", "--dump-outputs", "unused")
    assert failed and "--dump-outputs" in err


def test_multi_gpu_line_reports_the_collective_and_every_rank():
    d = load("round2_bench_4gpu_late.json")
    assert d["n_gpus"] == 4 and d["scaling"] == "weak"
    assert len(d["per_rank"]["ms_per_denoise"]) == 4 and len(d["per_rank"]["sm_mhz"]) == 4
    assert abs(max(d["per_rank"]["ms_per_denoise"]) - d["ms_per_step"]) < 0.5      # the headline is the max over ranks
    px = d["e2e_pixels"]
    assert "all_gather" in px["collective"] and px["scaling"] == "strong" and px["tiles_per_rank_max"] == 7
    assert "cpu_baseline" not in d
