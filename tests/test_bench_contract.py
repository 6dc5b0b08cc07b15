"""The bench.py JSON contract, checked on the committed record of the last B200 run (profiles/r2_bench_1gpu.json, or the
round-1 record while that does not exist) and on the argument parser; the output dump of --dump-outputs on the host
(writer, size budget) and, on the GPU, through a short bench run."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

REPO = Path(__file__).resolve().parents[1]


def _record():
    for name in ("r2_bench_1gpu.json", "r1_bench_1gpu.json"):
        p = REPO / "profiles" / name
        if p.exists():
            return json.loads(p.read_text()), name
    raise FileNotFoundError("no bench record under profiles/")


def test_recorded_line_has_every_contract_key():
    d, name = _record()
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"):
        assert k in d, k
    base = json.loads((REPO / "BASELINE.json").read_text())
    assert "samples/sec" in base["metric"] and d["metric"] == "audio_samples_per_sec" and d["unit"] == "samples/s"
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"] and "model" not in d["config"]
    assert abs(d["value"] - 32 * 312 * 256 / (d["ms_per_step"] / 1e3)) / d["value"] < 1e-6
    e = d["e2e"]
    assert e["unit"] == d["unit"] and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] == 32 * 312 * 256 * 4
    assert e["value"] != d["value"]                     # measured separately, through host buffers
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or r["traffic"] > 0
    c = d["cpu_baseline"]
    assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    assert d["gpu_launches"] > 0 and d["gpu_launches"] % d["steps"] == 0     # every step launches the same kernels, all ours
    if name.startswith("r2"):
        # round 2: the other BASELINE configs and the per-stage rooflines travel in the same line
        assert set(d["sweep"]) >= {"1", "8", "32", "128"} and d["strict_fp32"]["value"] > 0
        assert set(d["configs"]) >= {"c4", "c5"} and d["configs"]["c5"]["padding_frac"] <= 0.08
        assert {"nat_decoder_scan", "hifigan_stage0", "hifigan_stage3", "hifigan_conv_post", "melspec"} <= set(d["roofline_stages"])
        assert d["e2e"]["pageable_result"]["value"] > 0
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_bench_cli_flags():
    out = subprocess.run([sys.executable, str(REPO / "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--dump-outputs"):
        assert flag in out.stdout
    bad = subprocess.run([sys.executable, str(REPO / "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert bad.returncode != 0 and "--steps" in bad.stderr


def test_dump_outputs_budget_and_sample(tmp_path):
    import bench
    rng = np.random.default_rng(0)
    a, b = rng.standard_normal((3, 50, 8)), rng.standard_normal((3, 4000))
    bench.dump_outputs(tmp_path / "whole", dict(mel=a, wav=b))
    for name, x in (("mel", a), ("wav", b)):
        got = np.load(tmp_path / "whole" / f"{name}.npy")
        assert got.dtype == np.float32 and got.shape == x.shape and np.array_equal(got, x.astype(np.float32))
    budget = 16 << 10                                   # smaller than the 52.8 kB the two arrays take
    for run in ("s1", "s2"):
        bench.dump_outputs(tmp_path / run, dict(mel=a, wav=b), budget=budget)
    files = sorted((tmp_path / "s1").glob("*.npy"))
    assert [f.name for f in files] == ["mel.npy", "wav.npy"] and sum(f.stat().st_size for f in files) <= budget
    for f in files:
        got, again = np.load(f), np.load(tmp_path / "s2" / f.name)
        src = (a if f.stem == "mel" else b).astype(np.float32).reshape(-1)
        assert got.dtype == np.float32 and got.ndim == 1 and 0 < got.size < src.size
        assert np.array_equal(got, again) and np.isin(got, src).all()       # the same seeded positions every run


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    cmd = [sys.executable, str(REPO / "bench.py"), "--steps", "2", "--warmup", "1", "--batch", "2", "--no-cpu", "--no-callers",
           "--no-sweep", "--no-configs", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2
    n = d["config"]["mel_frames"]
    mel, wav = np.load(tmp_path / "mel.npy"), np.load(tmp_path / "wav.npy")
    assert mel.dtype == wav.dtype == np.float32 and mel.shape == (2, n, 80) and wav.shape == (2, 256 * n)
    assert np.isfinite(mel).all() and np.isfinite(wav).all() and np.abs(wav).max() > 0
