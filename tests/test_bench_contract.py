"""The bench.py JSON contract, checked on the lines committed under profiles/ (produced on a B200 by scripts/gpu_profile_r1b.sh), on
the argument parser and (GPU) on a short run: a missing key would make the recorded bench results unusable."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle.oracle import nmse

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "e2e"]


def _load(name):
    return json.load(open(os.path.join(ROOT, "profiles", name)))


def test_our_line_has_every_contract_key():
    d = _load("r1_bench_ours.json")
    for k in BASE_KEYS + ["clocks", "gpu_launches", "roofline", "cpu_baseline"]:
        assert k in d, k
    assert d["n_gpus"] == 1 and d["higher_is_better"] is True and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["warmup"] >= 3 and d["gpu_launches"] == d["roofline"]["launches_per_step"] * d["steps"] > 0
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in d["e2e"], k
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] < d["value"]
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["bound"] == "hbm" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert abs(d["value"] * d["ms_per_step"] - 1000.0) < 1e-6 * 1000                    # tok/s x ms/token
    assert abs(r["achieved"] - r["algorithmic_bytes_per_step"] * d["value"] / 1e9) < 1e-6 * r["achieved"]
    for k in ("sm_mhz", "sm_max_mhz", "reasons"):
        assert k in d["clocks"], k
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    c = d["cpu_baseline"]
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in c, k
    assert c["kind"] in ("reference", "port")
    pp = d["pp512"]
    assert pp["roofline"]["bound"] == "tensor" and pp["e2e"]["h2d_bytes_per_step"] == 512 * 4096 * 4


def test_reference_line_contract():
    d = _load("r1_bench_reference.json")
    for k in BASE_KEYS + ["impl", "cpu_baseline"]:
        assert k in d, k
    assert d["impl"] == "reference" and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"]
    ours = _load("r1_bench_ours.json")
    assert d["metric"] == ours["metric"] and d["unit"] == ours["unit"] and d["config"]["workload"] == ours["config"]["workload"]


def test_traffic_file_matches_the_algorithmic_bytes():
    t = _load("r1_traffic.json")
    ours = _load("r1_bench_ours.json")
    ratio = t["tg"]["dram_bytes_per_step"] / ours["roofline"]["algorithmic_bytes_per_step"]
    assert 0.98 <= ratio <= 1.05, ratio          # ncu DRAM bytes per token vs sum of ggml_row_size: no wasted re-reads


def test_bench_cli_defaults():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--dump-outputs"):
        assert flag in out.stdout, flag


@pytest.mark.gpu
def test_bench_steps_and_dump_outputs(tmp_path):
    """--steps is the number of timed steps of every timed loop; --dump-outputs writes what the timed paths computed in their last step,
    from inputs that are the same in every run.  All 32 layers: the outputs must not decay to zero on the way through the model."""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu", "--no-mix"]
    dumps = []
    for run in range(2):
        out = tmp_path / str(run)
        r = subprocess.run(cmd + ["--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and line["pp512"]["steps"] == 2 and line["gpu_launches"] == 2 * line["roofline"]["launches_per_step"]
        dumps.append({f.stem: np.load(f) for f in out.glob("*.npy")})
    assert sorted(dumps[0]) == ["pp512_hidden", "pp512_logits", "tg_logits"]
    shapes = {"tg_logits": (1, 128256), "pp512_logits": (1, 128256), "pp512_hidden": (512, 4096)}
    for name, a in dumps[0].items():
        assert a.dtype == np.float32 and a.shape == shapes[name] and np.isfinite(a).all(), name
        assert float(np.sqrt((a.astype(np.float64) ** 2).mean())) > 1e-2, (name, "outputs vanish")
        # same inputs, so only the order of the split-K GEMM's f32 atomic adds may differ (other inputs would give an NMSE near 1)
        e = nmse(dumps[1][name], a)
        assert e <= 1e-4, (name, e)
