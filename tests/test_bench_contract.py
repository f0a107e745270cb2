"""bench.py prints ONE JSON line with the keys the driver reads (metric, value, unit, n_gpus, steps, warmup, ms_per_step,
higher_is_better, scaling, vs_baseline, dtype, data, config.workload, roofline, cpu_baseline, e2e, gpu_launches, clocks).
CPU: the reference arm (oracle on the host cores).  GPU: our arm on a small batch."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
             "data", "config"}


def _run(args, timeout=900):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-sample", "8"])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "audio-sec/sec" and d["unit"] == "audio-s/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_argument_errors():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode == 2 and "error:" in r.stderr and r.stdout == ""


@pytest.mark.gpu
def test_gpu_arm_line_small_batch(tmp_path):
    d = _run(["--batch", "16", "--steps", "3", "--warmup", "3", "--cpu-sample", "8", "--dump-outputs", str(tmp_path)])
    assert d["dump_outputs"]["rows"] == list(range(16))                # the whole small batch fits the 64 MB budget
    shapes = {"mixed": (16, 15, 80, 20), "speech": (16, 15, 80, 20), "noise": (16, 15, 80, 20), "mixed_pcm": (16, 48000),
              "recon": (16, 47840)}
    for name, shape in shapes.items():
        a = np.load(str(tmp_path / (name + ".npy")))
        assert a.shape == shape and a.dtype == np.float32 and np.isfinite(a).all(), name
    assert BASE_KEYS <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] >= 3 and d["scaling"] == "weak" and d["dtype"] == "f32" and d["data"] == "synthetic"
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9 and rf["achieved"] > 0
    assert d["gpu_launches"] == 3 * d["steps"]
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 2 * 16 * 48000 * 4 and e["d2h_bytes_per_step"] == 3 * 16 * 15 * 1600 * 4 + 16 * 48000 * 4
    assert 0 < e["value"] < d["value"]                   # host copies inside the timed region: slower than the resident path
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert d["inverse"]["value"] > 0
    su = d["sustained"]                                   # >= 2 s of back-to-back steps beside the short headline region
    assert su["seconds"] >= 2.0 and su["steps"] >= d["steps"] and su["value"] > 0
    c = e["ceiling"]                                      # bare pinned-memcpy ceiling of the same buffers, measured live
    assert c["ms_per_step"] > 0 and c["h2d_alone_gbs"] > 0 and c["d2h_alone_gbs"] > 0 and 0 < e["frac_of_ceiling"] <= 1.5


@pytest.mark.gpu
def test_corpus_mode_line():
    """BASELINE configs[2] shape at a small size: a corpus sharded by utterance (strong scaling), one pass per step."""
    d = _run(["--corpus", "96", "--batch", "40", "--steps", "2", "--warmup", "3"])
    assert BASE_KEYS <= set(d) and d["scaling"] == "strong" and d["n_gpus"] == 1
    assert d["config"]["corpus_utterances"] == 96 and d["config"]["utterances_per_launch"] == 40
    assert d["gpu_launches"] == 3 * 3 * 2 and d["value"] > 0
