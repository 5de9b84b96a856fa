"""bench.py's command line.  CPU: the reference arm (`--impl reference`, the CPU oracle port) prints ONE JSON line with
the contract's keys -- same metric / unit / config as the GPU arm, `impl`, a `cpu_baseline` describing the run and an
`e2e` object with zero host<->device bytes -- and times exactly `--steps` steps.  GPU: `--dump-outputs`."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["unit"] == "steps/s" and d["higher_is_better"] is True and d["scaling"] == "strong"
    assert "IPR-DCGAN" in d["metric"] and "512" in d["metric"] and d["data"] == "synthetic"
    assert d["value"] > 0 and abs(d["ms_per_step"] * d["value"] - 1000.0) < 1e-3 * 1000.0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None


def _bench(*args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT)


def test_reference_arm_times_the_requested_steps():
    out = _bench("--impl", "reference", "--batch", "8", "--steps", "41", "--warmup", "1")
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 41


def test_bad_arguments_are_refused(tmp_path):
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)],
                 ["--workload", "verify", "--dump-outputs", str(tmp_path)]):
        out = _bench(*args, timeout=60)
        assert out.returncode == 2 and "error" in out.stderr, (args, out.stderr[-2000:])
    assert not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_step(tmp_path):
    """--dump-outputs writes the last timed step's metrics (the ones the JSON line reports), the generated batch and the
    generator / discriminator state as float32 / float64 .npy files, 64 MB at most."""
    out = _bench("--steps", "2", "--warmup", "1", "--batch", "64", "--skip-cpu-baseline", "--skip-eager-baseline",
                 "--dump-outputs", str(tmp_path), timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["steps"] == 2
    names = sorted(f[:-4] for f in os.listdir(tmp_path))
    assert all(f.endswith(".npy") for f in os.listdir(tmp_path))
    assert sum(os.path.getsize(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)) <= 64 * 10 ** 6
    arrays = {n: np.load(os.path.join(tmp_path, n + ".npy")) for n in names}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    metrics = {n[len("metric."):]: float(a) for n, a in arrays.items() if n.startswith("metric.")}
    assert metrics == {k.replace("/", "."): v for k, v in d["last_metrics"].items()}
    assert arrays["fake_sample"].shape == (64, 3, 32, 32) and np.isfinite(arrays["fake_sample"]).all()
    assert "G.module.fc.0.weight" in arrays and "D.module.net.0.0.weight_orig" in arrays
