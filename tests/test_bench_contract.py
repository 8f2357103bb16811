"""bench.py contract on the CPU side: the reference arm prints exactly ONE JSON line on stdout with the keys the driver
reads, and the B200 arm refuses to run without a GPU instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600):
    env = dict(os.environ, OMP_NUM_THREADS=str(min(8, os.cpu_count() or 1)))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout,
                          cwd=ROOT, env=env)


def test_reference_arm_prints_one_json_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/sec" and d["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data",
                "config", "e2e", "cpu_baseline", "gpu_launches"):
        assert key in d, key
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["config"]["per_step_batch"] == 16          # fixed sample: the denominator must not move between runs
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_both_arms_share_the_metric_string():
    """The driver divides the two arms only when their metric strings are equal (round-1 lost its anchor to a one-word
    difference)."""
    sys.path.insert(0, ROOT)
    import bench

    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][0])
    assert d["metric"] == bench.metric_label("resnet50") == "images/sec (ResNet-50 training step)"
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"metric": metric_label(') == 2      # both arms take the label from the one shared helper


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_b200_arm_fails_loudly_without_gpu():
    r = _run("--steps", "1", "--warmup", "1", "--no-cpu-baseline", timeout=300)
    assert r.returncode != 0
    assert r.stdout.strip() == ""          # no JSON line from a fallback path
    assert "no CUDA device" in r.stderr or "CUDA" in r.stderr


def test_dump_outputs_writes_a_fixed_float32_sample(tmp_path):
    """--dump-outputs: float32 .npy files, the same parameter sample on every call, its size capped whatever the model."""
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench

    flat_p = torch.randn(3 * bench.DUMP_PARAM_SAMPLE)
    loss, correct = torch.tensor([6.9]), torch.tensor([0, 1, 1, 0], dtype=torch.int32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), "m", loss, correct, flat_p)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["m_correct.npy", "m_loss.npy", "m_params_sample.npy"]
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float32 and np.array_equal(a, b), n
    sample = np.load(tmp_path / "a" / "m_params_sample.npy")
    assert 0 < sample.size <= bench.DUMP_PARAM_SAMPLE and np.isin(sample, flat_p.numpy()).all()
    assert np.array_equal(np.load(tmp_path / "a" / "m_correct.npy"), [0, 1, 1, 0])
