"""The reference arm of bench.py honours the output contract — exactly ONE JSON line on stdout with the keys a caller
reads (the GPU arm shares the same printing code); on a GPU, the cfg2 arm times exactly `--steps` updates and
`--dump-outputs` writes what the last of them computed."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "updates/s"
    assert d["metric"].startswith("metric-updates/sec") and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["config"]["workload"].startswith("MulticlassConfusionMatrix")


def test_reference_arm_non_zero_rank_exits_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], cwd=ROOT, capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_gpu_arm_times_k_steps_and_dumps_the_last_one(tmp_path):
    """`--steps K` times exactly K update() launches, and `--dump-outputs` writes the confusion matrix of the last of them:
    with K = 2 that is the host-generated seed-1 batch, checked against the numpy oracle."""
    import numpy as np

    from bench import make_batch
    from oracle.classification import multiclass_confusion_matrix

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-extras",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout)
    assert d["steps"] == 2 and d["gpu_launches"] == 2
    assert sorted(os.listdir(tmp_path)) == ["confmat.npy"]
    got = np.load(tmp_path / "confmat.npy")
    logits, target = make_batch(1)
    assert got.dtype == np.float64
    assert np.array_equal(got, multiclass_confusion_matrix(logits.float().numpy(), target.numpy(), 1000))


def test_dump_outputs_is_refused_outside_the_cfg2_gpu_line(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr and out.stdout.strip() == ""
    assert not os.listdir(tmp_path)
