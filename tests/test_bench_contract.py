"""bench.py contract on CPU: the reference arm prints exactly ONE JSON line on stdout with the agreed keys, and the
product arm refuses to run without a CUDA device (there is no CPU fallback).  Both arms run exactly --steps timed
steps, and --dump-outputs writes what the last of them returned."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]


def _run(*args, timeout=600):
    env = dict(os.environ, OMP_NUM_THREADS=os.environ.get("OMP_NUM_THREADS", "8"))
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=timeout,
                          env=env, cwd=str(ROOT))


def test_reference_arm_prints_one_json_line_with_contract_keys():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "images_per_sec" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "f32"
    assert d["value"] > 0 and d["steps"] >= 1 and d["ms_per_step"] > 0
    assert "workload" in d["config"] and "yolo11n" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def _bench_model():
    """The model bench.py times, built the same way (seeded init + randomised BN statistics)."""
    import bench
    from yololite.nn.tasks import DetectionModel

    torch.manual_seed(0)
    return bench.randomise_model_(DetectionModel("yolo11n.yaml", verbose=False)).eval()


def _load_dump(d):
    dets, counts = np.load(d / "dets.npy"), np.load(d / "counts.npy")
    assert dets.dtype == np.float32 and counts.dtype == np.float64
    assert dets.shape == (counts.shape[0], 300, 6)
    for i, n in enumerate(counts.astype(int)):
        assert not dets[i, n:].any()                     # rows past the count are zeroed
    return dets, counts.astype(int)


def test_reference_arm_runs_exactly_steps_and_dumps_its_last_step(tmp_path):
    import bench

    r = _run("--impl", "reference", "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    dets, counts = _load_dump(tmp_path)
    sd = {k: v.detach().clone() for k, v in _bench_model().state_dict().items()}
    want = bench.cpu_reference_step(sd, bench.synth_images(8, 1, seed=0)[0])
    assert counts.tolist() == [len(w) for w in want] and counts.sum() > 0
    for i, w in enumerate(want):
        np.testing.assert_array_equal(dets[i, :len(w)], w)


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(tmp_path):
    """With --steps 2 the last timed step ran on the second input batch: the dump equals infer_nms on that batch."""
    import bench

    r = _run("--steps", "2", "--warmup", "1", "--repeats", "1", "--no-extras", "--no-e2e", "--no-latency",
             "--no-roofline", "--no-cpu-baseline", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    dets, counts = _load_dump(tmp_path)
    x = bench.synth_images(64, 2, seed=0)[1].cuda()
    d, c = _bench_model().cuda().infer_nms(x, bench.CONF, bench.IOU, None, False, False, bench.MAX_DET)
    torch.cuda.synchronize()
    assert counts.tolist() == c.tolist() and counts.sum() > 0
    for i, n in enumerate(counts):
        np.testing.assert_array_equal(dets[i, :n], d[i, :n].cpu().numpy())


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a machine without CUDA")
def test_product_arm_fails_loudly_without_cuda():
    r = _run("--steps", "1", "--warmup", "3")
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout)
    assert not [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
