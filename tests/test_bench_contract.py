"""bench.py's command line: the reference arm prints one JSON line with the result's keys (runs the real CPU path on
one image); our arm's --dump-outputs files (GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--ref-images", "1"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "tokens/s" and d["higher_is_better"] is True
    assert d["metric"] == "vision tokens/s crop->patchify->ViT" and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "--steps must be at least 1" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_same_inputs_same_files(cuda, tmp_path):
    """--dump-outputs writes the last timed step's embeddings, grids and crop boxes as float32 / float64 .npy files
    (64 MiB at most), and two runs with the same arguments write the same values: the inputs are seeded."""
    import numpy as np
    runs = []
    for name in ("a", "b"):
        out = tmp_path / name
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--images", "2",
                            "--no-e2e", "--no-cpu", "--no-sharded", "--no-latency", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900, cwd=tmp_path)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert d["steps"] == 2 and d["config"]["images_per_step_per_gpu"] == 2
        files = sorted(os.listdir(out))
        assert files == ["crop_boxes.npy", "embeddings.npy", "image_grid_thw.npy"]
        assert sum(os.path.getsize(out / f) for f in files) <= 64 << 20
        arrays = {f: np.load(out / f) for f in files}
        assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
        runs.append(arrays)
    a = runs[0]
    assert a["embeddings.npy"].shape == (2 * 1225, 2048) and np.isfinite(a["embeddings.npy"]).all()
    assert a["image_grid_thw.npy"].tolist() == [[1, 70, 70]] * 2
    assert a["crop_boxes.npy"].tolist() == [[0, 0, 5000, 5000]] * 2
    for f in a:
        assert np.array_equal(a[f], runs[1][f]), f


def test_our_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
