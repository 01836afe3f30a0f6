"""GPU: `bench.py --dump-outputs DIR` writes what the timed path computed in its last timed step, from inputs that are
the same in every run with the same arguments."""
import json
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, keypoint_agreement, rel_err

pytestmark = pytest.mark.gpu


def test_bench_dump_outputs(tmp_path):
    cmd = [sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--images-per-step", "3",
           "--no-cpu-baseline", "--dump-outputs"]
    runs = []
    for k in range(2):
        out = subprocess.run(cmd + [str(tmp_path / f"run{k}")], capture_output=True, text=True, timeout=600, cwd=tmp_path)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 2 and line["warmup"] == 1
        runs.append({p.stem: np.load(p) for p in (tmp_path / f"run{k}").glob("*.npy")})
    a, b = runs
    assert sorted(a) == ["heatmap", "homographies", "keypoint_counts", "keypoints"]
    assert all(v.dtype == np.float32 for v in a.values())
    assert a["heatmap"].shape == (3, 240, 320) and a["homographies"].shape == (3, 99, 3, 3)
    counts = a["keypoint_counts"].astype(np.int64)
    assert counts.shape == (3,) and counts.min() > 0 and a["keypoints"].shape == (counts.sum(), 2)
    # every keypoint is a pixel of its image whose aggregated heat passed the detection threshold (0.015)
    img = np.repeat(np.arange(3), counts)
    r, c = a["keypoints"][:, 0].astype(np.int64), a["keypoints"][:, 1].astype(np.int64)
    assert (r >= 0).all() and (r < 240).all() and (c >= 0).all() and (c < 320).all()
    assert (a["heatmap"][img, r, c] >= 0.015).all()
    # same arguments, same inputs: the sampled homographies are identical and the outputs agree
    assert np.array_equal(a["homographies"], b["homographies"])
    assert rel_err(b["heatmap"], a["heatmap"]) < 1e-5
    splits = np.cumsum(counts)[:-1]
    for ka, kb in zip(np.split(a["keypoints"], splits), np.split(b["keypoints"], np.cumsum(b["keypoint_counts"].astype(np.int64))[:-1])):
        assert min(keypoint_agreement(ka, kb)) >= 0.99
