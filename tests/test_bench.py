"""bench.py --dump-outputs: what the last timed step computed, written so that two builds can be compared."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _load(d):
    return {n: np.load(os.path.join(d, n + ".npy")) for n in ("frame_pixels", "frame_pixel_index", "rays")}


def test_dump_outputs_samples_a_large_frame(tmp_path):
    """A 4K frame is larger than the dump may be: a fixed sample of its pixels, the same in every run, under 64 MB."""
    import bench

    h, w = 2160, 3840
    frame = np.random.default_rng(1).integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), frame, 123456789)
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    assert a["frame_pixels"].dtype == np.float32 and a["frame_pixel_index"].dtype == np.float64
    assert a["frame_pixels"].shape == (bench.DUMP_PIXELS, 3) and a["rays"].tolist() == [123456789.0]
    idx = a["frame_pixel_index"].astype(np.int64)
    assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < h * w
    assert np.array_equal(a["frame_pixels"], frame.reshape(-1, 3)[idx].astype(np.float32))
    for k in a:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.gpu
def test_dump_outputs_is_the_benchmarked_frame(tmp_path):
    """C2 fits the dump whole: the frame written equals the frame the run hashes, and the ray count is the step's."""
    out = tmp_path / "out"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
           "--workload", "C2", "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-800:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["gpu_launches"] == 2
    got = _load(str(out))
    w, h = line["config"]["width"], line["config"]["height"]
    assert np.array_equal(got["frame_pixel_index"], np.arange(w * h, dtype=np.float64))
    frame = got["frame_pixels"].astype(np.uint8)
    assert np.array_equal(got["frame_pixels"], frame.astype(np.float32))
    assert hashlib.sha256(frame.tobytes()).hexdigest() == line["frame_sha256"]
    assert got["rays"].tolist() == [line["rays_per_step"]]
