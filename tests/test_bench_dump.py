"""`bench.py --dump-outputs DIR`: the outputs of the last timed step as float .npy files, whole while they fit under
the size cap and as a fixed, seeded sample of records beyond it; on the GPU, the dumped frame is the frame the oracle
renders for the same workload."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_outputs_that_fit_are_written_whole(tmp_path):
    frame = np.arange(6 * 5 * 4, dtype=np.uint8).reshape(6, 5, 4)
    bench.dump_outputs(str(tmp_path), {"frame": frame, "count": np.array([3, 9], dtype=np.int64)})
    assert sorted(os.listdir(tmp_path)) == ["count.npy", "frame.npy"]
    got = np.load(tmp_path / "frame.npy")
    assert got.dtype == np.float32 and np.array_equal(got, frame)
    count = np.load(tmp_path / "count.npy")
    assert count.dtype == np.float64 and count.tolist() == [3, 9]


def test_outputs_over_the_cap_are_the_same_sample_every_run(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 40_000)
    rng = np.random.default_rng(5)
    arrays = {"frame": rng.integers(0, 256, (64, 64, 4), dtype=np.uint8),
              "light": rng.integers(0, 256, (16, 16, 16, 4), dtype=np.uint8),
              "count": np.array([7], dtype=np.int64)}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["count.npy", "frame.npy", "frame_index.npy", "light.npy", "light_index.npy"]
    assert sum(np.load(tmp_path / "a" / f).nbytes for f in files) <= 40_000
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    for name in ("frame", "light"):
        index = np.load(tmp_path / "a" / f"{name}_index.npy").astype(np.int64)
        assert len(index) > 0 and np.all(np.diff(index) > 0)
        assert np.array_equal(np.load(tmp_path / "a" / f"{name}.npy"), arrays[name].reshape(-1, 4)[index])


@pytest.mark.gpu
def test_dumped_frame_is_the_oracle_frame(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c0", "--steps", "2", "--warmup", "1",
                        "--cpu-seconds", "1", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    frame = np.load(tmp_path / "frame.npy")
    from aicb200 import scenes
    space, opts, w, h, _ = bench.make_workload("c0")
    cam = scenes.standard_camera(space, opts, w, h)
    prev = orc.get_libm()
    orc.set_libm(orc.LIBM_CR)   # powf / expf in f64, rounded once, as the device evaluates them
    try:
        ref = orc.OracleScene(space).render(cam, opts)["srgb8"].reshape(h, w, 4)
    finally:
        orc.set_libm(prev)
    assert frame.dtype == np.float32 and frame.shape == (h, w, 4)
    assert np.array_equal(frame, ref.astype(np.float32))
