"""`bench.py --dump-outputs DIR`: what the files hold, that the sample is fixed, and the argument checks.  CPU only:
the helper is fed a host tensor shaped like the headline decode's int32 [B, 2N] output."""
import os
import subprocess
import sys

import numpy as np
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_writes_a_fixed_sample(tmp_path):
    B = bench.DUMP_FRAMES + 1000
    bits = torch.from_numpy(np.random.RandomState(1).randint(0, 2, (B, 2 * bench.N_COUPLES)).astype(np.int32))
    counters = np.array([7, 3, B, B * 2 * bench.N_COUPLES], np.int64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), bits, counters)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["bits.npy", "counters.npy", "frame_index.npy"]
    total = 0
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)
        total += os.path.getsize(tmp_path / "a" / f)
    assert total <= 64 << 20
    idx = np.load(tmp_path / "a" / "frame_index.npy").astype(np.int64)
    assert len(idx) == bench.DUMP_FRAMES and np.all(np.diff(idx) > 0) and idx[-1] < B
    assert np.array_equal(np.load(tmp_path / "a" / "bits.npy"), bits.numpy()[idx].astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "a" / "counters.npy"), counters.astype(np.float64))


def test_dump_outputs_small_batch_keeps_every_frame(tmp_path):
    bits = torch.ones((16, 2 * bench.N_COUPLES), dtype=torch.int32)
    bench.dump_outputs(str(tmp_path), bits, np.zeros(4, np.int64))
    assert np.array_equal(np.load(tmp_path / "frame_index.npy"), np.arange(16, dtype=np.float64))
    assert np.load(tmp_path / "bits.npy").shape == (16, 2 * bench.N_COUPLES)


def test_bench_rejects_bad_arguments(tmp_path):
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), timeout=120)
        assert res.returncode == 2 and "error" in res.stderr, (extra, res.stderr[-500:])
    assert not os.listdir(tmp_path)
