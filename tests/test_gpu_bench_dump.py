"""`bench.py --dump-outputs DIR` end to end on the GPU: two runs with the same arguments write identical files, and
what they hold is the headline decode's own output — bits equal to the C oracle's decode of the same device-generated
frames, counters equal to the errors of those decisions summed over the timed steps."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from oracle import oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILES = ("bits.npy", "frame_index.npy", "counters.npy")


def test_bench_dump_repeats_and_matches_the_oracle(tmp_path):
    import torch
    from modulations_b200 import dvb_rcs2_turbo as turbo
    B, steps = 4096, 2
    for d in ("a", "b"):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--frames", str(B), "--steps", str(steps),
                              "--warmup", "0", "--dump-outputs", str(tmp_path / d)],
                             capture_output=True, text=True, cwd=ROOT, timeout=1200)
        assert res.returncode == 0, res.stderr[-2000:]
    got = {f: np.load(tmp_path / "a" / f) for f in FILES}
    for f in FILES:
        assert np.array_equal(got[f], np.load(tmp_path / "b" / f)), f
    idx = got["frame_index.npy"].astype(np.int64)
    assert np.array_equal(idx, np.arange(B))                 # a batch this small is dumped whole

    # the same frames as run_ours, regenerated on the device, decoded by the oracle
    codec = turbo.DVBRCS2_Turbo(bench.N_COUPLES, bench.RATE, bench.ITERS)
    h = codec.handle
    info = torch.empty((B, codec.k_info), dtype=torch.uint8, device="cuda")
    coded = torch.empty((B, h.n_llr), dtype=torch.uint8, device="cuda")
    llr = torch.empty((B, h.n_llr), dtype=torch.float32, device="cuda")
    h.mc_generate_bpsk(B, 1.0 / (2.0 * (1 / 3) * 10 ** (bench.EBN0_DB / 10)), bench.LLR_SEED, 0, info, coded, llr)
    o = oracle.OracleTurbo(bench.N_COUPLES, bench.RATE, bench.ITERS, perm=codec.perm, inv_perm=codec.inv_perm)
    ref = o.decode_batch(llr.cpu().numpy(), threads=os.cpu_count() or 1)
    assert np.array_equal(got["bits.npy"], ref[idx].astype(np.float32))
    err = ref != info.cpu().numpy()
    want = steps * np.array([err.sum(), np.any(err, axis=1).sum(), B, B * codec.k_info], np.float64)
    assert np.array_equal(got["counters.npy"], want)
