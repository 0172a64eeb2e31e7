#!/usr/bin/env python3
"""Observed float32-vs-complex128 error of the channel-state demapper (b200dvb_demap_csi) per table and noise variance,
on the random channel of tests/test_gpu_fading.py (|h| log-uniform in [1e-20, 1e3] plus zeros, y = h c + noise):
the largest |dLLR|, the largest |dLLR| / max(1, |h|^2) and that over the test's bound LLR_ATOL * max(1, |h|^2)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from tests import vectors
from tests.test_gpu_fading import LLR_ATOL, _tables, channel_case, csi_error

for name, kind, table in _tables():
    rs = np.random.RandomState(vectors.BPS[name] * 10 + (kind == 'natural'))
    for nv in vectors.DEMAP_NOISE_VARS + [0.0001]:
        y, h = channel_case(rs, table, 100_003, nv)
        got, want, bound = csi_error(name, table, y, h, nv)
        err = np.abs(got - want)
        print(f"{name:7s} {kind:8s} nv={nv:<7g} max|dLLR| {err.max():.3e}  max|dLLR|/max(1,|h|^2) "
              f"{(err / (bound / LLR_ATOL[name])).max():.3e}  of bound {(err / bound).max():.3f}", flush=True)
