#!/usr/bin/env python3
"""Observed float32-vs-float64 error of every waveform kernel instance, as a fraction of the bound that
tests/test_gpu_waveform_kernels.py asserts: (K + 1) * 2^-24 * sum_t |h_t| |x_{m,t}| per output and component.
Gaussian data at three scales, random taps and RRC taps (the test's float cases, 16 seeds per instance)."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.test_gpu_waveform_kernels import INSTANCES, float_case, float_error_ratio

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(f"# {smi} (nvidia-smi, read in the same call)")
print("# python tools/waveform_err.py: largest |kernel - float64| / ((K + 1) 2^-24 sum |h||x|) over 16 cases per instance")
for inst in INSTANCES:
    name, kind, sps, nt, r, var = inst
    worst = max(float_error_ratio(inst, *float_case(inst, seed)) for seed in range(16))
    print(f"{name:36s} sps {sps:2d} ntaps {nt:3d} residue {r} variant {var}   of bound {worst:.3f}", flush=True)
