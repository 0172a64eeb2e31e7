"""Drop-in for ``compute_llr`` (reference ``test_sdr_with_coding.py:200-225``):
max-log bit LLRs over a constellation enumerated from the mapper, sigma^2 floored
at 0.005, clipped to +-30, positive = bit 1 (SURVEY §0 F4).  Extended to 64QAM and
256QAM over the ``SDRModem`` constellations (the reference stops at 16QAM).

Runs in float32 on the GPU (``b200dvb_demap``); the reference computes in float64,
so results agree to a stated absolute tolerance (tests/test_gpu_modem.py).
"""
from __future__ import annotations

import numpy as np

from . import _lib
from .sdr_modem import gray_modem, ModemHandle


def compute_llr(syms, mod_type, noise_var, constellation=None, gain=None):
    """-> float64[n*bps] (numpy in) or float32 CUDA tensor (torch in).  `gain`: the complex channel gain of each
    symbol (received as h*c + noise); the LLRs are then over |y - h c|^2 (``b200dvb_demap_csi``)."""
    if mod_type not in _lib.MOD_IDS:
        raise KeyError(mod_type)                         # reference: MODULATIONS[mod_type] KeyError
    modem = gray_modem(mod_type) if constellation is None else ModemHandle(mod_type, constellation)
    torch = _lib.torch_mod()
    out = modem.llr(syms, noise_var, gain=gain)
    if isinstance(out, torch.Tensor):
        return out
    return out.astype(np.float64)


def decoder_llr(syms, mod_type, noise_var, gain=None):
    """LLRs in the DECODER's convention (positive = bit 0): -compute_llr, fused in
    the kernel as scale = -1 (SURVEY §0 F4)."""
    return gray_modem(mod_type).llr(syms, noise_var, scale=-1.0, gain=gain)


def estimate_noise_var(rx_symbols, mod_type, floor=0.02, default=0.05, modem=None):
    """Decision-directed noise-variance estimate of the reference's receive chain
    (``test_sdr_with_coding.py:460-467``): slice the received symbols to hard bits, re-map them, and take
    the mean squared distance to the re-mapped points, floored at 0.02; 0.05 when the re-mapped vector
    comes out longer than the input (the reference's guard, `:462-465`).  Slicing and re-mapping run on
    the GPU (``b200dvb_hard_demod`` / ``b200dvb_map``); ``modem`` defaults to ``SDRModem``."""
    from .sdr_modem import SDRModem
    modem = modem or SDRModem()
    rx = np.asarray(rx_symbols)
    bps = SDRModem.MODULATIONS[mod_type]['bps']
    rx_bits = modem.demodulate(rx, mod_type)
    const = modem.modulate(rx_bits[:len(rx) * bps], mod_type)
    if len(const) <= len(rx):
        nv = float(np.mean(np.abs(rx[:len(const)] - const) ** 2))
    else:
        nv = default
    return max(nv, floor)
