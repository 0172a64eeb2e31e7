"""Reference for the soft demapper with channel state (b200dvb_demap_csi), test infrastructure only: the max-log
rule of oracle.compute_llr over |s - h c|^2 for a known complex gain h per symbol, in complex128, vectorised and as a
per-symbol literal restatement to check it against (as oracle.compute_llr_literal does for compute_llr)."""
import numpy as np

from oracle.oracle import BPS, _label_bits, modulate


def compute_llr_csi_literal(syms, gain, mod_type, noise_var, constellation=None):
    """compute_llr_literal over a channel with a known complex gain per symbol: distances |s - h c|^2."""
    noise_var = max(noise_var, 0.005)
    bps = BPS[mod_type]
    all_bits = _label_bits(bps)
    if constellation is None:
        constellation = modulate(all_bits.flatten(), mod_type).reshape(-1)
    llr = np.zeros(len(syms) * bps)
    for i, (s, h) in enumerate(zip(syms, gain)):
        distances = np.abs(complex(s) - complex(h) * constellation.astype(np.complex128)) ** 2
        for b in range(bps):
            idx0 = np.where(all_bits[:, b] == 0)[0]
            idx1 = np.where(all_bits[:, b] == 1)[0]
            llr[i * bps + b] = (np.min(distances[idx0]) - np.min(distances[idx1])) / noise_var
    return np.clip(llr, -30, 30)


def compute_llr_csi(syms, gain, mod_type, noise_var, constellation=None, chunk=1 << 16):
    """compute_llr_csi_literal vectorised over symbols, in complex128."""
    noise_var = max(noise_var, 0.005)
    bps = BPS[mod_type]
    all_bits = _label_bits(bps)
    if constellation is None:
        constellation = modulate(all_bits.flatten(), mod_type).reshape(-1)
    c = np.asarray(constellation).astype(np.complex128)
    syms = np.asarray(syms).astype(np.complex128)
    gain = np.asarray(gain).astype(np.complex128)
    out = np.zeros((len(syms), bps))
    sets = [(np.where(all_bits[:, b] == 0)[0], np.where(all_bits[:, b] == 1)[0]) for b in range(bps)]
    for lo in range(0, len(syms), chunk):
        d = np.abs(syms[lo:lo + chunk, None] - gain[lo:lo + chunk, None] * c[None, :]) ** 2
        for b, (i0, i1) in enumerate(sets):
            out[lo:lo + chunk, b] = (d[:, i0].min(axis=1) - d[:, i1].min(axis=1)) / noise_var
    return np.clip(out.reshape(-1), -30, 30)
