"""Drop-in for the modulation part of the reference ``sdr_modem.SDRModem``
(``sdr_modem.py:29-36, 66-73, 101-266``): Gray-mapped BPSK/QPSK/8PSK/16/64/256QAM
bit->symbol mapping and hard slicing, executed by the table-driven CUDA kernels of
``libb200dvb.so``.  The SDR hardware I/O of the reference class (HackRF / RTL-SDR
subprocesses, pulse shaping, synchronisation: ``sdr_modem.py:77-97, 270-664``) is
out of scope (BASELINE.json north_star) and is not provided.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib

_GRAY = {2: [0, 1, 3, 2], 3: [0, 1, 3, 2, 6, 7, 5, 4],
         4: [0, 1, 3, 2, 6, 7, 5, 4, 12, 13, 15, 14, 10, 11, 9, 8]}   # sdr_modem.py:68-70
_QAM = {'16QAM': (2, 10), '64QAM': (3, 42), '256QAM': (4, 170)}


def gray_constellation(modulation):
    """Constellation indexed by MSB-first bit label, with the reference mapper's
    value and dtype: complex64 everywhere, complex128 for QPSK (sdr_modem.py:101-207)."""
    if modulation == 'BPSK':                                   # 2b - 1
        return np.array([-1.0, 1.0], dtype=np.complex64)
    if modulation == 'QPSK':                                   # ((1-2b0) + j(1-2b1)) / sqrt(2)
        pts = np.array([1 + 1j, 1 - 1j, -1 + 1j, -1 - 1j], dtype=np.complex64)
        return pts / np.sqrt(2)
    if modulation == '8PSK':                                   # exp(j*pi/4*gray3[label])
        return np.array([np.exp(1j * (g * np.pi / 4)) for g in _GRAY[3]], dtype=np.complex64)
    if modulation in _QAM:                                     # (2*gray[idx] - (L-1)) / sqrt(norm)
        half, norm = _QAM[modulation]
        L = 1 << half
        axis = [(2 * g - (L - 1)) / np.sqrt(norm) for g in _GRAY[half]]
        return np.array([axis[lab >> half] + 1j * axis[lab & (L - 1)] for lab in range(L * L)],
                        dtype=np.complex64)
    raise ValueError(f"Unknown modulation: {modulation}")


class ModemHandle:
    """One b200dvb_modem_t: a modulation id plus the constellation table it uses."""

    def __init__(self, modulation, table):
        if modulation not in _lib.MOD_IDS:
            raise ValueError(f"Unknown modulation: {modulation}")
        torch = _lib.require_cuda()
        self.device = torch.device("cuda", torch.cuda.current_device())
        self.modulation = modulation
        self.bps = _lib.BPS[modulation]
        self.table = np.asarray(table)
        t = np.ascontiguousarray(self.table.astype(np.complex128)).view(np.float64)
        h = ctypes.c_void_p()
        rc = _lib.load().b200dvb_modem_create(_lib.MOD_IDS[modulation], _lib.host_ptr(t), ctypes.byref(h))
        _lib.check(rc, modulation)
        self.h = h

    def __del__(self):
        try:
            if getattr(self, "h", None):
                _lib.load().b200dvb_modem_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # bits (any int array / CUDA tensor, length n_sym*bps) -> symbols
    def map(self, bits, out_complex128=False):
        torch = _lib.require_cuda()
        is_torch = isinstance(bits, torch.Tensor)
        b = _lib.to_device(bits, torch.uint8, self.device).reshape(-1)
        n = b.numel() // self.bps
        out = torch.empty(n, dtype=torch.complex128 if out_complex128 else torch.complex64,
                          device=self.device)
        with torch.cuda.device(self.device):
            rc = _lib.load().b200dvb_map(self.h, n, _lib.ptr(b), _lib.ptr(out), int(out_complex128),
                                         _lib.stream_ptr(self.device))
        _lib.check(rc, "map")
        return out if is_torch else out.cpu().numpy()

    def hard(self, symbols):
        torch = _lib.require_cuda()
        is_torch = isinstance(symbols, torch.Tensor)
        if not is_torch:
            symbols = np.asarray(symbols)
            f64 = symbols.dtype != np.complex64
            s = _lib.to_device(symbols.astype(np.complex128 if f64 else np.complex64),
                               torch.complex128 if f64 else torch.complex64, self.device)
        else:
            f64 = symbols.dtype == torch.complex128
            s = _lib.to_device(symbols, symbols.dtype if f64 else torch.complex64, self.device)
        n = s.numel()
        out = torch.empty(n * self.bps, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            rc = _lib.load().b200dvb_hard_demod(self.h, n, _lib.ptr(s), int(f64), _lib.ptr(out),
                                                _lib.stream_ptr(self.device))
        _lib.check(rc, "hard_demod")
        return out if is_torch else out.cpu().numpy()

    def llr(self, symbols, noise_var, scale=1.0, gain=None):
        """float32 max-log LLRs [n*bps], clipped to +-30 then multiplied by `scale`.  With `gain` (complex64, numpy
        or CUDA, one per symbol) the symbols were received as h*c + noise and the LLRs are over |y - h c|^2
        (b200dvb_demap_csi, perfect channel state)."""
        torch = _lib.require_cuda()
        is_torch = isinstance(symbols, torch.Tensor)
        s = _lib.to_device(symbols if is_torch else np.asarray(symbols).astype(np.complex64),
                           torch.complex64, self.device).reshape(-1)
        n = s.numel()
        if gain is not None:
            g = _lib.to_device(gain if isinstance(gain, torch.Tensor) else np.asarray(gain).astype(np.complex64),
                               torch.complex64, self.device).reshape(-1)
            if g.numel() != n:
                raise ValueError(f"gain has {g.numel()} elements for {n} symbols")
        out = torch.empty(n * self.bps, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            if gain is None:
                rc = _lib.load().b200dvb_demap(self.h, n, _lib.ptr(s), float(noise_var), float(scale),
                                               _lib.ptr(out), _lib.stream_ptr(self.device))
            else:
                rc = _lib.load().b200dvb_demap_csi(self.h, n, _lib.ptr(s), _lib.ptr(g), float(noise_var),
                                                   float(scale), _lib.ptr(out), _lib.stream_ptr(self.device))
        _lib.check(rc, "demap" if gain is None else "demap_csi")
        return out if is_torch else out.cpu().numpy()


    def llr_bf16(self, symbols_bf16, noise_var, scale=1.0):
        """The same for bf16x2 symbols: a CUDA (or CPU) torch.bfloat16 tensor [n, 2] (I, Q).  Each component is
        widened exactly to float32 on the device; 4 bytes per symbol are read instead of 8."""
        torch = _lib.require_cuda()
        s = symbols_bf16.to(device=self.device).contiguous()
        if s.dtype != torch.bfloat16 or s.dim() != 2 or s.shape[1] != 2:
            raise ValueError("symbols_bf16 must be a torch.bfloat16 tensor of shape [n, 2]")
        n = s.shape[0]
        out = torch.empty(n * self.bps, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            rc = _lib.load().b200dvb_demap_bf16(self.h, n, _lib.ptr(s), float(noise_var), float(scale),
                                                _lib.ptr(out), _lib.stream_ptr(self.device))
        _lib.check(rc, "demap_bf16")
        return out


_handles = {}


def gray_modem(modulation):
    """Cached ModemHandle over the SDRModem (Gray) constellation, one per CUDA device (its tables live in
    the memory of the device that was current when it was created)."""
    key = (_lib.require_cuda().cuda.current_device(), modulation)
    h = _handles.get(key)
    if h is None:
        h = ModemHandle(modulation, gray_constellation(modulation))
        _handles[key] = h
    return h


class SDRModem:
    """Modulation / demodulation half of the reference ``SDRModem``."""

    # sdr_modem.py:29-36
    MODULATIONS = {
        'BPSK':   {'bps': 1, 'order': 2,   'alpha': 0.02,  'n_rot': 2, 'rot_step': np.pi},
        'QPSK':   {'bps': 2, 'order': 4,   'alpha': 0.015, 'n_rot': 4, 'rot_step': np.pi / 2},
        '8PSK':   {'bps': 3, 'order': 8,   'alpha': 0.01,  'n_rot': 8, 'rot_step': np.pi / 4},
        '16QAM':  {'bps': 4, 'order': 16,  'alpha': 0.008, 'n_rot': 4, 'rot_step': np.pi / 2},
        '64QAM':  {'bps': 6, 'order': 64,  'alpha': 0.005, 'n_rot': 4, 'rot_step': np.pi / 2},
        '256QAM': {'bps': 8, 'order': 256, 'alpha': 0.003, 'n_rot': 4, 'rot_step': np.pi / 2},
    }

    def __init__(self, fc: float = 433e6, fs: float = 2e6, sps: int = 4,
                 tx_gain: int = 47, rx_gain: int = 49):
        self.fc, self.fs, self.sps, self.tx_gain, self.rx_gain = fc, fs, sps, tx_gain, rx_gain
        self.gray2, self.gray3, self.gray4 = _GRAY[2], _GRAY[3], _GRAY[4]
        self.inv_gray2 = [self.gray2.index(i) for i in range(4)]
        self.inv_gray3 = [self.gray3.index(i) for i in range(8)]
        self.inv_gray4 = [self.gray4.index(i) for i in range(16)]

    def modulate(self, bits, modulation: str = 'QPSK'):
        """Bits -> complex symbols (sdr_modem.py:222-243).  Zero-pads to a multiple of
        bps like the reference mappers; complex64, except QPSK which the reference
        returns as complex128."""
        if modulation not in self.MODULATIONS:
            raise ValueError(f"Unknown modulation: {modulation}")
        bps = self.MODULATIONS[modulation]['bps']
        bits = np.array(bits)
        pad = (bps - len(bits) % bps) % bps
        if pad:
            bits = np.append(bits, [0] * pad)
        return gray_modem(modulation).map(bits, out_complex128=(modulation == 'QPSK'))

    def demodulate(self, symbols, modulation: str = 'QPSK'):
        """Complex symbols -> hard bits (sdr_modem.py:245-266): nearest constellation
        point evaluated in float64, which is what the reference's per-modulation slicers
        (sign / rounded phase / rounded level index) compute."""
        if modulation not in self.MODULATIONS:
            raise ValueError(f"Unknown modulation: {modulation}")
        return gray_modem(modulation).hard(symbols).astype(int)

    def transmit(self, *a, **k):
        raise NotImplementedError("SDR hardware I/O is out of scope of modulations_b200")

    receive = transmit
