"""ctypes binding of libb200dvb.so (include/b200dvb.h) + device-buffer plumbing.

There is no CPU fallback anywhere in this package: if the shared library is
missing, or no CUDA device is visible, the first compute call raises.
PyTorch is used only to own device memory and streams.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200dvb.so")

OK, EINVAL, ENOSPEC, ECUDA, ENOMEM, EMOD = 0, -1, -2, -3, -4, -5
OPT_KERNEL, OPT_NO_ROW_STAGING, OPT_PHASE_TIMERS, OPT_DECODER_MODE = 1, 2, 3, 4
MODE_PARITY, MODE_NII, MODE_NII16 = 0, 1, 2
LLR_F32, LLR_F16, LLR_I8 = 0, 1, 2
KERNEL_AUTO, KERNEL_QUAD, KERNEL_TPF, KERNEL_LAT = 0, 1, 2, 3
MOD_IDS = {'BPSK': 0, 'QPSK': 1, '8PSK': 2, '16QAM': 3, '64QAM': 4, '256QAM': 5}
BPS = {'BPSK': 1, 'QPSK': 2, '8PSK': 3, '16QAM': 4, '64QAM': 6, '256QAM': 8}

_c_void_p, _c_int, _c_size_t = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t
_c_double, _c_float, _c_ll, _c_ull = ctypes.c_double, ctypes.c_float, ctypes.c_longlong, ctypes.c_ulonglong

# name -> (restype, argtypes); mirrors include/b200dvb.h one to one
SIGNATURES = {
    "b200dvb_version": (_c_int, []),
    "b200dvb_error_string": (ctypes.c_char_p, [_c_int]),
    "b200dvb_last_cuda_error": (ctypes.c_char_p, []),
    "b200dvb_device_count": (_c_int, []),
    "b200dvb_codec_create": (_c_int, [_c_int] + [_c_void_p] * 6 + [_c_int, _c_int, _c_double, _c_double, _c_void_p]),
    "b200dvb_codec_destroy": (_c_int, [_c_void_p]),
    "b200dvb_codec_n_llr": (_c_int, [_c_void_p]),
    "b200dvb_codec_frames_per_wave": (_c_int, [_c_void_p]),
    "b200dvb_codec_circular_lut": (_c_int, [_c_void_p, _c_void_p]),
    "b200dvb_codec_set_option": (_c_int, [_c_void_p, _c_int, _c_int]),
    "b200dvb_siso_workspace_bytes": (_c_size_t, [_c_void_p, _c_int]),
    "b200dvb_siso": (_c_int, [_c_void_p, _c_int] + [_c_void_p] * 6 + [_c_double] + [_c_void_p] * 3 + [_c_size_t, _c_void_p]),
    "b200dvb_decode_workspace_bytes": (_c_size_t, [_c_void_p, _c_int]),
    "b200dvb_decode": (_c_int, [_c_void_p, _c_int, _c_void_p, _c_ll] + [_c_void_p] * 5 + [_c_size_t, _c_void_p]),
    "b200dvb_decode_f16": (_c_int, [_c_void_p, _c_int, _c_void_p, _c_ll] + [_c_void_p] * 5 + [_c_size_t, _c_void_p]),
    "b200dvb_decode_i8": (_c_int, [_c_void_p, _c_int, _c_void_p, _c_ll, _c_float] + [_c_void_p] * 5 + [_c_size_t, _c_void_p]),
    "b200dvb_decode_app": (_c_int, [_c_void_p, _c_int, _c_void_p, _c_int, _c_float, _c_ll] + [_c_void_p] * 6
                           + [_c_size_t, _c_void_p]),
    "b200dvb_encode": (_c_int, [_c_void_p, _c_int, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "b200dvb_mc_generate_bpsk": (_c_int, [_c_void_p, _c_int, _c_float, _c_ull, _c_ull] + [_c_void_p] * 4),
    "b200dvb_awgn_complex": (_c_int, [_c_size_t, _c_float, _c_ull, _c_ull, _c_void_p, _c_void_p]),
    "b200dvb_fading_complex": (_c_int, [_c_size_t, _c_int, _c_float, _c_ull, _c_ull, _c_void_p, _c_void_p, _c_void_p]),
    "b200dvb_modem_create": (_c_int, [_c_int, _c_void_p, _c_void_p]),
    "b200dvb_modem_destroy": (_c_int, [_c_void_p]),
    "b200dvb_map": (_c_int, [_c_void_p, _c_size_t, _c_void_p, _c_void_p, _c_int, _c_void_p]),
    "b200dvb_demap": (_c_int, [_c_void_p, _c_size_t, _c_void_p, _c_float, _c_float, _c_void_p, _c_void_p]),
    "b200dvb_demap_bf16": (_c_int, [_c_void_p, _c_size_t, _c_void_p, _c_float, _c_float, _c_void_p, _c_void_p]),
    "b200dvb_demap_csi": (_c_int, [_c_void_p, _c_size_t, _c_void_p, _c_void_p, _c_float, _c_float, _c_void_p,
                                   _c_void_p]),
    "b200dvb_hard_demod": (_c_int, [_c_void_p, _c_size_t, _c_void_p, _c_int, _c_void_p, _c_void_p]),
    "b200dvb_pulse_shape": (_c_int, [_c_size_t, _c_void_p, _c_void_p, _c_int, _c_int, _c_void_p, _c_void_p]),
    "b200dvb_matched_filter": (_c_int, [_c_size_t, _c_void_p, _c_void_p, _c_int, _c_int, _c_ll, _c_size_t, _c_void_p, _c_void_p]),
    "b200dvb_debug_phase_cycles": (_c_int, [_c_void_p, _c_int]),
    "b200dvb_debug_set_option": (_c_int, [_c_int, _c_int]),
    "b200dvb_debug_tpf_cycles": (_c_int, [_c_void_p, _c_int]),
    "b200dvb_debug_nii_cycles": (_c_int, [_c_void_p, _c_int]),
    "b200dvb_debug_lat_cycles": (_c_int, [_c_void_p, _c_int]),
    "b200dvb_tmem_selftest": (_c_int, [_c_void_p]),
    "b200dvb_microbench": (_c_int, [_c_void_p]),
    "b200dvb_microbench2": (_c_int, [_c_void_p]),
}

_lib = None


def load():
    """Load libb200dvb.so (built by `python -m modulations_b200.build`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m modulations_b200.build` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the .so does not export it
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc, what=""):
    """Map a B200DVB_* return code to the exception the reference would raise."""
    if rc == OK:
        return
    lib = load()
    msg = lib.b200dvb_error_string(rc).decode()
    if rc == ECUDA:
        raise RuntimeError(f"{what}: {msg}: {lib.b200dvb_last_cuda_error().decode()}")
    if rc == ENOMEM:
        raise MemoryError(f"{what}: {msg}")
    if rc == EMOD:
        raise ValueError(f"Unknown modulation: {what}")
    raise ValueError(f"{what}: {msg}")


def torch_mod():
    import torch
    return torch


def require_cuda():
    torch = torch_mod()
    if not torch.cuda.is_available():
        raise RuntimeError("modulations_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def stream_ptr(device=None):
    """cudaStream_t of torch's current stream on `device` (default: the current device)."""
    torch = torch_mod()
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def to_device(x, dtype, device=None):
    """numpy / torch (any device) -> contiguous CUDA tensor of `dtype`."""
    torch = require_cuda()
    if isinstance(x, torch.Tensor):
        t = x
    else:
        t = torch.from_numpy(np.ascontiguousarray(x))
    if device is None:
        device = t.device if t.is_cuda else torch.device("cuda", torch.cuda.current_device())
    return t.to(device=device, dtype=dtype, non_blocking=True).contiguous()


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def host_ptr(a):
    return ctypes.c_void_p(a.ctypes.data)
