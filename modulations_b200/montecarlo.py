"""Monte-Carlo harness: the reference's per-frame AWGN loop
(``turbo_test_suite.py:121-199`` BPSK, ``test.py:34-103`` QPSK) as batched device
work, sharded by frame across the GPUs of one node, and the same over a Rayleigh
fading channel.

Per Eb/N0 point and batch: Philox info bits -> tail-biting encode -> map -> AWGN ->
LLR (-> soft demap for QPSK/8PSK/QAM) -> 8-iteration decode -> bit / frame error
counters accumulated by ``atomicAdd`` in the decode kernel's epilogue.  With
``channel="rayleigh"`` every modulation, BPSK included, goes map -> fading + AWGN
(``b200dvb_fading_complex``, one gain per ``coherence`` symbols) -> soft demap with
the known gains (``b200dvb_demap_csi``) -> decode.  Frames are
independent, so rank r of G simply owns a contiguous range of global frame
indices; the noise and data streams are keyed by the GLOBAL frame index, which
makes the summed counters independent of G.  The only exchange is one
``all_reduce(SUM)`` of ``int64[4 * n_points]`` (NCCL over NVLink), or one per batch
when adaptive stopping is on.
"""
from __future__ import annotations

import dataclasses
import time
from typing import List, Optional

import numpy as np

RATE = {'1/3': 1 / 3, '1/2': 1 / 2, '2/3': 2 / 3, '3/4': 3 / 4}
ALIGN = 16      # shard boundaries are multiples of 16 frames (whole Philox draws)
CHANNELS = ('awgn', 'rayleigh')


@dataclasses.dataclass
class SweepConfig:
    N: int = 212
    rate: str = '1/3'
    iterations: int = 8
    ebn0_db: List[float] = dataclasses.field(default_factory=lambda: [0.0, 1.0, 2.0])
    frames_per_point: int = 1 << 16
    batch: int = 1 << 16
    seed: int = 42
    modulation: str = 'BPSK'
    min_frame_errors: Optional[int] = None      # adaptive stopping (test.py:89-92 shape)
    channel: str = 'awgn'                       # 'awgn' or 'rayleigh' (block fading, perfect channel state)
    coherence: int = 1                          # rayleigh: symbols per fading block (1 = fast fading)

    def __post_init__(self):
        if self.channel not in CHANNELS:
            raise ValueError(f"unknown channel {self.channel!r}: one of {CHANNELS}")
        if isinstance(self.coherence, bool) or int(self.coherence) != self.coherence or self.coherence < 1:
            raise ValueError(f"coherence must be a whole number of symbols >= 1, got {self.coherence!r}")


def shard_range(total, rank, world, align=ALIGN):
    """Contiguous [lo, hi) of `total` frames owned by `rank`; boundaries are multiples
    of `align`; the ranges of all ranks tile [0, total) exactly."""
    units = (total + align - 1) // align
    lo = (units * rank) // world * align
    hi = (units * (rank + 1)) // world * align
    return min(lo, total), min(hi, total)


def noise_var(rate, ebn0_db, bps=1):
    """sigma^2 per real dimension: 1/(2 R bps Eb/N0) (turbo_test_suite.py:132-134; for
    unit-energy complex symbols carrying bps bits, test.py:36-38)."""
    return 1.0 / (2.0 * RATE[rate] * bps * 10 ** (ebn0_db / 10))


def fading_channel(iq, sigma, seed, offset, block_len=1, gain=None):
    """Rayleigh block fading plus AWGN in place on a CUDA complex64 tensor (``b200dvb_fading_complex``):
    iq[i] = h[b] iq[i] + sigma (n_re + j n_im), b = (offset + i) // block_len, h ~ CN(0, 1) keyed by (seed, b).
    `offset` (the global index of iq[0]) must be even.  `gain`, a CUDA complex64 tensor of iq's size, receives
    the h of every symbol.  Returns iq."""
    from . import _lib
    if gain is not None and gain.numel() != iq.numel():
        raise ValueError(f"gain has {gain.numel()} elements for {iq.numel()} symbols")
    _lib.check(_lib.load().b200dvb_fading_complex(iq.numel(), int(block_len), float(sigma), int(seed), int(offset),
                                                  _lib.ptr(iq), _lib.ptr(gain), _lib.stream_ptr(iq.device)),
               "fading_complex")
    return iq


def reduce_counters(counters, group=None):
    """SUM all-reduce of the error counters over the ranks (NCCL on GPUs, gloo in the
    CPU tests).  No-op when torch.distributed is not initialised."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(counters, op=dist.ReduceOp.SUM, group=group)
    return counters


def summarise(cfg, counters_host, seconds=None):
    out = []
    for i, e in enumerate(cfg.ebn0_db):
        be, fe, fr, bits = [int(v) for v in counters_host[4 * i:4 * i + 4]]
        out.append(dict(ebn0_db=e, bit_errors=be, frame_errors=fe, frames=fr, bits=bits,
                        ber=be / bits if bits else 0.0, fer=fe / fr if fr else 0.0))
    return dict(points=out, seconds=seconds)


def run_sweep(cfg: SweepConfig, rank=0, world=1, codec=None):
    """Runs this rank's shard of every Eb/N0 point, all-reduces the counters and
    returns ``summarise(...)`` (identical on every rank)."""
    import torch
    from . import _lib
    from .dvb_rcs2_turbo import DVBRCS2_Turbo
    from .sdr_modem import gray_modem
    lib = _lib.load()
    codec = codec or DVBRCS2_Turbo(cfg.N, cfg.rate, cfg.iterations)
    h = codec.handle
    dev = h.device
    bps = _lib.BPS[cfg.modulation]
    counters = torch.zeros(4 * len(cfg.ebn0_db), dtype=torch.int64, device=dev)
    bmax = max(ALIGN, (cfg.batch // ALIGN) * ALIGN)
    info = torch.empty((bmax, codec.k_info), dtype=torch.uint8, device=dev)
    coded = torch.empty((bmax, h.n_llr), dtype=torch.uint8, device=dev)
    llr = torch.empty((bmax, h.n_llr), dtype=torch.float32, device=dev)
    nsym = (h.n_llr + bps - 1) // bps
    gain = torch.empty(bmax * nsym, dtype=torch.complex64, device=dev) if cfg.channel == 'rayleigh' else None
    t0 = time.time()
    lo, hi = shard_range(cfg.frames_per_point, rank, world)
    shard_max = max(b - a for a, b in (shard_range(cfg.frames_per_point, r, world) for r in range(world)))
    n_batches = (shard_max + bmax - 1) // bmax          # same on every rank: collectives stay matched
    for pi, e in enumerate(cfg.ebn0_db):
        nv = noise_var(cfg.rate, e, bps)
        cnt = counters[4 * pi:4 * pi + 4]
        seed = cfg.seed * 1000003 + pi
        for b in range(n_batches):
            start = lo + b * bmax
            n = max(0, min(bmax, hi - start))
            if n > 0 and cfg.channel == 'rayleigh':
                # encode -> map -> fading + AWGN -> max-log demap over |y - h c|^2 with the decoder's sign (F4)
                h.mc_generate_bpsk(n, 1.0, seed, start, info, coded, llr)
                m = gray_modem(cfg.modulation)
                cb = coded[:n]
                if nsym * bps != h.n_llr:
                    cb = torch.nn.functional.pad(cb, (0, nsym * bps - h.n_llr))
                syms = m.map(cb.reshape(-1))
                g = gain[:syms.numel()]
                fading_channel(syms, float(np.sqrt(nv)), seed ^ 0x9E3779B9, start * nsym, cfg.coherence, gain=g)
                x = m.llr(syms, 2.0 * nv, scale=-1.0, gain=g).reshape(n, nsym * bps)
                codec.decode_batch(x, ref_bits=info[:n], counters=cnt, out="none")
            elif n > 0 and cfg.modulation == 'BPSK':
                h.mc_generate_bpsk(n, nv, seed, start, info, coded, llr)
                codec.decode_batch(llr[:n], ref_bits=info[:n], counters=cnt, out="none")
            elif n > 0:
                # encode -> map -> complex AWGN -> max-log demap with the decoder's sign (F4)
                h.mc_generate_bpsk(n, 1.0, seed, start, info, coded, llr)
                m = gray_modem(cfg.modulation)
                cb = coded[:n]
                if nsym * bps != h.n_llr:
                    cb = torch.nn.functional.pad(cb, (0, nsym * bps - h.n_llr))
                syms = m.map(cb.reshape(-1))
                _lib.check(lib.b200dvb_awgn_complex(syms.numel(), float(np.sqrt(nv)), seed ^ 0x9E3779B9,
                                                    start * nsym, _lib.ptr(syms), _lib.stream_ptr()), "awgn")
                x = m.llr(syms, 2.0 * nv, scale=-1.0).reshape(n, nsym * bps)
                codec.decode_batch(x, ref_bits=info[:n], counters=cnt, out="none")
            if cfg.min_frame_errors is not None:
                tot = reduce_counters(cnt.clone()).cpu()
                if int(tot[1]) >= cfg.min_frame_errors:
                    break
    reduce_counters(counters)
    host = counters.cpu().numpy()
    return summarise(cfg, host, time.time() - t0)
