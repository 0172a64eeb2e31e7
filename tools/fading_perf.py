#!/usr/bin/env python3
"""Kernel time of the Rayleigh channel and of the channel-state demapper, by CUDA events, on 2^27 resident symbols:

    python tools/fading_perf.py [--log2n 27] [--reps 20] [--out FILE]

* b200dvb_demap and b200dvb_demap_csi alternate three times each per modulation; algorithmic bytes per symbol are
  8 + 4 bps and 8 + 8 + 4 bps (symbol, gain, LLRs);
* b200dvb_fading_complex at block lengths 1 and 64, with the gain output (8 + 8 + 8 bytes per symbol) and without it
  (8 + 8), against b200dvb_awgn_complex (8 + 8);
* every rate is also given as a fraction of a device-to-device copy of >= 4 GB timed in the same run (read + write
  bytes over time).  The median of the three alternations is reported.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def timed(fn, reps):
    import torch
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=27)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from modulations_b200 import _lib
    from modulations_b200.sdr_modem import gray_modem
    lib = _lib.load()
    dev = torch.cuda.get_device_name(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    n = 1 << args.log2n
    st = _lib.stream_ptr()
    rows = [dict(device=dev, nvidia_smi=smi, n_sym=n, reps=args.reps)]

    src = torch.empty(1 << 30, dtype=torch.float32, device="cuda")          # 4 GiB
    dst = torch.empty_like(src)
    copy_s = sorted(timed(lambda: dst.copy_(src), 5) for _ in range(3))[1]
    copy_bw = 2 * src.numel() * 4 / copy_s
    rows.append(dict(what="device copy 4 GiB", seconds=copy_s, gbytes_per_s=copy_bw / 1e9))
    del src, dst

    def row(what, sec, bytes_per_sym, **kw):
        bw = n * bytes_per_sym / sec
        r = dict(what=what, seconds=sec, gsym_per_s=n / sec / 1e9, gbytes_per_s=bw / 1e9, of_copy=bw / copy_bw, **kw)
        rows.append(r)
        print(json.dumps(r), flush=True)

    y = torch.complex(torch.randn(n, device="cuda"), torch.randn(n, device="cuda"))
    g = torch.complex(torch.randn(n, device="cuda"), torch.randn(n, device="cuda"))
    for name in ('BPSK', 'QPSK', '8PSK', '16QAM', '64QAM', '256QAM'):
        m = gray_modem(name)
        out = torch.empty(n * m.bps, dtype=torch.float32, device="cuda")
        plain = lambda: _lib.check(lib.b200dvb_demap(m.h, n, _lib.ptr(y), 0.05, -1.0, _lib.ptr(out), st), "demap")
        csi = lambda: _lib.check(lib.b200dvb_demap_csi(m.h, n, _lib.ptr(y), _lib.ptr(g), 0.05, -1.0, _lib.ptr(out), st),
                                 "demap_csi")
        tp, tc = [], []
        for _ in range(3):
            tp.append(timed(plain, args.reps))
            tc.append(timed(csi, args.reps))
        row(f"demap {name}", sorted(tp)[1], 8 + 4 * m.bps, runs=tp)
        row(f"demap_csi {name}", sorted(tc)[1], 16 + 4 * m.bps, runs=tc)
        del out
    x = torch.zeros(n, dtype=torch.complex64, device="cuda")
    awgn = lambda: _lib.check(lib.b200dvb_awgn_complex(n, 0.1, 7, 0, _lib.ptr(x), st), "awgn")
    for L in (1, 64):
        fg = lambda: _lib.check(lib.b200dvb_fading_complex(n, L, 0.1, 7, 0, _lib.ptr(x), _lib.ptr(g), st), "fading")
        fn = lambda: _lib.check(lib.b200dvb_fading_complex(n, L, 0.1, 7, 0, _lib.ptr(x), None, st), "fading")
        ta, tg, tn = [], [], []
        for _ in range(3):
            ta.append(timed(awgn, args.reps))
            tg.append(timed(fg, args.reps))
            tn.append(timed(fn, args.reps))
        if L == 1:
            row("awgn_complex", sorted(ta)[1], 16, runs=ta)
        row(f"fading_complex L={L} with gain", sorted(tg)[1], 24, runs=tg)
        row(f"fading_complex L={L} without gain", sorted(tn)[1], 16, runs=tn)
    if args.out:
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")
    print(json.dumps(rows[:2]))


if __name__ == "__main__":
    main()
