#!/usr/bin/env python3
"""BER / FER sweep on the GPU path (BASELINE config 5 shape), one or more GPUs:

    python tools/ber_sweep.py [--N 212] [--rate 1/3] [--mod BPSK] [--ebn0 0 0.5 1 1.5 2] [--frames 1000000]
                              [--channel awgn|rayleigh] [--coherence L]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 tools/ber_sweep.py ...

Two runs are reported (SURVEY 8d): the PARITY run with the reference's committed interleaver table
(not a permutation: BER ~ 0.2, FER = 1 at every SNR — bit-exact with the reference, which decodes
the same way) and a labelled NON-PARITY run with a bijective interleaver through the same kernels.
The second is better but still floors: the reference trellis has parallel branches (SURVEY F3: inputs
00 and 11 give the same transition and the same parity), and the trellis is inside the parity scope.
Frames are sharded over the ranks; the only exchange is the all-reduce of the error counters.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=212)
    ap.add_argument("--rate", default="1/3")
    ap.add_argument("--mod", default="BPSK")
    ap.add_argument("--iters", type=int, default=8)
    ap.add_argument("--ebn0", type=float, nargs="+", default=[0.0, 0.5, 1.0, 1.5, 2.0])
    ap.add_argument("--frames", type=int, default=1 << 20, help="frame cap per Eb/N0 point (whole job)")
    ap.add_argument("--min-frame-errors", type=int, default=100, dest="mfe")
    ap.add_argument("--batch", type=int, default=1 << 17)
    ap.add_argument("--modes", nargs="+", default=["double-pass"], choices=["double-pass", "nii", "nii16"],
                    help="decoder modes for the bijective-interleaver runs (non-parity modes are labelled as such)")
    ap.add_argument("--channel", default="awgn", choices=["awgn", "rayleigh"],
                    help="rayleigh: block fading with perfect channel state at the demapper")
    ap.add_argument("--coherence", type=int, default=1, help="rayleigh: symbols per fading block (1 = fast fading)")
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from modulations_b200 import montecarlo as mc
    from modulations_b200.dvb_rcs2_turbo import DVBRCS2_Turbo, bijective_interleaver
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    cfg = mc.SweepConfig(N=args.N, rate=args.rate, iterations=args.iters, ebn0_db=args.ebn0,
                         frames_per_point=args.frames, batch=args.batch, modulation=args.mod,
                         min_frame_errors=args.mfe, channel=args.channel, coherence=args.coherence)
    out = {}
    runs = [("parity (committed interleaver table)", None, "double-pass")]
    for mode in args.modes:
        what = "reference decoder arithmetic" if mode == "double-pass" else f"NON-PARITY decoder mode {mode}"
        runs.append((f"non-parity (bijective interleaver), {what}", bijective_interleaver(args.N), mode))
    for label, perm, mode in runs:
        codec = DVBRCS2_Turbo(args.N, args.rate, args.iters, perm=perm, boundary=mode)
        out[label] = mc.run_sweep(cfg, rank, world, codec=codec)
        res = out[label]
        tot = sum(p["frames"] for p in res["points"])
        res["info_gbit_per_s_wall"] = tot * 2 * args.N / max(res["seconds"], 1e-9) / 1e9
    if rank == 0:
        print(json.dumps({"config": vars(args), "n_gpus": world, "runs": out}))
        for label, res in out.items():
            print(f"# {label}: {res['seconds']:.2f} s wall = {res['info_gbit_per_s_wall']:.2f} Gbit/s of information incl. the source", file=sys.stderr)
            for p in res["points"]:
                print(f"#   Eb/N0 {p['ebn0_db']:4.1f} dB  frames {p['frames']:9d}  BER {p['ber']:.3e}  FER {p['fer']:.3e}", file=sys.stderr)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
