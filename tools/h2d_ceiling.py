#!/usr/bin/env python3
"""Pinned-memory copy ceiling of the end-to-end decode path: every rank streams the bytes that
`DVBRCS2_Turbo.decode_batch_host` moves per step (H2D of the float32 LLRs, D2H of the hard bits) with
plain cudaMemcpyAsync on two streams and NO kernel, all ranks at once.  The aggregate is the most any
host-buffer decode can reach on this box: e2e Gbit/s <= frames/s at the ceiling x 2N.

    python tools/h2d_ceiling.py [FRAMES] [--llr-bytes 4|2|1]   (1 GPU)
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/h2d_ceiling.py

--llr-bytes 2: the LLRs cross as float16 (decode_batch_host with a float16 buffer), half the H2D bytes; --llr-bytes 1:
as int8 (an int8 buffer with llr_scale), a quarter; the default is float32.  Prints one JSON line per run (rank 0): per-direction GB/s per rank (min/max) and summed.
"""
import argparse
import json
import os

import torch
import torch.distributed as dist

N, N_LLR = 212, 1272


def measure(frames, esz, dev, world):
    """{layout: ceiling figures} for `frames` frames per rank and step, LLRs of `esz` bytes; all ranks at once."""
    out = {}
    for label, d2h_per_frame in (("int32_bits", 2 * N * 4), ("packed_bits", ((2 * N + 31) // 32) * 4)):
        hin = torch.empty((frames, N_LLR), dtype={4: torch.float32, 2: torch.float16, 1: torch.int8}[esz], pin_memory=True)
        hout = torch.empty(frames * d2h_per_frame, dtype=torch.uint8, pin_memory=True)
        din = torch.empty_like(hin, device=dev)
        dout = torch.empty_like(hout, device=dev)
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        chunk = 9472
        def step():
            for lo in range(0, frames, chunk):
                hi = min(frames, lo + chunk)
                with torch.cuda.stream(s_in):
                    din[lo:hi].copy_(hin[lo:hi], non_blocking=True)
                with torch.cuda.stream(s_out):
                    hout[lo * d2h_per_frame:hi * d2h_per_frame].copy_(dout[lo * d2h_per_frame:hi * d2h_per_frame], non_blocking=True)
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cur = torch.cuda.current_stream()
        steps = 5
        a.record(cur)
        s_in.wait_stream(cur); s_out.wait_stream(cur)
        for _ in range(steps):
            step()
        cur.wait_stream(s_in); cur.wait_stream(s_out)
        b.record(cur)
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        tmax = t.clone()
        if world > 1:
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms_max = float(tmax.item())
        h2d = frames * N_LLR * esz
        d2h = frames * d2h_per_frame
        out[label] = {"ms_per_step_max_over_ranks": ms_max, "h2d_gbs_per_rank": h2d / ms_max / 1e6,
                      "d2h_gbs_per_rank": d2h / ms_max / 1e6, "h2d_gbs_total": world * h2d / ms_max / 1e6,
                      "frames_per_s_total": world * frames / (ms_max * 1e-3),
                      "info_gbit_per_s_ceiling": world * frames * 2 * N / (ms_max * 1e-3) / 1e9}
        del hin, hout, din, dout
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("frames", nargs="?", type=int, default=262144)
    ap.add_argument("--llr-bytes", type=int, choices=(4, 2, 1), default=4,
                    help="bytes per LLR element: 4 float32, 2 float16, 1 int8")
    args = ap.parse_args()
    frames, esz = args.frames, args.llr_bytes
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    out = measure(frames, esz, dev, world)
    if rank == 0:
        try:
            aff = len(os.sched_getaffinity(0))
        except Exception:
            aff = None
        extra = {} if esz == 4 else {"llr_bytes": esz}
        print(json.dumps({"tool": "h2d_ceiling", "n_gpus": world, "frames_per_rank_per_step": frames, **extra,
                          "cpu_count": os.cpu_count(), "affinity": aff, **out}), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
