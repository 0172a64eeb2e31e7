#!/usr/bin/env python3
"""float32 against float16 (binary16) channel-LLR input of the decoder, on the same frames.

    python tools/llr16_perf.py [--runs 3]
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/llr16_perf.py

Prints one JSON line (rank 0) with:
  * the card's name, power limit and SM clock, read in this run;
  * resident decode rates (CUDA events, inputs already on the device, out="packed"), float32 and float16 runs
    alternated, `--runs` of each, with min / max: the thread-per-frame kernel at N=212 R=1/3 8 iterations on 2^20
    frames (5.3 GB of float32 LLRs: larger than L2), and the quad kernel at N=752 R=1/2 8 iterations on 4 waves of
    its global-record geometry (the prep re-reads the LLRs every half-iteration);
  * end to end: DVBRCS2_Turbo.decode_batch_host(out="packed") from pinned float32 / float16 buffers of 2^18 frames at
    N=212, host clock, alternated, and its fraction of the resident rate of the same format;
  * the pinned copy ceiling of those bytes (tools/h2d_ceiling.py) for 4- and 2-byte LLRs.
With several ranks every rank runs the same work on its own GPU at once; rates are summed over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from modulations_b200 import dvb_rcs2_turbo as turbo  # noqa: E402
import h2d_ceiling  # noqa: E402


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, pl, sm, smax = [v.strip() for v in r.stdout.strip().split(",")]
        return {"name": name, "power_limit": pl, "sm_clock": sm, "sm_clock_max": smax}
    except Exception as e:                                  # the name alone, from the runtime
        return {"name": torch.cuda.get_device_name(), "nvidia_smi": repr(e)}


def llrs(g, B, ebn0=2.0, seed=1234):
    h = g.handle
    info = torch.empty((B, g.k_info), dtype=torch.uint8, device="cuda")
    coded = torch.empty((B, h.n_llr), dtype=torch.uint8, device="cuda")
    llr = torch.empty((B, h.n_llr), dtype=torch.float32, device="cuda")
    h.mc_generate_bpsk(B, 1.0 / (2.0 * (g.k_info / h.n_llr) * 10 ** (ebn0 / 10)), seed, 0, info, coded, llr)
    del info, coded
    return llr


def barrier(world):
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()


def total(x, world):
    """sum of a per-rank float over ranks"""
    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t)
    return float(t.item())


def stats(v):
    return {"runs": v, "best": max(v), "min": min(v), "spread": max(v) - min(v)}


def resident(g, x32, runs, world, reps):
    """info Gbit/s (summed over ranks) of decode_batch(out="packed") on device-resident float32 / float16 LLRs; one run
    times `reps` back-to-back calls (a window of some 0.3 s)."""
    x16 = x32.half()
    B = x32.shape[0]
    out = {"float32": [], "float16": []}
    g.decode_batch(x32, out="packed")                        # warm both instances and the allocator
    p16 = g.decode_batch(x16, out="packed")
    same = bool(torch.equal(p16, g.decode_batch(x16.float(), out="packed")))
    del p16
    for _ in range(runs):
        for name, x in (("float32", x32), ("float16", x16)):
            barrier(world)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                g.decode_batch(x, out="packed")
            b.record()
            torch.cuda.synchronize()
            out[name].append(total(reps * B * g.k_info / (a.elapsed_time(b) * 1e-3) / 1e9, world))
    del x16
    return {k: stats(v) for k, v in out.items()}, same


def e2e(g, x32_dev, runs, world):
    """decode_batch_host(out="packed") info Gbit/s (summed over ranks) from pinned float32 / float16 buffers."""
    hosts = {"float32": x32_dev.cpu().pin_memory(), "float16": x32_dev.half().cpu().pin_memory()}
    B = x32_dev.shape[0]
    outs = {k: torch.empty((B, (g.k_info + 31) // 32), dtype=torch.int32, pin_memory=True) for k in hosts}
    res = {"float32": [], "float16": []}
    for k in hosts:                                          # warm: pipeline buffers, streams
        g.decode_batch_host(hosts[k], out_host=outs[k], out="packed")
    for _ in range(runs):
        for k in ("float32", "float16"):
            barrier(world)
            t0 = time.perf_counter()
            g.decode_batch_host(hosts[k], out_host=outs[k], out="packed")
            dt = time.perf_counter() - t0
            dt = dt if world == 1 else _max(dt, world)        # the slowest rank
            res[k].append(world * B * g.k_info / dt / 1e9)
    return {k: stats(v) for k, v in res.items()}


def _max(x, world):
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--tpf-frames", type=int, default=1 << 20)
    ap.add_argument("--e2e-frames", type=int, default=1 << 18)
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    res = {"tool": "llr16_perf", "n_gpus": world, "card": card(), "runs": args.runs}

    g = turbo.DVBRCS2_Turbo(212, '1/3', 8)
    x = llrs(g, args.tpf_frames)
    r, same = resident(g, x, args.runs, world, 3)
    res["tpf_n212_r13_8it"] = {"frames_per_rank": args.tpf_frames, "kernel": "tpf_kernel", "info_gbit_per_s": r,
                               "f16_over_f32_best": r["float16"]["best"] / r["float32"]["best"],
                               "outputs_equal_float32_of_widening": same}
    xe = x[:args.e2e_frames].clone()
    del x
    er = e2e(g, xe, args.runs, world)
    re_, _ = resident(g, xe, args.runs, world, 10)
    res["e2e_n212_r13_8it_packed"] = {
        "frames_per_rank": args.e2e_frames, "chunk": "one wave of the decode kernel (the default)", "api": 'decode_batch_host(out="packed"), pinned input, 3-stream pipeline',
        "h2d_bytes_per_frame": {"float32": g.n_llr * 4, "float16": g.n_llr * 2}, "d2h_bytes_per_frame": 56,
        "info_gbit_per_s": er, "resident_info_gbit_per_s_same_frames": re_,
        "frac_of_resident": {k: er[k]["best"] / re_[k]["best"] for k in er}}
    del xe
    torch.cuda.empty_cache()

    q = turbo.DVBRCS2_Turbo(752, '1/2', 8)
    B = 4 * 4736
    x = llrs(q, B)
    r, same = resident(q, x, args.runs, world, 20)
    res["quad_n752_r12_8it"] = {"frames_per_rank": B, "kernel": "quad_kernel (auto choice: global-record geometry)",
                                "info_gbit_per_s": r, "f16_over_f32_best": r["float16"]["best"] / r["float32"]["best"],
                                "outputs_equal_float32_of_widening": same}
    del x
    torch.cuda.empty_cache()

    res["copy_ceiling"] = {f"llr_bytes_{esz}": h2d_ceiling.measure(args.e2e_frames, esz, dev, world) for esz in (4, 2)}
    res["card_after"] = card()
    if rank == 0:
        print(json.dumps(res), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
