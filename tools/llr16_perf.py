#!/usr/bin/env python3
"""float32 against float16 (binary16) channel-LLR input of the decoder, on the same frames; with --int8 also int8.

    python tools/llr16_perf.py [--runs 3] [--int8]
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
--int8 adds int8 LLRs q = clamp(rint(4 x), -127, 127) decoded with llr_scale 0.25 (the nii16 mode's own quantisation
of x) as a third format in every comparison above, alternated with the other two, and the same resident and end-to-end
figures for the nii16 mode at N=212 R=1/3.  Without it the output is the float32 / float16 comparison alone.
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


I8_SCALE = 0.25                                             # int8 LLRs in 1/4 units (--int8)


def as_int8(x):
    return torch.clamp(torch.round(x / I8_SCALE), -127, 127).to(torch.int8)


def formats(x32, fmts):
    """{format: the same LLRs in that format} (same device)"""
    xs = {"float32": x32, "float16": x32.half()}
    if "int8" in fmts:
        xs["int8"] = as_int8(x32)
    return xs


def stats(v):
    return {"runs": v, "best": max(v), "min": min(v), "spread": max(v) - min(v)}


def resident(g, x32, runs, world, reps, fmts):
    """info Gbit/s (summed over ranks) of decode_batch(out="packed") on device-resident LLRs of each format in `fmts`;
    one run times `reps` back-to-back calls (a window of some 0.3 s).  Also whether the float16 outputs equal those
    of the float32 widening and (int8 in fmts, else None) the int8 outputs those of the float32 products."""
    xs = formats(x32, fmts)
    scale = {"int8": I8_SCALE}
    B = x32.shape[0]
    out = {k: [] for k in fmts}
    g.decode_batch(x32, out="packed")                        # warm every instance and the allocator
    p16 = g.decode_batch(xs["float16"], out="packed")
    same = bool(torch.equal(p16, g.decode_batch(xs["float16"].float(), out="packed")))
    del p16
    same8 = None
    if "int8" in fmts:
        p8 = g.decode_batch(xs["int8"], out="packed", llr_scale=I8_SCALE)
        same8 = bool(torch.equal(p8, g.decode_batch(xs["int8"].float() * I8_SCALE, out="packed")))
        del p8
    for _ in range(runs):
        for name in fmts:
            barrier(world)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                g.decode_batch(xs[name], out="packed", llr_scale=scale.get(name))
            b.record()
            torch.cuda.synchronize()
            out[name].append(total(reps * B * g.k_info / (a.elapsed_time(b) * 1e-3) / 1e9, world))
    del xs
    return {k: stats(v) for k, v in out.items()}, same, same8


def e2e(g, x32_dev, runs, world, fmts):
    """decode_batch_host(out="packed") info Gbit/s (summed over ranks) from pinned buffers of each format in `fmts`."""
    hosts = {k: v.cpu().pin_memory() for k, v in formats(x32_dev, fmts).items()}
    scale = {"int8": I8_SCALE}
    B = x32_dev.shape[0]
    outs = {k: torch.empty((B, (g.k_info + 31) // 32), dtype=torch.int32, pin_memory=True) for k in hosts}
    res = {k: [] for k in fmts}
    for k in hosts:                                          # warm: pipeline buffers, streams
        g.decode_batch_host(hosts[k], out_host=outs[k], out="packed", llr_scale=scale.get(k))
    for _ in range(runs):
        for k in fmts:
            barrier(world)
            t0 = time.perf_counter()
            g.decode_batch_host(hosts[k], out_host=outs[k], out="packed", llr_scale=scale.get(k))
            dt = time.perf_counter() - t0
            dt = dt if world == 1 else _max(dt, world)        # the slowest rank
            res[k].append(world * B * g.k_info / dt / 1e9)
    return {k: stats(v) for k, v in res.items()}


def _max(x, world):
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def int8_fields(r, same8):
    """the int8 figures of a resident comparison (none without --int8)"""
    if same8 is None:
        return {}
    return {"i8_over_f16_best": r["int8"]["best"] / r["float16"]["best"],
            "i8_over_f32_best": r["int8"]["best"] / r["float32"]["best"], "int8_scale": I8_SCALE,
            "int8_outputs_equal_float32_of_product": same8}


def e2e_entry(g, xe, args, world, fmts):
    """decode_batch_host from pinned buffers of each format, and the resident rate of the same frames"""
    er = e2e(g, xe, args.runs, world, fmts)
    re_, _, _ = resident(g, xe, args.runs, world, 10, fmts)
    esz = {"float32": 4, "float16": 2, "int8": 1}
    return {
        "frames_per_rank": args.e2e_frames, "chunk": "one wave of the decode kernel (the default)", "api": 'decode_batch_host(out="packed"), pinned input, 3-stream pipeline',
        "h2d_bytes_per_frame": {k: g.n_llr * esz[k] for k in fmts}, "d2h_bytes_per_frame": 56,
        "info_gbit_per_s": er, "resident_info_gbit_per_s_same_frames": re_,
        "frac_of_resident": {k: er[k]["best"] / re_[k]["best"] for k in er}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--tpf-frames", type=int, default=1 << 20)
    ap.add_argument("--e2e-frames", type=int, default=1 << 18)
    ap.add_argument("--int8", action="store_true", help="add int8 LLRs (scale 0.25) and the nii16 mode")
    args = ap.parse_args()
    fmts = ("float32", "float16", "int8") if args.int8 else ("float32", "float16")
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
    r, same, same8 = resident(g, x, args.runs, world, 3, fmts)
    res["tpf_n212_r13_8it"] = {"frames_per_rank": args.tpf_frames, "kernel": "tpf_kernel", "info_gbit_per_s": r,
                               "f16_over_f32_best": r["float16"]["best"] / r["float32"]["best"],
                               "outputs_equal_float32_of_widening": same, **int8_fields(r, same8)}
    xe = x[:args.e2e_frames].clone()
    del x
    res["e2e_n212_r13_8it_packed"] = e2e_entry(g, xe, args, world, fmts)
    del xe
    torch.cuda.empty_cache()

    q = turbo.DVBRCS2_Turbo(752, '1/2', 8)
    B = 4 * 4736
    x = llrs(q, B)
    r, same, same8 = resident(q, x, args.runs, world, 20, fmts)
    res["quad_n752_r12_8it"] = {"frames_per_rank": B, "kernel": "quad_kernel (auto choice: global-record geometry)",
                                "info_gbit_per_s": r, "f16_over_f32_best": r["float16"]["best"] / r["float32"]["best"],
                                "outputs_equal_float32_of_widening": same, **int8_fields(r, same8)}
    del x
    torch.cuda.empty_cache()

    if args.int8:
        n16 = turbo.DVBRCS2_Turbo(212, '1/3', 8, boundary="nii16")
        x = llrs(n16, args.tpf_frames)
        r, same, same8 = resident(n16, x, args.runs, world, 6, fmts)
        res["nii16_n212_r13_8it"] = {"frames_per_rank": args.tpf_frames, "kernel": "nii_kernel (nii16 mode)",
                                     "info_gbit_per_s": r, "outputs_equal_float32_of_widening": same,
                                     **int8_fields(r, same8)}
        xe = x[:args.e2e_frames].clone()
        del x
        res["nii16_e2e_n212_r13_8it_packed"] = e2e_entry(n16, xe, args, world, fmts)
        del xe
        torch.cuda.empty_cache()

    res["copy_ceiling"] = {f"llr_bytes_{esz}": h2d_ceiling.measure(args.e2e_frames, esz, dev, world)
                           for esz in ((4, 2, 1) if args.int8 else (4, 2))}
    res["card_after"] = card()
    if rank == 0:
        print(json.dumps(res), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
