#!/usr/bin/env python3
"""Cost of the soft output: hard-only decodes (packed words) against packed words + a-posteriori LLRs
(b200dvb_decode_app), on the same frames, one GPU.

    python tools/app_perf.py [--runs 3] > profiles/r03_app_perf_n1.txt

Resident cases time back-to-back decodes of device-resident float32 LLRs with CUDA events after a warm-up; the two
variants are alternated, `--runs` of each, on preallocated outputs and one workspace:
  * tpf:   N=212 R=1/3 8 iterations, 2^20 frames (2.7 GB of LLRs, 1.8 GB of app: larger than L2), thread-per-frame kernel;
  * quad:  N=752 R=1/2 8 iterations, 4 waves of the automatic choice (the global-record geometry);
  * nii16: N=212 R=1/3 8 iterations, 2^20 frames, nii kernel in the nii16 mode;
  * lat:   N=212 R=1/3 8 iterations, B=1 (the low-latency kernel), time per call over 2 000 calls (the frame fits L2).
End to end: decode_batch_host(out="packed") against decode_batch_host(out="app") from a pinned float32 buffer of 2^18
frames at N=212 (host clock; the call returns when the last copy has completed).
Prints the card's name, power limit and SM clock read in this run, one JSON line per case, and the card again.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from modulations_b200 import dvb_rcs2_turbo as turbo  # noqa: E402


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


def stats(v):
    return {"runs": v, "best": min(v), "worst": max(v), "spread": max(v) - min(v)}


def resident(g, x, runs, reps):
    """ms per decode call of `x` with out = packed, and packed + app, alternated; also whether the packed words of the
    two variants are equal"""
    h = g.handle
    B = x.shape[0]
    packed = torch.empty((B, (g.k_info + 31) // 32), dtype=torch.int32, device="cuda")
    packed2 = torch.empty_like(packed)
    app = torch.empty((B, g.k_info), dtype=torch.float32, device="cuda")
    ws = h.workspace("decode", B)
    variants = {"packed": dict(packed=packed), "packed+app": dict(packed=packed2, app=app)}
    for kw in variants.values():                              # warm both paths
        h.decode(x, ws=ws, **kw)
    torch.cuda.synchronize()
    same = bool(torch.equal(packed, packed2))
    ms = {k: [] for k in variants}
    for _ in range(runs):
        for name, kw in variants.items():
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                h.decode(x, ws=ws, **kw)
            b.record()
            torch.cuda.synchronize()
            ms[name].append(a.elapsed_time(b) / reps)
    del app, packed, packed2
    return ms, same


def report(case, g, B, ms, same, extra=None):
    s = {k: stats(v) for k, v in ms.items()}
    res = {"case": case, "frames": B, "ms_per_call": s,
           "info_gbit_per_s_best": {k: B * g.k_info / (v["best"] * 1e-3) / 1e9 for k, v in s.items()},
           "app_over_packed_time_best": s["packed+app"]["best"] / s["packed"]["best"],
           "app_bytes_per_frame": 4 * g.k_info, "packed_equal": same}
    res.update(extra or {})
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--frames", type=int, default=1 << 20)
    ap.add_argument("--e2e-frames", type=int, default=1 << 18)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    print(json.dumps({"tool": "app_perf", "card": card(), "runs": args.runs}), flush=True)

    g = turbo.DVBRCS2_Turbo(212, '1/3', 8, kernel="tpf")
    x = llrs(g, args.frames)
    ms, same = resident(g, x, args.runs, 3)
    report("tpf N=212 R=1/3 8 it", g, args.frames, ms, same, {"kernel": "tpf_kernel"})
    del x
    torch.cuda.empty_cache()

    q = turbo.DVBRCS2_Turbo(752, '1/2', 8)
    B = 4 * q.handle.frames_per_wave
    x = llrs(q, B)
    ms, same = resident(q, x, args.runs, 10)
    report("quad N=752 R=1/2 8 it", q, B, ms, same, {"kernel": "quad_kernel (automatic choice)", "waves": 4})
    del x
    torch.cuda.empty_cache()

    n16 = turbo.DVBRCS2_Turbo(212, '1/3', 8, boundary="nii16")
    x = llrs(n16, args.frames)
    ms, same = resident(n16, x, args.runs, 6)
    report("nii16 N=212 R=1/3 8 it", n16, args.frames, ms, same, {"kernel": "nii_kernel (nii16 mode)"})
    del x
    torch.cuda.empty_cache()

    lat = turbo.DVBRCS2_Turbo(212, '1/3', 8)
    x = llrs(lat, 16)[:1].contiguous()                       # the source generates whole draws of 16 frames
    ms, same = resident(lat, x, args.runs, 2000)
    report("lat N=212 R=1/3 8 it B=1", lat, 1, ms, same, {"kernel": "lat_kernel (automatic choice for B=1)"})
    del x

    xh = llrs(g, args.e2e_frames).cpu().pin_memory()
    outs = {"packed": torch.empty((args.e2e_frames, (g.k_info + 31) // 32), dtype=torch.int32, pin_memory=True),
            "app": torch.empty((args.e2e_frames, g.k_info), dtype=torch.float32, pin_memory=True)}
    g2 = turbo.DVBRCS2_Turbo(212, '1/3', 8)                   # the automatic kernel choice, as a user gets it
    e2e = {k: [] for k in outs}
    for k in outs:                                            # warm: pipeline buffers, streams
        g2.decode_batch_host(xh, out_host=outs[k], out=k)
    for _ in range(args.runs):
        for k in outs:
            g2.decode_batch_host(xh, out_host=outs[k], out=k)   # the pipeline is rebuilt per layout: time the second
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            g2.decode_batch_host(xh, out_host=outs[k], out=k)
            e2e[k].append((time.perf_counter() - t0) * 1e3)
    s = {k: stats(v) for k, v in e2e.items()}
    print(json.dumps({"case": "decode_batch_host N=212 R=1/3 8 it, pinned float32 in", "frames": args.e2e_frames,
                      "ms_per_call": s,
                      "info_gbit_per_s_best": {k: args.e2e_frames * g.k_info / (v["best"] * 1e-3) / 1e9
                                               for k, v in s.items()},
                      "app_over_packed_time_best": s["app"]["best"] / s["packed"]["best"],
                      "d2h_bytes_per_frame": {"packed": 4 * ((g.k_info + 31) // 32), "app": 4 * g.k_info}}), flush=True)
    print(json.dumps({"card_after": card()}), flush=True)


if __name__ == "__main__":
    main()
