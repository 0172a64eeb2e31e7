#!/usr/bin/env python3
"""bench.py — headline benchmark of the B200 baseband decode hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): turbo info Gbit/s for N=212-couple rate-1/3 frames decoded
with 8 max-log-MAP iterations.  One "step" = one decode pass over one batch of
synthetic frames (1 M frames per GPU, BPSK over AWGN at Eb/N0 = 2 dB, generated on
the device).  `value` is whole-job throughput with the LLRs already resident in HBM;
`e2e` is the same metric through `DVBRCS2_Turbo.decode_batch_host` with pinned HOST
buffers (H2D of the LLRs and D2H of the hard bits inside the timed region), next to
the pinned-copy ceiling of the box measured in the same run.

Prints ONE JSON line (rank 0).  See DESIGN.md §6 for how each field is derived.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_COUPLES, RATE, ITERS, EBN0_DB = 212, '1/3', 8, 2.0
ACS_PER_FRAME = 320 * N_COUPLES * 2 * ITERS          # SURVEY §8(d): 1 085 440
NOMINAL_ACS_PER_CLK_SM = 64.0                        # 1 FADD + 1 FMNMX per ACS at 128 issue slots/clk/SM
METRIC = "turbo_info_throughput_N212_R1/3_8it"
LLR_SEED = 20261018                                  # Philox seed of the headline frames (rank r: frames r*B ...)
WORKLOAD = "DVB-RCS2 rate-1/3 turbo, N=212 couples, BPSK AWGN Eb/N0=2 dB, max-log-MAP 8 iterations (BASELINE configs[1])"


_OUT = sys.stdout


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def lib_sha256():
    try:
        with open(os.path.join(ROOT, "modulations_b200", "libb200dvb.so"), "rb") as f:
            return hashlib.sha256(f.read()).hexdigest()
    except OSError:
        return None


def committed_ncu(sha):
    """profiles/r02_traffic.json: per-kernel figures read out of committed `ncu --set full` captures (DRAM bytes per
    frame, issue-slot and pipe utilisation), stamped with the sha256 of the library they were taken on and of the
    sources + flags it is built from (nvcc output is not byte-reproducible).  A figure from other kernels is NOT
    reported: the caller gets None plus the reason."""
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
    except Exception as e:
        return None, f"profiles/r02_traffic.json unreadable ({e!r})"
    if tr.get("lib_sha256") == sha:
        return tr, None
    try:        # the same SOURCES and flags compiled on another machine: identified by the hash of what the library is built from
        from modulations_b200.build import source_sha256
        if tr.get("src_sha256") == source_sha256():
            return tr, None
    except Exception:
        pass
    return None, ("profiles/r02_traffic.json was captured on another build of libb200dvb.so "
                  f"({str(tr.get('lib_sha256'))[:12]} != {str(sha)[:12]}, sources differ too): re-run tools/gpu_dram.sh")


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the reference's own numba decoder when baseline/_ref travelled and numba imports, else the C port
# ---------------------------------------------------------------------------------------------------
def host_frames(N, rate, frames, ebn0_db, seed, modulation="BPSK"):
    """Host-generated LLR frames with the reference's own channel model: BPSK `2y/sigma^2` clipped to +-50
    (turbo_test_suite.py:132-161) or QPSK `+2*sqrt(2)*y/N0` per component (test.py:62-78 with the correct sign,
    SURVEY F4).  The encoder is the oracle's (bit-exact with the reference's, tests/test_oracle_golden.py)."""
    from oracle import oracle
    o = oracle.OracleTurbo(N, rate, ITERS)
    rs = np.random.RandomState(seed)
    base = min(frames, 2048)
    info = rs.randint(0, 2, (base, 2 * N))
    coded = o.encode_batch(info).astype(np.float64)
    R = {'1/3': 1 / 3, '1/2': 1 / 2, '2/3': 2 / 3, '3/4': 3 / 4}[rate]
    reps = (frames + base - 1) // base
    tx = np.tile(1.0 - 2.0 * coded, (reps, 1))[:frames]
    if modulation == "BPSK":
        nv = 1.0 / (2.0 * R * 10 ** (ebn0_db / 10))
        llr = np.clip(2.0 * (tx + np.sqrt(nv) * rs.randn(*tx.shape)) / nv, -50, 50)
    else:                                                    # QPSK: unit-energy symbols, two bits each
        n0 = 1.0 / (2.0 * R * 10 ** (ebn0_db / 10))          # Es/N0 = 2 R Eb/N0
        y = tx / np.sqrt(2.0) + np.sqrt(n0 / 2.0) * rs.randn(*tx.shape)
        llr = np.clip(2.0 * np.sqrt(2.0) * y / n0, -50, 50)
    return np.tile(info, (reps, 1))[:frames].astype(np.uint8), llr.astype(np.float32)


def cpu_decode(N, rate, llr, threads=None):
    """-> (seconds, decoded uint8 [F, 2N], kind, detail).  kind "reference": the unmodified reference's
    `DVBRCS2_Turbo.decode` (numba) on one single-threaded process per core; "port": oracle/turbo_oracle.c on
    `threads` threads."""
    from baseline import ref_arm
    threads = threads or os.cpu_count() or 1
    ok, why = ref_arm.available()
    if ok:
        try:
            r = ref_arm.decode_timed(N, rate, ITERS, llr, procs=threads)
            return r["seconds"], r["decoded"], "reference", (
                f"/root/reference dvb_rcs2_turbo.DVBRCS2_Turbo.decode (numba, copy in baseline/_ref), {r['procs']} "
                f"single-threaded processes, JIT warm-up excluded")
        except Exception as e:                               # fall through to the port, and say why
            why = repr(e)
    from oracle import oracle
    o = oracle.OracleTurbo(N, rate, ITERS)
    t = time.time()
    dec = o.decode_batch(llr, threads=threads)
    return time.time() - t, dec.astype(np.uint8), "port", f"oracle/turbo_oracle.c on {threads} threads (reference arm unavailable: {why})"


def cpu_baseline(threads=None, seconds_of_cpu=20.0):
    """The reference decoder on the box's host cores over a bounded sample of the headline workload."""
    threads = threads or os.cpu_count() or 1
    from baseline import ref_arm
    per = 2.9e-3 if ref_arm.available()[0] else 1.0e-3       # s per frame per core: SURVEY §6 (numba) / round-1 port
    frames = int(max(threads * 16, min(seconds_of_cpu * threads / per / 4, 40000)))
    frames = (frames // threads) * threads
    _, llr = host_frames(N_COUPLES, RATE, frames, EBN0_DB, 7)
    dt, dec, kind, detail = cpu_decode(N_COUPLES, RATE, llr, threads)
    gbps = frames * 2 * N_COUPLES / dt / 1e9
    return {"value": gbps, "unit": "Gbit/s", "cores": threads, "kind": kind,
            "sample": f"{frames} frames N=212 R=1/3 8 it in {dt:.2f} s wall = {dt * threads / frames * 1e3:.2f} ms/frame/core; {detail}"}, dt


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on all host cores (rank 0 only)."""
    if rank != 0:
        return
    times = []
    base = None
    for i in range(args.warmup + args.steps):
        base, dt = cpu_baseline(seconds_of_cpu=max(4.0, 60.0 / max(1, args.warmup + args.steps)))
        if i >= args.warmup:
            times.append((base["value"], dt))
    val = float(np.mean([v for v, _ in times])) if times else base["value"]
    ms = float(np.mean([d for _, d in times])) * 1e3 if times else 0.0
    base["value"] = val
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Gbit/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": "bounded sample per step, see cpu_baseline.sample"},
            "cpu_baseline": base,
            "e2e": {"value": val, "unit": "Gbit/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), file=_OUT, flush=True)


DUMP_FRAMES = 16384            # 16384 frames x 424 bits as float32 = 27.8 MB: a dump stays small enough to keep and diff


def dump_outputs(out_dir, bits, counters):
    """--dump-outputs: what the headline decode handed its caller after the last timed step, for comparing two builds
    output for output.  bits.npy: the int32 hard decisions of a fixed, seeded sample of frames (all frames when
    there are at most DUMP_FRAMES), as float32 0/1 [S, 2N]; frame_index.npy: their rows in the batch (float64);
    counters.npy: the in-kernel counters (bit errors, frame errors, frames, bits; float64), accumulated over the
    timed steps as the caller's counter tensor holds them."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    B = bits.shape[0]
    idx = np.sort(np.random.RandomState(0).choice(B, min(B, DUMP_FRAMES), replace=False))
    sample = bits.index_select(0, torch.from_numpy(idx).to(bits.device)).cpu().numpy()
    np.save(os.path.join(out_dir, "bits.npy"), sample.astype(np.float32))
    np.save(os.path.join(out_dir, "frame_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "counters.npy"), np.asarray(counters, np.float64))


# ---------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from modulations_b200 import _lib
    from modulations_b200 import dvb_rcs2_turbo as turbo
    from modulations_b200 import montecarlo
    from modulations_b200.sdr_modem import gray_modem
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    codec = turbo.DVBRCS2_Turbo(N_COUPLES, RATE, ITERS)
    h = codec.handle
    B = args.frames
    nv = 1.0 / (2.0 * (1 / 3) * 10 ** (EBN0_DB / 10))
    info = torch.empty((B, codec.k_info), dtype=torch.uint8, device=dev)
    coded = torch.empty((B, h.n_llr), dtype=torch.uint8, device=dev)
    llr = torch.empty((B, h.n_llr), dtype=torch.float32, device=dev)
    h.mc_generate_bpsk(B, nv, LLR_SEED, rank * B, info, coded, llr)
    del coded
    bits = torch.empty((B, codec.k_info), dtype=torch.int32, device=dev)
    counters = torch.zeros(4, dtype=torch.int64, device=dev)
    ws = h.workspace("decode", B)
    stream = torch.cuda.current_stream()
    mp = measured_peaks()
    hbm = mp.get("hbm_gbs", 6650.0)
    hbm_src = "measured" if "hbm_gbs" in mp else "fallback"

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(fn, steps, warm):
        """`steps` calls of fn bracketed by barrier + synchronize, CUDA events on the launching stream, MAX over ranks.
        -> (total ms, per-step ms list of this rank)."""
        for _ in range(warm):
            fn()
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record(stream)
        for i in range(steps):
            fn()
            ev[i + 1].record(stream)
        barrier()
        t = torch.tensor([ev[0].elapsed_time(ev[-1])], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]

    def time_kernel(fn, reps=5, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream); fn(); b.record(stream)
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.mean(ts))

    # ---- headline: resident decode, one launch per step ---------------------------------------------------------
    def step():
        h.decode(llr, bits=bits, ref=info, counters=counters, ws=ws)

    for _ in range(args.warmup):
        step()
    barrier()
    counters.zero_()
    with ClockSampler(local_rank) as clk:
        total_ms, kernel_ms = timed_steps(step, args.steps, 0)
    if world > 1:
        dist.all_reduce(counters, op=dist.ReduceOp.SUM)          # the path's one real exchange (NCCL)
    ms_per_step = total_ms / args.steps
    frames_per_s = world * B / (ms_per_step * 1e-3)
    gbps = frames_per_s * codec.k_info / 1e9
    cnt = counters.cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, bits, cnt)

    # ---- roofline of the dominant kernel (tpf_kernel, the thread-per-frame decoder; one launch per step) ----
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    clocks = clk.summary()
    f_nom = (mp.get("sm_max_mhz") or 1965.0) * 1e6
    avg_kernel_s = float(np.mean(kernel_ms)) * 1e-3
    achieved = B * ACS_PER_FRAME / avg_kernel_s / 1e12          # T ACS/s on this GPU
    peak = NOMINAL_ACS_PER_CLK_SM * sms * f_nom / 1e12
    sha = lib_sha256()
    ncu, ncu_why = committed_ncu(sha)
    tpf_ncu = (ncu or {}).get("tpf_kernel", {})
    roof = {"bound": "alu", "achieved": achieved, "peak": peak, "unit": "TACS/s", "frac": achieved / peak,
            "traffic": tpf_ncu["dram_bytes_per_frame"] * B if "dram_bytes_per_frame" in tpf_ncu else None,
            "traffic_source": (f"dram__bytes_read+write of one tpf_kernel launch ({tpf_ncu.get('capture')}), per frame, "
                               "scaled to this batch; capture taken on the library with this sha256") if tpf_ncu else ncu_why,
            "algorithmic_io_bytes": 7208 * B,
            "issue_active": tpf_ncu.get("smsp__issue_active_pct"), "pipe_alu": tpf_ncu.get("pipe_alu_pct"),
            "pipe_fma": tpf_ncu.get("pipe_fma_pct"), "lib_sha256": sha,
            "note": "MODE: F3 merged-branch (SURVEY §0 F3: the reference trellis has parallel transitions and rounding is "
                    "monotone, so max(fl(a+g1), fl(a+g2)) == fl(a + max(g1,g2)) bit for bit; the kernel runs 32 FADD + 16 "
                    "FMNMX + 16 FSUB per recursion step instead of the reference's 64 + 64).  ACS = add-compare-select "
                    "of the REFERENCE algorithm (320*N per SISO, SURVEY 8d), so `achieved` is algorithmic ACS/s; peak = "
                    "64 ACS/clk/SM x SMs x max SM clock (issue-slot bound; FADD and FMNMX each measured at 128 "
                    "lane-ops/clk/SM on this part, profiles/r01_microbench.txt).  The kernel is bound by instruction "
                    "issue with ONE warp per scheduler, not by HBM, so MEASURED_PEAKS.json has no denominator for it.",
            "frac_at_measured_clock": (achieved / (NOMINAL_ACS_PER_CLK_SM * sms * clocks["sm_mhz"] * 1e6 / 1e12))
            if clocks.get("sm_mhz") else None}

    # ---- demapper + mapper (second half of the headline metric; BASELINE configs[3]): HBM-bound ---------------------
    demap, mapper = {}, {}
    nsym = 1 << 27
    chunks_for_1e10 = int(np.ceil(1e10 / nsym))
    iq = (torch.randn(nsym, 2, device=dev) * 0.7).view(torch.complex64).reshape(-1)
    demap_ncu = (ncu or {}).get("demap", {})
    for name in ("BPSK", "QPSK", "8PSK", "16QAM", "64QAM", "256QAM"):
        m = gray_modem(name)
        out = torch.empty(nsym * m.bps, dtype=torch.float32, device=dev)
        ms = time_kernel(lambda: _lib.check(lib.b200dvb_demap(m.h, nsym, _lib.ptr(iq), 0.05, 1.0, _lib.ptr(out),
                                                             _lib.stream_ptr()), "demap"))
        by = nsym * (8 + 4 * m.bps)
        gbs = by / (ms * 1e-3) / 1e9
        tr = demap_ncu.get(name, {}).get("dram_bytes_per_symbol")
        demap[name] = {"gsym_per_s": nsym / (ms * 1e-3) / 1e9, "bytes_per_symbol": 8 + 4 * m.bps, "symbols": nsym,
                       "seconds_for_1e10_symbols": ms * 1e-3 * 1e10 / nsym,
                       "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                                    "peak_source": hbm_src, "traffic": tr * nsym if tr else None}}
        if name in ("16QAM", "256QAM"):      # bf16x2 I/Q input (north_star "bf16x2 loads"), reported separately
            xb = torch.view_as_real(iq).to(torch.bfloat16).contiguous()
            ms = time_kernel(lambda: _lib.check(lib.b200dvb_demap_bf16(m.h, nsym, _lib.ptr(xb), 0.05, 1.0, _lib.ptr(out),
                                                                      _lib.stream_ptr()), "demap_bf16"))
            by = nsym * (4 + 4 * m.bps)
            gbs = by / (ms * 1e-3) / 1e9
            demap[name]["bf16x2_input"] = {"gsym_per_s": nsym / (ms * 1e-3) / 1e9, "bytes_per_symbol": 4 + 4 * m.bps,
                                           "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s",
                                                        "frac": gbs / hbm, "peak_source": hbm_src, "traffic": None}}
            del xb
        del out
        bits_in = torch.randint(0, 2, (nsym * m.bps,), dtype=torch.uint8, device=dev)
        sy = torch.empty(nsym, dtype=torch.complex64, device=dev)
        ms = time_kernel(lambda: _lib.check(lib.b200dvb_map(m.h, nsym, _lib.ptr(bits_in), _lib.ptr(sy), 0, _lib.stream_ptr()), "map"))
        by = nsym * (m.bps + 8)
        gbs = by / (ms * 1e-3) / 1e9
        mapper[name] = {"gsym_per_s": nsym / (ms * 1e-3) / 1e9, "bytes_per_symbol": m.bps + 8,
                        "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                                     "peak_source": hbm_src, "traffic": None},
                        "note": "one uint8 per bit in (the reference's layout), complex64 out"}
        del bits_in, sy
    del iq
    demap["_what"] = (f"BASELINE configs[3]: max-log LLR demap, 2^27 resident symbols per launch (larger than L2); 1e10 symbols = "
                      f"{chunks_for_1e10} such chunks (400 GB at 256QAM exceeds HBM), seconds_for_1e10_symbols = kernel time only")

    # ---- waveform stage next to the mapper / demapper (SURVEY 8(f) N4): HBM-bound streaming FIRs -------------
    waveform = {}
    try:
        from modulations_b200.modulators import Modulator
        mo = Modulator()                                           # reference defaults: sps 8, alpha 0.35, 49 taps
        nsw, nt, sps = 1 << 24, len(mo.rrc_filter), mo.sps
        taps_h = np.ascontiguousarray(mo.rrc_filter, np.float64)
        sy = (torch.randn(nsw, 2, device=dev) * 0.7).view(torch.complex64).reshape(-1)
        shaped = torch.empty((nsw - 1) * sps + nt, dtype=torch.complex64, device=dev)
        start = 2 * mo.filter_delay
        n_mf = (shaped.numel() + nt - 1 - start + sps - 1) // sps
        mf = torch.empty(n_mf, dtype=torch.complex64, device=dev)
        calls = (("pulse_shape", nsw * (8 + 8 * sps), lambda: lib.b200dvb_pulse_shape(
                      nsw, _lib.ptr(sy), _lib.host_ptr(taps_h), nt, sps, _lib.ptr(shaped), _lib.stream_ptr())),
                 ("matched_filter", n_mf * (8 * sps + 8), lambda: lib.b200dvb_matched_filter(
                      shaped.numel(), _lib.ptr(shaped), _lib.host_ptr(taps_h), nt, sps, start, n_mf, _lib.ptr(mf),
                      _lib.stream_ptr())))
        for name, by, call in calls:
            ms = time_kernel(lambda: _lib.check(call(), name))
            gbs = by / (ms * 1e-3) / 1e9
            waveform[name] = {"gsym_per_s": nsw / (ms * 1e-3) / 1e9, "symbols": nsw, "sps": sps, "taps": nt,
                              "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s",
                                           "frac": gbs / hbm, "peak_source": hbm_src, "traffic": None}}
        del sy, shaped, mf
    except Exception as e:                                         # never let the optional block break the headline line
        waveform = {"error": repr(e)}

    # ---- BASELINE configs[2]: 16QAM symbols -> soft demap -> turbo decode, device resident ---------
    Bc = min(B, 262144)
    nsym16 = (h.n_llr + 3) // 4
    m16 = gray_modem("16QAM")
    cb = torch.randint(0, 2, (Bc, nsym16 * 4), dtype=torch.uint8, device=dev)
    syms = m16.map(cb.reshape(-1))
    syms = syms + 0.1 * (torch.randn(syms.numel(), 2, device=dev).view(torch.complex64).reshape(-1))
    llr16 = torch.empty((Bc, nsym16 * 4), dtype=torch.float32, device=dev)
    cnt16 = torch.zeros(4, dtype=torch.int64, device=dev)
    ws16 = h.workspace("decode", Bc)

    def chain():
        _lib.check(lib.b200dvb_demap(m16.h, syms.numel(), _lib.ptr(syms), 0.02, -1.0, _lib.ptr(llr16), _lib.stream_ptr()), "demap")
        h.decode(llr16, ref=info[:Bc], counters=cnt16, ws=ws16)
    chain_total, _ = timed_steps(chain, args.steps, 2)
    chain_ms = chain_total / args.steps
    chain16 = {"info_gbit_per_s": world * Bc * codec.k_info / (chain_ms * 1e-3) / 1e9, "ms_per_step": chain_ms,
               "frames_per_gpu": Bc, "symbols_per_frame": nsym16,
               "what": "BASELINE configs[2]: 16QAM max-log demap (b200dvb_demap, decoder sign fused) + 8-iteration decode, resident"}
    del cb, syms, llr16

    # ---- non-parity decoder modes (SURVEY 8(f) N2): reported separately, never as `value` ---------------------------
    nonparity = {}
    try:
        Bn = min(B, 262144)
        cntp = torch.zeros(4, dtype=torch.int64, device=dev)
        wsp = h.workspace("decode", Bn)
        t_par, _ = timed_steps(lambda: h.decode(llr[:Bn], ref=info[:Bn], counters=cntp, ws=wsp), args.steps, 2)
        bpar = cntp.cpu().numpy().astype(float)
        what = {"nii": "single pass per SISO with next-iteration boundary metrics, float32 (csrc/decode_nii.cu, ArF32); bit-exact "
                       "against its own model oracle/nii_model.c",
                "nii16": "the same decoder in 16-bit fixed point, two frames per 32-bit register, add-compare-select as one DPX "
                         "instruction (VIADDMNMX.S16x2) per branch pair (csrc/nii16_core.cuh, ArS16); bit-exact against its own "
                         "integer model oracle/nii16_model.c"}
        for mode in ("nii", "nii16"):
            cn = turbo.DVBRCS2_Turbo(N_COUPLES, RATE, ITERS, boundary=mode)
            hn = cn.handle
            wsn = hn.workspace("decode", Bn)
            cntn = torch.zeros(4, dtype=torch.int64, device=dev)
            t_n, _ = timed_steps(lambda: hn.decode(llr[:Bn], ref=info[:Bn], counters=cntn, ws=wsn), args.steps, 2)
            a_ = cntn.cpu().numpy().astype(float)
            nonparity[mode] = {"info_gbit_per_s": world * Bn * codec.k_info / (t_n / args.steps * 1e-3) / 1e9,
                               "speedup_over_parity_mode": t_par / t_n, "frames_per_gpu": Bn,
                               "ber": a_[0] / max(a_[3], 1), "ber_parity_mode_same_frames": bpar[0] / max(bpar[3], 1),
                               "what": "NON-PARITY mode: " + what[mode]}
            del wsn
        nonparity["_note"] = ("BER here is on the committed interleaver, where every mode floors at ~0.2 (SURVEY F2); the comparison "
                              "that matters — bijective interleaver, same frames, binomial intervals — is tests/test_gpu_nii.py and "
                              "profiles/r02_ber_three_modes.txt")
        del wsp
    except Exception as e:
        nonparity = {"error": repr(e)}

    # ---- end to end with HOST buffers -----------------------------------------------------------------------------
    Be = min(B, args.e2e_frames)
    wpf = (codec.k_info + 31) // 32
    hin = torch.empty((Be, h.n_llr), dtype=torch.float32, pin_memory=True)
    hin.copy_(llr[:Be])
    torch.cuda.synchronize()
    e2e_modes = {}
    for mode, width, dt_ in (("packed", wpf, torch.int32), ("bits", codec.k_info, torch.int32)):
        hout = torch.empty((Be, width), dtype=dt_, pin_memory=True)
        tot, _ = timed_steps(lambda: codec.decode_batch_host(hin, hout, out=mode), args.steps, 2)
        val = world * Be * args.steps * codec.k_info / (tot * 1e-3) / 1e9
        got = turbo.unpack_bits(hout.numpy(), codec.k_info) if mode == "packed" else hout.numpy()
        same = bool(np.array_equal(got, bits[:Be].cpu().numpy()))
        e2e_modes[mode] = {"value": val, "d2h_bytes_per_step": Be * width * 4, "matches_resident_run": same}
        del hout
    # pinned-copy ceiling of this box, measured in the same run: the SAME bytes, plain cudaMemcpyAsync on two streams,
    # no kernel, all ranks at once (tools/h2d_ceiling.py is the stand-alone version)
    ceil = {}
    din = torch.empty((Be, h.n_llr), dtype=torch.float32, device=dev)
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    chunk = h.frames_per_wave
    for mode, width in (("packed", wpf), ("bits", codec.k_info)):
        hout = torch.empty((Be, width), dtype=torch.int32, pin_memory=True)
        dout = torch.empty((Be, width), dtype=torch.int32, device=dev)

        def copies():
            s_in.wait_stream(stream); s_out.wait_stream(stream)
            for lo in range(0, Be, chunk):
                hi = min(Be, lo + chunk)
                with torch.cuda.stream(s_in):
                    din[lo:hi].copy_(hin[lo:hi], non_blocking=True)
                with torch.cuda.stream(s_out):
                    hout[lo:hi].copy_(dout[lo:hi], non_blocking=True)
            stream.wait_stream(s_in); stream.wait_stream(s_out)
        tot, _ = timed_steps(copies, args.steps, 2)
        ms = tot / args.steps
        ceil[mode] = {"info_gbit_per_s": world * Be * codec.k_info / (ms * 1e-3) / 1e9,
                      "h2d_gbs_per_gpu": Be * h.n_llr * 4 / (ms * 1e-3) / 1e9,
                      "copy_gbs_all_gpus": world * Be * (h.n_llr * 4 + width * 4) / (ms * 1e-3) / 1e9}
        del hout, dout
    del din
    n_chunks = (Be + chunk - 1) // chunk
    e2e = {"value": e2e_modes["packed"]["value"], "unit": "Gbit/s", "h2d_bytes_per_step": Be * h.n_llr * 4,
           "d2h_bytes_per_step": e2e_modes["packed"]["d2h_bytes_per_step"], "frames_per_step": Be,
           "api": 'DVBRCS2_Turbo.decode_batch_host(out="packed"): pinned float32 LLRs in, the kernel\'s packed hard bits '
                  "(uint32 words, 56 B per frame) out, 3-stream pipeline, one kernel wave per chunk; the call returns after "
                  "its last device->host copy has completed",
           "matches_resident_run": e2e_modes["packed"]["matches_resident_run"],
           "copy_ceiling_gbit_per_s": ceil["packed"]["info_gbit_per_s"],
           "copy_ceiling_gbs": ceil["packed"]["copy_gbs_all_gpus"],
           "frac_of_ceiling": e2e_modes["packed"]["value"] / ceil["packed"]["info_gbit_per_s"],
           "frac_of_resident": e2e_modes["packed"]["value"] / gbps,
           "int32_layout": {"value": e2e_modes["bits"]["value"], "d2h_bytes_per_step": e2e_modes["bits"]["d2h_bytes_per_step"],
                            "matches_resident_run": e2e_modes["bits"]["matches_resident_run"],
                            "copy_ceiling_gbit_per_s": ceil["bits"]["info_gbit_per_s"],
                            "frac_of_ceiling": e2e_modes["bits"]["value"] / ceil["bits"]["info_gbit_per_s"],
                            "what": 'out="bits": the reference\'s int32[B, 2N] layout (1 696 B per frame device->host)'},
           "ceiling_what": "same bytes per step as plain pinned cudaMemcpyAsync H2D + D2H on two streams, no kernel, all "
                           "ranks concurrently, measured in this run"}

    # ---- e2e_mc: the reference's actual workflow (turbo_test_suite.py:121-199): device Philox source -> encode ->
    #      channel -> decode -> counters; 32 bytes cross PCIe per point --------------------------------------------
    Bm = min(B, 262144)
    cfg = montecarlo.SweepConfig(N=N_COUPLES, rate=RATE, iterations=ITERS, ebn0_db=[EBN0_DB],
                                 frames_per_point=world * Bm * 2, batch=Bm, seed=5)
    montecarlo.run_sweep(cfg, rank, world, codec=codec)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res_mc = montecarlo.run_sweep(cfg, rank, world, codec=codec)
    barrier()
    tm = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    mc_gbps = args.steps * cfg.frames_per_point * codec.k_info / float(tm.item()) / 1e9
    e2e_mc = {"value": mc_gbps, "unit": "Gbit/s", "frac_of_resident": mc_gbps / gbps,
              "frames_per_sweep": cfg.frames_per_point, "host_bytes_per_sweep": 32,
              "ber": res_mc["points"][0]["ber"], "fer": res_mc["points"][0]["fer"],
              "what": "montecarlo.run_sweep wall clock (max over ranks): Philox info bits -> encode -> BPSK/AWGN -> LLR -> "
                      "decode -> in-kernel counters -> one all_reduce; host sees 4 int64 per Eb/N0 point"}

    line_extra = {}
    if rank == 0 and world == 1:
        # ---- single-frame latency of the reference's call shape (turbo_test_suite.py:138-164) ---------------------
        x1 = llr[0].cpu().numpy()
        for _ in range(5):
            codec.decode(x1)
        ts = []
        for _ in range(30):
            t0 = time.perf_counter(); codec.decode(x1); ts.append(time.perf_counter() - t0)
        lat = {"decode_single_frame_us": float(np.median(ts) * 1e6), "what": "DVBRCS2_Turbo.decode(numpy llr) wall clock, "
               "median of 30 (H2D + one launch + D2H); small batches (up to min(6, N/50) passes of two CTAs per SM) run on the one-CTA-per-frame "
               "kernel (decode_lat.cu), batches up to one quad-kernel wave on the quad kernel, larger ones thread-per-frame"}
        for Bq in (1, 148, 256, 4096, 65536):
            xq = llr[:Bq]
            lat[f"resident_B{Bq}_us"] = time_kernel(lambda: codec.decode_batch(xq, out="packed"), reps=5, warm=2) * 1e3
        # ---- the reference's only runnable self-test configuration (test.py:12-14): N=752, R=1/2 -------------------
        c752 = turbo.DVBRCS2_Turbo(752, '1/2', ITERS)
        h752 = c752.handle
        B752 = 4 * h752.frames_per_wave
        i752 = torch.empty((B752, c752.k_info), dtype=torch.uint8, device=dev)
        c752c = torch.empty((B752, h752.n_llr), dtype=torch.uint8, device=dev)
        l752 = torch.empty((B752, h752.n_llr), dtype=torch.float32, device=dev)
        h752.mc_generate_bpsk(B752, 1.0 / (2 * 0.5 * 10 ** 0.2), 3, 0, i752, c752c, l752)
        cn752 = torch.zeros(4, dtype=torch.int64, device=dev)
        ms752 = time_kernel(lambda: c752.decode_batch(l752, ref_bits=i752, counters=cn752, out="none"), reps=3, warm=2)
        acs752 = 320 * 752 * 2 * ITERS
        a752 = B752 * acs752 / (ms752 * 1e-3) / 1e12
        _, l752h = host_frames(752, '1/2', 16 * (os.cpu_count() or 1), EBN0_DB, 11)
        dt752, dec752, kind752, det752 = cpu_decode(752, '1/2', l752h)
        g752 = c752.decode_batch(l752h)
        n752 = {"info_gbit_per_s": B752 * c752.k_info / (ms752 * 1e-3) / 1e9, "frames": B752, "ms": ms752,
                "roofline": {"bound": "alu", "achieved": a752, "peak": peak, "unit": "TACS/s", "frac": a752 / peak, "traffic": None},
                "kernel": "quad_kernel, global-record geometry (32 frames per SM, records in global memory fed through a cp.async ring: the records of longer frames do not fit on chip)",
                "cpu_baseline": {"value": len(l752h) * c752.k_info / dt752 / 1e9, "unit": "Gbit/s", "kind": kind752,
                                 "cores": os.cpu_count(), "sample": f"{len(l752h)} frames in {dt752:.2f} s; {det752}"},
                "matches_cpu_arm": bool(np.array_equal(g752, dec752)),
                "what": "N=752 couples, rate 1/2, 8 iterations: the configuration of the reference's only runnable self-test (test.py:12-14)"}
        del i752, c752c, l752
        # ---- BASELINE configs[0]: N=48 R=1/3 QPSK over AWGN, 100 000 IDENTICAL host-generated frames through the GPU
        #      (decode_batch_host) and through the CPU arm, both timed ------------------------------------------------
        c48 = turbo.DVBRCS2_Turbo(48, '1/3', ITERS)
        _, l48 = host_frames(48, '1/3', 100_000, EBN0_DB, 13, modulation="QPSK")
        p48 = torch.from_numpy(l48).pin_memory()
        o48 = torch.empty((len(l48), c48.k_info), dtype=torch.int32, pin_memory=True)
        for _ in range(2):
            c48.decode_batch_host(p48, o48)
        t0 = time.perf_counter()
        c48.decode_batch_host(p48, o48)
        gpu_s = time.perf_counter() - t0
        dt48, dec48, kind48, det48 = cpu_decode(48, '1/3', l48)
        cfg0 = {"frames": len(l48), "gpu_seconds": gpu_s, "gpu_info_gbit_per_s": len(l48) * 96 / gpu_s / 1e9,
                "cpu_seconds": dt48, "cpu_info_gbit_per_s": len(l48) * 96 / dt48 / 1e9, "cpu_kind": kind48, "cpu_detail": det48,
                "cpu_cores": os.cpu_count(), "speedup_e2e": dt48 / gpu_s,
                "outputs_identical": bool(np.array_equal(o48.numpy().astype(np.uint8), dec48)),
                "what": "BASELINE configs[0]: N=48 R=1/3 turbo, QPSK over AWGN (test.py:62-78 LLR with the correct sign), 8 iterations; "
                        "GPU = DVBRCS2_Turbo.decode_batch_host wall clock (pinned host LLRs -> int32 bits on the host)"}
        line_extra = {"latency": lat, "n752_r12": n752, "config0_n48_qpsk": cfg0}

    if rank == 0:
        base = cpu_baseline()[0] if world == 1 else None     # rank 0, N=1 only (tier contract)
        mb = np.zeros(8)
        lib.b200dvb_microbench(_lib.host_ptr(mb))
        line = {
            "metric": METRIC, "value": gbps, "unit": "Gbit/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "frames_per_gpu": B, "mframes_per_s": frames_per_s / 1e6,
                       "cache": "inputs larger than L2 (5.09 GB of LLRs per step)",
                       "output": "int32[B,2N] bits + in-kernel error counters",
                       "parallelism": f"frames sharded over {world} GPU(s); one NCCL all-reduce of int64[4] counters"},
            "roofline": roof, "cpu_baseline": base,
            "e2e": e2e, "e2e_mc": e2e_mc,
            "gpu_launches": args.steps, "gpu_launches_e2e": args.steps * n_chunks,
            "clocks": clocks,
            "counters": {"bit_errors": int(cnt[0]), "frame_errors": int(cnt[1]), "frames": int(cnt[2]),
                         "bits": int(cnt[3]), "note": "BER~0.2/FER=1 is the reference's behaviour (non-bijective "
                                                     "interleaver, SURVEY F2); parity is bit-exactness, not BER"},
            "demap": demap, "mapper": mapper, "waveform": waveform, "chain_16qam": chain16, "nonparity_modes": nonparity,
            "microbench_lane_ops_per_clk_sm": {k: float(v) for k, v in zip(
                ("fadd", "fmnmx", "acs_mix", "shfl", "dadd", "f2f", "fadd_x2", "clock_mhz"), mb)},
        }
        line.update(line_extra)
        print(json.dumps(line), file=_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=1_000_000, help="frames per GPU per step")
    ap.add_argument("--e2e-frames", type=int, default=262144, dest="e2e_frames")
    ap.add_argument("--dump-outputs", metavar="DIR", dest="dump_outputs",
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy "
                         "(bits.npy, frame_index.npy; counters.npy sums all --steps timed steps, so compare dumps "
                         "taken with the same arguments)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.frames = max(16, (args.frames // 16) * 16)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun with the contract's arguments
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29517"),
               os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    # stdout carries ONE JSON line.  Libraries write banners to file descriptor 1 behind Python's back (NCCL prints
    # "NCCL version ..." there on some boxes): fd 1 is pointed at stderr for the whole run and the line goes to a
    # private duplicate of the original stdout.
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
