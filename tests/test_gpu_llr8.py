"""GPU tests of the int8 channel-LLR input path (b200dvb_decode_i8, decode_batch / decode_batch_host with int8 input
and llr_scale).  The contract: decoding int8 LLRs q with scale s gives exactly what decoding the float32 array
float32(q) * float32(s) gives, bit for bit, in every decoder mode and for every kernel.  The oracle of every case is the
C oracle (or the non-parity mode's C model) fed that float32 array; the float32 GPU path fed the same values must match
too, on bits, packed words and the in-kernel error counters."""
import ctypes
import os

import numpy as np
import pytest

from oracle import oracle

pytestmark = pytest.mark.gpu

RATE = {'1/3': 1 / 3, '1/2': 1 / 2, '2/3': 2 / 3, '3/4': 3 / 4}
MODELS = {"double-pass": oracle.OracleTurbo, "nii": oracle.NiiModel, "nii16": oracle.Nii16Model}
# 0.37: the product q * 0.37 rounds; -0.6: a sign flip fused into the scale (and a rounding product)
SCALES = (1.0, 0.25, 0.37, -0.6)
THREADS = os.cpu_count() or 1


def _codec(N, rate, kernel="auto", boundary="double-pass"):
    from modulations_b200 import dvb_rcs2_turbo as turbo
    iters = 8 if N <= 212 else 4
    g = turbo.DVBRCS2_Turbo(N, rate, iters, kernel=kernel, boundary=boundary)
    g.handle                                              # ValueError where N has no geometry for the kernel
    return g, MODELS[boundary](N, rate, iters, perm=g.perm, inv_perm=g.inv_perm)


def _awgn(g, o, rate, B, ebn0, rs):
    """info bits [B, 2N] and float64 BPSK/AWGN LLRs clipped to +-50 [B, n_llr] (rate 2/3: n_coded is short of what the
    depuncturer consumes, the reference's truncation; the tail is zero-padded as tests/test_gpu_nii.py does)."""
    info = rs.randint(0, 2, (B, g.k_info))
    coded = np.asarray(o.encode_batch(info)).astype(np.float64)
    nv = 1.0 / (2.0 * RATE[rate] * 10 ** (ebn0 / 10))
    llr = np.clip(2.0 * ((1.0 - 2.0 * coded) + np.sqrt(nv) * rs.randn(*coded.shape)) / nv, -50, 50)
    if llr.shape[1] < g.n_llr:
        llr = np.pad(llr, ((0, 0), (0, g.n_llr - llr.shape[1])))
    return info.astype(np.uint8), llr


def _frames8(g, o, rate, B, ebn0, seed):
    """info bits and int8 LLRs q = clamp(rint(2.5 llr), -128, 127) [B, n_llr], with -128 planted in every frame."""
    rs = np.random.RandomState(seed)
    info, llr = _awgn(g, o, rate, B, ebn0, rs)
    q = np.clip(np.rint(2.5 * llr), -128, 127).astype(np.int8)
    cols = rs.randint(0, g.n_llr, (B, 3))
    q[np.arange(B)[:, None], cols] = -128
    return info, q


def _widen(q, s):
    """the float32 values the int8 contract names: float32(q) * float32(s), one IEEE float32 product each"""
    return q.astype(np.float32) * np.float32(s)


def _decode_all(g, x, info, llr_scale=None):
    """(bits, packed, counters) of one decode_batch call per layout on CUDA tensor x, counting against info."""
    import torch
    ref = torch.from_numpy(info).cuda()
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    bits = g.decode_batch(x, ref_bits=ref, counters=cnt, llr_scale=llr_scale)
    packed = g.decode_batch(x, out="packed", llr_scale=llr_scale)
    return bits.cpu().numpy(), packed.cpu().numpy(), cnt.cpu().numpy()


def _decode_as_laid_out(g, x, info, scale):
    """(bits, packed, counters) of ONE call of b200dvb_decode_i8 given int8 x's own data pointer and row stride.
    decode_batch would first copy a strided or offset view into a compact tensor; this hands the decoder the layout
    itself."""
    import torch
    from modulations_b200 import _lib
    h = g.handle
    B = x.shape[0]
    bits = torch.empty((B, g.k_info), dtype=torch.int32, device="cuda")
    packed = torch.empty((B, (g.k_info + 31) // 32), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    ref = torch.from_numpy(info).cuda()
    ws, need = h.workspace("decode", B)
    rc = _lib.load().b200dvb_decode_i8(h.h, B, ctypes.c_void_p(x.data_ptr()), x.stride(0), scale, _lib.ptr(bits),
                                       _lib.ptr(packed), _lib.ptr(ref), _lib.ptr(cnt), _lib.ptr(ws), need,
                                       ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc, "decode")
    return bits.cpu().numpy(), packed.cpu().numpy(), cnt.cpu().numpy()


def _assert_outputs(g, out8, out32, info, ref, what):
    from modulations_b200 import dvb_rcs2_turbo as turbo
    (b8, p8, c8), (b32, p32, c32) = out8, out32
    assert np.array_equal(b8, ref), f"{what}: {np.sum(b8 != ref)} bits differ from the oracle"
    assert np.array_equal(turbo.unpack_bits(p8, g.k_info), ref), f"{what}: packed words differ from the oracle"
    assert np.array_equal(b8, b32) and np.array_equal(p8, p32), f"{what}: int8 and float32 paths differ"
    assert np.array_equal(c8, c32), f"{what}: counters {c8} != {c32}"
    assert c8[0] == np.sum(ref != info) and c8[1] == np.sum(np.any(ref != info, axis=1))
    assert c8[2] == len(ref) and c8[3] == len(ref) * g.k_info


def _check_batches(g, o, q, info, what, big_scale):
    """Every scale on batches of 1, 16, 17 and 37 frames, and `big_scale` on the whole of q (one wave + 7 frames)."""
    import torch
    xq = torch.from_numpy(q).cuda()
    for s in SCALES:
        x32 = _widen(q[:37], s)
        ref = o.decode_batch(x32, threads=THREADS)
        x32d = torch.from_numpy(x32).cuda()
        for B in (1, 16, 17, 37):
            _assert_outputs(g, _decode_all(g, xq[:B], info[:B], s), _decode_all(g, x32d[:B], info[:B]), info[:B],
                            ref[:B], f"{what} scale={s} B={B}")
    x32 = _widen(q, big_scale)
    ref = o.decode_batch(x32, threads=THREADS)
    _assert_outputs(g, _decode_all(g, xq, info, big_scale), _decode_all(g, torch.from_numpy(x32).cuda(), info), info,
                    ref, f"{what} scale={big_scale} B={len(q)}")


CONFIGS = [(48, '1/3'), (64, '1/2'), (212, '1/3'), (212, '3/4'), (64, '2/3'), (424, '1/2'), (752, '1/2'), (848, '1/3')]
KERNEL_CASES = [(k, N, r) for k in ("auto", "quad", "tpf", "lat") for N, r in CONFIGS
                if not (k == "tpf" and N > 212)]                 # the thread-per-frame kernel has no geometry beyond 212


@pytest.mark.parametrize("kernel,N,rate", KERNEL_CASES)
def test_i8_every_kernel_equals_oracle_of_product(kernel, N, rate):
    """N=212 R=3/4 has n_llr = 583 (odd): contiguous rows cannot take the bulk-copy or paired loads, the per-element
    paths run.  The wave-sized batch takes one scale per case, in turn."""
    g, o = _codec(N, rate, kernel)
    big = g.handle.frames_per_wave + 7
    info, q = _frames8(g, o, rate, big, 2.0, 100 * N + len(kernel))
    _check_batches(g, o, q, info, f"{kernel} N={N} R={rate}", SCALES[KERNEL_CASES.index((kernel, N, rate)) % len(SCALES)])


@pytest.mark.parametrize("boundary", ["nii", "nii16"])
@pytest.mark.parametrize("N,rate", [(48, '1/3'), (212, '1/3'), (212, '3/4'), (64, '2/3')])
def test_i8_nonparity_modes_equal_their_models(boundary, N, rate):
    g, m = _codec(N, rate, boundary=boundary)
    big = g.handle.frames_per_wave + 7
    info, q = _frames8(g, m, rate, big, 2.0, 7 * N + len(boundary))
    _check_batches(g, m, q, info, f"{boundary} N={N} R={rate}", 0.37 if boundary == "nii" else 0.25)


@pytest.mark.parametrize("N,rate", [(212, '1/3'), (48, '1/3'), (212, '3/4')])
def test_i8_nii16_lossless_quarter_units(N, rate):
    """nii16 quantises every channel LLR x to clamp(rint(4 x), -127, 127) in 1/4 units.  Handing it exactly that int8
    with scale 0.25 decodes to the same result as x itself (the product q * 0.25 is exact and quantises back to q),
    on AWGN LLRs and on inputs saturated at +-50, against the nii16 model too."""
    import torch
    g, m = _codec(N, rate, boundary="nii16")
    B = g.handle.frames_per_wave + 7
    rs = np.random.RandomState(N + 16)
    info, llr = _awgn(g, m, rate, B, 1.0, rs)
    sat = np.where(rs.randint(0, 2, llr.shape) == 1, 50.0, -50.0)
    for what, x in (("awgn", llr.astype(np.float32)), ("saturated", sat.astype(np.float32))):
        q = np.clip(np.rint(4 * x), -127, 127).astype(np.int8)
        ref = m.decode_batch(x, threads=THREADS)
        out8 = _decode_all(g, torch.from_numpy(q).cuda(), info, 0.25)
        out32 = _decode_all(g, torch.from_numpy(x).cuda(), info)
        _assert_outputs(g, out8, out32, info, ref, f"nii16 N={N} R={rate} {what}")
        assert np.array_equal(g.decode_batch_host(torch.from_numpy(q).pin_memory(), llr_scale=0.25).numpy(), ref)


@pytest.mark.parametrize("kernel,boundary,N,rate", [("tpf", "double-pass", 212, '1/3'), ("quad", "double-pass", 212, '1/3'),
                                                    ("lat", "double-pass", 212, '1/3'), ("auto", "nii", 212, '1/3'),
                                                    ("auto", "nii16", 212, '1/3'), ("quad", "double-pass", 752, '1/2'),
                                                    ("tpf", "double-pass", 64, '1/2')])
def test_i8_row_pitch_and_alignment_paths(kernel, boundary, N, rate):
    """The decoder is handed each int8 layout as it is (pointer and row stride through the C ABI, no compacting copy):
    row pitches n_llr, n_llr + 1, n_llr + 3, n_llr + 16 and n_llr rounded up to 16 bytes, each with the rows starting
    0 / 1 / 2 / 3 / 16 bytes into a 256-byte aligned allocation.  This runs the bulk-copy (16-byte pitch and base) and
    the per-element transpositions of tpf / nii and the char2 (even pitch and base) and scalar loads of quad.  Every
    layout gives the oracle's decisions and exactly what the float32 path gives on the products."""
    import torch
    g, o = _codec(N, rate, kernel, boundary)
    B = 70
    info, q = _frames8(g, o, rate, B, 1.5, 4242 + N)
    s = 0.37
    x32 = _widen(q, s)
    ref = o.decode_batch(x32, threads=THREADS)
    out32 = _decode_all(g, torch.from_numpy(x32).cuda(), info)
    n = q.shape[1]
    src = torch.from_numpy(q).cuda()
    for pitch in (n, n + 1, n + 3, n + 16, (n + 15) // 16 * 16):
        for off in (0, 1, 2, 3, 16):
            buf = torch.zeros(B * pitch + off, dtype=torch.int8, device="cuda")
            assert buf.data_ptr() % 256 == 0
            x = buf.as_strided((B, n), (pitch, 1), off)
            x.copy_(src)
            assert x.data_ptr() == buf.data_ptr() + off and x.stride(0) == pitch
            _assert_outputs(g, _decode_as_laid_out(g, x, info, s), out32, info, ref,
                            f"{kernel}/{boundary} pitch n+{pitch - n}, offset {off} B")


@pytest.mark.parametrize("N,rate", [(212, '1/3'), (752, '1/2'), (212, '3/4')])
def test_i8_host_pipeline_all_layouts(N, rate):
    """decode_batch_host with a pinned int8 buffer of more frames than one chunk, for out = bits / packed / uint8,
    read on the host right after the call; equal to the float32 pipeline on the products and to the oracle."""
    import torch
    from modulations_b200 import dvb_rcs2_turbo as turbo
    g, o = _codec(N, rate)
    nfr, s = 50, -0.6
    info, q = _frames8(g, o, rate, nfr, 1.0, 77 + N)
    ref = o.decode_batch(_widen(q, s), threads=THREADS)
    reps = g.handle.frames_per_wave // nfr + 3                     # more frames than one chunk (one wave)
    x8 = torch.from_numpy(np.tile(q, (reps, 1))).pin_memory()
    x32 = torch.from_numpy(np.tile(_widen(q, s), (reps, 1))).pin_memory()
    want = np.tile(ref, (reps, 1))
    for out in ("bits", "packed", "uint8"):
        got8 = g.decode_batch_host(x8, out=out, llr_scale=s).numpy().copy()
        got32 = g.decode_batch_host(x32, out=out).numpy().copy()
        assert np.array_equal(got8, got32), out
        dec = turbo.unpack_bits(got8, g.k_info) if out == "packed" else got8.astype(np.int32)
        assert np.array_equal(dec, want), out
    # a numpy int8 array is accepted as well (the device gets the 8-bit values)
    assert np.array_equal(g.decode_batch_host(q, llr_scale=s).numpy(), ref)
    with pytest.raises(IndexError):
        g.decode_batch_host(x8.double())
    with pytest.raises(ValueError):
        g.decode_batch_host(x32, llr_scale=s)                      # a scale is never silently ignored


@pytest.mark.parametrize("N,rate", [(212, '1/3'), (64, '2/3')])
def test_i8_default_scale_is_todays_int8_decode(N, rate):
    """Without llr_scale, int8 input decodes as the values q themselves, which is what converting it to float32
    gives (the behaviour before int8 reached the device)."""
    import torch
    g, o = _codec(N, rate)
    info, q = _frames8(g, o, rate, 40, 2.0, 5 + N)
    want = g.decode_batch(q.astype(np.float32))
    assert np.array_equal(g.decode_batch(q), want)
    assert np.array_equal(g.decode_batch(torch.from_numpy(q).cuda()).cpu().numpy(), want)
    assert np.array_equal(g.decode_batch(q, llr_scale=1.0), want)


@pytest.mark.parametrize("kernel,N,rate,B", [("tpf", 212, '1/3', 100_000), ("quad", 752, '1/2', 100_000)])
def test_i8_randomised_large_batch_vs_oracle(kernel, N, rate, B):
    """10^5 DISTINCT device-generated frames (Philox source, Eb/N0 2 dB) quantised on the device to int8 with a scale
    whose products round, against the C oracle on every host thread; a second decode over the same workspace changes
    nothing."""
    import torch
    from modulations_b200 import dvb_rcs2_turbo as turbo
    g, o = _codec(N, rate, kernel)
    h = g.handle
    info = torch.empty((B, g.k_info), dtype=torch.uint8, device="cuda")
    coded = torch.empty((B, h.n_llr), dtype=torch.uint8, device="cuda")
    llr = torch.empty((B, h.n_llr), dtype=torch.float32, device="cuda")
    h.mc_generate_bpsk(B, 1.0 / (2.0 * (g.k_info / h.n_llr) * 10 ** 0.2), 2026 + N, 0, info, coded, llr)
    s = 0.37
    q = torch.clamp(torch.round(llr / s), -128, 127).to(torch.int8)
    got = turbo.unpack_bits(g.decode_batch(q, out="packed", llr_scale=s).cpu(), g.k_info)
    ref = o.decode_batch(_widen(q.cpu().numpy(), s), threads=THREADS)
    bad = np.flatnonzero(np.any(got != ref, axis=1))
    assert bad.size == 0, f"{bad.size} of {B} frames differ (first: {bad[:8]})"
    again = turbo.unpack_bits(g.decode_batch(q, out="packed", llr_scale=s).cpu(), g.k_info)
    assert np.array_equal(again, got)


def test_decode_i8_argument_errors():
    import torch
    from modulations_b200 import _lib
    g, _ = _codec(212, '1/3', "tpf")                              # checks its workspace size (a 32-frame batch would go to lat)
    h = g.handle
    lib = _lib.load()
    B, n = 32, h.n_llr
    x = torch.zeros((B, n + 1), dtype=torch.int8, device="cuda")
    bits = torch.empty((B, g.k_info), dtype=torch.int32, device="cuda")
    need = int(lib.b200dvb_decode_workspace_bytes(h.h, B))
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(ptr, stride, nbytes, scale=0.25):
        return lib.b200dvb_decode_i8(h.h, B, ptr, stride, scale, _lib.ptr(bits), None, None, None, _lib.ptr(ws),
                                     nbytes, st)

    assert call(None, n, need) == _lib.EINVAL                      # NULL llr
    assert call(_lib.ptr(x), n - 1, need) == _lib.EINVAL           # row stride shorter than n_llr
    assert call(_lib.ptr(x), n, need - 1) == _lib.ENOMEM           # workspace too small
    for bad in (0.0, -0.0, float("nan"), float("inf"), float("-inf")):
        assert call(_lib.ptr(x), n, need, bad) == _lib.EINVAL, bad
    assert call(ctypes.c_void_p(x.data_ptr() + 1), n, need) == _lib.OK   # no alignment requirement
    assert call(_lib.ptr(x), n, need, -2.0) == _lib.OK
    torch.cuda.synchronize()
    with pytest.raises(ValueError):
        g.decode_batch(x, llr_scale=float("nan"))
    with pytest.raises(ValueError):
        g.decode_batch(x.float(), llr_scale=0.25)                  # llr_scale with float input
    with pytest.raises(ValueError):
        g.decode_batch(x.half(), llr_scale=0.25)
