"""GPU tests of the binary16 (fp16) channel-LLR input path (b200dvb_decode_f16, decode_batch / decode_batch_host with
float16 input).  The contract: decoding fp16 LLRs h gives exactly what decoding float32(h) gives, bit for bit, in every
decoder mode and for every kernel.  The oracle of every case is the C oracle (or the non-parity mode's C model) fed
h.astype(np.float32); the float32 GPU path fed the same widened values must match too, on bits, packed words and the
in-kernel error counters."""
import ctypes
import os

import numpy as np
import pytest

from oracle import oracle

pytestmark = pytest.mark.gpu

RATE = {'1/3': 1 / 3, '1/2': 1 / 2, '2/3': 2 / 3, '3/4': 3 / 4}
MODELS = {"double-pass": oracle.OracleTurbo, "nii": oracle.NiiModel, "nii16": oracle.Nii16Model}


def _codec(N, rate, kernel="auto", boundary="double-pass"):
    from modulations_b200 import dvb_rcs2_turbo as turbo
    iters = 8 if N <= 212 else 4
    g = turbo.DVBRCS2_Turbo(N, rate, iters, kernel=kernel, boundary=boundary)
    g.handle                                              # ValueError where N has no geometry for the kernel
    return g, MODELS[boundary](N, rate, iters, perm=g.perm, inv_perm=g.inv_perm)


def _frames16(g, o, rate, B, ebn0, seed):
    """info bits [B, 2N] and BPSK/AWGN LLRs rounded to float16 [B, n_llr] (rate 2/3: n_coded is short of what the
    depuncturer consumes, the reference's truncation; the tail is zero-padded as tests/test_gpu_nii.py does)."""
    rs = np.random.RandomState(seed)
    info = rs.randint(0, 2, (B, g.k_info))
    coded = np.asarray(o.encode_batch(info)).astype(np.float64)
    nv = 1.0 / (2.0 * RATE[rate] * 10 ** (ebn0 / 10))
    llr = np.clip(2.0 * ((1.0 - 2.0 * coded) + np.sqrt(nv) * rs.randn(*coded.shape)) / nv, -50, 50).astype(np.float16)
    if llr.shape[1] < g.n_llr:
        llr = np.pad(llr, ((0, 0), (0, g.n_llr - llr.shape[1])))
    return info.astype(np.uint8), llr


def _decode_all(g, x, info):
    """(bits, packed, counters) of one decode_batch call per layout on CUDA tensor x, counting against info."""
    import torch
    ref = torch.from_numpy(info).cuda()
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    bits = g.decode_batch(x, ref_bits=ref, counters=cnt)
    packed = g.decode_batch(x, out="packed")
    return bits.cpu().numpy(), packed.cpu().numpy(), cnt.cpu().numpy()


def _decode_as_laid_out(g, x, info):
    """(bits, packed, counters) of ONE call of b200dvb_decode_f16 (float16 x) or b200dvb_decode (float32 x) given x's
    own data pointer and row stride.  decode_batch would first copy a strided or offset view into a compact tensor;
    this hands the decoder the layout itself."""
    import torch
    from modulations_b200 import _lib
    h = g.handle
    lib = _lib.load()
    fn = lib.b200dvb_decode_f16 if x.dtype == torch.float16 else lib.b200dvb_decode
    B = x.shape[0]
    bits = torch.empty((B, g.k_info), dtype=torch.int32, device="cuda")
    packed = torch.empty((B, (g.k_info + 31) // 32), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    ref = torch.from_numpy(info).cuda()
    ws, need = h.workspace("decode", B)
    rc = fn(h.h, B, ctypes.c_void_p(x.data_ptr()), x.stride(0), _lib.ptr(bits), _lib.ptr(packed), _lib.ptr(ref),
            _lib.ptr(cnt), _lib.ptr(ws), need, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc, "decode")
    return bits.cpu().numpy(), packed.cpu().numpy(), cnt.cpu().numpy()


def _check_against_f32(g, x16, info, ref, what):
    """x16: CUDA float16 [B, n_llr].  Outputs must equal the oracle's decisions `ref` and the float32 path's outputs on
    the widened values, on all three outputs."""
    _assert_outputs(g, _decode_all(g, x16, info), _decode_all(g, x16.float(), info), info, ref, what)


def _assert_outputs(g, out16, out32, info, ref, what):
    from modulations_b200 import dvb_rcs2_turbo as turbo
    (b16, p16, c16), (b32, p32, c32) = out16, out32
    assert np.array_equal(b16, ref), f"{what}: {np.sum(b16 != ref)} bits differ from the oracle"
    assert np.array_equal(turbo.unpack_bits(p16, g.k_info), ref), f"{what}: packed words differ from the oracle"
    assert np.array_equal(b16, b32) and np.array_equal(p16, p32), f"{what}: fp16 and float32 paths differ"
    assert np.array_equal(c16, c32), f"{what}: counters {c16} != {c32}"
    assert c16[0] == np.sum(ref != info) and c16[1] == np.sum(np.any(ref != info, axis=1))
    assert c16[2] == len(ref) and c16[3] == len(ref) * g.k_info


CONFIGS = [(48, '1/3'), (64, '1/2'), (212, '1/3'), (212, '3/4'), (64, '2/3'), (424, '1/2'), (752, '1/2'), (848, '1/3')]
KERNEL_CASES = [(k, N, r) for k in ("auto", "quad", "tpf", "lat") for N, r in CONFIGS
                if not (k == "tpf" and N > 212)]                 # the thread-per-frame kernel has no geometry beyond 212


@pytest.mark.parametrize("kernel,N,rate", KERNEL_CASES)
def test_f16_every_kernel_equals_oracle_of_widening(kernel, N, rate):
    """Batches of 1, 16, 17, 37 frames and one larger than a wave.  N=212 R=3/4 has n_llr = 583 (odd): contiguous
    rows cannot take the bulk-copy or paired loads, the per-element paths run."""
    import torch
    g, o = _codec(N, rate, kernel)
    big = g.handle.frames_per_wave + 7
    info, h = _frames16(g, o, rate, big, 2.0, 100 * N + len(kernel))
    ref = o.decode_batch(h.astype(np.float32), threads=os.cpu_count() or 1)
    x = torch.from_numpy(h).cuda()
    for B in (1, 16, 17, 37, big):
        _check_against_f32(g, x[:B], info[:B], ref[:B], f"{kernel} N={N} R={rate} B={B}")


@pytest.mark.parametrize("boundary", ["nii", "nii16"])
@pytest.mark.parametrize("N,rate", [(48, '1/3'), (212, '1/3'), (212, '3/4'), (64, '2/3')])
def test_f16_nonparity_modes_equal_their_models(boundary, N, rate):
    import torch
    g, m = _codec(N, rate, boundary=boundary)
    big = g.handle.frames_per_wave + 7
    info, h = _frames16(g, m, rate, big, 2.0, 7 * N + len(boundary))
    ref = m.decode_batch(h.astype(np.float32), threads=os.cpu_count() or 1)
    x = torch.from_numpy(h).cuda()
    for B in (1, 16, 17, 37, big):
        _check_against_f32(g, x[:B], info[:B], ref[:B], f"{boundary} N={N} R={rate} B={B}")


@pytest.mark.parametrize("kernel,boundary,N,rate", [("tpf", "double-pass", 212, '1/3'), ("quad", "double-pass", 212, '1/3'),
                                                    ("lat", "double-pass", 212, '1/3'), ("auto", "nii", 212, '1/3'),
                                                    ("auto", "nii16", 212, '1/3'), ("quad", "double-pass", 752, '1/2')])
def test_f16_row_pitch_and_alignment_paths(kernel, boundary, N, rate):
    """The decoder is handed each layout as it is (pointer and row stride through the C ABI, no compacting copy):
    row pitches n_llr, n_llr + 3, n_llr + 4 (16-byte rows for float32, not for float16: n_llr is a multiple of 8 here)
    and n_llr + 8 (16-byte rows with padding), each with the rows starting 0 / 1 / 2 / 4 / 8 elements into the
    allocation (float16 bases 16-, 2-, 4-, 8- and 16-byte aligned).  This runs the bulk-copy and the per-element
    transpositions of tpf / nii and the __half2 and scalar loads of quad.  Every layout gives the oracle's decisions
    and exactly what the float32 path gives on the same layout of the widened values."""
    import torch
    g, o = _codec(N, rate, kernel, boundary)
    B = 70
    info, h = _frames16(g, o, rate, B, 1.5, 4242 + N)
    ref = o.decode_batch(h.astype(np.float32), threads=os.cpu_count() or 1)
    n = h.shape[1]
    assert n % 8 == 0
    src = torch.from_numpy(h).cuda()
    for pitch in (n, n + 3, n + 4, n + 8):
        for off in (0, 1, 2, 4, 8):
            outs = []
            for dt in (torch.float16, torch.float32):
                buf = torch.zeros(B * pitch + off, dtype=dt, device="cuda")
                assert buf.data_ptr() % 256 == 0
                x = buf.as_strided((B, n), (pitch, 1), off)
                x.copy_(src.to(dt))
                assert x.data_ptr() == buf.data_ptr() + off * buf.element_size() and x.stride(0) == pitch
                outs.append(_decode_as_laid_out(g, x, info))
            _assert_outputs(g, outs[0], outs[1], info, ref, f"{kernel}/{boundary} pitch n+{pitch - n}, offset {off}")
    # numpy float16 input reaches the same path (the device gets the 16-bit values)
    assert np.array_equal(g.decode_batch(h), ref)


@pytest.mark.parametrize("N,rate", [(212, '1/3'), (752, '1/2'), (212, '3/4')])
def test_f16_host_pipeline_all_layouts(N, rate):
    """decode_batch_host with a pinned float16 buffer of more frames than one chunk, for out = bits / packed / uint8,
    read on the host right after the call; equal to the float32 pipeline on the widened buffer and to the oracle."""
    import torch
    from modulations_b200 import dvb_rcs2_turbo as turbo
    g, o = _codec(N, rate)
    nfr = 50
    info, h = _frames16(g, o, rate, nfr, 1.0, 77 + N)
    ref = o.decode_batch(h.astype(np.float32), threads=os.cpu_count() or 1)
    reps = g.handle.frames_per_wave // nfr + 3                     # more frames than one chunk (one wave)
    x16 = torch.from_numpy(np.tile(h, (reps, 1))).pin_memory()
    x32 = x16.float().pin_memory()
    want = np.tile(ref, (reps, 1))
    for out in ("bits", "packed", "uint8"):
        got16 = g.decode_batch_host(x16, out=out).numpy().copy()
        got32 = g.decode_batch_host(x32, out=out).numpy().copy()
        assert np.array_equal(got16, got32), out
        dec = turbo.unpack_bits(got16, g.k_info) if out == "packed" else got16.astype(np.int32)
        assert np.array_equal(dec, want), out
    with pytest.raises(IndexError):
        g.decode_batch_host(x16.double())


@pytest.mark.parametrize("kernel,N,rate,B", [("tpf", 212, '1/3', 100_000), ("quad", 752, '1/2', 100_000)])
def test_f16_randomised_large_batch_vs_oracle(kernel, N, rate, B):
    """10^5 DISTINCT device-generated frames (Philox source, Eb/N0 2 dB), rounded to float16, against the C oracle on
    every host thread; a second decode over the same workspace changes nothing."""
    import torch
    from modulations_b200 import dvb_rcs2_turbo as turbo
    g, o = _codec(N, rate, kernel)
    h = g.handle
    info = torch.empty((B, g.k_info), dtype=torch.uint8, device="cuda")
    coded = torch.empty((B, h.n_llr), dtype=torch.uint8, device="cuda")
    llr = torch.empty((B, h.n_llr), dtype=torch.float32, device="cuda")
    h.mc_generate_bpsk(B, 1.0 / (2.0 * (g.k_info / h.n_llr) * 10 ** 0.2), 2026 + N, 0, info, coded, llr)
    x16 = llr.half()
    got = turbo.unpack_bits(g.decode_batch(x16, out="packed").cpu(), g.k_info)
    ref = o.decode_batch(x16.float().cpu().numpy(), threads=os.cpu_count() or 1)
    bad = np.flatnonzero(np.any(got != ref, axis=1))
    assert bad.size == 0, f"{bad.size} of {B} frames differ (first: {bad[:8]})"
    again = turbo.unpack_bits(g.decode_batch(x16, out="packed").cpu(), g.k_info)
    assert np.array_equal(again, got)


def test_f16_rounding_costs_nothing_measurable():
    """The cost of the format: the same 2^17 frames at 2 / 5 / 8 dB with the bijective interleaver, decoded as float32
    LLRs and as their float16 rounding.  BER and FER must each lie inside the 99 % binomial interval (normal
    approximation, 2.576 sigma of the pooled estimate) of the other's, as in test_nii_ber_inside_parity_confidence_interval,
    with no allowance."""
    import torch
    from modulations_b200 import dvb_rcs2_turbo as turbo
    N, rate, B = 212, '1/3', 1 << 17
    g = turbo.DVBRCS2_Turbo(N, rate, 8, perm=turbo.bijective_interleaver(N))
    h = g.handle
    info = torch.empty((B, g.k_info), dtype=torch.uint8, device="cuda")
    coded = torch.empty((B, h.n_llr), dtype=torch.uint8, device="cuda")
    llr = torch.empty((B, h.n_llr), dtype=torch.float32, device="cuda")
    for ebn0 in (2.0, 5.0, 8.0):
        h.mc_generate_bpsk(B, 1.0 / (2.0 * (1 / 3) * 10 ** (ebn0 / 10)), 7 + int(ebn0), 0, info, coded, llr)
        c0 = torch.zeros(4, dtype=torch.int64, device="cuda")
        c1 = torch.zeros(4, dtype=torch.int64, device="cuda")
        g.decode_batch(llr, ref_bits=info, counters=c0, out="none")
        g.decode_batch(llr.half(), ref_bits=info, counters=c1, out="none")
        c0, c1 = c0.cpu().numpy().astype(float), c1.cpu().numpy().astype(float)
        assert c0[2] == B and c1[2] == B
        for what, e0, e1, n in (("BER", c0[0], c1[0], c0[3]), ("FER", c0[1], c1[1], c0[2])):
            p = (e0 + e1) / (2 * n)
            half = 2.576 * np.sqrt(max(p * (1 - p), 1e-12) * 2 / n)
            assert abs(e0 / n - e1 / n) <= half + 1e-12, (ebn0, what, e0 / n, e1 / n, half)


def test_decode_f16_argument_errors():
    import torch
    from modulations_b200 import _lib
    g, _ = _codec(212, '1/3', "tpf")                              # checks its workspace size (a 32-frame batch would go to lat)
    h = g.handle
    lib = _lib.load()
    B, n = 32, h.n_llr
    x = torch.zeros((B, n + 1), dtype=torch.float16, device="cuda")
    bits = torch.empty((B, g.k_info), dtype=torch.int32, device="cuda")
    need = int(lib.b200dvb_decode_workspace_bytes(h.h, B))
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(ptr, stride, nbytes):
        return lib.b200dvb_decode_f16(h.h, B, ptr, stride, _lib.ptr(bits), None, None, None, _lib.ptr(ws), nbytes, st)

    assert call(None, n, need) == _lib.EINVAL                      # NULL llr
    assert call(_lib.ptr(x), n - 1, need) == _lib.EINVAL           # row stride shorter than n_llr
    assert call(_lib.ptr(x), n, need - 1) == _lib.ENOMEM           # workspace too small
    assert call(ctypes.c_void_p(x.data_ptr() + 1), n, need) == _lib.EINVAL   # not 2-byte aligned
    assert call(_lib.ptr(x), n, need) == _lib.OK
    torch.cuda.synchronize()
