"""GPU tests of the soft output (b200dvb_decode_app, decode_batch / decode_batch_host with out="app").  The contract:
app[f][2k] / app[f][2k+1] is the a-posteriori LLR of bit A / B of couple k after the last iteration, the value whose
sign the hard decision takes.  Parity mode: float32 of the oracle's float64 Lfinal; "nii": the model's float32 sum;
"nii16": the model's 1/4-unit sum times 0.25; all bit for bit (compared as int32 views, so signed zeros count).  The
hard outputs of the same call (bits, packed words, counters) are exactly those of b200dvb_decode / _f16 / _i8.
The reference values come from what oracle/ already exports: orc_decode's nullable Lfinal for parity, and for the
non-parity modes the models' decode loop driven through their exported SISOs (nii_siso, nii16_siso_ext), whose
decisions must equal the models' own."""
import ctypes
import os

import numpy as np
import pytest

from oracle import oracle

pytestmark = pytest.mark.gpu

RATE = {'1/3': 1 / 3, '1/2': 1 / 2, '2/3': 2 / 3, '3/4': 3 / 4}
MODELS = {"double-pass": oracle.OracleTurbo, "nii": oracle.NiiModel, "nii16": oracle.Nii16Model}
THREADS = os.cpu_count() or 1
FMT = {"float32": 0, "float16": 1, "int8": 2}              # B200DVB_LLR_F32 / _F16 / _I8


def _codec(N, rate, kernel="auto", boundary="double-pass"):
    from modulations_b200 import dvb_rcs2_turbo as turbo
    iters = 8 if N <= 212 else 4
    g = turbo.DVBRCS2_Turbo(N, rate, iters, kernel=kernel, boundary=boundary)
    g.handle                                              # ValueError where N has no geometry for the kernel
    return g, MODELS[boundary](N, rate, iters, perm=g.perm, inv_perm=g.inv_perm)


def _awgn(g, o, rate, B, ebn0, seed):
    """info bits uint8 [B, 2N] and float32 BPSK/AWGN LLRs clipped to +-50 [B, n_llr] (rate 2/3: zero-padded tail)."""
    rs = np.random.RandomState(seed)
    info = rs.randint(0, 2, (B, g.k_info))
    coded = np.asarray(o.encode_batch(info)).astype(np.float64)
    nv = 1.0 / (2.0 * RATE[rate] * 10 ** (ebn0 / 10))
    llr = np.clip(2.0 * ((1.0 - 2.0 * coded) + np.sqrt(nv) * rs.randn(*coded.shape)) / nv, -50, 50)
    if llr.shape[1] < g.n_llr:
        llr = np.pad(llr, ((0, 0), (0, g.n_llr - llr.shape[1])))
    return info.astype(np.uint8), llr.astype(np.float32)


def _vp(a):
    return ctypes.c_void_p(a.ctypes.data)


def _tables(m):
    """int32 pointers the oracle's C functions take: next_st, out_W, out_Y, prev_st, prev_inp, perm, inv_perm"""
    return [_vp(np.ascontiguousarray(t, np.int32))
            for t in (m.next_state, m.out_W, m.out_Y, m.prev_state, m.prev_input, m.perm, m.inv_perm)], \
           [np.ascontiguousarray(t, np.int32) for t in (m.next_state, m.out_W, m.out_Y, m.prev_state, m.prev_input)]


def _chunks(B, f):
    """f(lo, hi) over B frames split across the host threads (ctypes drops the GIL inside the C calls)"""
    from concurrent.futures import ThreadPoolExecutor
    cuts = np.linspace(0, B, min(THREADS, B) + 1).astype(int)
    with ThreadPoolExecutor(len(cuts) - 1) as ex:
        list(ex.map(lambda i: f(int(cuts[i]), int(cuts[i + 1])), range(len(cuts) - 1)))


def _parity_ref(o, x):
    """(decisions, float32(Lfinal) [B, 2N] interleaved A, B per couple): orc_decode of every frame, whose nullable
    Lfinal output is the float64 sum (Lc + La) + Le1 of the hard decision (oracle/turbo_oracle.c)"""
    x = np.ascontiguousarray(x, np.float32)
    B, n = x.shape
    N = o.N
    dec = np.zeros((B, 2 * N), np.int32)
    lf = np.zeros((B, 2, N), np.float64)
    ptrs, _keep = _tables(o)
    punct = np.ascontiguousarray(o.punct_u8, np.uint8)
    fn = oracle.lib().orc_decode

    def run(lo, hi):
        for b in range(lo, hi):
            rc = fn(N, o.iterations, *ptrs, _vp(punct), o.period, _vp(x[b]), n, _vp(dec[b]), None, _vp(lf[b]))
            assert rc == 0
    _chunks(B, run)
    app = np.empty((B, 2 * N), np.float32)
    app[:, 0::2], app[:, 1::2] = lf[:, 0], lf[:, 1]
    return dec, app


def _nonparity_ref(m, x, fixed):
    """(decisions, float32 [B, 2N]) of the nii model (fixed=False) or the nii16 model (fixed=True) on float32 x: the
    decode loop of nii_decode / nii16_decode (depuncture, `iterations` x (SISO 1, interleave, SISO 2, de-interleave))
    driven through the models' exported SISOs nii_siso / nii16_siso_ext, ending in the sum (Lc + La) + Le1 whose sign
    they decide on: float32 for nii, integer 1/4-LLR units times 0.25 for nii16.  The caller checks the decisions
    against the model's own decode_batch, which pins this loop to the model."""
    x = np.ascontiguousarray(x, np.float32)
    B = x.shape[0]
    N, per = m.N, m.period
    dt = np.int32 if fixed else np.float32
    if fixed:                                                # nii16_model.c quant(): rint(4 x) clamped to +-127
        x = np.clip(np.rint(x * np.float32(4)), -127, 127).astype(np.int32)
    off, idx = np.full((6, N), -1, np.int64), 0              # A, B, W1, Y1, W2, Y2 positions in a row
    for i in range(N):
        off[0, i], off[1, i] = idx, idx + 1
        idx += 2
        for j in range(4):
            if m.punct_u8[j, i % per]:
                off[2 + j, i] = idx
                idx += 1
    chan = np.where(off[None] >= 0, x[:, np.maximum(off, 0)], 0).astype(dt)     # [B, 6, N]
    perm, inv = np.asarray(m.perm), np.asarray(m.inv_perm)
    ptrs, _keep = _tables(m)
    tab = ptrs[:5]
    lib = oracle.lib()
    dec = np.zeros((B, 2 * N), np.int32)
    app = np.zeros((B, 2 * N), np.float32)

    def run(lo, hi):
        scratch = np.zeros(N * 64 + 2 * (N + 1) * 16, dt)
        for b in range(lo, hi):
            A, Bb, W1, Y1, W2, Y2 = (np.ascontiguousarray(c) for c in chan[b])
            Ai, Bi = A[perm].copy(), Bb[perm].copy()
            La_A, La_B = np.zeros(N, dt), np.zeros(N, dt)
            st = np.zeros((4, 16), dt)
            Le1_A, Le1_B, Le2_A, Le2_B = (np.zeros(N, dt) for _ in range(4))
            for it in range(m.iterations):
                last = it == m.iterations - 1
                for k, (lA, lB, lW, lY, aA, aB, eA, eB) in enumerate((
                        (A, Bb, W1, Y1, La_A, La_B, Le1_A, Le1_B), (Ai, Bi, W2, Y2, None, None, Le2_A, Le2_B))):
                    if k == 1:
                        aA, aB = Le1_A[perm].copy(), Le1_B[perm].copy()
                    a0, b0 = st[2 * k], st[2 * k + 1]
                    if fixed:
                        rc = lib.nii16_siso_ext(*(_vp(v) for v in (lA, lB, lW, lY, aA, aB)), *tab, ctypes.c_int(N),
                                                ctypes.c_int(64 if last else 45), _vp(a0), _vp(b0), _vp(eA), _vp(eB),
                                                _vp(scratch))
                        assert rc == 0, "a 16-bit quantity of the nii16 format overflowed"
                    else:
                        lib.nii_siso(*(_vp(v) for v in (lA, lB, lW, lY, aA, aB)), *tab, ctypes.c_int(N),
                                     ctypes.c_float(1.0 if last else 0.7), _vp(a0), _vp(b0), _vp(eA), _vp(eB),
                                     _vp(scratch))
                La_A, La_B = Le2_A[inv].copy(), Le2_B[inv].copy()
            LA, LB = (A + La_A) + Le1_A, (Bb + La_B) + Le1_B
            dec[b, 0::2], dec[b, 1::2] = LA < 0, LB < 0
            if fixed:
                app[b, 0::2], app[b, 1::2] = np.float32(0.25) * LA.astype(np.float32), np.float32(0.25) * LB.astype(np.float32)
            else:
                app[b, 0::2], app[b, 1::2] = LA, LB
    _chunks(B, run)
    return dec, app


def _ref_app(m, x):
    """(decisions, float32 a-posteriori LLRs [B, 2N]) of the oracle / model on float32 x; the decisions are checked
    against the oracle's / model's own batch decode"""
    x = np.ascontiguousarray(x, np.float32)
    if isinstance(m, oracle.Nii16Model):
        dec, app = _nonparity_ref(m, x, True)
    elif isinstance(m, oracle.NiiModel):
        dec, app = _nonparity_ref(m, x, False)
    else:
        dec, app = _parity_ref(m, x)
    assert np.array_equal(dec, m.decode_batch(x, threads=THREADS)), "reference soft values disagree with the model"
    return dec, app


def _call(g, fn, x, info, ptr=None, stride=None, scale=1.0, app=True):
    """ONE call of b200dvb_decode_app (fn="app") or of the hard-only entry of x's dtype (fn="hard") on the CUDA tensor
    x, as laid out (its own data pointer and row stride unless given), with every output and error counting against
    info -> (app or None, bits, packed, counters) as numpy."""
    import torch
    from modulations_b200 import _lib
    h = g.handle
    lib = _lib.load()
    B = x.shape[0]
    fmt = str(x.dtype).removeprefix("torch.")
    ptr = ctypes.c_void_p(x.data_ptr()) if ptr is None else ptr
    stride = (x.stride(0) if B > 1 else x.shape[1]) if stride is None else stride
    a = torch.full((B, g.k_info), float("nan"), dtype=torch.float32, device="cuda")
    bits = torch.empty((B, g.k_info), dtype=torch.int32, device="cuda")
    packed = torch.empty((B, (g.k_info + 31) // 32), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    ref = torch.from_numpy(info).cuda()
    ws, need = h.workspace("decode", B)
    outs = (_lib.ptr(bits), _lib.ptr(packed), _lib.ptr(ref), _lib.ptr(cnt), _lib.ptr(ws), need,
            ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    if fn == "app":
        rc = lib.b200dvb_decode_app(h.h, B, ptr, FMT[fmt], scale, stride, _lib.ptr(a), *outs)
    elif fmt == "int8":
        rc = lib.b200dvb_decode_i8(h.h, B, ptr, stride, scale, *outs)
    else:
        rc = getattr(lib, "b200dvb_decode_f16" if fmt == "float16" else "b200dvb_decode")(h.h, B, ptr, stride, *outs)
    _lib.check(rc, fn)
    return (a.cpu().numpy() if fn == "app" else None), bits.cpu().numpy(), packed.cpu().numpy(), cnt.cpu().numpy()


def _same_app(got, want, what):
    bad = np.flatnonzero(np.any(got.view(np.int32) != want.view(np.int32), axis=1))
    assert bad.size == 0, f"{what}: app differs in {bad.size} of {len(got)} frames (first frame {bad[0]}: " \
                          f"{got[bad[0]][got[bad[0]].view(np.int32) != want[bad[0]].view(np.int32)][:4]} against " \
                          f"{want[bad[0]][got[bad[0]].view(np.int32) != want[bad[0]].view(np.int32)][:4]})"


def _check(g, x, info, dec, app, what, scale=1.0, ptr=None, stride=None, rows=None):
    """b200dvb_decode_app on x: app == `app`, bits == the oracle's `dec` (for the frames `rows` only when given: dec
    and app then hold those frames); bits / packed / counters == the hard-only entry's on the same input and
    workspace, for every frame."""
    from modulations_b200 import dvb_rcs2_turbo as turbo
    a, b, p, c = _call(g, "app", x, info, ptr, stride, scale)
    _, b0, p0, c0 = _call(g, "hard", x, info, ptr, stride, scale)
    sel = slice(None) if rows is None else rows
    _same_app(a[sel], app, what)
    assert np.array_equal(b[sel], dec), f"{what}: {np.sum(b[sel] != dec)} bits differ from the oracle"
    assert np.array_equal(b, b0) and np.array_equal(p, p0), f"{what}: hard outputs differ from the hard-only entry"
    assert np.array_equal(turbo.unpack_bits(p, g.k_info), b), f"{what}: packed words"
    assert np.array_equal(c, c0), f"{what}: counters {c} != {c0}"
    assert c[0] == np.sum(b != info) and c[2] == len(b) and c[3] == len(b) * g.k_info


CONFIGS = [(48, '1/3'), (64, '1/2'), (212, '1/3'), (212, '3/4'), (64, '2/3'), (424, '1/2'), (752, '1/2'), (848, '1/3')]
KERNEL_CASES = [(k, N, r) for k in ("auto", "quad", "tpf", "lat") for N, r in CONFIGS
                if not (k == "tpf" and N > 212)]                 # the thread-per-frame kernel has no geometry beyond 212


@pytest.mark.parametrize("kernel,N,rate", KERNEL_CASES)
def test_app_every_kernel_equals_oracle_lfinal(kernel, N, rate):
    """B = 1 (low-latency kernel under "auto"), 17 (a partial tile) and one wave + 7 frames."""
    import torch
    g, o = _codec(N, rate, kernel)
    big = g.handle.frames_per_wave + 7
    info, x = _awgn(g, o, rate, big, 1.5, 31 * N + len(kernel))
    dec, app = _ref_app(o, x)
    xd = torch.from_numpy(x).cuda()
    for B in (1, 17, big):
        _check(g, xd[:B], info[:B], dec[:B], app[:B], f"{kernel} N={N} R={rate} B={B}")


@pytest.mark.parametrize("boundary", ["nii", "nii16"])
@pytest.mark.parametrize("N,rate", [(48, '1/3'), (212, '1/3'), (212, '3/4'), (64, '2/3')])
def test_app_nonparity_modes_equal_their_models(boundary, N, rate):
    """nii: the model's float32 sum; nii16: its sum in 1/4 units times 0.25 (every value a multiple of 0.25).  B = 1,
    17, 33 (partial tiles; nii16 keeps two frames per lane) against the model on every frame; one wave + 7 frames
    against it on the first and last 40 frames and every 97th (the reference restates the model's decode loop in
    Python around its C SISOs, which is too slow for every frame of a wave)."""
    import torch
    g, m = _codec(N, rate, boundary=boundary)
    big = g.handle.frames_per_wave + 7
    info, x = _awgn(g, m, rate, big, 1.5, 11 * N + len(boundary))
    rows = np.unique(np.concatenate([np.arange(40), np.arange(0, big, 97), np.arange(big - 40, big)]))
    dec, app = _ref_app(m, x[rows])
    if boundary == "nii16":
        assert np.array_equal(app * 4, np.rint(app * 4)) and np.abs(app).max() <= 637 / 4
    xd = torch.from_numpy(x).cuda()
    for B in (1, 17, 33):
        _check(g, xd[:B], info[:B], dec[:B], app[:B], f"{boundary} N={N} R={rate} B={B}")
    _check(g, xd, info, dec, app, f"{boundary} N={N} R={rate} B={big}", rows=rows)


@pytest.mark.parametrize("kernel,boundary,N,rate", [("tpf", "double-pass", 212, '1/3'), ("quad", "double-pass", 212, '1/3'),
                                                    ("lat", "double-pass", 212, '1/3'), ("auto", "double-pass", 64, '2/3'),
                                                    ("quad", "double-pass", 752, '1/2'), ("auto", "nii", 212, '1/3'),
                                                    ("auto", "nii16", 212, '3/4')])
def test_app_narrow_inputs_equal_their_float32_widening(kernel, boundary, N, rate):
    """fp16 input and int8 input with scales 0.25 and -0.6 give the app (and the hard outputs) of decoding their
    float32 widening, which equals the oracle's on that widening."""
    import torch
    g, o = _codec(N, rate, kernel, boundary)
    B = 150
    info, x = _awgn(g, o, rate, B, 1.5, 5 * N + len(kernel))
    x16 = x.astype(np.float16)
    q = np.clip(np.rint(2.5 * x), -128, 127).astype(np.int8)
    for what, xn, s, wide in (("fp16", x16, 1.0, x16.astype(np.float32)),
                              ("int8 x 0.25", q, 0.25, q.astype(np.float32) * np.float32(0.25)),
                              ("int8 x -0.6", q, -0.6, q.astype(np.float32) * np.float32(-0.6))):
        dec, app = _ref_app(o, wide)
        a32, *_ = _call(g, "app", torch.from_numpy(wide).cuda(), info)
        _same_app(a32, app, f"{what} widening")
        _check(g, torch.from_numpy(xn).cuda(), info, dec, app, f"{kernel}/{boundary} N={N} {what}", scale=s)


@pytest.mark.parametrize("kernel,boundary,N,rate", [("tpf", "double-pass", 212, '1/3'), ("quad", "double-pass", 212, '1/3'),
                                                    ("lat", "double-pass", 212, '1/3'), ("auto", "nii", 212, '1/3'),
                                                    ("auto", "nii16", 212, '1/3'), ("quad", "double-pass", 752, '1/2')])
def test_app_row_pitch_and_alignment(kernel, boundary, N, rate):
    """Each format handed to the C ABI as laid out (pointer and row stride, no compacting copy): row pitches n_llr,
    n_llr + 1, n_llr + 3 and n_llr + 16 elements, rows starting 0 / 1 / 3 / 16 elements into a 256-byte aligned
    allocation (fp16: misaligned to 4 and 16 bytes; int8: to 2, 4 and 16).  Every layout gives the app of the compact
    float32 widening."""
    import torch
    g, o = _codec(N, rate, kernel, boundary)
    B = 70
    info, x = _awgn(g, o, rate, B, 1.5, 4242 + N)
    n = x.shape[1]
    q = np.clip(np.rint(2.5 * x), -128, 127).astype(np.int8)
    for xn, s in ((x, 1.0), (x.astype(np.float16), 1.0), (q, 0.37)):
        wide = xn.astype(np.float32) * np.float32(s) if xn.dtype == np.int8 else xn.astype(np.float32)
        dec, app = _ref_app(o, wide)
        src = torch.from_numpy(xn).cuda()
        for pitch in (n, n + 1, n + 3, n + 16):
            for off in (0, 1, 3, 16):
                buf = torch.zeros(B * pitch + off, dtype=src.dtype, device="cuda")
                assert buf.data_ptr() % 256 == 0
                xs = buf.as_strided((B, n), (pitch, 1), off)
                xs.copy_(src)
                _check(g, xs, info, dec, app, f"{kernel}/{boundary} {src.dtype} pitch n+{pitch - n} offset {off}", scale=s)


@pytest.mark.parametrize("N,rate", [(212, '1/3'), (752, '1/2'), (64, '2/3')])
def test_app_decode_batch_and_host_pipeline(N, rate):
    """decode_batch(out="app") on numpy and on torch input, decode_batch_host(out="app") over more frames than one
    chunk: float32 [B, 2N] equal to each other and to the oracle's; ref_bits / counters still count with out="app"."""
    import torch
    g, o = _codec(N, rate)
    nfr = 50
    info, x = _awgn(g, o, rate, nfr, 1.0, 77 + N)
    dec, app = _ref_app(o, x)
    got_np = g.decode_batch(x, out="app")
    assert isinstance(got_np, np.ndarray) and got_np.dtype == np.float32 and got_np.shape == (nfr, g.k_info)
    _same_app(got_np, app, "decode_batch numpy")
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    got_t = g.decode_batch(torch.from_numpy(x).cuda(), out="app", ref_bits=info, counters=cnt)
    assert isinstance(got_t, torch.Tensor) and got_t.is_cuda and got_t.dtype == torch.float32
    _same_app(got_t.cpu().numpy(), app, "decode_batch torch")
    assert cnt.cpu().numpy().tolist() == [int(np.sum(dec != info)), int(np.sum(np.any(dec != info, axis=1))), nfr,
                                          nfr * g.k_info]
    reps = g.handle.frames_per_wave // nfr + 3                     # more frames than one chunk (one wave)
    xh = torch.from_numpy(np.tile(x, (reps, 1))).pin_memory()
    got_h = g.decode_batch_host(xh, out="app")
    assert got_h.is_pinned() and got_h.dtype == torch.float32 and tuple(got_h.shape) == (reps * nfr, g.k_info)
    _same_app(got_h.numpy(), np.tile(app, (reps, 1)), "decode_batch_host")
    assert np.array_equal(g.decode_batch_host(xh, out="bits").numpy(), np.tile(dec, (reps, 1)))
    _same_app(g.decode_batch_host(x, out="app").numpy(), app, "decode_batch_host numpy")
    x16 = torch.from_numpy(x.astype(np.float16)).pin_memory()
    _same_app(g.decode_batch_host(x16, out="app").numpy(), g.decode_batch(x16.cuda(), out="app").cpu().numpy(),
              "decode_batch_host fp16")
    with pytest.raises(ValueError, match='"app"'):
        g.decode_batch(x, out="soft")
    with pytest.raises(ValueError, match='"app"'):
        g.decode_batch_host(xh, out="soft")


@pytest.mark.parametrize("kernel,N,rate,B", [("tpf", 212, '1/3', 100_000), ("quad", 752, '1/2', 100_000)])
def test_app_randomised_large_batch_vs_oracle(kernel, N, rate, B):
    """10^5 DISTINCT device-generated frames (Philox source, Eb/N0 2 dB) against the oracle's Lfinal on every host
    thread."""
    import torch
    g, o = _codec(N, rate, kernel)
    h = g.handle
    info = torch.empty((B, g.k_info), dtype=torch.uint8, device="cuda")
    coded = torch.empty((B, h.n_llr), dtype=torch.uint8, device="cuda")
    llr = torch.empty((B, h.n_llr), dtype=torch.float32, device="cuda")
    h.mc_generate_bpsk(B, 1.0 / (2.0 * (g.k_info / h.n_llr) * 10 ** 0.2), 4049 + N, 0, info, coded, llr)
    got = g.decode_batch(llr, out="app").cpu().numpy()
    _, app = _ref_app(o, llr.cpu().numpy())
    _same_app(got, app, f"{kernel} N={N} B={B}")


def test_decode_app_argument_errors():
    import torch
    from modulations_b200 import _lib
    g, _ = _codec(212, '1/3', "tpf")
    h = g.handle
    lib = _lib.load()
    B, n = 32, h.n_llr
    x = torch.zeros((B, n + 1), dtype=torch.float32, device="cuda")
    x16 = torch.zeros((B, n + 1), dtype=torch.float16, device="cuda")
    x8 = torch.zeros((B, n + 1), dtype=torch.int8, device="cuda")
    app = torch.empty((B, g.k_info + 2), dtype=torch.float32, device="cuda")
    need = int(lib.b200dvb_decode_workspace_bytes(h.h, B))
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(ptr, fmt, stride, a=_lib.ptr(app), scale=0.25):
        return lib.b200dvb_decode_app(h.h, B, ptr, fmt, scale, stride, a, None, None, None, None, _lib.ptr(ws), need, st)

    assert call(_lib.ptr(x), 0, n, a=None) == _lib.EINVAL                                      # app is required
    assert call(_lib.ptr(x), 0, n, a=ctypes.c_void_p(app.data_ptr() + 4)) == _lib.EINVAL       # 4-byte aligned app
    for fmt in (-1, 3, 7):
        assert call(_lib.ptr(x), fmt, n) == _lib.EINVAL, fmt                                   # unknown format
    for bad in (0.0, -0.0, float("nan"), float("inf"), float("-inf")):
        assert call(_lib.ptr(x8), 2, n, scale=bad) == _lib.EINVAL, bad                         # int8 scale
    assert call(ctypes.c_void_p(x16.data_ptr() + 1), 1, n) == _lib.EINVAL                      # odd fp16 pointer
    for fmt, t in ((0, x), (1, x16), (2, x8)):
        assert call(_lib.ptr(t), fmt, n - 1) == _lib.EINVAL, fmt                               # short row stride
        assert call(None, fmt, n) == _lib.EINVAL, fmt                                          # NULL llr
    # the scale is ignored for float32 and fp16 (any value, NaN included); int8 takes any alignment
    assert call(_lib.ptr(x), 0, n, scale=float("nan")) == _lib.OK
    assert call(_lib.ptr(x16), 1, n, scale=0.0) == _lib.OK
    assert call(ctypes.c_void_p(x8.data_ptr() + 1), 2, n) == _lib.OK
    assert call(_lib.ptr(x), 0, n, a=ctypes.c_void_p(app.data_ptr() + 8)) == _lib.OK           # 8-byte aligned app
    torch.cuda.synchronize()
