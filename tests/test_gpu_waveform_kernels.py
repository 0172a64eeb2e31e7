"""GPU: every pulse-shaping and matched-filter kernel instance of waveform.cu, called through the C ABI
(b200dvb_pulse_shape / b200dvb_matched_filter) on torch CUDA tensors, against a float64 reference.

Exact arithmetic: inputs with integer parts |x| <= 8 and dyadic taps k/4, |k| <= 16, make every product and partial
sum a multiple of 1/4 (1/16 for the matched filter of a pulse-shaped signal) far below 2^24 of those units, so the
float32 kernels must equal the float64 reference in any summation order.  A wrong index, a dropped tap, a stale or
missing staged sample, a tile or tail error shows as an inequality, not as a tolerance question.  Random Gaussian
data is checked against a derived bound, (K + 1) * 2^-24 * sum_t |h_t| |x_{m,t}| per output and component, K the length
of the output's FMA chain (the + 1 is the rounding of the taps to float32).

The dispatch (waveform.cu: launch_pulse_shape / launch_matched_filter) picks among 25 instances; INSTANCES names one
call per instance, and test_every_instance_runs checks with torch.profiler that they all run."""
import re

import numpy as np
import pytest

gpu = pytest.mark.gpu
EINVAL = -1
MAX_TAPS = 448
LENGTHS = (1, 2, 3, 4, 6, 7, 9, 10, 15, 16, 255, 256, 257, 511, 512, 513)   # symbols: QT - 1 and QT, tile edges
MF_LENGTHS = (1, 2, 3, 5, 255, 256, 257, 511, 512, 513)                     # outputs: tile edges
SPS_ALL = (1, 2, 3, 4, 5, 6, 8, 12, 16, 32, 34, 48, 49, 50, 64)
Q_EDGES = (1, 4, 5, 7, 8, 10, 11, 16, 17)       # taps per phase on both sides of the QT (4/7/10/16) and QW buckets


# ---- float64 reference ----------------------------------------------------------------------------------------------
def _conv(a, h, quarter=False):
    """np.convolve(a, h) for real a, h.  quarter=True states that the exact result is a multiple of 1/4 (integer
    samples, dyadic taps): long inputs then go through an FFT and are rounded back onto that grid, which is exact
    while the FFT's error stays below 1/8."""
    if len(a) == 0 or len(h) == 0:
        return np.zeros(max(len(a) + len(h) - 1, 0))
    if quarter and len(a) * len(h) > 20_000_000:
        from scipy.signal import fftconvolve
        return np.round(fftconvolve(a, h) * 4) / 4
    return np.convolve(a, h)


def ps_ref(sym, h, sps, absolute=False, quarter=False):
    """out[i] = sum_k sym[k] h[i - k sps], i < (n-1) sps + ntaps (scipy.signal.upfirdn(h, sym, up=sps)), per component
    in float64 (a complex product would turn Inf * 0 in the other component into NaN).  Polyphase: phase p of the
    output is sym convolved with h[p::sps].  absolute=True gives sum_k |sym[k]| |h[i - k sps]| instead."""
    sym, h = np.asarray(sym), np.asarray(h, np.float64)
    n, nt = len(sym), len(h)
    out = np.zeros((n - 1) * sps + nt, np.complex128)
    f = np.abs if absolute else (lambda v: v)
    for p in range(min(sps, nt)):
        hp = f(h[p::sps])
        out.real[p::sps] = _conv(f(sym.real.astype(np.float64)), hp, quarter)
        out.imag[p::sps] = _conv(f(sym.imag.astype(np.float64)), hp, quarter)
    return out


def mf_ref(x, h, sps, start, n_out, absolute=False, quarter=False):
    """out[m] = sum_t h[t] x[start + m sps - t], x = 0 outside [0, n): convolve(x, h, 'full')[start::sps], zero past
    the end; per component in float64.  absolute=True gives the sums of |h| |x| instead."""
    x, h = np.asarray(x), np.asarray(h, np.float64)
    out = np.zeros(n_out, np.complex128)
    idx = start + sps * np.arange(n_out, dtype=np.int64)
    f = np.abs if absolute else (lambda v: v)
    for part, src in ((out.real, x.real), (out.imag, x.imag)):
        full = _conv(f(src.astype(np.float64)), f(h), quarter)
        ok = idx < len(full)
        part[ok] = full[idx[ok]]
    return out


def dyadic_taps(rs, ntaps):
    return rs.randint(-16, 17, ntaps) / 4.0


def int_samples(rs, n):
    return (rs.randint(-8, 9, n) + 1j * rs.randint(-8, 9, n)).astype(np.complex64)


def mf_start(ntaps, sps, residue):
    """the smallest start >= ntaps - 1 with (start - ntaps + 1) mod sps = residue (Modulator uses residue 0)"""
    return ntaps - 1 + residue % sps


def mf_len(n_out, ntaps, sps, start):
    """the input length whose full convolution from `start` on has exactly n_out decimated outputs"""
    return max(0, start - ntaps + 2 + (n_out - 1) * sps)


def tap_counts(sps):
    """ntaps with ceil(ntaps / sps) on both sides of every bucket edge (full last row and a single tap in it), plus a
    count below sps (phases, and pair rows, without taps), 1 and 448."""
    out = {1, MAX_TAPS, max(1, sps // 2), max(1, sps - 1)}
    for q in Q_EDGES:
        for nt in (q * sps, (q - 1) * sps + 1):
            if 1 <= nt <= MAX_TAPS:
                out.add(nt)
    return sorted(out)


def test_reference_matches_the_oracle():
    """the references above are the oracle's upfirdn / convolve (no GPU needed)"""
    from oracle import oracle
    rs = np.random.RandomState(3)
    for sps, nt, n in ((8, 49, 37), (5, 3, 11), (2, 1, 1), (64, 385, 9), (3, 2, 5)):
        x = (rs.randn(n) + 1j * rs.randn(n)).astype(np.complex64)
        h = rs.randn(nt)
        assert np.allclose(ps_ref(x, h, sps), oracle.pulse_shape(x, h, sps), rtol=0, atol=1e-12)
        want = oracle.matched_filter(x, h, sps)
        got = mf_ref(x, h, sps, 2 * ((nt - 1) // 2), len(want))
        assert np.allclose(got, want, rtol=0, atol=1e-12)
        assert np.allclose(mf_ref(x, h, sps, 2 * ((nt - 1) // 2), len(want), absolute=True),
                           mf_ref(np.abs(x.real) + 1j * np.abs(x.imag), np.abs(h), sps, 2 * ((nt - 1) // 2), len(want)))


# ---- calls through the C ABI ----------------------------------------------------------------------------------------
GUARD = complex(1234.5, -4321.25)


def _lib():
    from modulations_b200 import _lib
    return _lib, _lib.load()


def _device(a, off):
    """complex64 CUDA copy of `a` starting `off` elements past a 512-byte aligned allocation"""
    import torch
    buf = torch.empty(len(a) + off + 1, dtype=torch.complex64, device="cuda")
    assert buf.data_ptr() % 512 == 0
    v = buf[off:off + len(a)]
    if len(a):
        v.copy_(torch.from_numpy(np.ascontiguousarray(a, np.complex64)))
    return v


def _out(n, off):
    """an output view `off` elements past a 32-byte boundary (element 4 of a 512-byte aligned allocation), with guard
    elements on both sides that must survive the call"""
    import torch
    buf = torch.full((n + off + 5,), GUARD, dtype=torch.complex64, device="cuda")
    return buf, buf[off + 4:off + 4 + n]


def _result(buf, n, off):
    import torch
    torch.cuda.synchronize()
    b = buf.cpu().numpy()
    assert np.all(b[:off + 4] == np.complex64(GUARD)) and np.all(b[off + 4 + n:] == np.complex64(GUARD)), \
        "wrote outside the output"
    return b[off + 4:off + 4 + n]


def pulse_shape(sym, h, sps, in_off=0, out_off=0):
    """b200dvb_pulse_shape; input and output `in_off` / `out_off` elements past an aligned address"""
    _l, lib = _lib()
    s = _device(sym, in_off)
    n_out = (len(sym) - 1) * sps + len(h)
    buf, o = _out(n_out, out_off)
    taps = np.ascontiguousarray(h, np.float64)
    _l.check(lib.b200dvb_pulse_shape(len(sym), _l.ptr(s), _l.host_ptr(taps), len(h), sps, _l.ptr(o), _l.stream_ptr()),
             "pulse_shape")
    return _result(buf, n_out, out_off)


def matched_filter(x, h, sps, start, n_out, in_off=0, out_off=0):
    _l, lib = _lib()
    xd = _device(x, in_off)
    buf, o = _out(n_out, out_off)
    taps = np.ascontiguousarray(h, np.float64)
    _l.check(lib.b200dvb_matched_filter(len(x), _l.ptr(xd), _l.host_ptr(taps), len(h), sps, start, n_out, _l.ptr(o),
                                        _l.stream_ptr()), "matched_filter")
    return _result(buf, n_out, out_off)


class mf_variant:
    """B200DVB_DBG_MF_VARIANT for the duration of a with-block, back to 0 (the default) whatever happens"""
    def __init__(self, v):
        self.v = v

    def __enter__(self):
        _l, lib = _lib()
        _l.check(lib.b200dvb_debug_set_option(1, self.v), "debug_set_option")

    def __exit__(self, *exc):
        _l, lib = _lib()
        _l.check(lib.b200dvb_debug_set_option(1, 0), "debug_set_option")


def assert_exact(got, want, what):
    bad = np.flatnonzero(got.astype(np.complex128) != want)
    assert bad.size == 0, f"{what}: {bad.size} of {len(want)} outputs differ, first at {bad[:5]}: " \
                          f"{got[bad[:3]]} vs {want[bad[:3]]}"


# ---- one call per instance: (instance, kind, sps, ntaps, residue, variant) ---------------------------------------------
# Aligned buffers.  Residue = (start - ntaps + 1) mod sps for the matched filter; variant = B200DVB_DBG_MF_VARIANT.
INSTANCES = (
    [(f"pulse_shape_sps_kernel<{s},{q}>", "ps", s, (q - 1) * s + 1, 0, 0) for s in (2, 4, 8) for q in (4, 7, 10, 16)]
    + [("pulse_shape_kernel", "ps", 5, 15, 0, 0)]
    + [(f"matched_filter4_kernel<{qw},{'true' if a else 'false'}>", "mf", 8, nt, r, int(a))
       for qw, nt, r in ((4, 25, 0), (6, 41, 0), (7, 49, 0), (8, 57, 0), (9, 64, 1)) for a in (False, True)]
    + [("matched_filter_kernel<2>", "mf", 5, 15, 0, 0), ("matched_filter_kernel<1>", "mf", 64, 385, 0, 0)]
)
ALL_INSTANCES = sorted({i[0] for i in INSTANCES})


def _kernel_names(prof):
    names = set()
    for e in prof.events():
        m = re.search(r"(pulse_shape_sps_kernel|pulse_shape_kernel|matched_filter4_kernel|matched_filter_kernel)"
                      r"(<[^>]*>)?", e.name.replace(" ", "").replace("(int)", ""))
        if m:
            names.add(m.group(0).replace("(bool)0", "false").replace("(bool)1", "true"))
    return names


@gpu
def test_every_instance_runs():
    """The dispatch reaches all 25 kernel instances, each from the call INSTANCES lists for it (torch.profiler's CUDA
    activity names the kernels that ran)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    assert len(ALL_INSTANCES) == 25
    rs = np.random.RandomState(1)
    for name, kind, sps, nt, r, var in INSTANCES:
        h = dyadic_taps(rs, nt)
        with mf_variant(var):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                if kind == "ps":
                    pulse_shape(int_samples(rs, 40), h, sps)
                else:
                    st = mf_start(nt, sps, r)
                    matched_filter(int_samples(rs, mf_len(600, nt, sps, st)), h, sps, st, 600)
                torch.cuda.synchronize()
        assert _kernel_names(prof) == {name}, (name, _kernel_names(prof))


# ---- exact arithmetic over the geometry grid --------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("sps", SPS_ALL)
def test_pulse_shape_exact(sps):
    """Every tap count of tap_counts(sps) and every length of LENGTHS, 32-byte aligned output (the per-period kernels
    for sps 2/4/8 up to 16 taps per phase, the generic kernel otherwise)."""
    rs = np.random.RandomState(100 + sps)
    for nt in tap_counts(sps):
        h = dyadic_taps(rs, nt)
        for n in LENGTHS:
            x = int_samples(rs, n)
            assert_exact(pulse_shape(x, h, sps), ps_ref(x, h, sps), f"sps {sps} ntaps {nt} n {n}")


@gpu
@pytest.mark.parametrize("sps", SPS_ALL)
def test_matched_filter_exact(sps):
    """Every tap count of tap_counts(sps) at residues 0, 1 and sps - 1, outputs on both sides of the 256 / 512-output
    tiles, and the three kernel variants."""
    rs = np.random.RandomState(200 + sps)
    for nt in tap_counts(sps):
        h = dyadic_taps(rs, nt)
        for r in sorted({0, 1 % sps, sps - 1}):
            st = mf_start(nt, sps, r)
            for n_out in MF_LENGTHS:
                x = int_samples(rs, mf_len(n_out, nt, sps, st))
                want = mf_ref(x, h, sps, st, n_out)
                for var in ((0, 1, 2) if n_out in (1, 257, 513) else (0,)):
                    with mf_variant(var):
                        got = matched_filter(x, h, sps, st, n_out)
                    assert_exact(got, want, f"sps {sps} ntaps {nt} residue {r} n_out {n_out} variant {var}")


@gpu
@pytest.mark.parametrize("sps", (2, 3, 6, 8, 12, 16, 50))
def test_matched_filter_every_residue(sps):
    """start - ntaps + 1 in every residue class mod sps: each moves the first output's staged origin, the pair-row
    tables and (for mf4) which QW instance runs."""
    rs = np.random.RandomState(300 + sps)
    for nt in sorted({2 * sps - 1, 4 * sps + 1, min(8 * sps, MAX_TAPS), 3}):
        h = dyadic_taps(rs, nt)
        for r in range(sps):
            st = mf_start(nt, sps, r) + sps * (r % 3)           # also starts a whole symbol or two later
            for n_out in (1, 257, 513):
                x = int_samples(rs, mf_len(n_out, nt, sps, st) + r % 2)
                assert_exact(matched_filter(x, h, sps, st, n_out), mf_ref(x, h, sps, st, n_out),
                             f"sps {sps} ntaps {nt} residue {r} start {st} n_out {n_out}")


@gpu
@pytest.mark.parametrize("sps,nt", [(8, 49), (8, 64), (5, 15), (6, 37), (64, 385), (2, 3), (32, 448)])
def test_matched_filter_start_and_length_edges(sps, nt):
    """start past the end (all zeros), n_out past the end of the full convolution (zero tail), an empty input with
    n_out > 0, and start = 0 (outputs before the filter has filled)."""
    rs = np.random.RandomState(sps * 1000 + nt)
    h = dyadic_taps(rs, nt)
    x = int_samples(rs, 3000)
    for var in (0, 1, 2):
        with mf_variant(var):
            for st, n_out in ((len(x) + nt - 1, 40), (len(x) + nt + 700, 600), (nt - 1, 700), (0, 517),
                              (5, (len(x) + nt) // sps + 300)):
                assert_exact(matched_filter(x, h, sps, st, n_out), mf_ref(x, h, sps, st, n_out),
                             f"start {st} n_out {n_out} variant {var}")
            _l, lib = _lib()                                        # n = 0 (a valid pointer: NULL is EINVAL)
            xd = _device(x[:1], 0)
            buf, o = _out(300, 1)
            _l.check(lib.b200dvb_matched_filter(0, _l.ptr(xd), _l.host_ptr(np.ascontiguousarray(h)), nt, sps, nt - 1,
                                                300, _l.ptr(o), _l.stream_ptr()), "matched_filter")
            assert np.all(_result(buf, 300, 1) == 0), f"empty input, variant {var}"


@gpu
@pytest.mark.parametrize("kind,sps,nt", [("ps", 8, 49), ("ps", 2, 7), ("ps", 4, 64), ("ps", 3, 10),
                                         ("mf", 8, 49), ("mf", 6, 25), ("mf", 5, 12), ("mf", 64, 100)])
def test_one_hot_taps(kind, sps, nt):
    """h = e_t: the output is a shifted copy of the input, which pins each tap position on its own (the expected
    output is built by indexing, not by a convolution)."""
    rs = np.random.RandomState(nt)
    x = int_samples(rs, 700)
    for t in sorted({0, 1, nt // 2, nt - 2, nt - 1} & set(range(nt))):
        h = np.zeros(nt)
        h[t] = 1.0
        if kind == "ps":
            want = np.zeros((len(x) - 1) * sps + nt, np.complex128)
            want[t + sps * np.arange(len(x))] = x
            assert_exact(pulse_shape(x, h, sps), want, f"tap {t}")
        else:
            for r in (0, sps - 1):
                st = mf_start(nt, sps, r)
                n_out = (len(x) + nt - 1 - st + sps - 1) // sps
                idx = st + sps * np.arange(n_out) - t
                want = np.where((idx >= 0) & (idx < len(x)), x[np.clip(idx, 0, len(x) - 1)], 0).astype(np.complex128)
                for var in (0, 1, 2):
                    with mf_variant(var):
                        assert_exact(matched_filter(x, h, sps, st, n_out), want, f"tap {t} residue {r} variant {var}")


@gpu
@pytest.mark.parametrize("off", (1, 2, 3))
def test_unaligned_buffers(off):
    """Input and output views 1, 2, 3 complex64 elements past an aligned allocation: the generic pulse-shaping
    kernel (output not 32-byte aligned), the matched filters' element-wise staging (input not 16-byte aligned) and
    scalar stores (output not 32-byte aligned)."""
    rs = np.random.RandomState(off)
    for sps, nt in ((2, 7), (4, 33), (8, 49), (8, 120)):
        h = dyadic_taps(rs, nt)
        for n in (1, 5, 257, 513):
            x = int_samples(rs, n)
            assert_exact(pulse_shape(x, h, sps, in_off=off, out_off=off), ps_ref(x, h, sps), f"ps sps {sps} n {n}")
    for sps, nt in ((8, 49), (8, 64), (6, 37), (2, 15), (5, 15), (16, 100), (64, 385), (8, 100)):
        h = dyadic_taps(rs, nt)
        for r in (0, 1):
            st = mf_start(nt, sps, r)
            for n_out in (1, 257, 513, 1100):
                x = int_samples(rs, mf_len(n_out, nt, sps, st))
                want = mf_ref(x, h, sps, st, n_out)
                for var in (0, 1, 2):
                    with mf_variant(var):
                        for io, oo in ((off, 0), (0, off), (off, off)):
                            assert_exact(matched_filter(x, h, sps, st, n_out, in_off=io, out_off=oo), want,
                                         f"mf sps {sps} ntaps {nt} n_out {n_out} variant {var} offsets {io}/{oo}")


@gpu
@pytest.mark.parametrize("inst", INSTANCES, ids=[i[0] for i in INSTANCES])
def test_every_block_runs_several_tiles(inst):
    """A length past the grid cap of the instance's launch (16, 6, 3 and 8 blocks per SM for pulse shaping, mf4, mf4
    with cp.async and the generic matched filter), so every persistent block loops at least twice and the cp.async
    double buffer is swapped; the matched-filter case runs under all three kernel variants."""
    import torch
    name, kind, sps, nt, r, var = inst
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rs = np.random.RandomState(7)
    if kind == "ps":
        per_block = 256 * (sps if "sps_kernel" in name else 1)        # output samples a block covers per tile
        n = (sms * 16 * per_block * 5 // 4) // sps + 1
        h = dyadic_taps(rs, nt)
        x = int_samples(rs, n)
        assert_exact(pulse_shape(x, h, sps), ps_ref(x, h, sps, quarter=True), name)
        return
    tile = 512 if sps <= 48 else 256
    n_out = sms * 8 * tile * 5 // 4 + 77                            # past all three caps
    nt = min(nt, 2 * sps + 1) if sps > 32 else nt                   # a cheap reference; the instance stays the same
    h = dyadic_taps(rs, nt)
    st = mf_start(nt, sps, r)
    x = int_samples(rs, mf_len(n_out, nt, sps, st) + 5)
    want = mf_ref(x, h, sps, st, n_out, quarter=True)
    for v in (0, 1, 2):
        with mf_variant(v):
            assert_exact(matched_filter(x, h, sps, st, n_out), want, f"{name}, variant {v}")


# ---- float data against the derived bound -------------------------------------------------------------------------------
def float_case(inst, seed):
    """Gaussian input and random (not float32-representable) taps, or the RRC taps of the instance's geometry"""
    from modulations_b200.modulators import rrcosfilter
    name, kind, sps, nt, r, var = inst
    rs = np.random.RandomState(seed)
    h = rs.randn(nt) if seed % 2 else rrcosfilter(-(-nt // sps), 0.35, 1, sps)[:nt]
    n = 1500 if kind == "ps" else mf_len(1500, len(h), sps, mf_start(len(h), sps, r))
    x = (rs.randn(n) + 1j * rs.randn(n)).astype(np.complex64) * np.float32(rs.choice([1e-3, 1.0, 1e3]))
    return h, x


def float_error_ratio(inst, h, x):
    """largest |kernel - float64| / ((K + 1) 2^-24 sum |h| |x|) over outputs and components"""
    name, kind, sps, nt, r, var = inst
    nt = len(h)
    if kind == "ps":
        got = pulse_shape(x, h, sps)
        want, s = ps_ref(x, h, sps), ps_ref(x, h, sps, absolute=True)
        k = -(-nt // sps)
    else:
        st = mf_start(nt, sps, r)
        n_out = (len(x) + nt - 1 - st + sps - 1) // sps
        with mf_variant(var):
            got = matched_filter(x, h, sps, st, n_out)
        want, s = mf_ref(x, h, sps, st, n_out), mf_ref(x, h, sps, st, n_out, absolute=True)
        k = nt
    worst = 0.0
    for g, w, b in ((got.real, want.real, s.real), (got.imag, want.imag, s.imag)):
        bound = (k + 1) * 2.0 ** -24 * b
        err = np.abs(g.astype(np.float64) - w)
        assert np.all(err <= bound), f"{name}: error {err.max():.3e} over the bound at {np.argmax(err - bound)}"
        worst = max(worst, float(np.max(np.where(bound > 0, err / np.where(bound > 0, bound, 1), 0))))
    return worst


@gpu
@pytest.mark.parametrize("inst", INSTANCES, ids=[i[0] for i in INSTANCES])
def test_float_error_within_derived_bound(inst):
    """tools/waveform_err.py prints the largest ratio per instance (profiles/r03_waveform_observed_error.txt)"""
    for seed in range(4):
        h, x = float_case(inst, seed)
        float_error_ratio(inst, h, x)


# ---- non-finite samples -----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("inst", INSTANCES, ids=[i[0] for i in INSTANCES])
def test_non_finite_samples_stay_in_their_window(inst):
    """An Inf and a NaN at chosen samples: every output whose window excludes them equals the reference (finite);
    those that include them are Inf or NaN exactly where the reference is.  Padded taps must not take part: 0 x Inf
    is NaN."""
    name, kind, sps, nt, r, var = inst
    rs = np.random.RandomState(11)
    h = dyadic_taps(rs, nt)
    h[h == 0] = 0.25                                                # every real tap touches its sample
    n = 900 if kind == "ps" else mf_len(300, nt, sps, mf_start(nt, sps, r))
    for a, b in ((n // 3, n // 3 + 1), (0, n - 1), (n // 2, n // 2 + 3 * sps + 1)):
        x = int_samples(rs, n)
        x.real[a] = np.inf
        x.imag[a] = -np.inf
        x.real[b] = np.nan
        if kind == "ps":
            got, want = pulse_shape(x, h, sps), ps_ref(x, h, sps)
        else:
            st = mf_start(nt, sps, r)
            n_out = (n + nt - 1 - st + sps - 1) // sps
            with mf_variant(var):
                got = matched_filter(x, h, sps, st, n_out)
            want = mf_ref(x, h, sps, st, n_out)
        assert np.isfinite(want).sum() > 0
        for part in ("real", "imag"):
            np.testing.assert_array_equal(getattr(got, part), getattr(want, part), err_msg=f"{name}, {part}, {a} {b}")


# ---- sizes past 2^31 elements --------------------------------------------------------------------------------------------
@gpu
def test_sizes_past_2_31():
    """Pulse shaping with more than 2^31 output samples (the per-period kernel, then the generic one on a shifted
    output), then the matched filter over those samples (more than 2^31 inputs) under all three variants.  Windows
    around the 2^31-byte, 2^32-byte, 2^33-byte and 2^31-element crossings and the tails equal the reference."""
    import torch
    if torch.cuda.mem_get_info()[0] < 40 * 2 ** 30:
        pytest.skip("needs about 40 GiB of free device memory")
    _l, lib = _lib()
    sps, nt = 8, 49
    h = dyadic_taps(np.random.RandomState(31), nt)
    taps = np.ascontiguousarray(h, np.float64)
    n_sym = (1 << 28) + 4099
    n_sh = (n_sym - 1) * sps + nt
    assert n_sh > 1 << 31
    g = torch.Generator(device="cuda").manual_seed(31)
    sym = torch.randint(-8, 9, (n_sym, 2), generator=g, device="cuda", dtype=torch.float32).view(torch.complex64)
    sym = sym.reshape(-1)
    buf = torch.empty(n_sh + 1, dtype=torch.complex64, device="cuda")
    crossings = [1 << 28, 1 << 29, 1 << 30, 1 << 31]

    def ps_windows(out, shift):
        for c in crossings + [n_sh - 300]:
            lo, hi = max(0, c - 700), min(n_sh, c + 700)
            k0, k1 = max(0, (lo - nt + 1) // sps), min(n_sym, hi // sps + 1)
            s = sym[k0:k1].cpu().numpy()
            want = ps_ref(s, h, sps)[lo - k0 * sps:hi - k0 * sps]
            assert_exact(out[lo + shift:hi + shift].cpu().numpy(), want, f"pulse shaping, window at {c}, shift {shift}")

    for shift in (1, 0):                                            # generic kernel first: the aligned result stays
        _l.check(lib.b200dvb_pulse_shape(n_sym, _l.ptr(sym), _l.host_ptr(taps), nt, sps, _l.ptr(buf[shift:]),
                                         _l.stream_ptr()), "pulse_shape")
        torch.cuda.synchronize()
        ps_windows(buf, shift)
    x = buf[:n_sh]
    st = nt - 1
    n_out = (n_sh + nt - 1 - st + sps - 1) // sps
    out = torch.empty(n_out, dtype=torch.complex64, device="cuda")
    for var in (0, 1, 2):
        out.fill_(complex(float("nan"), 0))
        with mf_variant(var):
            _l.check(lib.b200dvb_matched_filter(n_sh, _l.ptr(x), _l.host_ptr(taps), nt, sps, st, n_out, _l.ptr(out),
                                                _l.stream_ptr()), "matched_filter")
            torch.cuda.synchronize()
        for c in [c // sps for c in crossings] + [(1 << 31) // sps, n_out - 200]:
            lo, hi = max(0, c - 300), min(n_out, c + 300)
            s0, s1 = max(0, st + lo * sps - nt + 1), min(n_sh, st + (hi - 1) * sps + 1)
            want = mf_ref(x[s0:s1].cpu().numpy(), h, sps, st + lo * sps - s0, hi - lo)
            assert_exact(out[lo:hi].cpu().numpy(), want, f"matched filter, window at {c}, variant {var}")
    del sym, buf, out
    torch.cuda.empty_cache()


# ---- argument errors --------------------------------------------------------------------------------------------------
@gpu
def test_argument_errors_change_nothing():
    """EINVAL before any launch, output untouched: sps 0 or 65, ntaps 0 or 449, start < 0, NULL pointers."""
    import torch
    _l, lib = _lib()
    x = _device(int_samples(np.random.RandomState(5), 64), 0)
    taps = np.ascontiguousarray(np.full(MAX_TAPS + 1, 0.25), np.float64)
    tp = _l.host_ptr(taps)
    out = torch.full((2000,), GUARD, dtype=torch.complex64, device="cuda")
    o, xs, st = _l.ptr(out), _l.ptr(x), _l.stream_ptr()
    ps = [(64, xs, tp, 9, 0, o), (64, xs, tp, 9, 65, o), (64, xs, tp, 0, 8, o), (64, xs, tp, MAX_TAPS + 1, 8, o),
          (64, None, tp, 9, 8, o), (64, xs, None, 9, 8, o), (64, xs, tp, 9, 8, None)]
    for n, s, t, nt, sps, oo in ps:
        assert lib.b200dvb_pulse_shape(n, s, t, nt, sps, oo, st) == EINVAL, (nt, sps)
    mf = [(64, xs, tp, 9, 0, 8, 10, o), (64, xs, tp, 9, 65, 8, 10, o), (64, xs, tp, 0, 8, 8, 10, o),
          (64, xs, tp, MAX_TAPS + 1, 8, 8, 10, o), (64, xs, tp, 9, 8, -1, 10, o), (64, None, tp, 9, 8, 8, 10, o),
          (64, xs, None, 9, 8, 8, 10, o), (64, xs, tp, 9, 8, 8, 10, None)]
    for n, s, t, nt, sps, start, n_out, oo in mf:
        assert lib.b200dvb_matched_filter(n, s, t, nt, sps, start, n_out, oo, st) == EINVAL, (nt, sps, start)
    torch.cuda.synchronize()
    assert torch.all(out == GUARD)


@gpu
@pytest.mark.parametrize("sps,span", [(64, 6), (50, 8), (49, 9), (49, 7)])
def test_modulator_takes_every_sps(sps, span):
    """Modulator geometries past the 512-output tile's shared memory (sps >= 50, or sps 49 with more than 343 taps)
    filter like the oracle."""
    from modulations_b200.modulators import Modulator
    from oracle import oracle
    mo = Modulator(samples_per_symbol=sps, rrc_span=span)
    rs = np.random.RandomState(sps)
    syms = (rs.randn(1000) + 1j * rs.randn(1000)).astype(np.complex64)
    shaped = mo.apply_pulse_shaping(syms)
    tol = 2e-6 * np.sum(np.abs(mo.rrc_filter)) * np.max(np.abs(syms))
    assert np.max(np.abs(shaped - oracle.pulse_shape(syms, mo.rrc_filter, sps))) <= tol
    got = mo.matched_filter(shaped.astype(np.complex64))
    want = oracle.matched_filter(shaped.astype(np.complex64), mo.rrc_filter, sps)
    assert got.shape == want.shape
    assert np.max(np.abs(got - want)) <= 2e-6 * np.sum(np.abs(mo.rrc_filter)) * np.max(np.abs(shaped))
