"""GPU tests of the Rayleigh fading channel (b200dvb_fading_complex) and the soft demapper with channel state
(b200dvb_demap_csi): against the float64 oracle, against b200dvb_demap and b200dvb_awgn_complex where they must agree
bit for bit, the statistics of the gains, uncoded BER against the closed form, and the Monte-Carlo sweep."""
import numpy as np
import pytest

from oracle import oracle
from tests import csi_oracle, vectors

pytestmark = pytest.mark.gpu

# the float32 tolerance of the AWGN demapper (tests/test_gpu_modem.py), applied per symbol as LLR_ATOL * max(1, |h|^2):
# the LLR is |h|^2 / noise_var times a difference of distances to the equalised symbol
LLR_ATOL = {'BPSK': 9e-5, 'QPSK': 1e-5, '8PSK': 3.2e-5, '16QAM': 2.7e-5, '64QAM': 2.2e-5, '256QAM': 2.4e-5}
NATURAL = ['BPSK', 'QPSK', '8PSK', '16QAM', '64QAM']


def _lib():
    from modulations_b200 import _lib as L
    return L


def channel_case(rs, table, n, nv):
    """n received symbols y = h c + noise: c uniform over the table, |h| log-uniform in [1e-20, 1e3] with a uniform
    phase, 1 % of the gains exactly 0."""
    c = np.asarray(table).astype(np.complex128)[rs.randint(0, len(table), n)]
    h = 10 ** rs.uniform(-20, 3, n) * np.exp(2j * np.pi * rs.rand(n))
    h[rs.rand(n) < 0.01] = 0
    y = h * c + np.sqrt(nv / 2) * (rs.randn(n) + 1j * rs.randn(n))
    return y.astype(np.complex64), h.astype(np.complex64)


def csi_error(name, table, y, h, nv):
    """-> (GPU LLRs, oracle LLRs, per-LLR bound) for complex64 y, h."""
    from modulations_b200.soft_demod import compute_llr
    bps = vectors.BPS[name]
    got = compute_llr(y, name, nv, constellation=table, gain=h)
    want = csi_oracle.compute_llr_csi(y, h, name, nv, constellation=table)
    bound = np.repeat(LLR_ATOL[name] * np.maximum(1.0, np.abs(h.astype(np.complex128)) ** 2), bps)
    return got, want, bound


def _tables():
    from modulations_b200.modulators import natural_constellation
    from modulations_b200.sdr_modem import gray_constellation
    return ([(n, 'gray', gray_constellation(n)) for n in vectors.BPS]
            + [(n, 'natural', natural_constellation(n)) for n in NATURAL])


@pytest.mark.parametrize("name,kind", [(n, k) for n, k, _ in _tables()])
def test_csi_demap_vs_oracle(name, kind):
    """Random y and h (|h| from 1e-20 to 1e3, and 0) against the complex128 oracle: within LLR_ATOL * max(1, |h|^2)
    per LLR, the same hard decisions wherever the oracle's LLR is outside that bound, finite everywhere, 0 for h = 0."""
    table = dict(((n, k), t) for n, k, t in _tables())[(name, kind)]
    rs = np.random.RandomState(vectors.BPS[name] * 10 + (kind == 'natural'))
    for nv in vectors.DEMAP_NOISE_VARS + [0.0001]:
        y, h = channel_case(rs, table, 100_003, nv)
        got, want, bound = csi_error(name, table, y, h, nv)
        assert got.dtype == np.float64 and got.shape == want.shape and np.all(np.isfinite(got))
        err = np.abs(got - want)
        worst = np.argmax(err / bound)
        assert np.all(err <= bound), (name, kind, nv, "max |dLLR| / bound = %.3f at |h| = %.3e"
                                      % (err[worst] / bound[worst], abs(h[worst // vectors.BPS[name]])))
        bad = (got > 0) != (want > 0)
        assert np.all(np.abs(want[bad]) <= bound[bad])
        assert np.all(got.reshape(len(y), -1)[h == 0] == 0)


@pytest.mark.parametrize("name", list(vectors.BPS))
def test_csi_demap_extreme_inputs_are_finite(name):
    """Every finite y and h with |y|, |h| <= 1e6 gives a finite LLR within +-30 (no Inf * 0 in deep fades)."""
    from modulations_b200.soft_demod import compute_llr
    rs = np.random.RandomState(3)
    n = 20_000
    mag = lambda: np.concatenate([10 ** rs.uniform(-45, 6, n - 4), [0, 1e6, 1e-45, 1e-38]])
    y = (mag() * np.exp(2j * np.pi * rs.rand(n))).astype(np.complex64)
    h = (mag() * np.exp(2j * np.pi * rs.rand(n))).astype(np.complex64)
    got = compute_llr(y, name, 0.05, gain=h)
    assert np.all(np.isfinite(got)) and np.all(np.abs(got) <= 30)
    assert np.all(got.reshape(n, -1)[h == 0] == 0)


def _both_paths(name):
    """(label, ModemHandle) for the kernel paths a table can take: the Gray table (piecewise-linear for the square
    orders, generic for BPSK / 8PSK) and, for the square orders, the same table rotated by 1e-9 rad, which is not
    separable any more and takes the generic kernel (as in tests/test_gpu_modem.py)."""
    from modulations_b200.sdr_modem import ModemHandle, gray_constellation
    t = gray_constellation(name)
    out = [("gray", ModemHandle(name, t))]
    if name not in ('BPSK', '8PSK'):
        out.append(("generic", ModemHandle(name, t.astype(np.complex128) * np.exp(1j * 1e-9))))
    return out


@pytest.mark.parametrize("name", list(vectors.BPS))
def test_csi_demap_with_unit_gain_equals_demap(name):
    """h = 1 reproduces b200dvb_demap value for value, on every kernel path and length, and inside a mixed array
    the symbols whose gain is 1 get exactly b200dvb_demap's LLRs."""
    import torch
    bps = vectors.BPS[name]
    rs = np.random.RandomState(11 + bps)
    for label, m in _both_paths(name):
        for n in (1, 2, 3, 5, 31, 1000, 4097, 100_003):
            tx = oracle.modulate(rs.randint(0, 2, bps * n), name)
            y = (tx + 0.3 * (rs.randn(n) + 1j * rs.randn(n))).astype(np.complex64)
            for nv, scale in ((0.05, 1.0), (0.0001, -1.0), (0.5, 0.37)):
                ref = m.llr(y, nv, scale)
                assert np.array_equal(m.llr(y, nv, scale, gain=np.ones(n, np.complex64)), ref), (label, n, nv)
                h = (rs.randn(n) + 1j * rs.randn(n)).astype(np.complex64)
                one = rs.rand(n) < 0.5
                h[one] = 1
                got = m.llr(y, nv, scale, gain=h).reshape(n, bps)
                assert np.array_equal(got[one], ref.reshape(n, bps)[one]), (label, n, nv)
        # device tensors in and out
        yt = torch.from_numpy(y).cuda()
        out = m.llr(yt, 0.05, gain=torch.ones(n, dtype=torch.complex64, device="cuda"))
        assert out.dtype == torch.float32 and out.is_cuda and torch.equal(out, m.llr(yt, 0.05))


def test_csi_demap_argument_errors():
    import torch
    from modulations_b200.sdr_modem import gray_modem
    from modulations_b200.soft_demod import compute_llr, decoder_llr
    L = _lib()
    lib = L.load()
    m = gray_modem('16QAM')
    y = torch.zeros(64, dtype=torch.complex64, device="cuda")
    g = torch.ones(65, dtype=torch.complex64, device="cuda")
    out = torch.empty(64 * 4, dtype=torch.float32, device="cuda")
    assert lib.b200dvb_demap_csi(m.h, 64, L.ptr(y), None, 0.1, 1.0, L.ptr(out), None) == L.EINVAL
    assert lib.b200dvb_demap_csi(m.h, 64, None, L.ptr(g), 0.1, 1.0, L.ptr(out), None) == L.EINVAL
    assert lib.b200dvb_demap_csi(m.h, 64, L.ptr(y), L.ptr(g), 0.1, 1.0, None, None) == L.EINVAL
    assert lib.b200dvb_demap_csi(None, 64, L.ptr(y), L.ptr(g), 0.1, 1.0, L.ptr(out), None) == L.EINVAL
    assert lib.b200dvb_demap_csi(m.h, 64, L.ptr(y), L.ptr(g[1:]), 0.1, 1.0, L.ptr(out), None) == L.EINVAL  # 8 B
    assert lib.b200dvb_demap_csi(m.h, 0, L.ptr(y), L.ptr(g), 0.1, 1.0, L.ptr(out), None) == L.OK
    with pytest.raises(ValueError):
        m.llr(y, 0.1, gain=g)
    with pytest.raises(ValueError):
        compute_llr(np.zeros(4, np.complex64), 'QPSK', 0.1, gain=np.ones(3, np.complex64))
    rs = np.random.RandomState(1)
    yy, hh = channel_case(rs, oracle.sdr_constellation('QPSK'), 1001, 0.05)
    assert np.array_equal(decoder_llr(yy, 'QPSK', 0.05, gain=hh), -compute_llr(yy, 'QPSK', 0.05, gain=hh).astype(np.float32))


# ---- channel ---------------------------------------------------------------------------------------------------
def fading(n, block_len, sigma, seed, offset, iq=None, want_gain=True):
    import torch
    from modulations_b200 import montecarlo as mc
    iq = torch.zeros(n, dtype=torch.complex64, device="cuda") if iq is None else iq
    g = torch.empty(n, dtype=torch.complex64, device="cuda") if want_gain else None
    mc.fading_channel(iq, sigma, seed, offset, block_len, gain=g)
    return iq, g


def _bits(t):
    import torch
    return torch.view_as_real(t).contiguous().view(torch.int32)


@pytest.mark.parametrize("block_len", [1, 2, 7, 64])
def test_fading_noise_is_awgn_complex(block_len):
    """With iq all zeros the output is b200dvb_awgn_complex's, bit for bit, for any block length and offset."""
    import torch
    L = _lib()
    lib = L.load()
    for n, sigma, seed, offset in ((1, 0.3, 5, 0), (1001, 0.7, 9, 6), (1 << 20, 0.05, 123456789, 1 << 33)):
        a = torch.zeros(n, dtype=torch.complex64, device="cuda")
        L.check(lib.b200dvb_awgn_complex(n, sigma, seed, offset, L.ptr(a), L.stream_ptr()), "awgn")
        b, _ = fading(n, block_len, sigma, seed, offset)
        c, _ = fading(n, block_len, sigma, seed, offset, want_gain=False)
        assert torch.equal(_bits(a), _bits(b)) and torch.equal(_bits(a), _bits(c))


def test_fading_gain_statistics():
    """Fast fading: |h|^2 ~ Exp(1) (Kolmogorov-Smirnov), the mean of h within 5 standard errors of 0 and E|h|^2 within
    5 standard errors of 1 (sd of h's components sqrt(1/2), of |h|^2 1), adjacent gains uncorrelated
    (|mean(h_b conj(h_b+1))| within 5 / sqrt(n)), and the signal multiplied by exactly the reported gain."""
    import torch
    from scipy import stats
    n = 1 << 22
    x = torch.complex(torch.randn(n, device="cuda"), torch.randn(n, device="cuda"))
    y, g = fading(n, 1, 0.0, 77, 0, iq=x.clone())
    h = g.cpu().numpy().astype(np.complex128)
    p2 = np.abs(h) ** 2
    assert stats.kstest(p2, 'expon').pvalue > 1e-3
    se = np.sqrt(0.5 / n)
    assert abs(h.real.mean()) < 5 * se and abs(h.imag.mean()) < 5 * se
    assert abs(p2.mean() - 1) < 5 / np.sqrt(n)
    assert abs(np.mean(h[1:] * np.conj(h[:-1]))) < 5 / np.sqrt(n)
    xn, yn, gn = x.cpu().numpy(), y.cpu().numpy(), g.cpu().numpy()
    re, im = gn.real * xn.real - gn.imag * xn.imag, gn.real * xn.imag + gn.imag * xn.real    # float32 arithmetic
    assert np.array_equal(yn.real, re) and np.array_equal(yn.imag, im)


@pytest.mark.parametrize("block_len,offset", [(7, 0), (7, 6), (64, 1000), (3, 1 << 34)])
def test_fading_blocks(block_len, offset):
    """h is constant inside each block of block_len symbols, counted from the global index offset + i, and the
    gains of adjacent blocks are uncorrelated; the block gains are Exp(1) in power."""
    from scipy import stats
    n = 1 << 21
    _, g = fading(n, block_len, 0.1, 4242, offset)
    h = g.cpu().numpy().astype(np.complex128)
    b = (offset + np.arange(n)) // block_len
    first = np.r_[True, b[1:] != b[:-1]]
    hb = h[first]
    assert np.array_equal(h, np.repeat(hb, np.diff(np.r_[np.flatnonzero(first), n])))
    assert len(np.unique(hb)) == len(hb)
    inner = hb[1:-1]                                     # whole blocks only
    assert abs(np.mean(inner[1:] * np.conj(inner[:-1]))) < 5 / np.sqrt(len(inner))
    assert stats.kstest(np.abs(inner) ** 2, 'expon').pvalue > 1e-3


@pytest.mark.parametrize("block_len", [1, 5, 64])
def test_fading_split_calls_equal_one_call(block_len):
    """Two calls at offsets 0 and k draw exactly what one call draws (gains and noise keyed by the global index)."""
    import torch
    rs = np.random.RandomState(block_len)
    n = 100_001
    x = torch.from_numpy((rs.randn(n) + 1j * rs.randn(n)).astype(np.complex64)).cuda()
    whole, gw = fading(n, block_len, 0.4, 31, 0, iq=x.clone())
    for k in (2, 64, 50_000, 100_000):
        part = x.clone()
        gp = torch.empty(n, dtype=torch.complex64, device="cuda")
        from modulations_b200 import montecarlo as mc
        mc.fading_channel(part[:k], 0.4, 31, 0, block_len, gain=gp[:k])
        mc.fading_channel(part[k:], 0.4, 31, k, block_len, gain=gp[k:])
        assert torch.equal(_bits(part), _bits(whole)) and torch.equal(_bits(gp), _bits(gw))


def test_fading_argument_errors():
    import torch
    from modulations_b200 import montecarlo as mc
    L = _lib()
    lib = L.load()
    x = torch.ones(16, dtype=torch.complex64, device="cuda")
    g = torch.empty(16, dtype=torch.complex64, device="cuda")
    f = lib.b200dvb_fading_complex
    assert f(16, 1, 0.1, 1, 0, None, L.ptr(g), None) == L.EINVAL
    assert f(16, 1, -0.1, 1, 0, L.ptr(x), L.ptr(g), None) == L.EINVAL
    assert f(16, 1, float("nan"), 1, 0, L.ptr(x), L.ptr(g), None) == L.EINVAL
    assert f(16, 0, 0.1, 1, 0, L.ptr(x), L.ptr(g), None) == L.EINVAL
    assert f(16, -3, 0.1, 1, 0, L.ptr(x), L.ptr(g), None) == L.EINVAL
    assert f(16, 1, 0.1, 1, 7, L.ptr(x), L.ptr(g), None) == L.EINVAL
    assert f(0, 1, 0.1, 1, 0, L.ptr(x), L.ptr(g), None) == L.OK
    torch.cuda.synchronize()
    assert torch.equal(x, torch.ones_like(x))
    with pytest.raises(ValueError):
        mc.fading_channel(x, 0.1, 1, 0, gain=g[:8])
    with pytest.raises(ValueError):
        mc.fading_channel(x, 0.1, 1, 1)


# ---- end to end ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ['BPSK', 'QPSK'])
@pytest.mark.parametrize("coherence", [1, 64])
def test_uncoded_ber_matches_rayleigh_closed_form(name, coherence):
    """map -> fading + AWGN -> CSI demap -> sign over Rayleigh fading: the BER is 1/2 (1 - sqrt(g / (1 + g))) with
    g = Eb/N0, for any coherence length.  This pins the noise normalisation, the gain statistics and the CSI
    weighting together.  Bits that share a gain are not independent, so the 99 % interval is the binomial one over
    the independent fading blocks (bps * coherence bits each; a block's error fraction lies in [0, 1], so its variance
    is at most p (1 - p)): exact for BPSK with coherence 1, conservative otherwise."""
    import torch
    from modulations_b200.sdr_modem import gray_modem
    bps = vectors.BPS[name]
    nbits = 1 << 25
    m = gray_modem(name)
    gen = torch.Generator(device="cuda").manual_seed(2024 + coherence)
    gain = torch.empty(nbits // bps, dtype=torch.complex64, device="cuda")
    for pi, ebn0_db in enumerate((0.0, 5.0, 10.0, 15.0)):
        g = 10 ** (ebn0_db / 10)
        nv = 1.0 / (2 * bps * g)                                    # per real dimension, unit-energy symbols
        bits = torch.randint(0, 2, (nbits,), dtype=torch.uint8, device="cuda", generator=gen)
        syms = m.map(bits)
        from modulations_b200 import montecarlo as mc
        mc.fading_channel(syms, float(np.sqrt(nv)), 99 + pi, 0, coherence, gain=gain)
        llr = m.llr(syms, 2 * nv, gain=gain)
        errors = int(((llr > 0).to(torch.uint8) != bits).sum())
        p = 0.5 * (1 - np.sqrt(g / (1 + g)))
        n_eff = nbits // (bps * coherence)
        half = 2.5758 * np.sqrt(p * (1 - p) / n_eff)
        assert abs(errors / nbits - p) <= half, (name, coherence, ebn0_db, errors / nbits, p, half)


@pytest.mark.parametrize("mod", ["BPSK", "16QAM"])
@pytest.mark.parametrize("coherence", [1, 7])
def test_rayleigh_sweep_independent_of_batching(mod, coherence):
    """test_sweep_independent_of_batching for channel="rayleigh": the counters depend only on (seed, global frame
    index), also when fading blocks straddle frames (coherence 7), and two half-shards sum to the whole run."""
    from modulations_b200 import montecarlo as mc
    kw = dict(N=48, rate='1/2', iterations=4, ebn0_db=[1.0, 6.0], frames_per_point=4096, seed=5, modulation=mod,
              channel="rayleigh", coherence=coherence)
    a = mc.run_sweep(mc.SweepConfig(batch=4096, **kw))
    b = mc.run_sweep(mc.SweepConfig(batch=1024, **kw))
    assert a["points"] == b["points"]
    halves = [mc.run_sweep(mc.SweepConfig(batch=2048, **kw), rank=r, world=2) for r in range(2)]
    for p, (x, y) in zip(a["points"], zip(halves[0]["points"], halves[1]["points"])):
        for key in ("bit_errors", "frame_errors", "frames", "bits"):
            assert p[key] == x[key] + y[key]
    assert a["points"][0]["frames"] == 4096 and a["points"][0]["bits"] == 4096 * 96
