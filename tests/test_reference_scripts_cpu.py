"""The reference's own scripts, UNMODIFIED, against the drop-in module (SURVEY 8(f) N3).

The reference's `d_test.py` and `turbo_test_suite.py` import `dvb_rcs2_turbo` (names `DVB_RCS2_TurboCodec`,
`bcjr_decode`) and walk the facade: `.encode/.decode`, `.interleaver.{perm,inv_perm,N,interleave}`,
`.encoder1/2.encode`, `.decoder1/2.decode`, `.k_info/.n_coded/.N/.code_rate`.  Here `sys.modules
['dvb_rcs2_turbo']` is pointed at `modulations_b200.dvb_rcs2_turbo` and the scripts' `main()` is run.

The scripts are not part of this repository: those two tests run when $REFERENCE_DIR (by default the same directory
as oracle/make_golden.py's) holds a checkout of the reference project and skip otherwise.  The calls the scripts make
on the drop-in are replayed by `test_facade_calls_of_the_scripts`, which runs everywhere.  No GPU is needed: the
tests exercise the HOST side of
the drop-in (names, argument handling, shapes, dtypes, the facade objects): the one class through which
the package reaches the device (`_CodecHandle`) is replaced by a stand-in that answers with the C oracle.
That stand-in lives here, in tests/; nothing under modulations_b200/ knows about it.  The device side of
the same calls is covered by the `-m gpu` tests (tests/test_gpu_codec.py::test_facade_and_circular_state).
"""
import builtins
import importlib.util
import os
import sys
import types

import numpy as np
import pytest

REF = os.environ.get("REFERENCE_DIR", "/root/reference")
needs_scripts = pytest.mark.skipif(not os.path.exists(os.path.join(REF, "d_test.py")),
                                   reason="the reference's scripts are not part of this repository: set $REFERENCE_DIR "
                                          "to a checkout of the reference project")


class _OracleHandle:
    """Stand-in for modulations_b200.dvb_rcs2_turbo._CodecHandle: same methods, computed by oracle/ on CPU tensors."""

    def __init__(self, N, next_state, out_W, out_Y, perm, inv_perm, punct_u8, period, iterations,
                 sf_inner=0.7, sf_last=1.0, kernel=None, mode=None):
        import torch
        from oracle import oracle
        rate = None
        pu = np.asarray(punct_u8, np.uint8)
        for r, p in oracle.PUNCTURE_PATTERNS.items():
            if p['period'] == period and np.array_equal(np.array([p[k] for k in ('W1', 'Y1', 'W2', 'Y2')], np.uint8), pu):
                rate = r
        assert rate is not None
        self.o = oracle.OracleTurbo(int(N), rate, int(iterations), perm=np.asarray(perm, np.int32),
                                    inv_perm=np.asarray(inv_perm, np.int32))
        self.device = torch.device("cpu")
        self.N, self.k_info, self.n_llr = int(N), 2 * int(N), self.o.n_emit
        self.frames_per_wave = 16
        self.h = None

    def set_option(self, option, value):
        pass

    def encode(self, info, want_circ=False):
        import torch
        x = info.numpy().astype(np.int32)
        coded = self.o.encode_batch(x).astype(np.uint8)
        circ = None
        if want_circ:
            circ = np.stack([self.o.encode(r, return_circ=True)[1] for r in x]).astype(np.uint8)
        return torch.from_numpy(coded), (torch.from_numpy(circ) if want_circ else None)

    def decode(self, x, bits=None, packed=None, ref=None, counters=None, stream=None, ws=None):
        import torch
        dec = self.o.decode_batch(np.ascontiguousarray(x.numpy()[:, :self.n_llr]))
        if bits is not None:
            bits.copy_(torch.from_numpy(dec))

    def siso(self, f4, d2, sf):
        import torch
        A, B = [], []
        for i in range(f4[0].shape[0]):
            a, b = self.o.siso(*[t[i].numpy() for t in f4], *[t[i].numpy() for t in d2], sf)
            A.append(a); B.append(b)
        return torch.from_numpy(np.stack(A)), torch.from_numpy(np.stack(B))


@pytest.fixture
def dropin(monkeypatch):
    import torch
    from modulations_b200 import _lib, dvb_rcs2_turbo as turbo

    def to_device(x, dtype, device=None):
        t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
        return t.to(dtype=dtype).contiguous()
    monkeypatch.setattr(_lib, "require_cuda", lambda: torch)
    monkeypatch.setattr(_lib, "to_device", to_device)
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    monkeypatch.setattr(turbo, "_CodecHandle", _OracleHandle)
    monkeypatch.setattr(turbo, "_siso_handles", {})
    monkeypatch.setattr(turbo, "_component_handles", {})
    monkeypatch.setitem(sys.modules, "dvb_rcs2_turbo", turbo)
    plt = types.ModuleType("matplotlib.pyplot")
    for name in ("figure", "subplots", "savefig", "show", "tight_layout", "close", "plot", "semilogy", "grid",
                 "xlabel", "ylabel", "title", "legend", "subplot", "ylim", "xlim"):
        setattr(plt, name, lambda *a, **k: None)
    mpl = types.ModuleType("matplotlib")
    mpl.pyplot = plt
    mpl.use = lambda *a, **k: None
    monkeypatch.setitem(sys.modules, "matplotlib", mpl)
    monkeypatch.setitem(sys.modules, "matplotlib.pyplot", plt)
    return turbo


def _load(name):
    spec = importlib.util.spec_from_file_location("ref_" + name, os.path.join(REF, name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)                  # runs `from dvb_rcs2_turbo import DVB_RCS2_TurboCodec, bcjr_decode`
    return mod


@needs_scripts
def test_d_test_runs_unmodified(dropin, capsys):
    mod = _load("d_test")
    assert mod.bcjr_decode is dropin.bcjr_decode
    mod.main()
    out = capsys.readouterr().out
    assert "DEBUG COMPLETE" in out and "TURBO ITERATION ANALYSIS" in out


@needs_scripts
def test_turbo_test_suite_runs_unmodified(dropin, monkeypatch, capsys):
    mod = _load("turbo_test_suite")
    # setup(): rate 1 = '1/3', block 48, 3 blocks, SNR 0..1 dB step 1 (a negative start makes the reference's own
    # np.random.seed(int(snr*1000)+42) raise, turbo_test_suite.py:136), 2 iterations; Enter; no plots
    answers = iter(["1", "48", "3", "0", "1", "1", "2", "", "n"])
    monkeypatch.setattr(builtins, "input", lambda *a: next(answers))
    tester = mod.TurboCodeTester()
    tester.run()
    out = capsys.readouterr().out
    assert "Test completed" in out
    assert tester.codec.k_info == 96 and tester.codec.n_coded == 288 and abs(tester.codec.code_rate - 1 / 3) < 1e-12


def test_facade_calls_of_the_scripts(dropin):
    """The calls d_test.py and turbo_test_suite.py make on the drop-in (the two names they import, the facade's
    attributes, encode / decode, the interleaver, both constituent encoders and SISO decoders; INTEGRATION.md), at the
    scripts' own configuration (N=48, rate 1/3, 2 iterations), each checked against the C oracle."""
    from oracle import oracle
    from tests import vectors
    N = 48
    c = dropin.DVB_RCS2_TurboCodec(block_length=N, code_rate='1/3', n_iterations=2)
    assert (c.k_info, c.n_coded, c.N, c.interleaver.N) == (96, 288, N, N) and abs(c.code_rate - 1 / 3) < 1e-12
    o = oracle.OracleTurbo(N, '1/3', 2, perm=c.interleaver.perm, inv_perm=c.interleaver.inv_perm)
    rs = np.random.RandomState(5)
    info = rs.randint(0, 2, c.k_info)
    coded = c.encode(info)
    assert np.array_equal(coded, o.encode(info))
    A, B = info[0::2], info[1::2]
    Ai, Bi = c.interleaver.interleave(A, B)
    assert np.array_equal(Ai, A[o.perm]) and np.array_equal(Bi, B[o.perm])
    full = np.asarray(coded).reshape(N, 6)                  # rate 1/3: A, B, W1, Y1, W2, Y2 per couple
    for enc, a, b, cols in ((c.encoder1, A, B, (2, 3)), (c.encoder2, Ai, Bi, (4, 5))):
        W, Y = enc.encode(a, b)
        assert np.array_equal(W, full[:, cols[0]]) and np.array_equal(Y, full[:, cols[1]])
    llr = vectors.awgn_llr(rs, np.asarray(coded), '1/3', 2.0)
    Lc = vectors.depuncture(llr, N, o.punct)
    La = vectors.siso_apriori(N)
    for dec, w, y in ((c.decoder1, Lc[2], Lc[3]), (c.decoder2, Lc[4], Lc[5])):
        got, want = dec.decode(Lc[0], Lc[1], w, y, *La), o.siso(Lc[0], Lc[1], w, y, *La, 0.7)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    got, want = dropin.bcjr_decode(Lc[0], Lc[1], Lc[2], Lc[3], *La, 1.0), o.siso(Lc[0], Lc[1], Lc[2], Lc[3], *La, 1.0)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    assert np.array_equal(c.decode(llr), o.decode(llr))
