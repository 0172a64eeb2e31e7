"""Drop-in for the reference ``dvb_rcs2_turbo`` module, running on B200.

Same names, arguments, array layouts and error behaviour as the reference
(``dvb_rcs2_turbo.py``); all trellis work — SISO recursions, the 8-iteration
decoder, the tail-biting encoder with its GF(2) circular-state solve — runs in
hand-written sm_100a kernels behind ``libb200dvb.so`` (``include/b200dvb.h``).
There is no CPU fallback.

Host code here only builds the small tables exactly as the reference does
(interleaver ``:311-325``, trellis ``:327-396``, puncturing ``:21-26``) and moves
arrays.  ``perm`` is not a permutation for any table entry and ``inv_perm`` is
``np.argsort(perm)`` with the host's tie order (SURVEY §0 F2), so both are handed
to the device as opaque gather tables.

Batched entry points (``encode_batch`` / ``decode_batch`` / 2-D inputs to
``bcjr_max_log_map``) accept numpy arrays or CUDA torch tensors and are what the
Monte-Carlo harness uses; the single-frame methods are the reference's API.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib

# dvb_rcs2_turbo.py:12-17 — N_couples: (P, Q0, Q1, Q2, Q3)
INTERLEAVER_PARAMS = {
    48: (31, 4, 2, 0, 3), 64: (41, 2, 6, 4, 1),
    212: (137, 0, 6, 4, 9), 220: (143, 4, 2, 8, 5),
    424: (277, 2, 4, 0, 7), 752: (491, 0, 8, 2, 5),
    848: (553, 4, 6, 0, 3),
}

# dvb_rcs2_turbo.py:21-26 — 1 = transmitted, 0 = punctured
PUNCTURE_PATTERNS = {
    '1/3': {'period': 1, 'W1': [1], 'Y1': [1], 'W2': [1], 'Y2': [1]},
    '1/2': {'period': 2, 'W1': [1, 0], 'Y1': [0, 1], 'W2': [1, 0], 'Y2': [0, 1]},
    '2/3': {'period': 3, 'W1': [1, 0, 0], 'Y1': [0, 1, 0], 'W2': [0, 0, 1], 'Y2': [0, 0, 0]},
    '3/4': {'period': 4, 'W1': [1, 0, 0, 0], 'Y1': [0, 1, 0, 0], 'W2': [0, 0, 1, 0], 'Y2': [0, 0, 0, 0]},
}


# ---------------------------------------------------------------------------
# small host helpers with the reference's names (dvb_rcs2_turbo.py:32-114)
# ---------------------------------------------------------------------------
def max_star(a, b):
    """Max-log approximation max(a, b) (dvb_rcs2_turbo.py:32-35)."""
    return a if a > b else b


def _pack_rows(M):
    M = np.asarray(M, dtype=np.int64) & 1
    return [int(sum(int(M[i, j]) << j for j in range(4))) for i in range(4)]


def _unpack_rows(rows):
    return np.array([[(r >> j) & 1 for j in range(4)] for r in rows], dtype=np.int32)


def mat_mul_gf2(A, B):
    """4x4 product over GF(2) (dvb_rcs2_turbo.py:37-48), rows bit-packed."""
    a, Bt = _pack_rows(A), _pack_rows(np.asarray(B).T)
    return np.array([[bin(a[i] & Bt[j]).count("1") & 1 for j in range(4)] for i in range(4)], dtype=np.int32)


def mat_pow_gf2(A, power):
    """Square-and-multiply over GF(2) (dvb_rcs2_turbo.py:50-61)."""
    res = np.eye(4, dtype=np.int32)
    base = np.array(A, dtype=np.int32)
    power = int(power)
    while power > 0:
        if power & 1:
            res = mat_mul_gf2(res, base)
        base = mat_mul_gf2(base, base)
        power >>= 1
    return res


def solve_circular_state_gf2(G_pow_N, Z_N):
    """Solve (I + G^N) Sc = Z_N over GF(2) (dvb_rcs2_turbo.py:63-114): Gaussian
    elimination on bit-packed augmented rows, same pivoting order as the reference."""
    rows = _pack_rows((np.eye(4, dtype=np.int64) + np.asarray(G_pow_N, dtype=np.int64)) % 2)
    rows = [r | (((int(Z_N) >> i) & 1) << 4) for i, r in enumerate(rows)]
    for i in range(4):
        if not (rows[i] >> i) & 1:
            for k in range(i + 1, 4):
                if (rows[k] >> i) & 1:
                    rows[i], rows[k] = rows[k], rows[i]
                    break
        if (rows[i] >> i) & 1:
            for k in range(i + 1, 4):
                if (rows[k] >> i) & 1:
                    rows[k] ^= rows[i]
    x = 0
    for i in range(3, -1, -1):
        s = (rows[i] >> 4) & 1
        for j in range(i + 1, 4):
            s ^= ((rows[i] >> j) & 1) & ((x >> j) & 1)
        x |= s << i
    return x


def build_trellis():
    """Historic name (SURVEY Appendix A): -> (next_state, out_w, out_y) of the
    committed 16-state trellis (dvb_rcs2_turbo.py:327-370)."""
    t = _trellis_tables()
    return t["next_state"], t["out_W"], t["out_Y"]


def _trellis_tables():
    s = np.arange(16)[:, None]
    u = np.arange(4)[None, :]
    ab = ((u >> 1) ^ u) & 1
    s0, s1, s2, s3 = s & 1, (s >> 1) & 1, (s >> 2) & 1, (s >> 3) & 1
    dk = ab ^ s2 ^ s3                                   # :351
    out_W = (dk ^ s0 ^ s1 ^ s3).astype(np.int32)        # :355
    out_Y = (dk ^ s1 ^ s2 ^ s3).astype(np.int32)        # :359
    next_state = ((s2 << 3) | (s1 << 2) | (s0 << 1) | dk).astype(np.int32)   # :366
    prev_state = np.full((16, 4), -1, np.int32)
    prev_input = np.full((16, 4), -1, np.int32)
    fill = [0] * 16
    for st in range(16):                                # :389-396
        for inp in range(4):
            ns = int(next_state[st, inp])
            if fill[ns] < 4:
                prev_state[ns, fill[ns]] = st
                prev_input[ns, fill[ns]] = inp
                fill[ns] += 1
    G = np.zeros((4, 4), np.int32)                      # :380-383
    G[0, 2] = G[0, 3] = G[1, 0] = G[2, 1] = G[3, 2] = 1
    return dict(next_state=next_state, out_W=out_W, out_Y=out_Y, prev_state=prev_state,
                prev_input=prev_input, G_matrix=G)


# ---------------------------------------------------------------------------
# device handle: every call into libb200dvb.so for the codec goes through this class
# ---------------------------------------------------------------------------
class _CodecHandle:
    """Owns one b200dvb_codec_t on the device that was current at construction, plus its cached
    workspaces (one per kind and CUDA stream, so calls on different streams never share scratch).
    All launches run with that device current and on ITS current stream, whatever device the caller
    has selected meanwhile."""

    def __init__(self, N, next_state, out_W, out_Y, perm, inv_perm, punct_u8, period, iterations,
                 sf_inner=0.7, sf_last=1.0, kernel=None, mode=None):
        torch = _lib.require_cuda()
        lib = _lib.load()
        self.device = torch.device("cuda", torch.cuda.current_device())
        arrs = [np.ascontiguousarray(a, np.int32) for a in (next_state, out_W, out_Y, perm, inv_perm)]
        pu = np.ascontiguousarray(punct_u8, np.uint8)
        h = ctypes.c_void_p()
        rc = lib.b200dvb_codec_create(int(N), *[_lib.host_ptr(a) for a in arrs], _lib.host_ptr(pu),
                                      int(period), int(iterations), float(sf_inner), float(sf_last),
                                      ctypes.byref(h))
        _lib.check(rc, f"codec_create(N={N})")
        self.h = h
        self.N = int(N)
        self.k_info = 2 * int(N)
        self.n_llr = int(lib.b200dvb_codec_n_llr(h))
        self._ws = {}
        if kernel is not None:
            self.set_option(_lib.OPT_KERNEL, {"auto": _lib.KERNEL_AUTO, "quad": _lib.KERNEL_QUAD,
                                              "tpf": _lib.KERNEL_TPF, "lat": _lib.KERNEL_LAT}[kernel])
        if mode is not None:
            self.set_option(_lib.OPT_DECODER_MODE, mode)
        self.frames_per_wave = int(lib.b200dvb_codec_frames_per_wave(h))    # depends on the decoder mode

    def set_option(self, option, value):
        _lib.check(_lib.load().b200dvb_codec_set_option(self.h, int(option), int(value)), "codec_set_option")

    def stream(self):
        return _lib.torch_mod().cuda.current_stream(self.device)

    def workspace(self, kind, B, stream=None):
        torch = _lib.torch_mod()
        lib = _lib.load()
        fn = lib.b200dvb_decode_workspace_bytes if kind == "decode" else lib.b200dvb_siso_workspace_bytes
        need = int(fn(self.h, int(B)))
        key = (kind, (stream or self.stream()).cuda_stream)
        cur = self._ws.get(key)
        if cur is None or cur.numel() < need:
            cur = torch.empty(need, dtype=torch.uint8, device=self.device)
            self._ws[key] = cur
        return cur, need

    # -- the three device operations of the codec -------------------------------------------------
    def encode(self, info, want_circ=False):
        """info uint8 CUDA [B, 2N] -> (coded uint8 [B, n_llr], circ uint8 [B, 2] or None)."""
        torch = _lib.torch_mod()
        B = info.shape[0]
        with torch.cuda.device(self.device):
            coded = torch.empty((B, self.n_llr), dtype=torch.uint8, device=self.device)
            circ = torch.empty((B, 2), dtype=torch.uint8, device=self.device) if want_circ else None
            rc = _lib.load().b200dvb_encode(self.h, B, _lib.ptr(info), _lib.ptr(coded), _lib.ptr(circ),
                                            ctypes.c_void_p(self.stream().cuda_stream))
        _lib.check(rc, "encode")
        return coded, circ

    def decode(self, x, bits=None, packed=None, ref=None, counters=None, stream=None, ws=None, llr_scale=1.0, app=None):
        """x float32, float16 or int8 CUDA [B, >= n_llr] (row stride in elements taken from the tensor).  float16 goes
        to b200dvb_decode_f16: the decode of its exact float32 widening, bit for bit.  int8 goes to b200dvb_decode_i8:
        the decode of float32(q) * float32(llr_scale), bit for bit; ``llr_scale`` is not read for other dtypes.
        ``app`` (float32 CUDA [B, 2N], contiguous): the call goes to b200dvb_decode_app, which also writes the
        a-posteriori LLRs there; the other outputs are the same."""
        torch = _lib.torch_mod()
        B = x.shape[0]
        st = stream or self.stream()
        entry, scaled, code = _LLR_FORMATS[_dtype_name(x.dtype)]
        lib = _lib.load()
        with torch.cuda.device(self.device):
            buf, need = ws if ws is not None else self.workspace("decode", B, st)
            stride = x.stride(0) if B > 1 else x.shape[1]     # a length-1 axis may report stride 0
            outs = (_lib.ptr(bits), _lib.ptr(packed), _lib.ptr(ref), _lib.ptr(counters), _lib.ptr(buf), need,
                    ctypes.c_void_p(st.cuda_stream))
            if app is not None:
                rc = lib.b200dvb_decode_app(self.h, B, _lib.ptr(x), code, float(llr_scale) if scaled else 1.0, stride,
                                            _lib.ptr(app), *outs)
            else:
                scale = (float(llr_scale),) if scaled else ()
                rc = getattr(lib, entry)(self.h, B, _lib.ptr(x), stride, *scale, *outs)
        _lib.check(rc, "decode")

    def siso(self, f4, d2, sf):
        """f4: four float32 CUDA [B, N] (Lc_A, Lc_B, Lc_W, Lc_Y); d2: two float64 (La_A, La_B)."""
        torch = _lib.torch_mod()
        B = f4[0].shape[0]
        with torch.cuda.device(self.device):
            LeA = torch.empty((B, self.N), dtype=torch.float64, device=self.device)
            LeB = torch.empty_like(LeA)
            ws, need = self.workspace("siso", B)
            rc = _lib.load().b200dvb_siso(self.h, B, *[_lib.ptr(t) for t in f4], *[_lib.ptr(t) for t in d2],
                                          float(sf), _lib.ptr(LeA), _lib.ptr(LeB), _lib.ptr(ws), need,
                                          ctypes.c_void_p(self.stream().cuda_stream))
        _lib.check(rc, "bcjr_max_log_map")
        return LeA, LeB

    def mc_generate_bpsk(self, B, noise_var, seed, frame_offset, info, coded, llr):
        """Monte-Carlo source (b200dvb_mc_generate_bpsk): Philox info bits -> encode -> BPSK + AWGN -> LLR, written
        into caller-owned CUDA buffers info uint8 [>=B, 2N], coded uint8 [>=B, n_llr], llr float32 [>=B, n_llr]."""
        torch = _lib.torch_mod()
        with torch.cuda.device(self.device):
            rc = _lib.load().b200dvb_mc_generate_bpsk(self.h, int(B), float(noise_var), int(seed), int(frame_offset),
                                                      _lib.ptr(info), _lib.ptr(coded), _lib.ptr(llr),
                                                      ctypes.c_void_p(self.stream().cuda_stream))
        _lib.check(rc, "mc_generate_bpsk")

    def __del__(self):
        try:
            if getattr(self, "h", None):
                _lib.load().b200dvb_codec_destroy(self.h)
                self.h = None
        except Exception:
            pass


_siso_handles = {}


def _siso_handle(N, next_st, out_W, out_Y):
    dev = _lib.require_cuda().cuda.current_device()
    key = (dev, int(N), np.asarray(next_st).tobytes(), np.asarray(out_W).tobytes(), np.asarray(out_Y).tobytes())
    h = _siso_handles.get(key)
    if h is None:
        ident = np.arange(int(N), dtype=np.int32)
        h = _CodecHandle(N, next_st, out_W, out_Y, ident, ident, np.ones((4, 1), np.uint8), 1, 1)
        _siso_handles[key] = h
    return h


def _as_2d(x, N):
    """[N'] or [B, N'] -> [B, N]; like the reference's loops (``for k in range(N)``) only the first N
    entries of each row are read."""
    torch = _lib.torch_mod()
    if not isinstance(x, torch.Tensor):
        x = np.asarray(x)
    if x.ndim == 1:
        x = x[None, :]
    if x.shape[-1] < N:
        raise IndexError(f"SISO input has {x.shape[-1]} entries per frame, N = {N}")
    return x[..., :N]


def bcjr_max_log_map(Lc_A, Lc_B, Lc_W, Lc_Y, La_A, La_B, next_st, out_W, out_Y, prev_st, prev_inp,
                     N, scaling_factor):
    """Max-log-MAP SISO half-iteration, double pass for the circular trellis with
    extrinsic scaling — same signature and return as the reference
    (dvb_rcs2_turbo.py:116-281): ``(Le_A, Le_B)`` float64[N].

    Bit-exact with the reference's arithmetic (float64 branch-metric sums rounded
    to float32, float32 recursions normalised by state 0, float64 extrinsic).
    Inputs may also be ``[B, N]`` (numpy or CUDA torch) for B independent frames.

    Narrower than the reference in three documented ways: (1) ``prev_st`` / ``prev_inp`` are accepted
    for signature parity but not read — the kernel derives the reverse trellis from ``next_st``; (2) only
    the committed 16-state trellis (``_trellis_tables()``) has a kernel specialisation, any other table
    raises ``ValueError`` (B200DVB_ENOSPEC) instead of being emulated; (3) N must be a multiple of 4 in
    [8, 2048] (every N of the reference's table is).
    """
    torch = _lib.require_cuda()
    N = int(N)
    h = _siso_handle(N, next_st, out_W, out_Y)
    is_torch = isinstance(Lc_A, torch.Tensor)
    single = (not is_torch and np.asarray(Lc_A).ndim == 1) or (is_torch and Lc_A.dim() == 1)
    f = [_lib.to_device(_as_2d(x, N), torch.float32, h.device) for x in (Lc_A, Lc_B, Lc_W, Lc_Y)]
    d = [_lib.to_device(_as_2d(x, N), torch.float64, h.device) for x in (La_A, La_B)]
    LeA, LeB = h.siso(f, d, scaling_factor)
    if is_torch:
        return (LeA[0], LeB[0]) if single else (LeA, LeB)
    a, b = LeA.cpu().numpy(), LeB.cpu().numpy()
    return (a[0], b[0]) if single else (a, b)


def bcjr_decode_circular(*args):
    """Historic alias (SURVEY Appendix A).  13 arguments: the committed signature;
    7 arguments ``(Lc_A, Lc_B, Lc_W, Lc_Y, La_A, La_B, scaling)``: committed trellis.
    Always the COMMITTED arithmetic of ``bcjr_max_log_map``."""
    if len(args) == 13:
        return bcjr_max_log_map(*args)
    if len(args) == 7:
        t = _trellis_tables()
        N = np.asarray(args[0]).shape[-1] if not hasattr(args[0], "dim") else args[0].shape[-1]
        return bcjr_max_log_map(*args[:6], t["next_state"], t["out_W"], t["out_Y"], t["prev_state"],
                                t["prev_input"], N, args[6])
    raise TypeError("bcjr_decode_circular takes 13 or 7 positional arguments")


def bcjr_decode(*args):
    """Historic name imported by the reference's ``d_test.py:9`` (revisions 12-15 10:39 … 12-16 11:00 of
    ``dvb_rcs2_turbo.py``, SURVEY Appendix A; 7 arguments ``(6 LLR arrays, scaling)``).  Served by the
    committed arithmetic like the other aliases."""
    return bcjr_decode_circular(*args)


def max_log_map_decode(*args):
    """Historic alias.  11 arguments ``(6 arrays, next_st, prev_st, out_w, out_y,
    scaling)`` or 7 ``(6 arrays, scaling)``; committed arithmetic."""
    if len(args) == 11:
        a6, next_st, prev_st, out_w, out_y, sc = args[:6], args[6], args[7], args[8], args[9], args[10]
        N = a6[0].shape[-1]
        return bcjr_max_log_map(*a6, next_st, out_w, out_y, prev_st, None, N, sc)
    if len(args) == 7:
        return bcjr_decode_circular(*args)
    raise TypeError("max_log_map_decode takes 11 or 7 positional arguments")


# ---------------------------------------------------------------------------
# DVBRCS2_Turbo (dvb_rcs2_turbo.py:287-537)
# ---------------------------------------------------------------------------
def bijective_interleaver(N):
    """An almost-regular-permutation interleaver that IS a permutation (extension for non-parity runs):
    pi(i) = (P i + 4 d(i mod 4) + 3) mod N with P the table's period made coprime to N."""
    from math import gcd
    P = INTERLEAVER_PARAMS[N][0] if N in INTERLEAVER_PARAMS else 13
    while gcd(P, N) != 1:
        P += 2
    i = np.arange(N, dtype=np.int64)
    d = np.array([0, 3, 5, 2], dtype=np.int64)[i % 4]
    perm = ((P * i + 4 * d + 3) % N).astype(np.int32)
    while len(np.unique(perm)) != N:                          # 4 d(i mod 4) keeps residues apart unless 4 | P's orbit
        P += 2
        while gcd(P, N) != 1:
            P += 2
        perm = ((P * i + 4 * d + 3) % N).astype(np.int32)
    return perm


class DVBRCS2_Turbo:
    BOUNDARIES = {"double-pass": _lib.MODE_PARITY, "nii": _lib.MODE_NII, "nii16": _lib.MODE_NII16}

    def __init__(self, N_couples, code_rate, iterations=8, perm=None, kernel=None, boundary="double-pass"):
        """``perm`` (extension, NOT reference behaviour): a user-supplied interleaver table of length N
        replacing the committed one, whose formula is not a permutation (SURVEY F2: BER ~ 0.2 at every
        SNR).  With a bijective ``perm`` the same kernels decode properly; results are then compared with
        the oracle given the same table, and reported as a labelled non-parity run (SURVEY 8f N2).
        ``kernel`` (development / tests): "auto" (default), "quad", "tpf" or "lat" forces one decode kernel.
        ``boundary`` (extension): "double-pass" (default) is the reference's decoder, bit-exact
        (dvb_rcs2_turbo.py:162-230: every recursion runs twice around the circular trellis).  "nii" is a
        NON-PARITY mode: one pass per SISO, alpha[0] / beta[N] initialised from the metrics the same constituent
        decoder reached in the previous iteration, float32 extrinsics (csrc/nii_core.cuh).  Its hard decisions
        differ from the reference's in isolated bits; it is judged on BER/FER and checked bit for bit against
        its own model (oracle/nii_model.c).  "nii16" is the same decoder in 16-bit fixed point, two frames per
        32-bit register with DPX add-compare-select instructions (csrc/nii16_core.cuh; model oracle/nii16_model.c).
        ``decode`` / ``decode_batch`` / ``decode_batch_host`` follow it;
        ``bcjr_max_log_map`` and the encoder are unaffected."""
        if boundary not in self.BOUNDARIES:
            raise ValueError(f"boundary must be one of {sorted(self.BOUNDARIES)}")
        self.boundary = boundary
        self.N = N_couples
        self.k_info = N_couples * 2
        self._iterations = iterations
        self._kernel = kernel
        self.punct = PUNCTURE_PATTERNS[code_rate]               # KeyError for unknown rates (:292)
        if self.N not in INTERLEAVER_PARAMS:                    # :295-296
            raise ValueError(f"Block size {self.N} not in standard tables.")
        self._init_interleaver()
        if perm is not None:
            perm = np.ascontiguousarray(perm, np.int32)
            if perm.shape != (self.N,) or perm.min() < 0 or perm.max() >= self.N:
                raise ValueError("perm must hold N indices in [0, N)")
            self.perm = perm
            self.inv_perm = np.argsort(self.perm).astype(np.int32)
        for k, v in _trellis_tables().items():
            setattr(self, k, v)
        self._calc_coded_size()
        self._punct_u8 = np.array([self.punct[k] for k in ('W1', 'Y1', 'W2', 'Y2')], np.uint8)
        self._handles = {}
        self._e2e = None
        self._one = {}             # decode(): pinned staging + device buffers per (handle, stream)

    @property
    def iterations(self):
        """Read on every decode like the reference's attribute (:493): assigning a new value takes effect
        on the next call (the device handle is rebuilt for it)."""
        return self._iterations

    @iterations.setter
    def iterations(self, value):
        self._iterations = int(value)

    # -- tables -------------------------------------------------------------
    def _init_interleaver(self):
        """perm[i] = P*(i + d(i%4) + Q3*(i//4)) mod N, inv_perm = argsort(perm) (:311-325)."""
        P, Q0, Q1, Q2, Q3 = INTERLEAVER_PARAMS[self.N]
        i = np.arange(self.N, dtype=np.int64)
        d = np.array([0, Q0, Q1, Q2], dtype=np.int64)[i % 4]
        self.perm = ((P * (i + d + Q3 * (i // 4))) % self.N).astype(np.int32)
        self.inv_perm = np.argsort(self.perm).astype(np.int32)

    def _calc_coded_size(self):
        """n_coded = (N // period) * bits_per_period — keeps the reference's
        truncation for N % period != 0 (:398-402)."""
        p = self.punct
        per = 2 * p['period'] + sum(p['W1']) + sum(p['Y1']) + sum(p['W2']) + sum(p['Y2'])
        self.n_coded = (self.N // p['period']) * per

    @property
    def handle(self):
        """The device handle for (current CUDA device, current ``iterations``)."""
        torch = _lib.require_cuda()
        key = (torch.cuda.current_device(), int(self._iterations))
        h = self._handles.get(key)
        if h is None:
            h = _CodecHandle(self.N, self.next_state, self.out_W, self.out_Y, self.perm, self.inv_perm,
                             self._punct_u8, self.punct['period'], self._iterations, kernel=self._kernel,
                             mode=self.BOUNDARIES[self.boundary] if self.boundary != "double-pass" else None)
            self._handles[key] = h
        return h

    @property
    def n_llr(self):
        """LLRs the depuncturer consumes (= bits ``encode`` emits)."""
        return self.handle.n_llr

    # -- encoder ------------------------------------------------------------
    def encode_batch(self, bits, return_circ=False):
        """bits [B, 2N] (numpy or CUDA torch, any integer dtype) -> uint8 [B, n_llr]."""
        torch = _lib.require_cuda()
        h = self.handle
        is_torch = isinstance(bits, torch.Tensor)
        info = _lib.to_device(bits, torch.uint8, h.device).reshape(-1, self.k_info)
        coded, circ = h.encode(info, return_circ)
        if not is_torch:
            coded = coded.cpu().numpy()
            circ = circ.cpu().numpy() if return_circ else None
        return (coded, circ) if return_circ else coded

    def encode(self, bits):
        """Encode 2N info bits into the punctured codeword, int32 (:431-462)."""
        bits = np.array(bits, dtype=np.int32)
        if bits.shape[0] < self.k_info:
            raise IndexError("encode needs 2*N info bits")
        return self.encode_batch(bits[None, :self.k_info])[0].astype(np.int32)

    # -- decoder ------------------------------------------------------------
    def decode_batch(self, llr, ref_bits=None, counters=None, out="bits", llr_scale=None):
        """llr [B, >= n_llr] float32 (numpy or CUDA torch) -> hard decisions.

        float16 input (``torch.float16`` or ``np.float16``) reaches the device as 16 bits and is decoded by the
        binary16 path: fp16 in = decode of its exact float32 widening, bit for bit, in every mode and kernel.
        int8 input (``torch.int8`` or ``np.int8``) reaches the device as 8 bits: q is decoded as the float32 LLR
        float32(q) * float32(llr_scale), bit for bit (``llr_scale`` defaults to 1.0; it must be finite and non-zero,
        and is an error with any other dtype).  Any other dtype is converted to float32.

        out="bits": int32 [B, 2N] (reference layout); "packed": uint32 [B, ceil(2N/32)], bit i of a frame at
        word i//32, bit i%32; "app": float32 [B, 2N], the a-posteriori LLR of each info bit after the last
        iteration in the layout of "bits", positive = bit 0 (b200dvb_decode_app: parity mode gives the float32 of
        the reference's float64 sum, "nii" its float32 sum, "nii16" its 1/4-unit sum times 0.25); "none": nothing
        (error counting only).  ``ref_bits`` (anything reshapeable to uint8 [B, 2N]) and ``counters`` (CUDA
        int64/uint64 tensor, >= 4 elements) enable in-kernel error counting: counters += {bit errors, frame errors,
        frames, info bits}.
        """
        torch = _lib.require_cuda()
        h = self.handle
        if out not in ("bits", "packed", "app", "none"):
            raise ValueError('out must be "bits", "packed", "app" or "none"')
        is_torch = isinstance(llr, torch.Tensor)
        if not is_torch:
            llr = np.asarray(llr)
        fmt, kw = _llr_format(llr.dtype, llr_scale)
        x = _lib.to_device(llr, getattr(torch, fmt or "float32"), h.device)
        if x.dim() == 1:
            x = x[None, :]
        if x.dim() != 2 or x.shape[1] < h.n_llr:
            raise IndexError(f"llr has {x.shape[-1]} values per frame, the depuncturer needs {h.n_llr}")
        if x.stride(1) != 1:
            x = x.contiguous()
        B = x.shape[0]
        bits = packed = app = None
        if out == "bits":
            bits = torch.empty((B, self.k_info), dtype=torch.int32, device=h.device)
        elif out == "packed":
            packed = torch.empty((B, (self.k_info + 31) // 32), dtype=torch.int32, device=h.device)
        elif out == "app":
            app = kw["app"] = torch.empty((B, self.k_info), dtype=torch.float32, device=h.device)
        ref = None
        if ref_bits is not None:
            ref = _lib.to_device(ref_bits, torch.uint8, h.device)
            if ref.numel() != B * self.k_info:
                raise ValueError(f"ref_bits holds {ref.numel()} bits, the batch has {B} x {self.k_info}")
            ref = ref.reshape(B, self.k_info)
        if counters is not None and not (isinstance(counters, torch.Tensor) and counters.is_cuda
                                         and counters.dtype in (torch.int64, torch.uint64)
                                         and counters.numel() >= 4 and counters.is_contiguous()
                                         and counters.device == h.device):
            raise ValueError("counters must be a contiguous CUDA int64/uint64 tensor with >= 4 elements on the codec's device")
        h.decode(x, bits=bits, packed=packed, ref=ref, counters=counters, **kw)
        res = {"bits": bits, "packed": packed, "app": app}.get(out)
        if res is not None and not is_torch:
            res = res.cpu().numpy()
        return res

    def decode_batch_host(self, llr_host, out_host=None, chunk=None, out="bits", llr_scale=None):
        """End-to-end decode of HOST buffers: pinned ``llr_host`` float32, float16 or int8 [B, >= n_llr] -> pinned
        ``out_host``.

        float16 rows cross PCIe as 16 bits (half the bytes) and are decoded by the binary16 path: fp16 in = decode of
        its exact float32 widening, bit for bit.  int8 rows cross as 8 bits (a quarter of the bytes) and q is decoded
        as float32(q) * float32(llr_scale), bit for bit, as in ``decode_batch``.

        out="bits": int32 [B, 2N], the reference's layout (1 696 B per N=212 frame over PCIe);
        out="packed": int32 words [B, ceil(2N/32)], bit i of a frame at word i//32, bit i%32 (56 B per frame:
        the kernel's packed output copied as it is — ``unpack_bits`` expands it lazily on the host);
        out="uint8": uint8 [B, 2N], expanded from the packed words on the device (424 B per frame);
        out="app": float32 [B, 2N], the a-posteriori LLRs of ``decode_batch(out="app")`` (8 N bytes per frame).

        Chunks are pipelined over three CUDA streams so the host->device copy of chunk i+1, the decode of
        chunk i and the device->host copy of chunk i-1 overlap.  ``chunk`` defaults to one wave of the decode
        kernel (tools/e2e_chunks.py).  The call returns after the last device->host copy has COMPLETED: the
        returned CPU tensor can be read at once."""
        torch = _lib.require_cuda()
        h = self.handle
        if out not in ("bits", "packed", "uint8", "app"):
            raise ValueError('out must be "bits", "packed", "uint8" or "app"')
        if chunk is None:
            chunk = max(16, h.frames_per_wave)
        is_torch = isinstance(llr_host, torch.Tensor)
        x = llr_host if is_torch else np.asarray(llr_host)
        fmt, kw = _llr_format(x.dtype, llr_scale)
        if not is_torch:
            fmt = fmt or "float32"
            x = torch.from_numpy(np.ascontiguousarray(x, fmt))
        if x.dim() != 2 or x.shape[1] < h.n_llr or fmt is None:
            raise IndexError(f"llr needs float32, float16 or int8 shape [B, >= {h.n_llr}]")
        B, width = x.shape
        wpf = (self.k_info + 31) // 32
        oshape, odtype = {"bits": ((self.k_info,), torch.int32), "packed": ((wpf,), torch.int32),
                          "uint8": ((self.k_info,), torch.uint8), "app": ((self.k_info,), torch.float32)}[out]
        if out_host is None:
            out_host = torch.empty((B,) + oshape, dtype=odtype, pin_memory=True)
        elif tuple(out_host.shape) != (B,) + oshape or out_host.dtype != odtype:
            raise ValueError(f"out_host must be {odtype} of shape {(B,) + oshape}")
        nstage = 3
        key = (h, chunk, width, out, x.dtype)
        if self._e2e is None or self._e2e[0] != key:
            with torch.cuda.device(h.device):
                streams = [torch.cuda.Stream(device=h.device) for _ in range(nstage)]
                din = [torch.empty((chunk, width), dtype=x.dtype, device=h.device) for _ in range(nstage)]
                dout = [torch.empty((chunk,) + oshape, dtype=odtype, device=h.device) for _ in range(nstage)]
                dpk = [torch.empty((chunk, wpf), dtype=torch.int32, device=h.device) if out == "uint8" else None
                       for _ in range(nstage)]
                wss = [h.workspace("decode", chunk, st) for st in streams]
                done = [torch.cuda.Event() for _ in range(nstage)]
            self._e2e = (key, streams, din, dout, dpk, wss, done)
        _, streams, din, dout, dpk, wss, done = self._e2e
        cur = h.stream()
        for st in streams:
            st.wait_stream(cur)
        for i, lo in enumerate(range(0, B, chunk)):
            n = min(chunk, B - lo)
            j = i % nstage
            with torch.cuda.stream(streams[j]):
                din[j][:n].copy_(x[lo:lo + n], non_blocking=True)
                if out == "bits":
                    h.decode(din[j][:n], bits=dout[j], stream=streams[j], ws=wss[j], **kw)
                elif out == "packed":
                    h.decode(din[j][:n], packed=dout[j], stream=streams[j], ws=wss[j], **kw)
                elif out == "app":
                    h.decode(din[j][:n], app=dout[j], stream=streams[j], ws=wss[j], **kw)
                else:
                    h.decode(din[j][:n], packed=dpk[j], stream=streams[j], ws=wss[j], **kw)
                    _unpack_bits_device(dpk[j][:n], dout[j][:n], self.k_info)
                out_host[lo:lo + n].copy_(dout[j][:n], non_blocking=True)
                done[j].record(streams[j])
        for j, st in enumerate(streams):
            cur.wait_stream(st)
        for ev in done:                       # the copies land in host memory: block the HOST, not only the stream
            ev.synchronize()
        return out_host

    def decode(self, llr):
        """Decode one frame of LLRs (positive = bit 0) into 2N info bits, int32 (:464-537).

        The reference's call shape (turbo_test_suite.py:138-164): one frame per call, so the host side counts.  Pinned
        staging buffers and the device tensors are kept per (handle, stream); a call is one copy into pinned memory,
        an asynchronous host-to-device copy, the kernel, an asynchronous copy back and one stream synchronisation.
        Not re-entrant per object and stream (neither is the reference's numba decoder)."""
        llr = np.array(llr, dtype=np.float32)
        torch = _lib.require_cuda()
        h = self.handle
        if llr.ndim != 1 or llr.shape[0] < h.n_llr or getattr(h.device, "type", "cuda") != "cuda":
            return self.decode_batch(llr[None, :] if llr.ndim == 1 else llr)[0]      # (short input: raises like the batch path)
        with torch.cuda.device(h.device):
            st = torch.cuda.current_stream(h.device)
            key = (h, st.cuda_stream)
            one = self._one.get(key)
            if one is None:
                hin = torch.empty((1, h.n_llr), dtype=torch.float32, pin_memory=True)
                hout = torch.empty((1, self.k_info), dtype=torch.int32, pin_memory=True)
                one = (hin, hin.numpy(), torch.empty((1, h.n_llr), dtype=torch.float32, device=h.device),
                       torch.empty((1, self.k_info), dtype=torch.int32, device=h.device), hout, hout.numpy())
                self._one[key] = one
            hin, hin_np, din, dbits, hout, hout_np = one
            np.copyto(hin_np[0], llr[:h.n_llr])
            din.copy_(hin, non_blocking=True)
            h.decode(din, bits=dbits, stream=st)
            hout.copy_(dbits, non_blocking=True)
            st.synchronize()
        return hout_np[0].copy()


# Channel LLR element formats the decoder takes, by dtype name (numpy's and torch's alike; the name is also the torch
# dtype on the device): the C entry point, whether it takes a scale (int8 q is the float32 LLR q * llr_scale), and the
# format code of b200dvb_decode_app.
_LLR_FORMATS = {"float32": ("b200dvb_decode", False, _lib.LLR_F32),
                "float16": ("b200dvb_decode_f16", False, _lib.LLR_F16),
                "int8": ("b200dvb_decode_i8", True, _lib.LLR_I8)}


def _dtype_name(dtype):
    return str(dtype).removeprefix("torch.")


def _llr_format(dtype, llr_scale):
    """-> (name in _LLR_FORMATS, or None for a dtype the decoder does not take; _CodecHandle.decode keywords).  int8
    takes its scale (1.0 when not given); a scale given with any other dtype is an error, not silently ignored."""
    fmt = _dtype_name(dtype)
    fmt = fmt if fmt in _LLR_FORMATS else None
    if fmt is None or not _LLR_FORMATS[fmt][1]:
        if llr_scale is not None:
            raise ValueError("llr_scale applies to int8 LLRs only")
        return fmt, {}
    return fmt, {"llr_scale": 1.0 if llr_scale is None else float(llr_scale)}


def _unpack_bits_device(packed, out_u8, k_info):
    """packed int32 [n, W] -> out_u8 uint8 [n, k_info] on the device (plain tensor ops: plumbing, not the hot path)."""
    torch = _lib.torch_mod()
    sh = torch.arange(32, device=packed.device, dtype=torch.int32)
    b = (packed.unsqueeze(-1) >> sh) & 1
    out_u8.copy_(b.reshape(packed.shape[0], -1)[:, :k_info])


def unpack_bits(packed, k_info):
    """Host-side expansion of ``decode_batch_host(..., out="packed")`` words into the reference's int32 [B, 2N]."""
    a = packed.numpy() if hasattr(packed, "numpy") else np.asarray(packed)
    b = np.unpackbits(np.ascontiguousarray(a).view(np.uint8), axis=1, bitorder="little")
    return b[:, :k_info].astype(np.int32)


# ---------------------------------------------------------------------------
# Facade used by turbo_test_suite.py / d_test.py / test_sdr_with_coding.py
# (class missing from the committed reference source, SURVEY §0 F1)
# ---------------------------------------------------------------------------
class _Interleaver:
    def __init__(self, perm, inv_perm):
        self.perm, self.inv_perm, self.N = perm, inv_perm, len(perm)

    def interleave(self, A, B):
        return np.asarray(A)[self.perm], np.asarray(B)[self.perm]


_component_handles = {}


def _component_handle(N):
    """Codec handle of ONE constituent code (identity interleaver, nothing punctured), per device."""
    dev = _lib.require_cuda().cuda.current_device()
    h = _component_handles.get((dev, int(N)))
    if h is None:
        t = _trellis_tables()
        ident = np.arange(N, dtype=np.int32)
        h = _CodecHandle(N, t["next_state"], t["out_W"], t["out_Y"], ident, ident, np.ones((4, 1), np.uint8), 1, 1)
        _component_handles[(dev, int(N))] = h
    return h


def _component_encode(N, A, B):
    """-> (coded uint8 numpy [N, 6], circ uint8 numpy [2]) of the constituent encoder for couples (A, B)."""
    torch = _lib.require_cuda()
    h = _component_handle(N)
    bits = np.stack([np.asarray(A), np.asarray(B)], axis=1).reshape(1, -1)
    coded, circ = h.encode(_lib.to_device(bits, torch.uint8, h.device), True)
    return coded.cpu().numpy()[0].reshape(N, 6), circ.cpu().numpy()[0]


class _ConstituentEncoder:
    def __init__(self, N):
        self.N = N

    def encode(self, A, B):
        """Tail-biting constituent encode of couples (A, B) -> (W, Y) int32[N]."""
        c, _ = _component_encode(self.N, A, B)
        c = c.astype(np.int32)
        return c[:, 2].copy(), c[:, 3].copy()


class _ConstituentDecoder:
    def __init__(self, N, scaling_factor):
        self._t = _trellis_tables()
        self.N, self.scaling_factor = N, scaling_factor

    def decode(self, Lc_A, Lc_B, Lc_W, Lc_Y, La_A, La_B):
        t = self._t
        return bcjr_max_log_map(Lc_A, Lc_B, Lc_W, Lc_Y, La_A, La_B, t["next_state"], t["out_W"],
                                t["out_Y"], t["prev_state"], t["prev_input"], self.N,
                                self.scaling_factor)


class DVB_RCS2_TurboCodec:
    """``DVB_RCS2_TurboCodec(block_length=, code_rate=, n_iterations=)``: the API the
    reference's scripts import (turbo_test_suite.py:406-410, d_test.py:18,
    test_sdr_with_coding.py:258-262) over the committed codec arithmetic."""

    def __init__(self, block_length, code_rate, n_iterations=8):
        self._codec = DVBRCS2_Turbo(block_length, code_rate, n_iterations)
        num, den = code_rate.split('/')
        self.code_rate = float(num) / float(den)
        self.N = self._codec.N
        self.k_info = self._codec.k_info
        self.n_coded = self._codec.n_coded
        self.n_iterations = n_iterations
        self.interleaver = _Interleaver(self._codec.perm, self._codec.inv_perm)
        self.encoder1 = self.encoder2 = _ConstituentEncoder(self.N)
        self.decoder1 = self.decoder2 = _ConstituentDecoder(self.N, 0.7)

    def encode(self, bits):
        return self._codec.encode(bits)

    def decode(self, llr):
        return self._codec.decode(llr)


def determine_circular_state(A, B):
    """Historic name: circular start state of the constituent encoder for couples (A, B)."""
    _, circ = _component_encode(len(A), A, B)
    return int(circ[0])
