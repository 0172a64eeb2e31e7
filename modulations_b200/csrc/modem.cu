// modem.cu — table-driven mapper, hard slicer and max-log soft demapper.
//
// Reference: SDRModem.modulate / demodulate (sdr_modem.py:101-266), Modulator
// (modulators.py:119-200) and compute_llr (test_sdr_with_coding.py:200-225):
//     llr[i*bps+b] = (min_{c: bit_b(c)=0} |s_i - c|^2 - min_{c: bit_b(c)=1} |s_i - c|^2) / max(nv, 0.005)
//     clipped to +-30, bit b = 0 is the MSB of the label, positive LLR <=> bit 1.
//
// Two demapper kernels, both HBM-streaming (8 B in, 4*bps B out per symbol):
//   * demap_generic<BPS>: any constellation.  Table in shared memory, one thread
//     per symbol, all M distances, per-bit minima with compile-time label bits.
//   * demap_pwl<HALF>: square constellations whose label splits into an I half and
//     a Q half (all of the reference's QAM tables and QPSK).  |s-c|^2 = dI^2 + dQ^2,
//     the other axis' term is common to both minima and cancels, so each bit's
//     max-log LLR depends on one coordinate only and is piecewise linear in it:
//     between consecutive mid-points of the axis levels the nearest level of each
//     subset is fixed and (x-Xa)^2 - (x-Xb)^2 = 2(Xb-Xa)x + (Xa^2-Xb^2).  The host
//     tabulates (slope, intercept) per bit and segment from the table it is given —
//     2L-2 segments per axis — so 256QAM costs ~10 flops per LLR instead of 256
//     distances (SURVEY §7 H4): the kernel stays on the HBM roofline.
#include "common.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <vector>

namespace b200dvb {

namespace {

constexpr int kThreads = 256;

template <typename OutT> struct Cplx;
template <> struct Cplx<float> { using type = float2; };
template <> struct Cplx<double> { using type = double2; };

template <typename OutT>
__global__ void map_kernel(size_t n, int bps, const uint8_t *__restrict__ bits,
                           const double *__restrict__ table, typename Cplx<OutT>::type *__restrict__ iq)
{
    __shared__ double2 tab[256];
    const int M = 1 << bps;
    for (int i = threadIdx.x; i < M; i += blockDim.x) tab[i] = make_double2(table[2 * i], table[2 * i + 1]);
    __syncthreads();
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        int lab = 0;
        for (int b = 0; b < bps; ++b) lab = (lab << 1) | (bits[i * bps + b] & 1);
        const double2 p = tab[lab];
        typename Cplx<OutT>::type o;
        o.x = (OutT)p.x; o.y = (OutT)p.y;       // complex128 -> complex64 rounds exactly like np.array(.., complex64)
        iq[i] = o;
    }
}

// The same mapping for complex64 output, written for the memory system: the generic kernel above keeps ONE symbol per
// thread in flight behind a dependent byte load (2.6 symbols per clock and SM: 53 - 64 % of the HBM roofline).  Here a
// thread takes FOUR CONSECUTIVE symbols at a time — 4 BPS bit-bytes = BPS aligned words in (one to three vector loads,
// no symbol straddles the group), 32 bytes out (two 16-byte stores; a warp writes 1 KB contiguous) — with kMapU such
// groups in flight, and gathers a label (first bit = MSB, sdr_modem.py:260-274) from the byte LSBs with one multiply:
// ((w & 0x01010101) * 0x08040201) >> 24 = 8 b0 + 4 b1 + 2 b2 + b3 (the partial products occupy distinct bits).
constexpr int kMapU = 2;

__device__ __forceinline__ unsigned lab4(unsigned w) { return ((w & 0x01010101u) * 0x08040201u) >> 24; }

template <int BPS>
__device__ __forceinline__ void load_words(const uint8_t *__restrict__ p, unsigned (&w)[BPS])
{
    if constexpr (BPS == 1) w[0] = *reinterpret_cast<const unsigned *>(p);
    else if constexpr (BPS == 2) { const uint2 v = *reinterpret_cast<const uint2 *>(p); w[0] = v.x; w[1] = v.y; }
    else if constexpr (BPS == 3) {
        const unsigned *q = reinterpret_cast<const unsigned *>(p);
        w[0] = q[0]; w[1] = q[1]; w[2] = q[2];
    } else if constexpr (BPS == 4) {
        const uint4 v = *reinterpret_cast<const uint4 *>(p); w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    } else if constexpr (BPS == 6) {
        const uint2 *q = reinterpret_cast<const uint2 *>(p);
        const uint2 a = q[0], b = q[1], c = q[2];
        w[0] = a.x; w[1] = a.y; w[2] = b.x; w[3] = b.y; w[4] = c.x; w[5] = c.y;
    } else {
        static_assert(BPS == 8, "orders of the reference: 1, 2, 3, 4, 6, 8 bits per symbol");
        const uint4 *q = reinterpret_cast<const uint4 *>(p);
        const uint4 a = q[0], b = q[1];
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
    }
}
// the four bytes starting at byte Q of the group (compile-time Q; bytes past the group read as 0)
template <int BPS, int Q>
__device__ __forceinline__ unsigned bytes4(const unsigned (&w)[BPS])
{
    constexpr int i = Q >> 2, sh = 8 * (Q & 3);
    const unsigned lo = i < BPS ? w[i < BPS ? i : 0] : 0u, hi = i + 1 < BPS ? w[i + 1 < BPS ? i + 1 : 0] : 0u;
    return sh ? __funnelshift_r(lo, hi, sh) : lo;
}
template <int BPS, int J>
__device__ __forceinline__ unsigned group_label(const unsigned (&w)[BPS])
{
    constexpr int Q = J * BPS;
    if constexpr (BPS <= 4) {
        constexpr unsigned mask = BPS == 4 ? 0x01010101u : (1u << (8 * BPS)) - 1u;
        return lab4(bytes4<BPS, Q>(w) & mask) >> (4 - BPS);
    } else {
        constexpr unsigned mask = BPS == 8 ? 0x01010101u : (1u << (8 * (BPS - 4))) - 1u;
        return (lab4(bytes4<BPS, Q>(w)) << (BPS - 4)) | (lab4(bytes4<BPS, Q + 4>(w) & mask) >> (8 - BPS));
    }
}

template <int BPS>
__global__ void __launch_bounds__(kThreads)
map_words_kernel(size_t n, const uint8_t *__restrict__ bits, const double *__restrict__ table, float2 *__restrict__ iq)
{
    __shared__ float2 tab[1 << BPS];
    for (int i = threadIdx.x; i < (1 << BPS); i += blockDim.x)       // complex128 -> complex64 rounds like np.array(.., complex64)
        tab[i] = make_float2((float)table[2 * i], (float)table[2 * i + 1]);
    __syncthreads();
    const size_t groups = n >> 2;                                    // whole groups of 4 symbols
    const size_t stride = (size_t)gridDim.x * blockDim.x * kMapU;
    for (size_t base = (size_t)blockIdx.x * blockDim.x * kMapU + threadIdx.x; base < groups; base += stride) {
        unsigned w[kMapU][BPS];
#pragma unroll
        for (int u = 0; u < kMapU; ++u) {
            const size_t g = base + (size_t)u * blockDim.x;
            if (g < groups) load_words<BPS>(bits + g * (4 * BPS), w[u]);
            else
#pragma unroll
                for (int q = 0; q < BPS; ++q) w[u][q] = 0u;
        }
#pragma unroll
        for (int u = 0; u < kMapU; ++u) {
            const size_t g = base + (size_t)u * blockDim.x;
            if (g < groups) {
                const float2 s0 = tab[group_label<BPS, 0>(w[u])], s1 = tab[group_label<BPS, 1>(w[u])];
                const float2 s2 = tab[group_label<BPS, 2>(w[u])], s3 = tab[group_label<BPS, 3>(w[u])];
                // one 256-bit store (sm_100: STG.E.ENL2.256): the lane's four symbols are exactly one 32-byte sector;
                // as two 16-byte stores every sector was written in two partial pieces (59 - 74 % instead of 8x %)
                asm volatile("st.global.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(iq + 4 * g),
                             "l"(*reinterpret_cast<const unsigned long long *>(&s0)), "l"(*reinterpret_cast<const unsigned long long *>(&s1)),
                             "l"(*reinterpret_cast<const unsigned long long *>(&s2)), "l"(*reinterpret_cast<const unsigned long long *>(&s3)) : "memory");
            }
        }
    }
    // the last n % 4 symbols, bit by bit
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const size_t i = 4 * groups + threadIdx.x;
        unsigned lab = 0;
        for (int b = 0; b < BPS; ++b) lab = (lab << 1) | (bits[i * BPS + b] & 1u);
        iq[i] = tab[lab];
    }
}

// One symbol per lane and store (8 bytes per lane, 256 contiguous bytes per warp store), kSymU symbols per thread in
// flight: the symbol's BPS bit-bytes are one aligned load for BPS = 1, 2, 4, 8.
constexpr int kSymU = 4;
template <int BPS>
__device__ __forceinline__ unsigned load_label(const uint8_t *__restrict__ bits, size_t i)
{
    const size_t o = i * BPS;
    if constexpr (BPS == 1) return bits[o] & 1u;
    else if constexpr (BPS == 2) {
        const unsigned w = *reinterpret_cast<const uint16_t *>(bits + o);
        return ((w & 1u) << 1) | ((w >> 8) & 1u);
    } else if constexpr (BPS == 4) return lab4(*reinterpret_cast<const unsigned *>(bits + o));
    else {
        static_assert(BPS == 8, "aligned orders only");
        const uint2 w = *reinterpret_cast<const uint2 *>(bits + o);
        return (lab4(w.x) << 4) | lab4(w.y);
    }
}
template <int BPS>
__global__ void __launch_bounds__(kThreads)
map_sym_kernel(size_t n, const uint8_t *__restrict__ bits, const double *__restrict__ table, float2 *__restrict__ iq)
{
    __shared__ float2 tab[1 << BPS];
    for (int i = threadIdx.x; i < (1 << BPS); i += blockDim.x)
        tab[i] = make_float2((float)table[2 * i], (float)table[2 * i + 1]);
    __syncthreads();
    const size_t stride = (size_t)gridDim.x * blockDim.x * kSymU;
    for (size_t base = (size_t)blockIdx.x * blockDim.x * kSymU + threadIdx.x; base < n; base += stride) {
        unsigned lab[kSymU];
#pragma unroll
        for (int u = 0; u < kSymU; ++u) {
            const size_t i = base + (size_t)u * blockDim.x;
            lab[u] = i < n ? load_label<BPS>(bits, i) : 0u;
        }
#pragma unroll
        for (int u = 0; u < kSymU; ++u) {
            const size_t i = base + (size_t)u * blockDim.x;
            if (i < n) iq[i] = tab[lab[u]];
        }
    }
}

template <typename InT>
__global__ void hard_kernel(size_t n, int bps, const typename Cplx<InT>::type *__restrict__ iq,
                            const double *__restrict__ table, uint8_t *__restrict__ bits)
{
    __shared__ double2 tab[256];
    const int M = 1 << bps;
    for (int i = threadIdx.x; i < M; i += blockDim.x) tab[i] = make_double2(table[2 * i], table[2 * i + 1]);
    __syncthreads();
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const double x = (double)iq[i].x, y = (double)iq[i].y;
        double best = 1e300; int arg = 0;
        for (int c = 0; c < M; ++c) {
            const double dr = x - tab[c].x, di = y - tab[c].y;
            const double d = dr * dr + di * di;
            if (d < best) { best = d; arg = c; }
        }
        for (int b = 0; b < bps; ++b) bits[i * bps + b] = (uint8_t)((arg >> (bps - 1 - b)) & 1);
    }
}

// ---- soft demapper ---------------------------------------------------------------
// One thread computes SPT consecutive symbols (8*SPT bytes in, 4*SPT*BPS bytes out).
// When a thread's output chunk is exactly 16 bytes the float4 stores of a warp are
// already contiguous; larger chunks are staged through shared memory so that every
// global store instruction of a warp still writes 512 contiguous bytes.
template <int BPS> struct GenericLlr {
    const float2 *tab;          // shared memory
    float inv_nv, scale;
    __device__ __forceinline__ void operator()(const float2 s, float (&v)[BPS]) const {
        constexpr int M = 1 << BPS;
        float d0[BPS], d1[BPS];
#pragma unroll
        for (int b = 0; b < BPS; ++b) { d0[b] = 3.0e38f; d1[b] = 3.0e38f; }
#pragma unroll
        for (int c = 0; c < M; ++c) {
            const float dr = s.x - tab[c].x, di = s.y - tab[c].y;
            const float d = fmaf(di, di, dr * dr);
#pragma unroll
            for (int b = 0; b < BPS; ++b) {
                if ((c >> (BPS - 1 - b)) & 1) d1[b] = fminf(d1[b], d);
                else                          d0[b] = fminf(d0[b], d);
            }
        }
#pragma unroll
        for (int b = 0; b < BPS; ++b)
            v[b] = fminf(fmaxf((d0[b] - d1[b]) * inv_nv, -30.f), 30.f) * scale;
    }
};

template <int BPS> struct PwlLlr {          // BPS = 2 * HALF
    const float2 *sc;           // shared memory: float2[2][HALF][nseg]
    int nseg, first_is_q;
    float x0a, invda, x0b, invdb, inv_nv, scale;
    __device__ __forceinline__ void operator()(const float2 s, float (&v)[BPS]) const {
        constexpr int HALF = BPS / 2;
        const float xa = first_is_q ? s.y : s.x, xb = first_is_q ? s.x : s.y;
        const int ua = min(max(__float2int_rd((xa - x0a) * invda), 0), nseg - 1);
        const int ub = min(max(__float2int_rd((xb - x0b) * invdb), 0), nseg - 1);
#pragma unroll
        for (int b = 0; b < HALF; ++b) {
            const float2 ca = sc[b * nseg + ua], cb = sc[(HALF + b) * nseg + ub];
            v[b] = fminf(fmaxf(fmaf(ca.x, xa, ca.y) * inv_nv, -30.f), 30.f) * scale;
            v[HALF + b] = fminf(fmaxf(fmaf(cb.x, xb, cb.y) * inv_nv, -30.f), 30.f) * scale;
        }
    }
};

// Symbol input formats of the demapper: complex64 (float2, the reference's dtype) or bf16x2 (4 bytes per symbol,
// BASELINE north_star "bf16x2 loads of I/Q": widened exactly to float32, then the same arithmetic).
// kCsi: the symbols come with a complex64 channel gain h each (InCsi below).
struct InF32 {
    static constexpr bool kCsi = false;
    typedef float2 sym_t;
    static __device__ __forceinline__ float2 one(const sym_t *p, size_t i) { return __ldcs(p + i); }
    static __device__ __forceinline__ void two(const sym_t *p, size_t i, float2 &a, float2 &b)
    {
        const float4 t = __ldcs(reinterpret_cast<const float4 *>(p + i));
        a = make_float2(t.x, t.y); b = make_float2(t.z, t.w);
    }
};
struct InBf16 {
    static constexpr bool kCsi = false;
    typedef unsigned sym_t;                                // low half = I, high half = Q (a little-endian bf16 pair)
    static __device__ __forceinline__ float2 widen(unsigned w) { return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u)); }
    static __device__ __forceinline__ float2 one(const sym_t *p, size_t i) { return widen(__ldcs(p + i)); }
    static __device__ __forceinline__ void two(const sym_t *p, size_t i, float2 &a, float2 &b)
    {
        const uint2 t = __ldcs(reinterpret_cast<const uint2 *>(p + i));
        a = widen(t.x); b = widen(t.y);
    }
};
// complex64 symbols y with a complex64 gain h each (b200dvb_demap_csi): |y - hc|^2 = |h|^2 |z - c|^2 with
// z = y conj(h) / |h|^2, so each symbol runs the arithmetic of InF32 on z with inv_nv scaled by |h|^2.
struct InCsi : InF32 {
    static constexpr bool kCsi = true;
};

// y <- z = y conj(h) / |h|^2 and inv_nv <- |h|^2 inv_nv.  z is formed in float64, where the products of float32
// values are exact: in float32 the two terms of a component cancel, and the error of the sum is relative to |z|, not
// to the component.  With h = 1 every step is exact, so the symbol's LLRs are those of b200dvb_demap.  Deep fades
// produce no Inf * 0: the float64 z is finite for every finite y and h != 0, h = 0 gives z = 0 and LLR 0, and z's
// components are clamped to +-1e18 (reached only where |y| > 1e18 |h|) so that |z - c|^2 stays finite in float32.
__device__ __forceinline__ void equalise(float2 &y, const float2 h, float &inv_nv)
{
    const double hx = h.x, hy = h.y, h2 = hx * hx + hy * hy;
    const double r = h2 > 0.0 ? 1.0 / h2 : 0.0;
    const double zx = ((double)y.x * hx + (double)y.y * hy) * r, zy = ((double)y.y * hx - (double)y.x * hy) * r;
    y = make_float2((float)fmin(fmax(zx, -1e18), 1e18), (float)fmin(fmax(zy, -1e18), 1e18));
    inv_nv *= (float)h2;
}

template <int BPS, int SPT, class IN, class F>
__device__ __forceinline__ void demap_body(size_t n, const typename IN::sym_t *__restrict__ iq,
                                           const float2 *__restrict__ gain, float *__restrict__ llr,
                                           const F &f, float *stage)
{
    constexpr int CH = BPS * SPT;                       // floats per thread
    constexpr bool kStage = (CH != 4);
    const size_t tile = (size_t)blockDim.x * SPT;       // symbols per block iteration
    for (size_t base = (size_t)blockIdx.x * tile; base < n; base += (size_t)gridDim.x * tile) {
        const size_t i0 = base + (size_t)threadIdx.x * SPT;
        const bool full = base + tile <= n;
        float2 s[SPT], h[SPT];
        if (full && (SPT % 2) == 0) {
#pragma unroll
            for (int j = 0; j < SPT; j += 2) {
                IN::two(iq, i0 + j, s[j], s[j + 1 < SPT ? j + 1 : j]);
                if constexpr (IN::kCsi) InF32::two(gain, i0 + j, h[j], h[j + 1 < SPT ? j + 1 : j]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < SPT; ++j) {
                s[j] = (i0 + j < n) ? IN::one(iq, i0 + j) : make_float2(0.f, 0.f);
                if constexpr (IN::kCsi) h[j] = (i0 + j < n) ? InF32::one(gain, i0 + j) : make_float2(0.f, 0.f);
            }
        }
        float v[SPT][BPS];
#pragma unroll
        for (int j = 0; j < SPT; ++j) {
            if constexpr (IN::kCsi) {
                F g = f;
                equalise(s[j], h[j], g.inv_nv);
                g(s[j], v[j]);
            } else {
                f(s[j], v[j]);
            }
        }
        if (!kStage) {
            if (full || i0 + SPT <= n) {
                const float *p = &v[0][0];
                __stcs(reinterpret_cast<float4 *>(llr + i0 * BPS), make_float4(p[0], p[1], p[2], p[3]));
            } else {
#pragma unroll
                for (int j = 0; j < SPT; ++j)
#pragma unroll
                    for (int b = 0; b < BPS; ++b)
                        if (i0 + j < n) llr[(i0 + j) * BPS + b] = v[j][b];
            }
        } else {
            float *mine = stage + threadIdx.x * CH;
#pragma unroll
            for (int j = 0; j < SPT; ++j)
#pragma unroll
                for (int b = 0; b < BPS; ++b) mine[j * BPS + b] = v[j][b];
            __syncthreads();
            const size_t remain = (n - base) * BPS;                         // floats left from `base`
            const size_t tot = remain < (size_t)blockDim.x * CH ? remain : (size_t)blockDim.x * CH;
            float *out = llr + base * BPS;                                   // 16-byte aligned: tile*BPS % 4 == 0
            for (size_t q = threadIdx.x; q * 4 + 3 < tot; q += blockDim.x)
                __stcs(reinterpret_cast<float4 *>(out) + q, reinterpret_cast<const float4 *>(stage)[q]);
            for (size_t q = (tot / 4) * 4 + threadIdx.x; q < tot; q += blockDim.x) out[q] = stage[q];
            __syncthreads();
        }
    }
}

template <int BPS, int SPT, class IN>
__global__ void __launch_bounds__(kThreads)
demap_generic(size_t n, const typename IN::sym_t *__restrict__ iq, const float *__restrict__ table,
              float inv_nv, float scale, float *__restrict__ llr, const float2 *__restrict__ gain)
{
    constexpr int M = 1 << BPS;
    __shared__ float2 tab[M];
    __shared__ __align__(16) float stage[(BPS * SPT != 4) ? kThreads * BPS * SPT : 4];
    for (int i = threadIdx.x; i < M; i += blockDim.x) tab[i] = make_float2(table[2 * i], table[2 * i + 1]);
    __syncthreads();
    GenericLlr<BPS> f{tab, inv_nv, scale};
    demap_body<BPS, SPT, IN>(n, iq, gain, llr, f, stage);
}

// Per-axis piecewise-linear demapper.  coef: float2[2][HALF][nseg].
template <int HALF, int SPT, class IN>
__global__ void __launch_bounds__(kThreads)
demap_pwl(size_t n, const typename IN::sym_t *__restrict__ iq, const float2 *__restrict__ coef, int nseg,
          float x0a, float invda, float x0b, float invdb, int first_is_q, float inv_nv, float scale,
          float *__restrict__ llr, const float2 *__restrict__ gain)
{
    constexpr int BPS = 2 * HALF;
    __shared__ float2 sc[2 * 4 * 30];
    __shared__ __align__(16) float stage[(BPS * SPT != 4) ? kThreads * BPS * SPT : 4];
    for (int i = threadIdx.x; i < 2 * HALF * nseg; i += blockDim.x) sc[i] = coef[i];
    __syncthreads();
    PwlLlr<BPS> f{sc, nseg, first_is_q, x0a, invda, x0b, invdb, inv_nv, scale};
    demap_body<BPS, SPT, IN>(n, iq, gain, llr, f, stage);
}

// 256QAM (4 bits per axis): one thread per (symbol, axis) writes one float4, so a warp's
// stores are 512 contiguous bytes with no staging; both threads of a symbol read the same
// 8 input bytes (and the same gain, for InCsi).
template <class IN>
__global__ void __launch_bounds__(kThreads)
demap_pwl_axis4(size_t n, const typename IN::sym_t *__restrict__ iq, const float2 *__restrict__ coef, int nseg,
                float x0a, float invda, float x0b, float invdb, int first_is_q, float inv_nv_, float scale,
                float4 *__restrict__ llr4, const float2 *__restrict__ gain)
{
    __shared__ float2 sc[2 * 4 * 30];
    for (int i = threadIdx.x; i < 2 * 4 * nseg; i += blockDim.x) sc[i] = coef[i];
    __syncthreads();
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < 2 * n; t += (size_t)gridDim.x * blockDim.x) {
        float2 s = IN::one(iq, t >> 1);
        float inv_nv = inv_nv_;
        if constexpr (IN::kCsi) equalise(s, InF32::one(gain, t >> 1), inv_nv);
        const int ax = (int)(t & 1);                    // 0: first half of the label, 1: second half
        const float x = (ax ^ first_is_q) ? s.y : s.x;
        const float x0 = ax ? x0b : x0a, invd = ax ? invdb : invda;
        const int u = min(max(__float2int_rd((x - x0) * invd), 0), nseg - 1);
        const float2 *c = sc + ax * 4 * nseg + u;
        float v[4];
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const float2 cc = c[b * nseg];
            v[b] = fminf(fmaxf(fmaf(cc.x, x, cc.y) * inv_nv, -30.f), 30.f) * scale;
        }
        __stcs(llr4 + t, make_float4(v[0], v[1], v[2], v[3]));
    }
}

int grid_for(size_t n, int threads, int per_sm)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    size_t need = (n + threads - 1) / threads;
    size_t cap = (size_t)sms * per_sm;
    return (int)std::max<size_t>(1, std::min(need, cap));
}

}  // namespace

// Host: tabulate (slope, intercept) per axis, bit and segment (see header comment).
int modem_build_pwl(Modem &m)
{
    const int L = m.nlev, half = m.half;
    m.pwl = 0;
    if (!m.separable || L < 2) return B200DVB_OK;
    const int nseg = 2 * L - 2;
    std::vector<float> coef((size_t)2 * half * nseg * 2);
    for (int ax = 0; ax < 2; ++ax) {
        // ax 0 = axis selected by the first half of the label, ax 1 = second half
        std::vector<double> lev(L);
        for (int j = 0; j < L; ++j) {
            const int lab = (ax == 0) ? j * L : j;
            const bool is_q = (ax == 0) ? (m.separable == 2) : (m.separable == 1);
            lev[j] = m.h_table[2 * lab + (is_q ? 1 : 0)];
        }
        std::vector<double> sorted = lev;
        std::sort(sorted.begin(), sorted.end());
        const double span = sorted[L - 1] - sorted[0];
        if (!(span > 0)) return B200DVB_OK;
        const double step = span / (L - 1);
        for (int j = 0; j < L; ++j)
            if (fabs(sorted[j] - (sorted[0] + step * j)) > 1e-6 * span) return B200DVB_OK;   // not uniform: generic path
        const double delta = step * 0.5, x0 = sorted[0];
        m.pwl_x0[ax] = (float)x0;
        m.pwl_invd[ax] = (float)(1.0 / delta);
        for (int b = 0; b < half; ++b)
            for (int u = 0; u < nseg; ++u) {
                const double xc = (u == 0) ? x0 : (u == nseg - 1 ? sorted[L - 1] : x0 + delta * (u + 0.5));
                int a0 = -1, a1 = -1;
                for (int j = 0; j < L; ++j) {
                    const int bit = (j >> (half - 1 - b)) & 1;
                    int &best = bit ? a1 : a0;
                    if (best < 0 || fabs(xc - lev[j]) < fabs(xc - lev[best])) best = j;
                }
                if (a0 < 0 || a1 < 0) return B200DVB_OK;
                const double Xa = lev[a0], Xb = lev[a1];
                const size_t o = (((size_t)ax * half + b) * nseg + u) * 2;
                coef[o] = (float)(2.0 * (Xb - Xa));
                coef[o + 1] = (float)(Xa * Xa - Xb * Xb);
            }
    }
    B2_CUDA(cudaMalloc(&m.d_pwl, coef.size() * sizeof(float)));
    B2_CUDA(cudaMemcpy(m.d_pwl, coef.data(), coef.size() * sizeof(float), cudaMemcpyHostToDevice));
    m.nseg = nseg;
    m.pwl = 1;
    return B200DVB_OK;
}

static int g_map_variant = 0;      // development: 0 = per-order choice, 1 = one symbol per lane, 2 = four per lane
void set_map_variant(int v) { g_map_variant = v; }

int launch_map(const Modem &m, size_t n, const uint8_t *bits, void *iq, int out_f64, cudaStream_t s)
{
    if (n == 0) return B200DVB_OK;
    // complex64 out, both pointers 32-byte aligned, one of the six orders of the reference: the word-load kernel;
    // anything else: the generic one
    if (!out_f64 && ((reinterpret_cast<uintptr_t>(bits) | reinterpret_cast<uintptr_t>(iq)) & 31) == 0) {
        const int gridg = grid_for((n + 3) / 4, kThreads * kMapU, 8), grids = grid_for(n, kThreads * kSymU, 8);
        float2 *o = (float2 *)iq;
        const bool grp = g_map_variant == 2 || (g_map_variant == 0 && m.bps >= 3);   // measured per order: profiles/r02_mapper.txt
        switch (m.bps) {
        case 1: if (grp) map_words_kernel<1><<<gridg, kThreads, 0, s>>>(n, bits, m.d_table64, o); else map_sym_kernel<1><<<grids, kThreads, 0, s>>>(n, bits, m.d_table64, o); break;
        case 2: if (grp) map_words_kernel<2><<<gridg, kThreads, 0, s>>>(n, bits, m.d_table64, o); else map_sym_kernel<2><<<grids, kThreads, 0, s>>>(n, bits, m.d_table64, o); break;
        case 4: if (grp) map_words_kernel<4><<<gridg, kThreads, 0, s>>>(n, bits, m.d_table64, o); else map_sym_kernel<4><<<grids, kThreads, 0, s>>>(n, bits, m.d_table64, o); break;
        case 8: if (grp) map_words_kernel<8><<<gridg, kThreads, 0, s>>>(n, bits, m.d_table64, o); else map_sym_kernel<8><<<grids, kThreads, 0, s>>>(n, bits, m.d_table64, o); break;
        case 3: map_words_kernel<3><<<gridg, kThreads, 0, s>>>(n, bits, m.d_table64, o); break;
        case 6: map_words_kernel<6><<<gridg, kThreads, 0, s>>>(n, bits, m.d_table64, o); break;
        default: map_kernel<float><<<grid_for(n, kThreads, 8), kThreads, 0, s>>>(n, m.bps, bits, m.d_table64, o); break;
        }
        B2_CUDA(cudaGetLastError());
        return B200DVB_OK;
    }
    const int grid = grid_for(n, kThreads, 8);
    if (out_f64) map_kernel<double><<<grid, kThreads, 0, s>>>(n, m.bps, bits, m.d_table64, (double2 *)iq);
    else         map_kernel<float><<<grid, kThreads, 0, s>>>(n, m.bps, bits, m.d_table64, (float2 *)iq);
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

int launch_hard(const Modem &m, size_t n, const void *iq, int in_f64, uint8_t *bits, cudaStream_t s)
{
    if (n == 0) return B200DVB_OK;
    const int grid = grid_for(n, kThreads, 8);
    if (in_f64) hard_kernel<double><<<grid, kThreads, 0, s>>>(n, m.bps, (const double2 *)iq, m.d_table64, bits);
    else        hard_kernel<float><<<grid, kThreads, 0, s>>>(n, m.bps, (const float2 *)iq, m.d_table64, bits);
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

template <class IN>
static int launch_demap_t(const Modem &m, size_t n, const void *iq_, const float2 *gain, float noise_var, float scale,
                          float *llr, cudaStream_t s)
{
    if (n == 0) return B200DVB_OK;
    const typename IN::sym_t *iq = (const typename IN::sym_t *)iq_;
    if ((reinterpret_cast<uintptr_t>(iq_) & 15) || (reinterpret_cast<uintptr_t>(gain) & 15) ||
        (reinterpret_cast<uintptr_t>(llr) & 15))
        return B200DVB_EINVAL;                               // vector loads/stores need 16-byte alignment
    const float nv = noise_var > 0.005f ? noise_var : 0.005f;      // test_sdr_with_coding.py:202
    const float inv_nv = 1.0f / nv;
    if (m.pwl) {
        const float2 *coef = (const float2 *)m.d_pwl;
        const int fq = (m.separable == 2);
#define PWL(H, S) demap_pwl<H, S, IN><<<grid_for(n, kThreads * S, 8), kThreads, 0, s>>>(                \
        n, iq, coef, m.nseg, m.pwl_x0[0], m.pwl_invd[0], m.pwl_x0[1], m.pwl_invd[1], fq, inv_nv, scale, llr, gain)
        switch (m.half) {
        case 1: PWL(1, 2); break;
        case 2: PWL(2, 1); break;
        case 3: PWL(3, 2); break;
        case 4:
            demap_pwl_axis4<IN><<<grid_for(2 * n, kThreads, 8), kThreads, 0, s>>>(
                n, iq, coef, m.nseg, m.pwl_x0[0], m.pwl_invd[0], m.pwl_x0[1], m.pwl_invd[1], fq, inv_nv, scale,
                reinterpret_cast<float4 *>(llr), gain);
            break;
        default: return B200DVB_ENOSPEC;
        }
#undef PWL
    } else {
        switch (m.bps) {
#define GEN(B, S) demap_generic<B, S, IN><<<grid_for(n, kThreads * S, 8), kThreads, 0, s>>>(n, iq, m.d_table32, inv_nv, scale, llr, gain)
        case 1: GEN(1, 4); break;
        case 2: GEN(2, 2); break;
        case 3: GEN(3, 4); break;
        case 4: GEN(4, 1); break;
        case 6: GEN(6, 2); break;
        case 8: GEN(8, 1); break;
#undef GEN
        default: return B200DVB_ENOSPEC;
        }
    }
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

int launch_demap(const Modem &m, size_t n, const void *iq, float noise_var, float scale, float *llr, cudaStream_t s)
{
    return launch_demap_t<InF32>(m, n, iq, nullptr, noise_var, scale, llr, s);
}
int launch_demap_bf16(const Modem &m, size_t n, const void *iq, float noise_var, float scale, float *llr, cudaStream_t s)
{
    return launch_demap_t<InBf16>(m, n, iq, nullptr, noise_var, scale, llr, s);
}
int launch_demap_csi(const Modem &m, size_t n, const void *iq, const void *gain, float noise_var, float scale,
                     float *llr, cudaStream_t s)
{
    return launch_demap_t<InCsi>(m, n, iq, (const float2 *)gain, noise_var, scale, llr, s);
}

}  // namespace b200dvb
