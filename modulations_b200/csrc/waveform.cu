// waveform.cu — the stage on either side of the mapper / demapper (SURVEY §8(f) N4):
// root-raised-cosine pulse shaping of symbols (modulators.py:85-100: upfirdn(h, syms, up=sps))
// and the receive matched filter + symbol-rate decimation (modulators.py:102-117:
// convolve(samples, h, 'full')[2*delay::sps]).  Both are HBM-streaming FIRs over complex64:
//
//   pulse shaping   8 B of symbol in, 8*sps B of samples out per symbol: write bound.  Polyphase:
//                   out[q*sps + p] = sum_j s[q-j] * h[p + j*sps]; a thread owns one output sample,
//                   the <= ceil(ntaps/sps) symbols it needs are shared by the sps threads around it
//                   (L1); for sps 2/4/8 a thread owns a whole symbol period instead (see below).
//   matched filter  8*sps B of samples in, 8 B of symbol out per symbol: read bound.  A block owns
//                   512 consecutive outputs (two per thread); the samples they span are staged in shared memory
//                   PHASE-MAJOR ([i mod sps][i / sps]): for a given tap every thread of a warp then
//                   reads consecutive 8-byte words (no bank conflicts — sample-major staging would be
//                   a 2*sps-word stride), and every input sample is read from HBM once (plus the taps' reach
//                   at tile boundaries: 48 of 4140 samples at sps 8).
//
// The taps arrive as a HOST float64 array (the reference's rrc_filter), are rounded once to float32 and travel in the
// kernel's parameter space (constant bank).
// Arithmetic: float32 FMAs, taps rounded once to float32; the reference convolves in float64, so
// parity is a stated tolerance (tests/test_gpu_waveform.py), not bit-exactness.
#include "common.cuh"

#include <string.h>

namespace b200dvb {

namespace {

constexpr int kMfThreads = 256;     // one or two outputs per thread (two share the constant reads and the loop)

// Taps travel as a kernel argument: the parameter space is a constant bank, so a tap (and, for the matched filter,
// the staged offset of the sample it multiplies) is a uniform constant-cache read, not a shared-memory wavefront.
struct FirTaps {
    float h[kMaxFirTaps];
    int off[kMaxFirTaps];           // matched filter: staged offset of tap t for thread 0 (see matched_filter_kernel)
};

__global__ void __launch_bounds__(256)
pulse_shape_kernel(size_t n_sym, const float2 *__restrict__ sym, const __grid_constant__ FirTaps T, int ntaps,
                   int sps, size_t n_out, float2 *__restrict__ out)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_out; i += (size_t)gridDim.x * blockDim.x) {
        const size_t q = i / sps;
        const int p = (int)(i - q * sps);
        float ar = 0.f, ai = 0.f;
        for (int j = 0, t = p; t < ntaps; ++j, t += sps) {
            if (q >= (size_t)j && q - j < n_sym) {
                const float2 s = __ldg(sym + (q - j));
                ar = fmaf(s.x, T.h[t], ar);
                ai = fmaf(s.y, T.h[t], ai);
            }
        }
        out[i] = make_float2(ar, ai);
    }
}

// Compile-time sps: a thread owns ALL sps output samples of one symbol period q — the Q = ceil(ntaps/sps) symbols
// they depend on are loaded once (coalesced: consecutive threads, consecutive symbols) and the sps*Q complex MACs run
// out of registers; the thread's sps samples are 8*sps contiguous bytes, stored 16 B at a time.  Only taps below ntaps
// take part: an FMA with a zero-padded tap would turn an Inf or NaN symbol into a NaN in outputs whose window (the real
// taps) does not contain it.
template <int SPS, int QT>
__global__ void __launch_bounds__(256)
pulse_shape_sps_kernel(size_t n_sym, const float2 *__restrict__ sym, const __grid_constant__ FirTaps T, int ntaps,
                       size_t n_out, float2 *__restrict__ out)
{
    // QT = compile-time bound of the symbols an output period depends on (ceil(ntaps / SPS) <= QT).  Interior periods
    // (every one of the QT symbols exists) take a path without per-load bounds checks and 64-bit compares: the round-1
    // kernel spent 75 % of its issue slots on the ALU pipe doing exactly those (profiles/r02_waveform_ncu.txt) and was
    // ALU-bound, not HBM-bound.
    const size_t nq = (n_out + SPS - 1) / SPS;                      // symbol periods that hold output samples
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (size_t)gridDim.x * blockDim.x) {
        float2 s[QT];
        if (q >= (size_t)(QT - 1) && q < n_sym) {
            const float2 *p = sym + q;
#pragma unroll
            for (int j = 0; j < QT; ++j) s[j] = __ldg(p - j);
        } else {
#pragma unroll
            for (int j = 0; j < QT; ++j)
                s[j] = (q >= (size_t)j && q - j < n_sym) ? __ldg(sym + (q - j)) : make_float2(0.f, 0.f);
        }
        float2 acc[SPS];
#pragma unroll
        for (int p = 0; p < SPS; ++p) acc[p] = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < QT; ++j) {
            const int real = ntaps - j * SPS;                       // taps j*SPS + p with p < real exist (uniform)
            if (real >= SPS) {
#pragma unroll
                for (int p = 0; p < SPS; ++p) {
                    acc[p].x = fmaf(s[j].x, T.h[j * SPS + p], acc[p].x);
                    acc[p].y = fmaf(s[j].y, T.h[j * SPS + p], acc[p].y);
                }
            } else if (real > 0) {
#pragma unroll
                for (int p = 0; p < SPS; ++p) {
                    if (p < real) {
                        acc[p].x = fmaf(s[j].x, T.h[j * SPS + p], acc[p].x);
                        acc[p].y = fmaf(s[j].y, T.h[j * SPS + p], acc[p].y);
                    }
                }
            }
        }
        float2 *o = out + q * SPS;
        if ((q + 1) * SPS <= n_out && (SPS % 4) == 0) {             // whole period in range: 32-byte stores = full sectors
#pragma unroll                                                      // (out is 32-byte aligned on this path)
            for (int p = 0; p < SPS; p += 4)
                asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                             :: "l"(o + p), "f"(acc[p].x), "f"(acc[p].y), "f"(acc[p + 1].x), "f"(acc[p + 1].y),
                                "f"(acc[p + 2 < SPS ? p + 2 : p].x), "f"(acc[p + 2 < SPS ? p + 2 : p].y),
                                "f"(acc[p + 3 < SPS ? p + 3 : p].x), "f"(acc[p + 3 < SPS ? p + 3 : p].y) : "memory");
        } else if ((q + 1) * SPS <= n_out && (SPS % 2) == 0) {
#pragma unroll
            for (int p = 0; p < SPS; p += 2)
                *reinterpret_cast<float4 *>(o + p) = make_float4(acc[p].x, acc[p].y, acc[p + 1].x, acc[p + 1].y);
        } else {
#pragma unroll
            for (int p = 0; p < SPS; ++p)
                if (q * SPS + p < n_out) o[p] = acc[p];
        }
    }
}

// out[m] = sum_t h[t] * x[start + m*sps - t],  x[i] = 0 outside [0, n).
// Staging is phase-major: sample i of the tile sits at xs[((i - base) mod sps) * pitch + (i - base) / sps] with base a
// multiple of sps, so that for one tap the threads of a warp (consecutive outputs, i.e. samples sps apart) read
// consecutive 8-byte words.  The staged index of the sample that tap t multiplies for the tile's first output is
// r0 - t with r0 = ntaps - 1 + ((start - ntaps + 1) mod sps) — the same for every tile — so its offset T.off[t] is a
// per-launch constant the host tabulates.
// NOUT outputs per thread: 2 (a 512-output tile) unless the tile's staging exceeds the shared memory a block may take
// (sps >= 50, or sps 49 with more than 343 taps); then 1 (a 256-output tile, half the staging).
template <int NOUT>
__global__ void __launch_bounds__(kMfThreads, 4)
matched_filter_kernel(size_t n, const float2 *__restrict__ x, const __grid_constant__ FirTaps T, int ntaps,
                      int sps, long long start, size_t n_out, float2 *__restrict__ out, int pitch, int r0)
{
    constexpr int kTile = NOUT * kMfThreads;
    extern __shared__ float2 xs[];                                  // [sps][pitch], phase-major
    const bool even = (kMfThreads % sps) == 0;                      // then a thread's phase never changes while staging
    const bool fast = even && (sps % 2) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
    for (size_t m0 = (size_t)blockIdx.x * kTile; m0 < n_out; m0 += (size_t)gridDim.x * kTile) {
        const long long base = start + (long long)m0 * sps - r0;    // staged index 0 <-> sample `base` (a multiple of sps)
        const int span = (kTile - 1) * sps + r0 + 1;
        __syncthreads();                                            // previous tile fully consumed
        if (fast && base >= 0 && (size_t)(base + span + 1) <= n) {
            // interior tile, even sps, 16-byte aligned input: 16-byte loads (two samples: phases ph, ph + 1 of the same
            // position), all of a thread's loads in flight before its first shared-memory store, 32-bit indexing
            const float2 *xb = x + base;
            const int ph = (2 * threadIdx.x) % sps, step = 2 * kMfThreads / sps;
            const int pos0 = (2 * threadIdx.x) / sps;
            constexpr int kIt = 5;                                  // loads in flight per thread and pass
            for (int r = 2 * threadIdx.x, pos = pos0; r < span; r += kIt * 2 * kMfThreads, pos += kIt * step) {
                float4 buf[kIt];
#pragma unroll
                for (int u = 0; u < kIt; ++u)
                    if (r + u * 2 * kMfThreads < span) buf[u] = __ldg(reinterpret_cast<const float4 *>(xb + r + u * 2 * kMfThreads));
#pragma unroll
                for (int u = 0; u < kIt; ++u)
                    if (r + u * 2 * kMfThreads < span) {
                        xs[ph * pitch + pos + u * step] = make_float2(buf[u].x, buf[u].y);
                        xs[(ph + 1) * pitch + pos + u * step] = make_float2(buf[u].z, buf[u].w);
                    }
            }
        } else if (even) {
            // eight loads in flight per thread before the first shared-memory store: the staging pass is the only
            // place this kernel touches HBM, and a rolled load-store loop would pay one memory latency per iteration
            const int ph = threadIdx.x % sps, step = kMfThreads / sps;
            int pos = threadIdx.x / sps;
            for (int r = threadIdx.x; r < span; r += 8 * kMfThreads, pos += 8 * step) {
                float2 buf[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const long long i = base + r + u * kMfThreads;
                    buf[u] = (r + u * kMfThreads < span && i >= 0 && (size_t)i < n) ? __ldg(x + i) : make_float2(0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    if (r + u * kMfThreads < span) xs[ph * pitch + pos + u * step] = buf[u];
            }
        } else {
            for (int r = threadIdx.x; r < span; r += kMfThreads) {
                const long long i = base + r;
                xs[(r % sps) * pitch + r / sps] = (i >= 0 && (size_t)i < n) ? __ldg(x + i) : make_float2(0.f, 0.f);
            }
        }
        __syncthreads();
        const float2 *xt = xs + threadIdx.x;                        // outputs m0 + tid (and m0 + tid + 256)
        float ar = 0.f, ai = 0.f, br = 0.f, bi = 0.f;
        for (int t = 0; t < ntaps; ++t) {
            const int o = T.off[t];
            const float hh = T.h[t];
            const float2 v0 = xt[o];
            ar = fmaf(v0.x, hh, ar); ai = fmaf(v0.y, hh, ai);
            if (NOUT == 2) {
                const float2 v1 = xt[o + kMfThreads];
                br = fmaf(v1.x, hh, br); bi = fmaf(v1.y, hh, bi);
            }
        }
        const size_t m = m0 + threadIdx.x;
        if (m < n_out) out[m] = make_float2(ar, ai);
        if (NOUT == 2 && m + kMfThreads < n_out) out[m + kMfThreads] = make_float2(br, bi);
    }
}


// ---- matched filter, four CONSECUTIVE outputs per thread, phase PAIRS, double-buffered (the default path) ---------
// profiles/r01_mf_ncu.txt: with one LDS.64 per tap and output the tap loop read 392 B of shared memory per output
// (49 taps) against 72 B of HBM: the LSU data pipe, not HBM, was the wall (80 % busy, 55 % of the copy bandwidth).
//  * Consecutive outputs of one phase row read consecutive staged positions, so a thread that owns outputs
//    4 tid .. 4 tid + 3 needs, per row, a window of (taps per row + 3) entries for 4 x (taps per row) MACs.
//  * Two neighbouring samples (phases 2 pp, 2 pp + 1 of one position) are staged as ONE 16-byte entry: a 16-byte
//    global read lands with one 16-byte shared-memory write, and one LDS.128 of the tap loop serves two phase rows:
//    11 LDS.128 per phase pair and four outputs at 49 taps / sps 8 — 176 B per output instead of 392.
//  * To keep the window loads conflict-free each pair row is staged in FOUR interleaved sub-rows, position q at
//    [q mod 4][q div 4]: entry e of every thread's window then sits at [(b+e) mod 4][(b+e) div 4 + tid], consecutive
//    16-byte words across the warp.
//  * Staging is asynchronous (cp.async, 16 bytes) into the other of two buffers while the current tile is computed:
//    the load-then-compute phases of a block no longer alternate, HBM requests stay in flight all the time.
// The host tabulates, per pair row, the first staged position its taps touch and both phases' taps in position order
// (zero padded to QW, with a mask of the real ones).  Even sps only; odd sps takes matched_filter_kernel.
constexpr int kMf4Threads = 128;
constexpr int kMf4Tile = 4 * kMf4Threads;
constexpr int kMf4MaxPairs = 16;    // sps <= 32
constexpr int kMf4MaxQ = 9;
struct FirRows {
    float h[kMf4MaxPairs][2][kMf4MaxQ + 1];   // [pair row][phase in pair][position within the pair row's window]
    unsigned real[kMf4MaxPairs][2];           // bit q set: h[..][..][q] is a tap, not padding
    int base[kMf4MaxPairs];
};
__device__ __forceinline__ int mf4_idx(int pos, int q4) { return (pos & 3) * q4 + (pos >> 2); }

// acc[j] += (x_j, y_j) * h for the four outputs when `real`: predicated FMAs.  Written as a C++ branch, ptxas made
// it one (with the tap's constant load moved inside it), which cost the matched filter 5 % of its bandwidth.
__device__ __forceinline__ void fma4_if(unsigned real, float2 (&acc)[4], float x0, float y0, float x1, float y1,
                                        float x2, float y2, float x3, float y3, float h)
{
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %17, 0;\n\t"
        "@p fma.rn.f32 %0, %8, %16, %0;\n\t@p fma.rn.f32 %1, %9, %16, %1;\n\t"
        "@p fma.rn.f32 %2, %10, %16, %2;\n\t@p fma.rn.f32 %3, %11, %16, %3;\n\t"
        "@p fma.rn.f32 %4, %12, %16, %4;\n\t@p fma.rn.f32 %5, %13, %16, %5;\n\t"
        "@p fma.rn.f32 %6, %14, %16, %6;\n\t@p fma.rn.f32 %7, %15, %16, %7;\n\t}"
        : "+f"(acc[0].x), "+f"(acc[0].y), "+f"(acc[1].x), "+f"(acc[1].y),
          "+f"(acc[2].x), "+f"(acc[2].y), "+f"(acc[3].x), "+f"(acc[3].y)
        : "f"(x0), "f"(y0), "f"(x1), "f"(y1), "f"(x2), "f"(y2), "f"(x3), "f"(y3), "f"(h), "r"(real));
}

template <int QW, bool ASYNC>
__global__ void __launch_bounds__(kMf4Threads, ASYNC ? 3 : 6)
matched_filter4_kernel(size_t n, const float2 *__restrict__ x, const __grid_constant__ FirRows T, int sps,
                       long long start, size_t n_out, float2 *__restrict__ out, int pitch, int q4, int r0, int span,
                       int pair_shift)
{
    extern __shared__ float4 xs4[];                                 // [2 buffers (ASYNC) | 1][sps / 2][4][q4]
    const int npair = sps >> 1;
    const int bufsz = npair * pitch;
    const bool aligned = (reinterpret_cast<uintptr_t>(x) & 15) == 0;
    const int span2 = span >> 1;                                    // 16-byte entries per tile (span is a multiple of sps)
    auto tile_base = [&](size_t m0) { return start + (long long)m0 * sps - r0; };   // sample of staged position 0, phase 0
    auto interior = [&](size_t m0) {
        const long long base = tile_base(m0);
        return aligned && base >= 0 && (size_t)(base + span) <= n && (base & 1) == 0;
    };
    auto stage_async = [&](size_t m0, float4 *buf) {
        const float4 *xb = reinterpret_cast<const float4 *>(x + tile_base(m0));
        const unsigned sbase = (unsigned)__cvta_generic_to_shared(buf);
#pragma unroll 4
        for (int i = threadIdx.x; i < span2; i += kMf4Threads) {
            const int pp = pair_shift >= 0 ? (i & (npair - 1)) : i % npair, pos = pair_shift >= 0 ? (i >> pair_shift) : i / npair;
            const unsigned d = sbase + 16u * (unsigned)(pp * pitch + mf4_idx(pos, q4));
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(d), "l"(xb + i) : "memory");
        }
    };
    // interior tile staged through registers: every 16-byte load of a thread in flight before its first store
    auto stage_regs = [&](size_t m0, float4 *buf) {
        const float4 *xb = reinterpret_cast<const float4 *>(x + tile_base(m0));
        constexpr int kIt = 6;
        for (int i0 = threadIdx.x; i0 < span2; i0 += kIt * kMf4Threads) {
            float4 v[kIt];
#pragma unroll
            for (int u = 0; u < kIt; ++u)
                if (i0 + u * kMf4Threads < span2) v[u] = __ldg(xb + i0 + u * kMf4Threads);
#pragma unroll
            for (int u = 0; u < kIt; ++u) {
                const int i = i0 + u * kMf4Threads;
                if (i < span2) {
                    const int pp = pair_shift >= 0 ? (i & (npair - 1)) : i % npair, pos = pair_shift >= 0 ? (i >> pair_shift) : i / npair;
                    buf[pp * pitch + mf4_idx(pos, q4)] = v[u];
                }
            }
        }
    };
    auto stage_sync = [&](size_t m0, float4 *buf) {
        const long long base = tile_base(m0);
        for (int i = threadIdx.x; i < span2; i += kMf4Threads) {
            const int pp = i % npair, pos = i / npair;
            const long long i0 = base + 2 * (long long)i, i1 = i0 + 1;
            const float2 a = (i0 >= 0 && (size_t)i0 < n) ? __ldg(x + i0) : make_float2(0.f, 0.f);
            const float2 c = (i1 >= 0 && (size_t)i1 < n) ? __ldg(x + i1) : make_float2(0.f, 0.f);
            buf[pp * pitch + mf4_idx(pos, q4)] = make_float4(a.x, a.y, c.x, c.y);
        }
    };
    const size_t stride = (size_t)gridDim.x * kMf4Tile;
    size_t m0 = (size_t)blockIdx.x * kMf4Tile;
    int cur = 0;
    if (ASYNC) {
        if (m0 < n_out && interior(m0)) stage_async(m0, xs4);
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    for (; m0 < n_out; m0 += stride, cur ^= ASYNC ? 1 : 0) {
        float4 *buf = xs4 + cur * bufsz;
        if (ASYNC) {
            const size_t m1 = m0 + stride;
            if (m1 < n_out && interior(m1)) stage_async(m1, xs4 + (cur ^ 1) * bufsz);   // the other buffer was released by the
            asm volatile("cp.async.commit_group;" ::: "memory");                         // barrier at the end of the last tile
            if (!interior(m0)) stage_sync(m0, buf);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            if (interior(m0)) stage_regs(m0, buf); else stage_sync(m0, buf);
        }
        __syncthreads();
        float2 acc[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[j] = make_float2(0.f, 0.f);
        const float4 *xt = buf + threadIdx.x;
        for (int pp = 0; pp < npair; ++pp) {
            const int b = T.base[pp];
            const unsigned ra = T.real[pp][0], rb = T.real[pp][1];
            const float4 *row = xt + pp * pitch;
            float4 w[QW + 3];
#pragma unroll
            for (int e = 0; e < QW + 3; ++e) w[e] = row[mf4_idx(b + e, q4)];
            // padded taps take no part: 0 x (an Inf or NaN sample outside this output's window) would be NaN
#pragma unroll
            for (int q = 0; q < QW; ++q) {
                fma4_if(ra & (1u << q), acc, w[q].x, w[q].y, w[q + 1].x, w[q + 1].y, w[q + 2].x, w[q + 2].y,
                        w[q + 3].x, w[q + 3].y, T.h[pp][0][q]);
                fma4_if(rb & (1u << q), acc, w[q].z, w[q].w, w[q + 1].z, w[q + 1].w, w[q + 2].z, w[q + 2].w,
                        w[q + 3].z, w[q + 3].w, T.h[pp][1][q]);
            }
        }
        const size_t m = m0 + 4 * (size_t)threadIdx.x;
        if (m + 4 <= n_out && (reinterpret_cast<uintptr_t>(out) & 31) == 0) {
            asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                         :: "l"(out + m), "f"(acc[0].x), "f"(acc[0].y), "f"(acc[1].x), "f"(acc[1].y),
                            "f"(acc[2].x), "f"(acc[2].y), "f"(acc[3].x), "f"(acc[3].y) : "memory");
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (m + j < n_out) out[m + j] = acc[j];
        }
        __syncthreads();                                            // this tile's buffer may be refilled now
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

int fill_taps(FirTaps &T, const double *taps_h, int ntaps)
{
    if (ntaps < 1 || ntaps > kMaxFirTaps) return B200DVB_EINVAL;
    for (int i = 0; i < kMaxFirTaps; ++i) { T.h[i] = i < ntaps ? (float)taps_h[i] : 0.f; T.off[i] = 0; }
    return B200DVB_OK;
}

}  // namespace

// development: 0 = default (four outputs per thread, phase pairs, staged through registers), 1 = the same with
// double-buffered cp.async staging, 2 = the round-1 kernel (two strided outputs per thread)
static int g_mf_variant = 0;
void set_mf_variant(int v) { g_mf_variant = v; }

int launch_pulse_shape(size_t n_sym, const void *sym, const double *taps_h, int ntaps, int sps, void *out, cudaStream_t s)
{
    if (n_sym == 0) return B200DVB_OK;
    FirTaps T;
    if (int rc = fill_taps(T, taps_h, ntaps)) return rc;
    const size_t n_out = (n_sym - 1) * (size_t)sps + ntaps;
    int dev = 0, sms = 148;
    B2_CUDA(cudaGetDevice(&dev));
    B2_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int Q = (ntaps + sps - 1) / sps;
    const bool al16 = (reinterpret_cast<uintptr_t>(out) & 31) == 0;   // 32-byte stores on the per-period path
    const float2 *sy = reinterpret_cast<const float2 *>(sym);
    float2 *o = reinterpret_cast<float2 *>(out);
    if ((sps == 8 || sps == 4 || sps == 2) && Q <= 16 && al16) {
        size_t blocks = ((n_out + sps - 1) / sps + 255) / 256;
        if (blocks > (size_t)sms * 16) blocks = (size_t)sms * 16;
#define B2_PS(S, QQ) pulse_shape_sps_kernel<S, QQ><<<(unsigned)blocks, 256, 0, s>>>(n_sym, sy, T, ntaps, n_out, o)
#define B2_PSQ(S) do { if (Q <= 4) B2_PS(S, 4); else if (Q <= 7) B2_PS(S, 7); else if (Q <= 10) B2_PS(S, 10); else B2_PS(S, 16); } while (0)
        if (sps == 8)      B2_PSQ(8);
        else if (sps == 4) B2_PSQ(4);
        else               B2_PSQ(2);
#undef B2_PSQ
#undef B2_PS
        B2_CUDA(cudaGetLastError());
        return B200DVB_OK;
    }
    size_t blocks = (n_out + 255) / 256;
    if (blocks > (size_t)sms * 16) blocks = (size_t)sms * 16;
    pulse_shape_kernel<<<(unsigned)blocks, 256, 0, s>>>(n_sym, sy, T, ntaps, sps, n_out, o);
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

int launch_matched_filter(size_t n, const void *x, const double *taps_h, int ntaps, int sps, long long start,
                          size_t n_out, void *out, cudaStream_t s)
{
    if (n_out == 0) return B200DVB_OK;
    if (ntaps < 1 || ntaps > kMaxFirTaps) return B200DVB_EINVAL;
    int dev = 0, sms = 148;
    B2_CUDA(cudaGetDevice(&dev));
    B2_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int Qrow = (ntaps + sps - 1) / sps;                       // taps per phase row (at most)
    if (Qrow + 1 <= kMf4MaxQ && (sps % 2) == 0 && sps / 2 <= kMf4MaxPairs) {
        // four consecutive outputs per thread, phase pairs, double-buffered (matched_filter4_kernel)
        const long long lo4 = start - (ntaps - 1);
        const int r04 = ntaps - 1 + (int)(((lo4 % sps) + sps) % sps);   // staged sample index of the first output's tap 0
        FirRows R;
        memset(&R, 0, sizeof R);
        int omax = 0, qw = 1;
        for (int pp = 0; pp < sps / 2; ++pp) {
            int bmin = 1 << 30, bmax = -1;
            for (int t = 0; t < ntaps; ++t)
                if (((r04 - t) % sps) >> 1 == pp) {
                    const int o = (r04 - t) / sps;
                    if (o < bmin) bmin = o;
                    if (o > bmax) bmax = o;
                }
            if (bmax < 0) { bmin = 0; bmax = 0; }                   // a pair row without taps (ntaps < sps)
            R.base[pp] = bmin;
            for (int t = 0; t < ntaps; ++t)
                if (((r04 - t) % sps) >> 1 == pp) {
                    const int ph = (r04 - t) % sps & 1, q = (r04 - t) / sps - bmin;
                    R.h[pp][ph][q] = (float)taps_h[t];
                    R.real[pp][ph] |= 1u << q;
                }
            if (bmin > omax) omax = bmin;
            if (bmax - bmin + 1 > qw) qw = bmax - bmin + 1;
        }
        const int qsel = qw <= 4 ? 4 : qw <= 6 ? 6 : qw <= 7 ? 7 : qw <= 8 ? 8 : 9;
        // Bank layout of the staging stores.  A 16-byte shared-memory access is served per QUARTER warp (8 consecutive
        // lanes = 8 consecutive 16-byte entries of the input = 8 / npair consecutive positions x npair phase pairs),
        // and those 8 must fall into 8 different 16-byte bank groups: entry (pp, pos) sits at pp * pitch + (pos mod 4)
        // * q4 + pos div 4, so the residues of q4 and of the row pitch mod 8 are chosen per npair (the first version
        // used one choice for all and ran at 2 wavefronts per store and 82 % LSU load: profiles/r02_waveform_ncu.txt).
        const int np = sps / 2;
        const int q4_res = np == 1 ? 2 : 1;                          // npair 1: 8 positions -> {0,2,4,6} + {0,1}
        const int pitch_res = np == 2 ? 4 : np == 4 ? 2 : 1;         // npair 2: {0..3} + {0,4}; 4: {0,1} + {0,2,4,6}; >= 8: odd pitch
        int q4 = (kMf4Tile + omax + qsel + 3 + 3) / 4 + 1;          // entries per sub-row: the tile + the windows' reach
        while ((q4 & 7) != q4_res) ++q4;
        int pitch4 = 4 * q4;
        while ((pitch4 & 7) != pitch_res) ++pitch4;
        const bool use_async = g_mf_variant == 1;
        const size_t smem4 = (size_t)(use_async ? 2 : 1) * (sps / 2) * pitch4 * sizeof(float4);
        int pair_shift = -1;
        for (int b = 0; b < 5; ++b) if ((sps / 2) == (1 << b)) pair_shift = b;
        const int span4 = (omax + kMf4Tile - 1 + qsel + 3) * sps;   // all positions any window reads, in samples
        if (smem4 <= 200 * 1024 && g_mf_variant != 2) {
            size_t blocks = (n_out + kMf4Tile - 1) / kMf4Tile;
            const size_t per_sm = use_async ? 3 : 6;                // persistent blocks per SM
            if (blocks > (size_t)sms * per_sm) blocks = (size_t)sms * per_sm;
            const float2 *xi = reinterpret_cast<const float2 *>(x);
            float2 *oo = reinterpret_cast<float2 *>(out);
#define B2_MF4K(Q, A)                                                                                                  \
            do {                                                                                                       \
                if (smem4 > 48 * 1024)                                                                                 \
                    B2_CUDA(cudaFuncSetAttribute(matched_filter4_kernel<Q, A>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4)); \
                matched_filter4_kernel<Q, A><<<(unsigned)blocks, kMf4Threads, smem4, s>>>(n, xi, R, sps, start, n_out, oo, pitch4, q4, r04, span4, pair_shift); \
            } while (0)
#define B2_MF4(Q) do { if (use_async) B2_MF4K(Q, true); else B2_MF4K(Q, false); } while (0)
            if (qsel == 4) B2_MF4(4); else if (qsel == 6) B2_MF4(6); else if (qsel == 7) B2_MF4(7); else if (qsel == 8) B2_MF4(8); else B2_MF4(9);
#undef B2_MF4
#undef B2_MF4K
            B2_CUDA(cudaGetLastError());
            return B200DVB_OK;
        }
    }
    FirTaps T;
    if (int rc = fill_taps(T, taps_h, ntaps)) return rc;
    // staged positions per phase: the tile's outputs + the taps' reach + the rounding of the origin; odd pitch (in
    // 8-byte words) spreads the sps rows of the staging pass over the banks.  A 512-output tile fits for every
    // sps <= 48; above that the 256-output tile keeps every (sps <= 64, ntaps <= 448) within 136 KB.
    auto pitch_for = [&](int tile) { return (tile + (ntaps + sps - 1) / sps + 2) | 1; };
    const int nout = (size_t)sps * pitch_for(2 * kMfThreads) * sizeof(float2) <= 200 * 1024 ? 2 : 1;
    const int tile = nout * kMfThreads, pitch = pitch_for(tile);
    const long long lo = start - (ntaps - 1);                       // first sample of the first output
    const int r0 = ntaps - 1 + (int)(((lo % sps) + sps) % sps);     // its staged index with the origin on a multiple of sps
    for (int t = 0; t < ntaps; ++t) T.off[t] = ((r0 - t) % sps) * pitch + (r0 - t) / sps;
    const size_t smem = (size_t)sps * pitch * sizeof(float2);
    size_t blocks = (n_out + tile - 1) / tile;
    if (blocks > (size_t)sms * 8) blocks = (size_t)sms * 8;
    const float2 *xi = reinterpret_cast<const float2 *>(x);
    float2 *oo = reinterpret_cast<float2 *>(out);
#define B2_MFK(K)                                                                                                      \
    do {                                                                                                               \
        if (smem > 48 * 1024)                                                                                          \
            B2_CUDA(cudaFuncSetAttribute(matched_filter_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        matched_filter_kernel<K><<<(unsigned)blocks, kMfThreads, smem, s>>>(n, xi, T, ntaps, sps, start, n_out, oo, pitch, r0); \
    } while (0)
    if (nout == 2) B2_MFK(2); else B2_MFK(1);
#undef B2_MFK
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

}  // namespace b200dvb
