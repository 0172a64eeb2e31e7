// decode_quad.cu — batched max-log-MAP decoder for the 16-state duo-binary
// circular turbo code, bit-exact with the reference's mixed fp64/fp32 arithmetic
// (reference: dvb_rcs2_turbo.py:116-281 bcjr_max_log_map, :464-537 decode).
//
// Mapping (DESIGN.md §4 has the derivation and the numbers):
//   * One CTA = 2 warps = 8 frames.  Warp 0 runs the forward (alpha) recursion,
//     warp 1 the backward (beta) recursion of the same 8 frames.
//   * One frame and direction = a "quad" of 4 lanes, 4 states per lane.  The
//     trellis is a shift register (ns = 2*(s&7) + dk), so two trellis steps are
//     lane-local (a radix-4 butterfly) and the 16 metrics are re-dealt by a 4x4
//     transpose through shared memory every second step.  The per-step
//     normalisation by state 0 (:178-179) is a 4-wide shuffle broadcast.
//   * Branch metrics are kept in shared memory as ONE 32-byte record per step:
//     the 8 merged values GP[c] = max(g(00), g(11)), GM[c] = max(g(01), g(10)) for
//     the four (W,Y) classes c.  The reference trellis has parallel branches
//     (SURVEY §0 F3) and fp32 rounding is monotone, so max(fl(a+g1), fl(a+g2)) ==
//     fl(a + max(g1,g2)) exactly: the 4-way ACS collapses to 2-way.  The smaller
//     member of each pair is -GP[~c] / -GM[~c], so the extrinsic stage recovers
//     all 16 signed branch metrics from the same record.
//   * The reference stores a full alpha and a full beta array (:163,:200).  Here
//     the two warps meet in the middle: each stores a checkpoint every 8 steps on
//     its way in, and on the way out re-computes the other direction 8 steps at a
//     time into registers (exact: same operations, same order).  Shared memory
//     per frame is 32 B/step + 2 x 64 B per 8 steps instead of 160 B/step.
//   * a-priori / extrinsic values stay float64 (:233-234, :267-279) in an
//     L2-resident global workspace; interleaving is a gather through the host's
//     perm / inv_perm tables (never assumed bijective, SURVEY §0 F2).
#include "common.cuh"

#include <stdlib.h>

namespace b200dvb {

namespace {

struct QuadArgs {
    QuadGeom g;
    int B, iterations, n_groups;
    double sf_inner, sf_last;
    const int16_t *tab;
    // full decode
    const void *llr;      // [B][llr_stride] elements of the kernel's LlrT (float32, binary16 or int8)
    long long llr_stride;
    int32_t *bits;
    uint32_t *packed;
    const uint8_t *ref_bits;
    unsigned long long *counters;
    // single SISO
    const float *LcA, *LcB, *LcW, *LcY;
    const double *LaA, *LaB;
    double *LeA, *LeB;
    double siso_sf;
    int vec_ab, vec_wy;   // two-element loads of (A,B) / (W,Y) pairs are legal for this codec + stride
    int timed;            // development: add this launch's per-phase cycles to g_phase_cycles
    // workspace
    double2 *Le1, *Le2, *Y;
    float *grec;          // geometry `grec`: [CTA][frame slot][rec_stride] branch-metric records
    float llr_scale;      // int8 element q is the LLR q * llr_scale (last: the other members keep their offsets)
    float *app;           // full decode: [B][2N] a-posteriori LLRs (float2 per couple) or NULL; last, for the same reason
};

// phase timers (SM cycles summed over CTAs): 0 prep, 1 recursion in (pass 1 + pass 2 to the
// crossing point), 2 recursion out (windows + extrinsic), 3 epilogue, 4 hard decision, 5 CTA total
__device__ unsigned long long g_phase_cycles[8];

constexpr int kXchFloats = 144;
constexpr int kBatch = 4;          // positions per thread whose loads are issued together (prep / epilogue)   // one exchange buffer (8 quads, skewed), see xbase()

// flat position index -> (frame slot f, step k); magic = floor(2^32 / N) + 1 (exact for i*N < 2^32)
__device__ __forceinline__ void split_pos(int i, int N, unsigned magic, int &f, int &k)
{
    f = (int)__umulhi((unsigned)i, magic);
    k = i - f * N;
}

// The same for the global-record geometry: a warp takes 8 frames x 4 consecutive steps, so that its record stores (and
// the reads of the extrinsic maxima) cover 4 x 256 contiguous bytes of the [group][step][8 frames] layout, and its LLR /
// Y / extrinsic accesses 32 or 64 contiguous bytes per frame (N is a multiple of 4).
template <bool GREC>
__device__ __forceinline__ void pos_of(int i, int N, unsigned magic, int &f, int &k)
{
    split_pos(i, N, magic, f, k);
    if (GREC) {
        const int idx = (f & 7) * N + k;
        k = 4 * (idx >> 5) + (idx & 3);
        f = (f & ~7) + ((idx >> 2) & 7);
    }
}

__device__ __forceinline__ int cls2(int s)
{   // 2 * class(s): class = 2*(s0^s1^s2) + s1  (w = A^B^s0^s1^s2, y = A^B^s1)
    int s0 = s & 1, s1 = (s >> 1) & 1, s2 = (s >> 2) & 1;
    return 2 * (2 * (s0 ^ s1 ^ s2) + s1);
}

struct Lane {
    int q;         // quad (frame within CTA, or the scratch area for idle quads)
    int p;         // lane within quad
    int oA[2];     // float offset of butterfly A's (g0,g1) pair inside a record, by parity of k
    int oB[2];     // same for butterfly B
    int xw;        // float offset of this lane's float4 slot in an exchange buffer
    int xr;        // float offset of column p, row 0 of this quad in an exchange buffer
    int role_word; // record word this lane writes in the extrinsic reduction
};

// exchange buffer: quad q occupies 16 floats at 16q + 4(q>>1): float4 stores of a
// quarter-warp and the column reads of a full warp are both bank-conflict free.
__device__ __forceinline__ int xbase(int q) { return 16 * q + 4 * (q >> 1); }

// Branch-metric pairs of one lane for two consecutive steps (even k, then k+1), and
// the complementary-class pairs the extrinsic stage needs.
struct G2 { float2 a0, b0, a1, b1; };
struct GH { float2 gA, gB, hA, hB; };

template <int SS>       // SS: floats between the records of consecutive steps (8: frame-major; 64: 8 frames interleaved)
struct Recs {           // per-lane pointers into this frame's records
    const float *pA0, *pB0, *pA1, *pB1;     // (g0,g1) of butterfly A/B in record k (even) / k+1
    int dA0, dB0, dA1, dB1;                 // float distance from the g pair to the h pair (class ~c)
    __device__ __forceinline__ G2 pair(int k_even) const {
        G2 g;
        g.a0 = *reinterpret_cast<const float2 *>(pA0 + k_even * SS);
        g.b0 = *reinterpret_cast<const float2 *>(pB0 + k_even * SS);
        g.a1 = *reinterpret_cast<const float2 *>(pA1 + k_even * SS);
        g.b1 = *reinterpret_cast<const float2 *>(pB1 + k_even * SS);
        return g;
    }
    template <int KPAR> __device__ __forceinline__ void one(int k, float2 &gA, float2 &gB) const {
        const int e = (k - KPAR) * SS;
        gA = *reinterpret_cast<const float2 *>((KPAR ? pA1 : pA0) + e);
        gB = *reinterpret_cast<const float2 *>((KPAR ? pB1 : pB0) + e);
    }
    template <int KPAR> __device__ __forceinline__ GH ext(int k) const {
        const int e = (k - KPAR) * SS;
        const float *a = (KPAR ? pA1 : pA0) + e, *b = (KPAR ? pB1 : pB0) + e;
        GH g;
        g.gA = *reinterpret_cast<const float2 *>(a);
        g.gB = *reinterpret_cast<const float2 *>(b);
        g.hA = *reinterpret_cast<const float2 *>(a + (KPAR ? dA1 : dA0));
        g.hB = *reinterpret_cast<const float2 *>(b + (KPAR ? dB1 : dB0));
        return g;
    }
};

__device__ __forceinline__ void norm4(float (&r)[4])
{   // alpha[k+1,:] -= alpha[k+1,0]  (dvb_rcs2_turbo.py:178-179, :212-213)
    float n = __shfl_sync(0xffffffffu, r[0], 0, 4);
    r[0] = __fsub_rn(r[0], n); r[1] = __fsub_rn(r[1], n);
    r[2] = __fsub_rn(r[2], n); r[3] = __fsub_rn(r[3], n);
}

// One trellis step on the 4 states of a lane: butterfly A on (r0,r2) with (g0,g1) =
// (gA.x,gA.y), butterfly B on (r1,r3) with (g0,g1) = (gB.y,gB.x); then normalise.
__device__ __forceinline__ void stepg(float (&r)[4], const float2 gA, const float2 gB)
{
    float o0 = fmaxf(__fadd_rn(r[0], gA.x), __fadd_rn(r[2], gA.y));
    float o1 = fmaxf(__fadd_rn(r[0], gA.y), __fadd_rn(r[2], gA.x));
    float o2 = fmaxf(__fadd_rn(r[1], gB.y), __fadd_rn(r[3], gB.x));
    float o3 = fmaxf(__fadd_rn(r[1], gB.x), __fadd_rn(r[3], gB.y));
    r[0] = o0; r[1] = o1; r[2] = o2; r[3] = o3;
    norm4(r);
}

// 4x4 transpose inside each quad through shared memory.
__device__ __forceinline__ void transpose_fwd(float (&r)[4], float *xb, const Lane &L)
{
    *reinterpret_cast<float4 *>(xb + L.xw) = make_float4(r[0], r[1], r[2], r[3]);
    __syncwarp();
    r[0] = xb[L.xr]; r[1] = xb[L.xr + 4]; r[2] = xb[L.xr + 8]; r[3] = xb[L.xr + 12];
}
__device__ __forceinline__ void transpose_bwd(float (&r)[4], float *xb, const Lane &L)
{   // same transpose applied to the register tuple (r0, r2, r1, r3)
    *reinterpret_cast<float4 *>(xb + L.xw) = make_float4(r[0], r[2], r[1], r[3]);
    __syncwarp();
    r[0] = xb[L.xr]; r[2] = xb[L.xr + 4]; r[1] = xb[L.xr + 8]; r[3] = xb[L.xr + 12];
}

// Recursion checkpoints (one float4 per lane): in shared memory, or — when that frees
// enough room for a fourth group of frames — in tensor memory.  TMEM is lane-private,
// but the alpha and beta warp of a group sit in the same lane quadrant (warp ids g and
// g + 4), so lane l of one reads what lane l of the other wrote (tcgen05.st/ld .32x32b).
template <bool TMEM> struct Ckpt;
template <> struct Ckpt<false> {
    float *base;                                   // this lane's float4 slot of checkpoint 0
    __device__ __forceinline__ void store(int idx, const float (&r)[4]) const {
        *reinterpret_cast<float4 *>(base + idx * 16) = make_float4(r[0], r[1], r[2], r[3]);
    }
    __device__ __forceinline__ void load(int idx, float (&r)[4]) const {
        const float4 c = *reinterpret_cast<const float4 *>(base + idx * 16);
        r[0] = c.x; r[1] = c.y; r[2] = c.z; r[3] = c.w;
    }
    __device__ __forceinline__ void publish() const {}
    __device__ __forceinline__ void acquire() const {}
};
template <> struct Ckpt<true> {
    unsigned taddr;                                // TMEM address of column 0 in this warp's lane quadrant
    __device__ __forceinline__ void store(int idx, const float (&r)[4]) const {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
                     ::"r"(taddr + 4u * idx), "r"(__float_as_uint(r[0])), "r"(__float_as_uint(r[1])),
                       "r"(__float_as_uint(r[2])), "r"(__float_as_uint(r[3])) : "memory");
    }
    __device__ __forceinline__ void load(int idx, float (&r)[4]) const {
        unsigned a, b, c, d;
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(taddr + 4u * idx) : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        r[0] = __uint_as_float(a); r[1] = __uint_as_float(b); r[2] = __uint_as_float(c); r[3] = __uint_as_float(d);
    }
    __device__ __forceinline__ void publish() const {      // before the CTA barrier that hands checkpoints over
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __device__ __forceinline__ void acquire() const {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
};

struct Xch {            // two alternating exchange buffers: one __syncwarp per use
    float *b0, *b1;
    __device__ __forceinline__ float *next() { float *t = b0; b0 = b1; b1 = t; return t; }
};

// Extrinsic for step k (dvb_rcs2_turbo.py:239-248) fused with the owning
// direction's recursion step.  a = alpha[k], b = beta[k+1] in matching layouts.
// Writes (U0, U3, V1, V2) = max over states of the four branch-pair metrics into
// words 0..3 of record k (gamma[k] is dead after this step; its values were
// loaded into `G` before the call).
template <int KPAR, bool OWN_ALPHA>
__device__ __forceinline__ void ext_step(float (&a)[4], float (&b)[4], const GH G, float *rec,
                                         const Lane &L, Xch &x)
{
    const float2 gA = G.gA, gB = G.gB, hA = G.hA, hB = G.hB;
    // butterfly A: x = (a0,a2) y = (b0,b2) g = (gA.x,gA.y) h = (hA.x,hA.y)
    const float a0g0 = __fadd_rn(a[0], gA.x), a2g0 = __fadd_rn(a[2], gA.x);
    const float a0g1 = __fadd_rn(a[0], gA.y), a2g1 = __fadd_rn(a[2], gA.y);
    float AE0 = fmaxf(__fadd_rn(a0g0, b[0]), __fadd_rn(a2g0, b[2]));
    float AE1 = fmaxf(__fadd_rn(a0g1, b[2]), __fadd_rn(a2g1, b[0]));
    float AF0 = fmaxf(__fadd_rn(__fsub_rn(a[0], hA.x), b[0]), __fadd_rn(__fsub_rn(a[2], hA.x), b[2]));
    float AF1 = fmaxf(__fadd_rn(__fsub_rn(a[0], hA.y), b[2]), __fadd_rn(__fsub_rn(a[2], hA.y), b[0]));
    // butterfly B: x = (a1,a3) y = (b1,b3) g = (gB.y,gB.x) h = (hB.y,hB.x)
    const float a1g0 = __fadd_rn(a[1], gB.y), a3g0 = __fadd_rn(a[3], gB.y);
    const float a1g1 = __fadd_rn(a[1], gB.x), a3g1 = __fadd_rn(a[3], gB.x);
    float BE0 = fmaxf(__fadd_rn(a1g0, b[1]), __fadd_rn(a3g0, b[3]));
    float BE1 = fmaxf(__fadd_rn(a1g1, b[3]), __fadd_rn(a3g1, b[1]));
    float BF0 = fmaxf(__fadd_rn(__fsub_rn(a[1], hB.y), b[1]), __fadd_rn(__fsub_rn(a[3], hB.y), b[3]));
    float BF1 = fmaxf(__fadd_rn(__fsub_rn(a[1], hB.x), b[3]), __fadd_rn(__fsub_rn(a[3], hB.x), b[1]));
    float4 T;
    if (KPAR == 0) {   // even k: butterfly B has t = 1 -> its roles are (V1,U0,V2,U3)
        T = make_float4(fmaxf(AE0, BE1), fmaxf(AE1, BE0), fmaxf(AF0, BF1), fmaxf(AF1, BF0));
    } else {           // odd k: both butterflies share t = p1 (resolved by the reader)
        T = make_float4(fmaxf(AE0, BE0), fmaxf(AE1, BE1), fmaxf(AF0, BF0), fmaxf(AF1, BF1));
    }
    // own recursion step (shares the x+g sums when the owner is alpha)
    if (OWN_ALPHA) {
        float o0 = fmaxf(a0g0, a2g1), o1 = fmaxf(a0g1, a2g0);
        float o2 = fmaxf(a1g0, a3g1), o3 = fmaxf(a1g1, a3g0);
        a[0] = o0; a[1] = o1; a[2] = o2; a[3] = o3;
        norm4(a);
    } else {
        stepg(b, gA, gB);
    }
    // cross-lane max by reduce-scatter over the quad: lane p ends up with role p of
    // (U0,V1,U3,V2).  On odd k lanes 2,3 (p1 = 1) hold their partials as (V1,U0,V2,U3),
    // so what they send and keep is swapped pairwise.  Pure register traffic: no
    // barrier, and independent steps of a window overlap their shuffles.
    const bool p1 = (L.p & 2) != 0, p0 = (L.p & 1) != 0;
    float s0, s1, k0, k1;
    if (KPAR == 0) {
        s0 = p1 ? T.x : T.z; s1 = p1 ? T.y : T.w;
        k0 = p1 ? T.z : T.x; k1 = p1 ? T.w : T.y;
    } else {
        s0 = p1 ? T.y : T.z; s1 = p1 ? T.x : T.w;
        k0 = p1 ? T.w : T.x; k1 = p1 ? T.z : T.y;
    }
    k0 = fmaxf(k0, __shfl_xor_sync(0xffffffffu, s0, 2));
    k1 = fmaxf(k1, __shfl_xor_sync(0xffffffffu, s1, 2));
    const float snd = p0 ? k0 : k1, kp = p0 ? k1 : k0;
    const float v = fmaxf(kp, __shfl_xor_sync(0xffffffffu, snd, 1));
    rec[L.role_word] = v;
}

// ---------------------------------------------------------------------------
// One SISO over the frames of this CTA.  Records must be complete and a
// __syncthreads() must have been executed before the call; on return (after the
// trailing __syncthreads) words 0..3 of every record hold (U0,U3,V1,V2).
// Branch metrics are always loaded one step (or one step pair) ahead of their use:
// the exchange-buffer stores in between would otherwise pin the loads behind them.
// ---------------------------------------------------------------------------
template <int LEN, int SS, class CK>
__device__ __forceinline__ void window_alpha(float (&r)[4], float *grec, const Recs<SS> &R,
                                             const CK &ck, int ck_idx, int j0, const Lane &L, Xch &x)
{
    float wb[LEN][4];
    ck.load(ck_idx, wb[LEN - 1]);
    float2 gA, gB, nA, nB;
    R.template one<(LEN - 1) & 1>(j0 + LEN - 1, gA, gB);
#pragma unroll
    for (int i = LEN - 2; i >= 0; --i) {   // beta[j0+2+i] -> beta[j0+1+i] uses gamma[j0+1+i]
#pragma unroll
        for (int t = 0; t < 4; ++t) wb[i][t] = wb[i + 1][t];
        if (i > 0) {
            if (i & 1) R.template one<1>(j0 + i, nA, nB); else R.template one<0>(j0 + i, nA, nB);
        }
        stepg(wb[i], gA, gB);
        if (((i + 1) & 1) == 0) transpose_bwd(wb[i], x.next(), L);
        gA = nA; gB = nB;
    }
    GH G = R.template ext<0>(j0), Gn = G;
#pragma unroll
    for (int i = 0; i < LEN; ++i) {
        float *rec = grec + (j0 + i) * SS;
        if (i + 1 < LEN) {
            if ((i + 1) & 1) Gn = R.template ext<1>(j0 + i + 1); else Gn = R.template ext<0>(j0 + i + 1);
        }
        if (i & 1) {
            ext_step<1, true>(r, wb[i], G, rec, L, x);
            transpose_fwd(r, x.next(), L);
        } else {
            ext_step<0, true>(r, wb[i], G, rec, L, x);
        }
        G = Gn;
    }
}

template <int SS, class CK>
__device__ __forceinline__ void window_beta(float (&r)[4], float *grec, const Recs<SS> &R,
                                            const CK &ck, int ck_idx, int j0, const Lane &L, Xch &x)
{
    float wa[kWin][4];
    ck.load(ck_idx, wa[0]);
    float2 gA, gB, nA, nB;
    R.template one<0>(j0, gA, gB);
#pragma unroll
    for (int i = 1; i < kWin; ++i) {       // alpha[j0+i-1] -> alpha[j0+i] uses gamma[j0+i-1]
#pragma unroll
        for (int t = 0; t < 4; ++t) wa[i][t] = wa[i - 1][t];
        if (i + 1 < kWin) {
            if (i & 1) R.template one<1>(j0 + i, nA, nB); else R.template one<0>(j0 + i, nA, nB);
        }
        stepg(wa[i], gA, gB);
        if ((i - 1) & 1) transpose_fwd(wa[i], x.next(), L);
        gA = nA; gB = nB;
    }
    GH G = R.template ext<1>(j0 + kWin - 1), Gn = G;
#pragma unroll
    for (int i = kWin - 1; i >= 0; --i) {
        float *rec = grec + (j0 + i) * SS;
        if (i > 0) {
            if ((i - 1) & 1) Gn = R.template ext<1>(j0 + i - 1); else Gn = R.template ext<0>(j0 + i - 1);
        }
        if (i & 1) {
            ext_step<1, false>(wa[i], r, G, rec, L, x);
        } else {
            ext_step<0, false>(wa[i], r, G, rec, L, x);
            transpose_bwd(r, x.next(), L);
        }
        G = Gn;
    }
}

// Records in global memory (GREC, long frames): [group][step][8 frames][8 floats], so that the records of one step of
// a warp's 8 frames are 256 contiguous bytes.  The recursion warps do not read them from global memory (through L1
// every first touch of a sector was a miss whatever prefetch.global.L1 was issued ahead: measured, 51 % L1 hit rate,
// long-scoreboard stalls 37 %) but from a private shared-memory ring that cp.async keeps kFeedAhead step pairs ahead:
// one 16-byte LDGSTS per lane and step pair.  The loops read "their" pair at its ring position, the frame-major code
// path reads it at its step index: the same Recs arithmetic serves both.
constexpr int kGrecStep = 64;        // floats between the records of consecutive steps
constexpr int kRingSteps = 32;       // ring capacity in steps (8 KB per recursion warp)
constexpr int kFeedAhead = 8;        // step pairs in flight ahead of the one being read (kFeedAhead + 2 <= kRingSteps / 2)

__device__ __forceinline__ void q_cpa16(void *dst, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void q_cpa_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int K> __device__ __forceinline__ void q_cpa_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(K) : "memory"); }

// Step pairs of the "in" phase in the order the warp consumes them: alpha 0, 2, .. N-2 (pass 1), 0, 2, .. M (pass 2 and
// its last look-ahead); beta N-2, N-4, .. 0 (pass 1), N-2, .. (pass 2).
struct Feed {
    float *ring;              // this warp's ring
    const float *src;         // this group's records in global memory
    int N, lane, beta, total, iss, rd;
    __device__ __forceinline__ int pair_k(int i) const {
        const int h = N >> 1;
        const int j = i < h ? i : i - h;
        return beta ? N - 2 - 2 * j : 2 * j;
    }
    __device__ __forceinline__ void issue() {
        if (iss < total) {
            int k = pair_k(iss);
            k = k < 0 ? 0 : k;
            const int st = ((iss * 2) & (kRingSteps - 1)) + (lane >> 4);
            q_cpa16(ring + st * kGrecStep + (lane & 15) * 4, src + (size_t)(k + (lane >> 4)) * kGrecStep + (lane & 15) * 4);
        }
        q_cpa_commit();       // (an empty group keeps the wait arithmetic uniform)
        ++iss;
    }
    __device__ __forceinline__ void start() {
        iss = rd = 0;
        for (int i = 0; i <= kFeedAhead; ++i) issue();
    }
    // ring step index of the next pair to read; its data is complete when this returns
    __device__ __forceinline__ int next_slot() {
        issue();
        q_cpa_wait<kFeedAhead + 1>();
        __syncwarp();
        const int st = (rd * 2) & (kRingSteps - 1);
        ++rd;
        return st;
    }
};

// does every lane of the warp hold, bit for bit, what checkpoint idx holds?
template <class CK>
__device__ __forceinline__ bool rejoined(const CK &ck, int idx, const float (&r)[4])
{
    float o[4];
    ck.load(idx, o);
    const bool eq = __float_as_uint(o[0]) == __float_as_uint(r[0]) && __float_as_uint(o[1]) == __float_as_uint(r[1]) &&
                    __float_as_uint(o[2]) == __float_as_uint(r[2]) && __float_as_uint(o[3]) == __float_as_uint(r[3]);
    return __all_sync(0xffffffffu, eq);
}

template <bool PF, class CK>
__device__ __forceinline__ void siso_core(const QuadGeom &g, float *gam, const CK &ck, float *xch, float *rings,
                                          int warp, int xslot, const Lane &L, long long &t_mid)
{
    const int N = g.N, M = g.M;
    constexpr int SS = PF ? kGrecStep : 8;
    float *ggrp = gam + (size_t)(L.q >> 3) * N * kGrecStep;                  // (GREC) this group's records
    float *grec = PF ? ggrp + (L.q & 7) * 8 : gam + L.q * g.rec_stride;     // this frame's records (written by ext_step)
    float *ring = rings + xslot * (kRingSteps * kGrecStep);
    float *rbase = PF ? ring + (L.q & 7) * 8 : grec;                        // what the recursion reads
    Xch x{xch + xslot * 2 * kXchFloats, xch + xslot * 2 * kXchFloats + kXchFloats};
    Recs<SS> R;
    R.pA0 = rbase + L.oA[0];      R.pB0 = rbase + L.oB[0];
    R.pA1 = rbase + SS + L.oA[1]; R.pB1 = rbase + SS + L.oB[1];
    R.dA0 = 6 - 2 * L.oA[0]; R.dB0 = 6 - 2 * L.oB[0];
    R.dA1 = 6 - 2 * L.oA[1]; R.dB1 = 6 - 2 * L.oB[1];
    Feed F;
    F.ring = ring; F.src = ggrp; F.N = N; F.lane = threadIdx.x & 31; F.beta = warp;
    F.total = warp ? (N >> 1) + ((N - M) >> 1) + 1 : (N >> 1) + (M >> 1) + 1;
    if (PF) F.start();
    // the pair at step k (frame-major records) or the next pair of the feed (ring)
    auto pair_at = [&](int k) -> G2 { return PF ? R.pair(F.next_slot()) : R.pair(k); };
    float r[4] = {0.f, 0.f, 0.f, 0.f};
    if (warp == 0) {
        // pass 1 (convergence, :167-179) from zeros, then alpha[0] <- alpha[N] (:182-183)
        // GREC (long frames): pass 1 leaves its own checkpoints over [0, M) and keeps alpha[M]; pass 2 then stops at the
        // first checkpoint where the 8 frames of the warp hold, bit for bit, what pass 1 held there — from that point
        // on it would only reproduce pass 1 (same records, deterministic recursion), whose checkpoints are in place.
        // Exact (a warp that never re-joins runs all of pass 2); the second laps re-join after ~50 steps on average
        // (decode_lat.cu), pass 2 is N/2 steps.
        float rM[4] = {0.f, 0.f, 0.f, 0.f};
        G2 cur = pair_at(0);
#pragma unroll 2
        for (int k = 0; k < N; k += 2) {
            const G2 nxt = pair_at(k + 2 < N ? k + 2 : 0);
            if (PF) {
                if ((k & (kWin - 1)) == 0 && k < M) ck.store(k / kWin, r);
                if (k == M) { rM[0] = r[0]; rM[1] = r[1]; rM[2] = r[2]; rM[3] = r[3]; }
            }
            stepg(r, cur.a0, cur.b0);
            stepg(r, cur.a1, cur.b1);
            transpose_fwd(r, x.next(), L);
            cur = nxt;
        }
        if (PF) ck.publish();                               // (the stores above are complete before pass 2 reads them back)
        // pass 2 up to the crossing point M (a multiple of kWin), checkpoint every kWin steps
        for (int k = 0; k < M; k += kWin) {
            if (PF && rejoined(ck, k / kWin, r)) { r[0] = rM[0]; r[1] = rM[1]; r[2] = rM[2]; r[3] = rM[3]; break; }
            ck.store(k / kWin, r);
#pragma unroll
            for (int j = 0; j < kWin; j += 2) {
                const G2 nxt = pair_at(k + j + 2);         // k + j + 2 <= M < N
                stepg(r, cur.a0, cur.b0);
                stepg(r, cur.a1, cur.b1);
                transpose_fwd(r, x.next(), L);
                cur = nxt;
            }
        }
    } else {
        // beta pass 1 (:203-213): j = N..2, then beta[N] <- beta[0] (:216-217)
        float rM[4] = {0.f, 0.f, 0.f, 0.f};
        const int ragged = (N - M) & (kWin - 1);           // 0 or 4
        G2 cur = pair_at(N - 2);
#pragma unroll 2
        for (int j = N; j > 0; j -= 2) {
            const G2 nxt = pair_at(j >= 4 ? j - 4 : N - 2);
            if (PF) {                                       // (GREC: checkpoints of pass 1 over (M, N], see the alpha warp)
                if (j > M && ((j - M) & (kWin - 1)) == 0) ck.store(g.nckA + (j - M) / kWin - 1, r);
                if (ragged && j == N) ck.store(g.nckA + g.nckB - 1, r);
                if (j == M) { rM[0] = r[0]; rM[1] = r[1]; rM[2] = r[2]; rM[3] = r[3]; }
            }
            stepg(r, cur.a1, cur.b1);      // gamma[j-1] (odd)
            stepg(r, cur.a0, cur.b0);      // gamma[j-2] (even)
            transpose_bwd(r, x.next(), L);
            cur = nxt;
        }
        if (PF) ck.publish();
        // pass 2 down to M: a checkpoint at the end of every alpha-warp window
        int j = N;
        bool done = false;
        if (ragged) {
            if (PF && rejoined(ck, g.nckA + g.nckB - 1, r)) done = true;
            else {
                ck.store(g.nckA + g.nckB - 1, r);
                for (int t = 0; t < ragged; t += 2, j -= 2) {
                    const G2 nxt = pair_at(j - 4);
                    stepg(r, cur.a1, cur.b1);
                    stepg(r, cur.a0, cur.b0);
                    transpose_bwd(r, x.next(), L);
                    cur = nxt;
                }
            }
        }
        for (; !done && j > M; j -= kWin) {
            if (PF && rejoined(ck, g.nckA + (j - M) / kWin - 1, r)) { done = true; break; }
            ck.store(g.nckA + (j - M) / kWin - 1, r);
#pragma unroll
            for (int t = 0; t < kWin; t += 2) {
                const G2 nxt = pair_at(j - t - 4);          // >= M - 4 >= 4
                stepg(r, cur.a1, cur.b1);
                stepg(r, cur.a0, cur.b0);
                transpose_bwd(r, x.next(), L);
                cur = nxt;
            }
        }
        if (done) { r[0] = rM[0]; r[1] = rM[1]; r[2] = rM[2]; r[3] = rM[3]; }
    }
    if (PF) { q_cpa_wait<0>(); __syncwarp(); }
    ck.publish();
    __syncthreads();
    ck.acquire();
    t_mid = clock64();
    // "out" phase.  GREC: the 8 records of a window are staged in the ring (two 2 KB halves, the next window's copy in
    // flight while this one computes); R is re-based so that step k of the window reads ring step (half * 8 + k - j0).
    auto stage = [&](int j0, int len, int half) {
        if (PF) {
            const int lane = threadIdx.x & 31;
#pragma unroll
            for (int q = 0; q < kWin / 2; ++q) {
                const int st = 2 * q + (lane >> 4);
                if (st < len)
                    q_cpa16(ring + (half * kWin + st) * kGrecStep + (lane & 15) * 4,
                            ggrp + (size_t)(j0 + st) * kGrecStep + (lane & 15) * 4);
            }
            q_cpa_commit();
        }
    };
    auto rebased = [&](int j0, int half) -> Recs<SS> {
        Recs<SS> W = R;
        if (PF) {
            const int d = (half * kWin - j0) * kGrecStep;
            W.pA0 += d; W.pB0 += d; W.pA1 += d; W.pB1 += d;
        }
        return W;
    };
    if (warp == 0) {
        int half = 0;
        stage(M, N - M >= kWin ? kWin : 4, 0);
        for (int w = 0; w < g.nckB; ++w) {
            const int j0 = M + w * kWin;
            if (PF) {
                __syncwarp();
                const int jn = j0 + kWin;
                if (w + 1 < g.nckB) stage(jn, N - jn >= kWin ? kWin : 4, half ^ 1); else q_cpa_commit();
                q_cpa_wait<1>();
                __syncwarp();
            }
            const Recs<SS> W = rebased(j0, half);
            if (N - j0 >= kWin) window_alpha<kWin, SS>(r, grec, W, ck, g.nckA + w, j0, L, x);
            else                window_alpha<4, SS>(r, grec, W, ck, g.nckA + w, j0, L, x);
            half ^= 1;
        }
    } else {
        int half = 0;
        stage((g.nckA - 1) * kWin, kWin, 0);
        for (int w = g.nckA - 1; w >= 0; --w) {
            if (PF) {
                __syncwarp();
                if (w > 0) stage((w - 1) * kWin, kWin, half ^ 1); else q_cpa_commit();
                q_cpa_wait<1>();
                __syncwarp();
            }
            const Recs<SS> W = rebased(w * kWin, half);
            window_beta<SS>(r, grec, W, ck, w, w * kWin, L, x);
            half ^= 1;
        }
    }
    if (PF) q_cpa_wait<0>();
    __syncthreads();
}

// Branch-metric record for one trellis step (dvb_rcs2_turbo.py:131-160): float64
// left-to-right sums rounded once to float32, then merged per (W,Y) class.
__device__ __forceinline__ void make_record(int k, double YA, double YB, float pW, float pY,
                                            float4 &lo4, float4 &hi4)
{
    const double a = YA * 0.5, b = YB * 0.5;
    const double w = (double)pW * 0.5, y = (double)pY * 0.5;
    const double s = __dadd_rn(a, b), d = __dsub_rn(a, b);
    float P[4], Mv[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const double sw = (c & 2) ? -w : w, sy = (c & 1) ? -y : y;
        P[c] = __double2float_rn(__dadd_rn(__dadd_rn(s, sw), sy));
        Mv[c] = __double2float_rn(__dadd_rn(__dadd_rn(d, sw), sy));
    }
    float o[8];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const float GP = fmaxf(P[c], -P[3 - c]);
        const float GM = fmaxf(Mv[3 - c], -Mv[c]);
        const bool swap = (k & 1) && (((c >> 1) ^ c) & 1);
        o[2 * c] = swap ? GM : GP;
        o[2 * c + 1] = swap ? GP : GM;
    }
    lo4 = make_float4(o[0], o[1], o[2], o[3]);
    hi4 = make_float4(o[4], o[5], o[6], o[7]);
}

// Extrinsic epilogue for one step (dvb_rcs2_turbo.py:250-279).
__device__ __forceinline__ double2 make_extrinsic(const float4 uv, double YA, double YB, double sf)
{
    const double a = YA * 0.5, b = YB * 0.5;
    const bool sP = __dadd_rn(a, b) < 0.0, sM = __dsub_rn(a, b) < 0.0;
    const float app0 = sP ? uv.y : uv.x, app3 = sP ? uv.x : uv.y;
    const float app1 = sM ? uv.w : uv.z, app2 = sM ? uv.z : uv.w;
    const float LA = __fsub_rn(fmaxf(app0, app1), fmaxf(app2, app3));
    const float LB = __fsub_rn(fmaxf(app0, app2), fmaxf(app1, app3));
    double ea = __dmul_rn(__dsub_rn((double)LA, YA), sf);
    double eb = __dmul_rn(__dsub_rn((double)LB, YB), sf);
    ea = ea > 300.0 ? 300.0 : ea; ea = ea < -300.0 ? -300.0 : ea;
    eb = eb > 300.0 ? 300.0 : eb; eb = eb < -300.0 ? -300.0 : eb;
    return make_double2(ea, eb);
}

template <bool SISO_ONLY, bool TMEM, bool GREC = false, class LlrT = float>
__global__ void __launch_bounds__(kMaxCtaThreads)
quad_kernel(const QuadArgs A)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const QuadGeom g = A.g;
    const int N = g.N;
    const int tid = threadIdx.x, lane = tid & 31;
    const int NT = blockDim.x;                       // recursion warps + helper warps (prep / epilogue only)
    const int wid = tid >> 5;
    // warp roles.  smem checkpoints: alpha warps 0..G-1, beta warps G..2G-1.  TMEM checkpoints
    // (G <= 4): alpha warp g and beta warp 4+g share lane quadrant g.  Everything else helps
    // with the data-parallel phases only.
    const int bfirst = TMEM ? 4 : g.groups;
    const bool isA = wid < g.groups, isB = wid >= bfirst && wid < bfirst + g.groups;
    const bool helper = !(isA || isB);
    const int warp = isB;                            // 0: forward (alpha) warps, 1: backward (beta) warps
    const int wgrp = helper ? 0 : (isB ? wid - bfirst : wid);      // 8-frame group this warp serves
    const int xslot = helper ? 0 : (isB ? g.groups + wgrp : wgrp); // exchange-buffer slot
    // ---- shared memory carve-up -------------------------------------------------
    int16_t *tab = reinterpret_cast<int16_t *>(smem_raw);
    const int tab_bytes = ((7 * N * 2 + 15) / 16) * 16;
    const int FR = g.frames;                         // frames this CTA decodes at a time
    const int areas = FR + (FR < 8 * g.groups);      // idle quads (frame slot >= FR) share one scratch area
    // GREC (long frames): the records of 32 frames do not fit in shared memory, so they live in this CTA's slice of
    // the global workspace and reach the SM through L1 (which gets the shared memory this geometry does not use) and
    // L2; only this CTA reads or writes its slice, so the SM's own L1 stays coherent with it.
    float *smf = reinterpret_cast<float *>(smem_raw + tab_bytes);
    float *gam = smf;
    if constexpr (GREC) gam = A.grec + (size_t)blockIdx.x * areas * g.rec_stride;
    float *ckbuf = GREC ? smf : gam + areas * g.rec_stride;
    float *xch = ckbuf + (TMEM ? 0 : areas * g.ck_stride);
    int *flags = reinterpret_cast<int *>(xch + 4 * g.groups * kXchFloats);
    unsigned *tmem_slot = reinterpret_cast<unsigned *>(flags + 64);
    float *rings = reinterpret_cast<float *>(flags + 68);            // GREC: one record ring per recursion warp
    unsigned char *hb = reinterpret_cast<unsigned char *>(gam);   // hard-bit pairs: the records are dead by then
    if (TMEM && wid == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"((unsigned)__cvta_generic_to_shared(tmem_slot)), "r"(g.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (TMEM) asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");   // [8][N] hard-bit pairs

    for (int i = tid; i < 7 * N; i += NT) tab[i] = A.tab[i];
    __syncthreads();
    unsigned tmem_base = 0;
    if (TMEM) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        tmem_base = *tmem_slot;
    }
    // Y = Lc + La (float64) of a thread's own positions lives in its TMEM lane between prep and
    // epilogue; the four warps of a lane quadrant use disjoint column ranges.
    const bool YTMEM = TMEM && g.y_slots > 0;
    const unsigned ytaddr = tmem_base + (((unsigned)(wid & 3) * 32u) << 16) +
                            4u * (g.nckA + g.nckB) + 4u * g.y_slots * (unsigned)(wid >> 2);
    const int P = FR * N;                   // (frame, step) positions of this CTA, dealt out flat
    // positions per thread whose loads are issued together in prep / epilogue: with the records in global memory these
    // phases are a string of L2 / HBM round trips on 14 warps, so twice as many are kept in flight
    constexpr int KB = GREC ? 2 * kBatch : kBatch;
    const unsigned magic = g.magic;
    const int16_t *t_perm = tab, *t_inv = tab + N, *t_offA = tab + 2 * N;

    Lane L;
    L.q = min(wgrp * 8 + (lane >> 2), FR); L.p = lane & 3;
    L.oA[0] = cls2(L.p);     L.oB[0] = cls2(L.p + 4);
    L.oA[1] = cls2(2 * L.p); L.oB[1] = cls2(2 * L.p + 1);
    L.xw = xbase(lane >> 2) + 4 * L.p;
    L.xr = xbase(lane >> 2) + L.p;
    L.role_word = ((L.p & 1) << 1) | (L.p >> 1);      // roles (U0,V1,U3,V2) -> words (0,2,1,3)

    unsigned long long bit_err = 0, frm_err = 0, frames_done = 0;
    long long ph[6] = {0, 0, 0, 0, 0, 0};
    const long long t_start = clock64();
    const size_t slot0 = (size_t)blockIdx.x * FR * N;
    double2 *Le1 = A.Le1 + slot0, *Le2 = A.Le2 + slot0, *Yb = A.Y + slot0;

    for (int grp = blockIdx.x; grp < A.n_groups; grp += gridDim.x) {
        const long long frame0 = (long long)grp * FR;
        const int n_half = SISO_ONLY ? 1 : 2 * A.iterations;
        for (int h = 0; h < n_half; ++h) {
            const int second = h & 1;                      // 0: SISO1 (natural), 1: SISO2 (interleaved)
            const bool first = (h == 0);
            const double sf = SISO_ONLY ? A.siso_sf
                                        : ((h >> 1) < A.iterations - 1 ? A.sf_inner : A.sf_last);
            const double2 *LePrev = second ? Le1 : Le2;
            double2 *LeOut = second ? Le2 : Le1;
            const int16_t *t_oW = tab + (3 + 2 * second) * N, *t_oY = tab + (4 + 2 * second) * N;
            __syncthreads();   // tables loaded / previous phase finished with gam, Le
            const long long t0 = clock64();
            // ---- prep: gather, a-priori add, branch-metric records ------------------
            // KB positions per thread are loaded before any is consumed, so the
            // dependent smem-index -> L2 gather round trips overlap.
            for (int it = 0; it * KB * NT < P; ++it) {       // warp-uniform trip count
                const int i0 = tid + it * KB * NT;
                float sA[KB], sB[KB], pW[KB], pY[KB];
                double2 La[KB];
#pragma unroll
                for (int u = 0; u < KB; ++u) {
                    int f, k; const int i = i0 + u * NT; pos_of<GREC>(i, N, magic, f, k);
                    const long long frame = frame0 + f;
                    sA[u] = sB[u] = pW[u] = pY[u] = 0.f;
                    La[u] = make_double2(0.0, 0.0);
                    if (i < P && frame < A.B) {
                        if (SISO_ONLY) {
                            const size_t e = (size_t)frame * N + k;
                            sA[u] = __ldg(A.LcA + e); sB[u] = __ldg(A.LcB + e);
                            pW[u] = __ldg(A.LcW + e); pY[u] = __ldg(A.LcY + e);
                            if (A.LaA) La[u].x = __ldg(A.LaA + e);
                            if (A.LaB) La[u].y = __ldg(A.LaB + e);
                        } else {
                            const LlrT *Lf = static_cast<const LlrT *>(A.llr) + frame * A.llr_stride;
                            const int src = second ? t_perm[k] : k;
                            const int oa = t_offA[src];
                            if (A.vec_ab) {
                                const float2 v = llr_ldg2(Lf + oa, A.llr_scale);
                                sA[u] = v.x; sB[u] = v.y;
                            } else {
                                sA[u] = llr_ldg(Lf + oa, A.llr_scale); sB[u] = llr_ldg(Lf + oa + 1, A.llr_scale);
                            }
                            const int ow = t_oW[k], oy = t_oY[k];
                            if (A.vec_wy) {          // both parities present, adjacent and aligned to two elements
                                const float2 v = llr_ldg2(Lf + ow, A.llr_scale);
                                pW[u] = v.x; pY[u] = v.y;
                            } else {
                                if (ow >= 0) pW[u] = llr_ldg(Lf + ow, A.llr_scale);
                                if (oy >= 0) pY[u] = llr_ldg(Lf + oy, A.llr_scale);
                            }
                            if (!first) La[u] = __ldcg(LePrev + (size_t)f * N + (second ? src : (int)t_inv[k]));
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < KB; ++u) {
                    int f, k; const int i = i0 + u * NT; pos_of<GREC>(i, N, magic, f, k);
                    // computed unconditionally (one basic block, so the independent
                    // float64 chains of the batch interleave); only the stores are guarded
                    const double YA = __dadd_rn((double)sA[u], La[u].x);   // Lc_A[k] + La_A[k] (:135)
                    const double YB = __dadd_rn((double)sB[u], La[u].y);
                    float4 lo4, hi4;
                    make_record(k, YA, YB, pW[u], pY[u], lo4, hi4);
                    if (i < P) {
                        float *rec = GREC ? gam + ((size_t)(f >> 3) * N + k) * kGrecStep + (f & 7) * 8 : gam + f * g.rec_stride + k * 8;
                        *reinterpret_cast<float4 *>(rec) = lo4;
                        *reinterpret_cast<float4 *>(rec + 4) = hi4;
                        if (!YTMEM) __stcg(Yb + (size_t)f * N + k, make_double2(YA, YB));
                    }
                    if (YTMEM)          // Y stays on chip: this thread's TMEM lane, slot = it*KB + u
                        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
                                     ::"r"(ytaddr + 4u * (it * KB + u)), "r"(__double2loint(YA)), "r"(__double2hiint(YA)),
                                       "r"(__double2loint(YB)), "r"(__double2hiint(YB)) : "memory");
                }
            }
            if (YTMEM) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            __syncthreads();
            const long long t1 = clock64();
            long long t2;
            if (!helper) {
                Ckpt<TMEM> ck;
                if constexpr (TMEM) ck.taddr = tmem_base + (((unsigned)(wid & 3) * 32u) << 16);
                else ck.base = ckbuf + L.q * g.ck_stride + 4 * L.p;
                siso_core<GREC>(g, gam, ck, xch, rings, warp, xslot, L, t2);
            } else {
                __syncthreads();
                t2 = clock64();
                __syncthreads();
            }
            const long long t3 = clock64();
            // ---- epilogue: extrinsic LLRs (float64) ---------------------------------
            for (int it = 0; it * KB * NT < P; ++it) {
                const int i0 = tid + it * KB * NT;
                double2 Y[KB];
                float4 uv[KB];
#pragma unroll
                for (int u = 0; u < KB; ++u) {
                    int f, k; const int i = i0 + u * NT; pos_of<GREC>(i, N, magic, f, k);
                    Y[u] = make_double2(0.0, 0.0); uv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (i < P && frame0 + f < A.B) {
                        if (!YTMEM) Y[u] = __ldcg(Yb + (size_t)f * N + k);
                        uv[u] = *reinterpret_cast<const float4 *>(GREC ? gam + ((size_t)(f >> 3) * N + k) * kGrecStep + (f & 7) * 8 : gam + f * g.rec_stride + k * 8);
                    }
                    if (YTMEM) {
                        int a, b, c, d;
                        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                                     : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(ytaddr + 4u * (it * KB + u)) : "memory");
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                        Y[u] = make_double2(__hiloint2double(b, a), __hiloint2double(d, c));
                    }
                }
#pragma unroll
                for (int u = 0; u < KB; ++u) {
                    int f, k; const int i = i0 + u * NT; pos_of<GREC>(i, N, magic, f, k);
                    const long long frame = frame0 + f;
                    const double2 e = make_extrinsic(uv[u], Y[u].x, Y[u].y, sf);
                    if (i < P && frame < A.B) {
                        if (SISO_ONLY) {
                            A.LeA[(size_t)frame * N + k] = e.x;
                            A.LeB[(size_t)frame * N + k] = e.y;
                        } else {
                            __stcg(LeOut + (size_t)f * N + k, e);
                        }
                    }
                }
            }
            ph[0] += t1 - t0; ph[1] += t2 - t1; ph[2] += t3 - t2; ph[3] += clock64() - t3;
        }
        if (SISO_ONLY) continue;
        __syncthreads();
        const long long t5 = clock64();
        // ---- hard decision (dvb_rcs2_turbo.py:526-537) + optional error counting ----
        if (tid < FR) flags[tid] = 0;
        __syncthreads();
        for (int i0 = tid; i0 < P; i0 += kBatch * NT) {
            double2 La[kBatch], e1[kBatch];
            float sA[kBatch], sB[kBatch];
            uchar2 rb[kBatch];
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                int f, j; const int i = i0 + u * NT; split_pos(i, N, magic, f, j);
                const long long frame = frame0 + f;
                La[u] = e1[u] = make_double2(0.0, 0.0); sA[u] = sB[u] = 0.f; rb[u] = make_uchar2(0, 0);
                if (i < P && frame < A.B) {
                    const LlrT *Lf = static_cast<const LlrT *>(A.llr) + frame * A.llr_stride;
                    const int oa = t_offA[j];
                    La[u] = __ldcg(Le2 + (size_t)f * N + t_inv[j]);
                    e1[u] = __ldcg(Le1 + (size_t)f * N + j);
                    sA[u] = llr_ldg(Lf + oa, A.llr_scale); sB[u] = llr_ldg(Lf + oa + 1, A.llr_scale);
                    if (A.ref_bits)
                        rb[u] = *reinterpret_cast<const uchar2 *>(A.ref_bits + (size_t)frame * 2 * N + 2 * j);
                }
            }
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                int f, j; const int i = i0 + u * NT; split_pos(i, N, magic, f, j);
                const long long frame = frame0 + f;
                if (i < P && frame < A.B) {
                    const double LA = __dadd_rn(__dadd_rn((double)sA[u], La[u].x), e1[u].x);
                    const double LB = __dadd_rn(__dadd_rn((double)sB[u], La[u].y), e1[u].y);
                    const int bA = LA < 0.0, bB = LB < 0.0;
                    if (A.bits)
                        *reinterpret_cast<int2 *>(A.bits + (size_t)frame * 2 * N + 2 * j) = make_int2(bA, bB);
                    if (A.app)
                        *reinterpret_cast<float2 *>(A.app + (size_t)frame * 2 * N + 2 * j) =
                            make_float2(__double2float_rn(LA), __double2float_rn(LB));
                    hb[f * N + j] = (unsigned char)(bA | (bB << 1));
                    if (A.ref_bits) {
                        const int errs = (bA != rb[u].x) + (bB != rb[u].y);
                        bit_err += errs;
                        if (errs) atomicOr(&flags[f], 1);
                    }
                }
            }
        }
        __syncthreads();
        if (A.packed) {
            const int wpf = (2 * N + 31) / 32;
            for (int i = tid; i < FR * wpf; i += NT) {
                const int f = i / wpf, w = i - f * wpf;
                if (frame0 + f >= A.B) continue;
                unsigned v = 0;
                for (int t = 0; t < 16; ++t) {
                    const int j = w * 16 + t;
                    if (j < N) v |= (unsigned)hb[f * N + j] << (2 * t);
                }
                A.packed[(size_t)(frame0 + f) * wpf + w] = v;
            }
        }
        ph[4] += clock64() - t5;
        if (tid < FR && frame0 + tid < A.B) {
            frames_done += 1;
            frm_err += flags[tid];
        }
    }
    if (tid == 0) {
        ph[5] = clock64() - t_start;
        if (A.timed)
            for (int i = 0; i < 6; ++i) atomicAdd(&g_phase_cycles[i], (unsigned long long)ph[i]);
    }
    if (!SISO_ONLY && A.counters) {
        // one atomic per warp and counter at kernel end
        for (int o = 16; o > 0; o >>= 1) {
            bit_err += __shfl_xor_sync(0xffffffffu, bit_err, o);
            frm_err += __shfl_xor_sync(0xffffffffu, frm_err, o);
            frames_done += __shfl_xor_sync(0xffffffffu, frames_done, o);
        }
        if (lane == 0) {
            if (bit_err) atomicAdd(A.counters + 0, bit_err);
            if (frm_err) atomicAdd(A.counters + 1, frm_err);
            if (frames_done) {
                atomicAdd(A.counters + 2, frames_done);
                atomicAdd(A.counters + 3, frames_done * 2ull * N);
            }
        }
    }
    if (TMEM) {
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (wid == 0)
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(g.tmem_cols) : "memory");
    }
}

}  // namespace

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static size_t quad_smem_bytes(const QuadGeom &g)
{
    const int areas = g.frames + (g.frames < 8 * g.groups);
    size_t tab = ((size_t)7 * g.N * 2 + 15) / 16 * 16;
    if (g.grec) return tab + (size_t)4 * g.groups * kXchFloats * 4 + 68 * 4 + (size_t)2 * g.groups * kRingSteps * kGrecStep * 4;
    size_t fl = (size_t)areas * g.rec_stride + (g.use_tmem ? 0 : (size_t)areas * g.ck_stride) +
                4 * g.groups * kXchFloats;
    return tab + fl * 4 + 68 * 4;
}

int quad_configure(Codec &c, size_t smem_optin)
{
    QuadGeom &g = c.geom;
    const int N = c.N;
    if (N < 8 || N > kMaxN || (N % 4) != 0) return B200DVB_ENOSPEC;
    g.N = N;
    g.M = ((N / 2) / kWin) * kWin;
    if (g.M == 0) g.M = kWin <= N - 4 ? kWin : 0;
    if (g.M <= 0 || g.M >= N) return B200DVB_ENOSPEC;
    g.nckA = g.M / kWin;
    g.nckB = (N - g.M + kWin - 1) / kWin;
    g.magic = (unsigned)((1ull << 32) / (unsigned)N) + 1u;
    g.rec_stride = 8 * N + 8;                       // == 8 (mod 32): 4 frames tile the 32 banks
    int ck = (g.nckA + g.nckB) * 16;
    if ((ck % 32) == 0) ck += 16;                   // == 16 (mod 32)
    g.ck_stride = ck;
    // One CTA per SM: `groups` pairs of (alpha warp, beta warp), 8 frames per pair, all warps
    // in the same phase so they share the instruction cache.  Two placements of the recursion
    // checkpoints are tried and the one that keeps more frames resident wins: shared memory
    // (up to 7 groups when N is small) or tensor memory (up to 4 groups: one per lane quadrant).
    const size_t cap = smem_optin;
    const int want_groups = kMaxGroups;
    QuadGeom best{};
    best.frames = 0;
    for (int tm = 0; tm < 2; ++tm) {
        QuadGeom t = g;
        t.use_tmem = tm;
        t.tmem_cols = 32;
        t.y_slots = 0;
        while (t.tmem_cols < 4 * (t.nckA + t.nckB)) t.tmem_cols *= 2;
        if (tm && t.tmem_cols > 512) continue;
        const int gmax = tm ? 4 : kMaxGroups;
        int gr = want_groups < 1 ? 1 : (want_groups > gmax ? gmax : want_groups);
        bool ok = false;
        for (; gr >= 1 && !ok; --gr) {
            t.groups = gr;
            for (t.frames = 8 * gr; t.frames > 8 * (gr - 1) && t.frames >= 1; --t.frames) {
                t.smem_bytes = quad_smem_bytes(t);
                if (t.smem_bytes <= cap) { ok = true; break; }
            }
        }
        if (ok && t.frames > best.frames) best = t;
    }
    if (best.frames < 1) return B200DVB_ENOSPEC;
    g = best;
    const bool want_y = true;
    {
        int t = kMaxCtaThreads;
        if (t < kCtaThreads * g.groups) t = kCtaThreads * g.groups;
        if (t > kMaxCtaThreads) t = kMaxCtaThreads;
        g.threads = t;
    }
    if (g.use_tmem && want_y) {
        // 4 words per position, ceil(P / threads) positions per thread, 4 warps per lane quadrant
        const int slots = (g.frames * N + g.threads - 1) / g.threads;
        const int slots4 = ((slots + kBatch - 1) / kBatch) * kBatch;
        const int warps_per_quadrant = (g.threads / 32 + 3) / 4;
        const int need = 4 * (g.nckA + g.nckB) + 4 * slots4 * warps_per_quadrant;
        if (need <= 512) {
            g.y_slots = slots4;
            while (g.tmem_cols < need) g.tmem_cols *= 2;
        }
    }
    B2_CUDA(cudaFuncSetAttribute(quad_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap));   // SISO (float32)
    B2_CUDA(cudaFuncSetAttribute(quad_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap));
    B2_CHECK(for_each_llr_type([&](auto t) {
        using L = decltype(t);
        B2_CUDA(cudaFuncSetAttribute(quad_kernel<false, false, false, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap));
        B2_CUDA(cudaFuncSetAttribute(quad_kernel<false, true, false, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap));
        return B200DVB_OK;
    }));
    int occ = 0;
    if (g.use_tmem) {
        B2_CHECK(occupancy_all_formats(&occ, [](auto t) { return quad_kernel<false, true, false, decltype(t)>; }, g.threads, g.smem_bytes));
        if (occ > 1 && g.tmem_cols > 256) occ = 1;      // two CTAs must both get their TMEM columns
        if (occ > 512 / g.tmem_cols) occ = 512 / g.tmem_cols;
    } else {
        B2_CHECK(occupancy_all_formats(&occ, [](auto t) { return quad_kernel<false, false, false, decltype(t)>; }, g.threads, g.smem_bytes));
    }
    if (occ < 1) return B200DVB_ENOSPEC;
    g.ctas_per_sm = occ;
    // Long frames: when shared memory holds the records of fewer than three groups (N >= 296: 2 x 8 frames at N=424, 8
    // at N=752: two recursion warps on an SM), a second geometry keeps the records in global memory and runs the full
    // four groups (32 frames, 8 recursion warps) per SM.
    c.geom_g = QuadGeom{};
    if (g.frames <= 16 && 4 * (g.nckA + g.nckB) <= 512) {
        QuadGeom t = g;
        t.grec = 1; t.use_tmem = 1; t.groups = 4; t.frames = 32; t.y_slots = 0;   // (Y stays in global memory: KB != kBatch)
        t.threads = kMaxCtaThreads;
        t.tmem_cols = 32;
        while (t.tmem_cols < 4 * (t.nckA + t.nckB)) t.tmem_cols *= 2;
        t.smem_bytes = quad_smem_bytes(t);
        // the shared memory this geometry leaves unused is worth more as L1 for the records
        const int carve = (int)((t.smem_bytes * 100 + cap - 1) / cap) + 4;
        B2_CHECK(for_each_llr_type([&](auto l) {
            B2_CUDA(cudaFuncSetAttribute(quad_kernel<false, true, true, decltype(l)>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap));
            B2_CUDA(cudaFuncSetAttribute(quad_kernel<false, true, true, decltype(l)>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
            return B200DVB_OK;
        }));
        int og = 0;
        B2_CHECK(occupancy_all_formats(&og, [](auto l) { return quad_kernel<false, true, true, decltype(l)>; }, t.threads, t.smem_bytes));
        if (og > 512 / t.tmem_cols) og = 512 / t.tmem_cols;
        if (og > 1) og = 1;
        if (og >= 1) { t.ctas_per_sm = og; c.geom_g = t; }
    }
    return B200DVB_OK;
}

// Geometry that serves a full decode of B frames: whichever needs less time for its waves.  One wave of the
// global-record geometry (32 frames per SM) takes 2.3 x as long as one of the shared-memory geometry with 8 frames per
// SM (N=752: 4.15 ms against 1.84 ms) and 1.85 x one with 16 frames per SM (N=424: 2.08 against 1.15 ms;
// profiles/r02_long.txt), so small batches, which the shared-memory geometry spreads over more SMs, stay there.  A pure
// function of (codec, B): the workspace query and the launch agree.
static const QuadGeom &decode_geom(const Codec &c, int B)
{
    if (c.geom_g.frames <= 0) return c.geom;
    const long long sw = (long long)c.num_sms * c.geom.ctas_per_sm * c.geom.frames;
    const long long gw = (long long)c.num_sms * c.geom_g.ctas_per_sm * c.geom_g.frames;
    const long long waves_s = (B + sw - 1) / sw, waves_g = (B + gw - 1) / gw;
    const long long r100 = c.geom.frames <= 8 ? 230 : 185;
    return waves_g * r100 < waves_s * 100 ? c.geom_g : c.geom;
}

static int grid_for(const Codec &c, const QuadGeom &g, int B)
{
    const int groups = (B + g.frames - 1) / g.frames;
    const int cap = c.num_sms * g.ctas_per_sm;
    return groups < cap ? groups : cap;
}
static size_t grec_floats(const QuadGeom &g, int grid)
{
    const int areas = g.frames + (g.frames < 8 * g.groups);
    return g.grec ? (size_t)grid * areas * g.rec_stride : 0;
}

size_t quad_workspace_bytes(const Codec &c, int B)
{
    const QuadGeom &g = decode_geom(c, B);
    const int grid = grid_for(c, g, B);
    return (size_t)3 * grid * g.frames * c.N * sizeof(double2) + grec_floats(g, grid) * sizeof(float) + 512;
}
size_t siso_workspace_bytes(const Codec &c, int B)
{
    return (size_t)grid_for(c, c.geom, B) * c.geom.frames * c.N * sizeof(double2) + 256;
}

static inline unsigned char *align256(void *p)
{
    return reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(p) + 255) & ~(uintptr_t)255);
}

int quad_launch_decode(const Codec &c, const DecodeIo &io)
{
    if (io.ws_bytes < quad_workspace_bytes(c, io.B)) return B200DVB_ENOMEM;
    const QuadGeom &G = decode_geom(c, io.B);
    const int grid = grid_for(c, G, io.B);
    const size_t per = (size_t)grid * G.frames * c.N;
    QuadArgs A{};
    fill_decode_args(A, c, io);
    A.g = G;
    A.n_groups = (io.B + G.frames - 1) / G.frames;
    const uintptr_t pair_bytes = 2 * llr_bytes(io.fmt);
    const bool even = (io.llr_stride % 2 == 0) && ((reinterpret_cast<uintptr_t>(io.llr) & (pair_bytes - 1)) == 0);
    A.vec_ab = even && c.vec_ab;
    A.vec_wy = even && c.vec_wy;
    A.timed = c.opt_phase_timers;
    A.Le1 = reinterpret_cast<double2 *>(align256(io.ws));
    A.Le2 = A.Le1 + per; A.Y = A.Le2 + per;
    A.grec = reinterpret_cast<float *>(align256(A.Y + per));
    with_llr_type(io.fmt, [&](auto t) {
        using L = decltype(t);
        if (G.grec)          quad_kernel<false, true, true, L><<<grid, G.threads, G.smem_bytes, io.stream>>>(A);
        else if (G.use_tmem) quad_kernel<false, true, false, L><<<grid, G.threads, G.smem_bytes, io.stream>>>(A);
        else                 quad_kernel<false, false, false, L><<<grid, G.threads, G.smem_bytes, io.stream>>>(A);
    });
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

int launch_siso(const Codec &c, int B, const float *Lc_A, const float *Lc_B, const float *Lc_W,
                const float *Lc_Y, const double *La_A, const double *La_B, double sf,
                double *Le_A, double *Le_B, void *ws, size_t ws_bytes, cudaStream_t s)
{
    if (B == 0) return B200DVB_OK;
    if (ws_bytes < siso_workspace_bytes(c, B)) return B200DVB_ENOMEM;
    const int grid = grid_for(c, c.geom, B);
    QuadArgs A{};
    A.g = c.geom; A.B = B; A.iterations = 1;
    A.n_groups = (B + c.geom.frames - 1) / c.geom.frames;
    A.tab = c.d_tab;
    A.LcA = Lc_A; A.LcB = Lc_B; A.LcW = Lc_W; A.LcY = Lc_Y; A.LaA = La_A; A.LaB = La_B;
    A.LeA = Le_A; A.LeB = Le_B; A.siso_sf = sf;
    A.Y = reinterpret_cast<double2 *>(align256(ws));
    A.Le1 = A.Y; A.Le2 = A.Y;
    if (c.geom.use_tmem) quad_kernel<true, true><<<grid, c.geom.threads, c.geom.smem_bytes, s>>>(A);
    else                 quad_kernel<true, false><<<grid, c.geom.threads, c.geom.smem_bytes, s>>>(A);
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

int quad_read_phase_cycles(double *out_h, int reset) { return read_phase_cycles(g_phase_cycles, out_h, reset); }

}  // namespace b200dvb
