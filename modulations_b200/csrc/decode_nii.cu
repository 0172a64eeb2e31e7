// decode_nii.cu — the NON-PARITY decoder mode "nii" (SURVEY 8(f) N2, BASELINE north_star "windows ... use
// next-iteration circular-state initialisation"): a thread-per-frame max-log-MAP turbo decoder that makes ONE pass
// per SISO.  Selected only by an explicit flag (B200DVB_OPT_DECODER_MODE = B200DVB_MODE_NII); its results are not the
// reference's bit for bit and are judged on BER/FER; the kernel itself is checked bit for bit against its own
// plain-C model oracle/nii_model.c.  nii_core.cuh states the arithmetic.
//
// What changes against decode_tpf.cu (the parity mode, dvb_rcs2_turbo.py:116-281):
//   * no pass 1: alpha[0] / beta[N] of a SISO are the boundary metrics the same constituent decoder reached one
//     iteration earlier (zeros in the first iteration), kept per lane in the workspace.  Of the reference's five
//     sweeps per SISO (alpha x2, beta x2, extrinsic) three remain; per lane 0.5 N "in" steps + 0.5 N recomputed +
//     0.5 N extrinsic steps instead of 1.5 N + 0.5 N + 0.5 N;
//   * float32 a-priori / extrinsic values and branch-metric sums: no FP64 pipe, no F2F conversions (the 16-lane
//     XU pipe was the largest term of the parity kernel's prep stage), half the scratch traffic;
//   * a-posteriori maxima taken per parity class BEFORE the branch metric is added (48 FADD + 36 FMNMX per step
//     instead of 128 + 60).
// Unchanged: the mapping (a warp owns 16 frames, lanes 0-15 forward, lanes 16-31 backward threads in bit-reversed
// labels, one warp per SM sub-partition), the record pool (tensor memory for the outer T steps of either frame end,
// shared memory for the middle), meet in the middle with a checkpoint every 4 steps, recompute windows, the
// group-staged transposition and the fused hard decision / error counters.
#include "common.cuh"
#include "nii_core.cuh"
#include "nii16_core.cuh"
#include "tpf_dev.cuh"

#include <math.h>

namespace b200dvb {

namespace {

using namespace tpf;

// ---- arithmetic policies: the kernel below moves every value through `float` registers and float2 / float4
//      containers; a policy decides what the 32 bits mean.  ArF32 = mode "nii" (one float32 frame per lane),
//      ArS16 = mode "nii16" (two int16 frames per lane, nii16_core.cuh; the casts are register renames) --------------
struct ArF32 {
    static constexpr int kFpl = 1;                                  // frames per lane
    typedef float sf_t;
    static __device__ __forceinline__ void make_record(float YA, float YB, float W, float Y, float (&g)[8]) { nii::make_record(YA, YB, W, Y, g); }
    static __device__ __forceinline__ void pass_step(float (&v)[16], const float (&g)[8], bool isb) { tpf::pass_step(v, g, isb); }
    static __device__ __forceinline__ void bwd_step(float (&z)[16], const float (&g)[8]) { tpf::bwd_step(z, g); }
    static __device__ __forceinline__ void app_maxima(const float (&x)[16], const float (&zs)[16], const float (&g)[8], float (&uv)[4]) { nii::app_maxima(x, zs, g, uv); }
    static __device__ __forceinline__ void make_extrinsic(const float (&uv)[4], float YA, float YB, sf_t sf, float &ea, float &eb) { nii::make_extrinsic(uv, YA, YB, sf, ea, eb); }
    static __device__ __forceinline__ float add(float a, float b) { return f_add(a, b); }
    static __device__ __forceinline__ float chan(float lo, float) { return lo; }             // channel LLR of the lane's frame(s)
    static __device__ __forceinline__ int neg(float L, int) { return L < 0.f; }             // hard decision of sub-frame i
};
struct ArS16 {
    static constexpr int kFpl = 2;
    typedef int sf_t;
    template <int K> static __device__ __forceinline__ void in(const float (&a)[K], nii16::p16 (&b)[K])
    {
#pragma unroll
        for (int i = 0; i < K; ++i) b[i] = nii16::bits(a[i]);
    }
    template <int K> static __device__ __forceinline__ void out(const nii16::p16 (&b)[K], float (&a)[K])
    {
#pragma unroll
        for (int i = 0; i < K; ++i) a[i] = nii16::fl(b[i]);
    }
    static __device__ __forceinline__ void make_record(float YA, float YB, float W, float Y, float (&g)[8])
    {
        nii16::p16 pg[8];
        nii16::make_record(nii16::bits(YA), nii16::bits(YB), nii16::bits(W), nii16::bits(Y), pg);
        out(pg, g);
    }
    static __device__ __forceinline__ void pass_step(float (&v)[16], const float (&g)[8], bool isb)
    {
        nii16::p16 pv[16], pg[8];
        in(v, pv); in(g, pg);
        nii16::pass_step(pv, pg, isb);
        out(pv, v);
    }
    static __device__ __forceinline__ void bwd_step(float (&z)[16], const float (&g)[8])
    {
        nii16::p16 pz[16], pg[8];
        in(z, pz); in(g, pg);
        nii16::bwd_step(pz, pg);
        out(pz, z);
    }
    static __device__ __forceinline__ void app_maxima(const float (&x)[16], const float (&zs)[16], const float (&g)[8], float (&uv)[4])
    {
        nii16::p16 px[16], pz[16], pg[8], pu[4];
        in(x, px); in(zs, pz); in(g, pg);
        nii16::app_maxima(px, pz, pg, pu);
        out(pu, uv);
    }
    static __device__ __forceinline__ void make_extrinsic(const float (&uv)[4], float YA, float YB, sf_t sf, float &ea, float &eb)
    {
        nii16::p16 pu[4], a, b;
        in(uv, pu);
        nii16::make_extrinsic(pu, nii16::bits(YA), nii16::bits(YB), sf, a, b);
        ea = nii16::fl(a); eb = nii16::fl(b);
    }
    static __device__ __forceinline__ float add(float a, float b) { return nii16::fl(nii16::add2(nii16::bits(a), nii16::bits(b))); }
    static __device__ __forceinline__ float chan(float lo, float hi) { return nii16::fl(nii16::pack16(nii16::quant(lo), nii16::quant(hi))); }
    static __device__ __forceinline__ int neg(float L, int i) { return (i ? nii16::hi16(nii16::bits(L)) : nii16::lo16(nii16::bits(L))) < 0; }
};

constexpr int kW = kTpfWin;
constexpr int kHdrBytes = 64 + kTpfWarps * kRingPairs * 8;   // after the tables: slots, one mbarrier per warp, kRingPairs ring mbarriers per warp

// phase timers (SM cycles summed over warps): 0 transpose-in, 1 "in" pass (+prep), 2 boundary load/store + crossing,
// 3 unused, 4 out-phase windows in shared memory, 5 out-phase windows in tensor memory, 6 hard decision, 7 warp total
__device__ unsigned long long g_nii_cycles[8];

struct NiiArgs {
    TpfGeom g;
    int B, iterations, n_tiles, n_llr, vec4;
    float sf_inner, sf_last;
    int sf_inner_q, sf_last_q;       // the same in Q6 for the fixed-point mode
    const int16_t *tab;
    const void *llr;                 // [B][llr_stride] elements of the kernel's LlrT (float32, binary16 or int8)
    long long llr_stride;
    int32_t *bits;
    uint32_t *packed;
    const uint8_t *ref_bits;
    unsigned long long *counters;
    unsigned char *ws;
    float llr_scale;                 // int8 element q is the LLR q * llr_scale (last: the other members keep their offsets)
};

struct Ctx {
    int N, M, T;
    int f, isb, lane, h8;            // frame within the tile, 0 = alpha lane / 1 = beta lane, byte offset of this frame's float2 in a 16-byte chunk
    unsigned tq;                     // TMEM address of this warp's lane quadrant, column 0
    unsigned ycol;                   // first of the 2 kW spare TMEM columns that park the window's Y
    float4 *srec;                    // this warp's shared-memory records: [(k - T) * 2 + half][16 frames]
    unsigned char *stage;            // this warp's staging area (kStageBytes)
    const int16_t *perm, *inv;       // shared-memory copies of the interleaver tables
    float4 *L1A, *L2A;               // de-punctured channel LLRs [j][32 lanes]
    float2 *Le, *LeF;                // extrinsics [k][16] (in place; last half-iteration -> LeF)
    float4 *Yb;                      // Y = Lc + La, [k/2][16]: (YA, YB) of step k (even) and of step k+1
    float4 *CK;                      // checkpoints [slot][4][32 lanes]
    float4 *INIT;                    // boundary metrics [siso][4][32 lanes], natural labels, indexed by the lane that READS them
    unsigned long long pol;          // L2 evict-first policy for the channel LLRs
    unsigned one;                    // 1, opaque to the compiler (see cpa16)
    unsigned rmbar;                  // shared-memory address of this warp's kRingPairs ring mbarriers (bulk channel loads)
    __device__ __forceinline__ float4 *wstore() const { return reinterpret_cast<float4 *>(stage); }
    __device__ __forceinline__ float4 *slotZ() const { return reinterpret_cast<float4 *>(stage + 8192); }
    __device__ __forceinline__ float4 *slotX() const { return reinterpret_cast<float4 *>(stage + 10240); }
};

__device__ __forceinline__ void smem_get(const Ctx &c, int k, float (&g)[8])
{
    const float4 lo = c.srec[((k - c.T) * 2) * 16 + c.f], hi = c.srec[((k - c.T) * 2 + 1) * 16 + c.f];
    g[0] = lo.x; g[1] = lo.y; g[2] = lo.z; g[3] = lo.w; g[4] = hi.x; g[5] = hi.y; g[6] = hi.z; g[7] = hi.w;
}
__device__ __forceinline__ void smem_put(const Ctx &c, int k, const float (&g)[8])
{
    c.srec[((k - c.T) * 2) * 16 + c.f] = make_float4(g[0], g[1], g[2], g[3]);
    c.srec[((k - c.T) * 2 + 1) * 16 + c.f] = make_float4(g[4], g[5], g[6], g[7]);
}

struct Buf { float a[8], b[8]; };

__device__ __forceinline__ void ck_store(const Ctx &c, int slot, const float (&v)[16])
{   // always in natural state order: the beta lanes hold rho4 labels during the "in" pass
    float n[16];
#pragma unroll
    for (int s = 0; s < 16; ++s) n[s] = c.isb ? v[rho4(s)] : v[s];
#ifdef NII_CK256
    // two 32-byte stores per checkpoint instead of four 16-byte ones: slot layout [2 halves][32 lanes] x 32 B
    unsigned char *p = reinterpret_cast<unsigned char *>(c.CK) + slot * 2048 + c.lane * 32;
#pragma unroll
    for (int h = 0; h < 2; ++h)
        asm volatile("st.global.cg.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                     :: "l"(p + h * 1024), "f"(n[8 * h]), "f"(n[8 * h + 1]), "f"(n[8 * h + 2]), "f"(n[8 * h + 3]),
                        "f"(n[8 * h + 4]), "f"(n[8 * h + 5]), "f"(n[8 * h + 6]), "f"(n[8 * h + 7]) : "memory");
#else
#pragma unroll
    for (int q = 0; q < 4; ++q)
        st_ws(c.CK + (slot * 4 + q) * 32 + c.lane, make_float4(n[4 * q], n[4 * q + 1], n[4 * q + 2], n[4 * q + 3]));
#endif
}
__device__ __forceinline__ void issue_ckpt(const Ctx &c, int slot)
{   // alpha lanes need their alpha checkpoint as X, beta lanes their beta checkpoint as Z
    float4 *dst = (c.isb ? c.slotZ() : c.slotX()) + c.lane;
#ifdef NII_CK256
    const unsigned char *p = reinterpret_cast<const unsigned char *>(c.CK) + slot * 2048 + c.lane * 32;
#pragma unroll
    for (int q = 0; q < 4; ++q) cpa16(dst + q * 32, p + (q >> 1) * 1024 + (q & 1) * 16, c.one);
#else
#pragma unroll
    for (int q = 0; q < 4; ++q) cpa16(dst + q * 32, c.CK + (slot * 4 + q) * 32 + c.lane, c.one);
#endif
}
__device__ __forceinline__ void slot_get(const float4 *slot, int lane, float (&v)[16])
{
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 t = slot[q * 32 + lane];
        v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
    }
}
__device__ __forceinline__ void slot_put(float4 *slot, int lane, const float (&v)[16])
{
#pragma unroll
    for (int q = 0; q < 4; ++q) slot[q * 32 + lane] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}

// ---- Y = Lc + La (float32) of the current window, parked in 2 kW spare TMEM columns of this lane -------------
__device__ __forceinline__ void tm_ld2(unsigned taddr, float (&y)[2])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=f"(y[0]), "=f"(y[1]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tm_wait_ld2(float (&y)[2])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(y[0]), "+f"(y[1]) :: "memory");
}
__device__ __forceinline__ float4 ld_ws4(const float4 *p)
{   // workspace load: L2 only (the workspace is rewritten by other phases; L1 is not coherent with those stores)
    float4 v;
    asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
struct YQ { float4 y[2]; };                                          // steps (w0, w0+1) and (w0+2, w0+3)
__device__ __forceinline__ void yq_load(const Ctx &c, int w0, int len, YQ &q)
{   // global loads issued a whole window ahead of their use (w0 is even for both half-warps)
    static_assert(kW == 4, "two pair entries per window");
    q.y[0] = ld_ws4(c.Yb + (w0 >> 1) * 16 + c.f);
    q.y[1] = ld_ws4(c.Yb + ((len > 2 ? w0 + 2 : w0) >> 1) * 16 + c.f);
}
__device__ __forceinline__ void yq_park(const Ctx &c, const YQ &q, int w0, int len, int ck_slot)
{
    const float y[8] = {q.y[0].x, q.y[0].y, q.y[0].z, q.y[0].w, q.y[1].x, q.y[1].y, q.y[1].z, q.y[1].w};
#pragma unroll
    for (int u = 0; u < kW; ++u)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};"
                     :: "r"(c.tq + c.ycol + 2u * u), "f"(y[2 * u]), "f"(y[2 * u + 1]) : "memory");
    tm_wait_st();
    // the values are in TMEM now.  ONE predicated discard instruction drops the dead scratch of this window:
    // lanes 0-7 the 2 x 2 x 2 lines of Y (lane = half-warp, pair, half of the pair's 256 bytes), lanes 16-31 the 16
    // lines of the checkpoint slot the finished window consumed
    const int dir = (c.lane >> 2) & 1, pr = (c.lane >> 1) & 1, l16 = c.lane & 15;
    const int w0d = __shfl_sync(0xffffffffu, w0, dir << 4);         // w0 of the alpha (lane 0) / beta (lane 16) half
    const void *line = c.lane < 16
        ? static_cast<const void *>(c.Yb + ((w0d >> 1) + pr) * 16 + (c.lane & 1) * 8)
        : static_cast<const void *>(c.CK + (ck_slot * 4 + (l16 >> 2)) * 32 + (l16 & 3) * 8);
    if (c.lane < 16 ? (c.lane < 8 && 2 * pr < len) : ck_slot >= 0) l2_discard(line);
}

// the float32 epilogue of a window's LAST step, carried into the next window (as in decode_tpf.cu: its dependent
// chain fills the load latencies of the next window's start)
struct Pend { float uv[4], y[2]; int idx; };
template <class AR>
__device__ __forceinline__ void pend_flush(const Ctx &c, Pend &p, typename AR::sf_t sf, float2 *LeOut)
{
    float ea, eb;
    AR::make_extrinsic(p.uv, p.y[0], p.y[1], sf, ea, eb);
    if (p.idx >= 0) st_ws(LeOut + p.idx * 16 + c.f, make_float2(ea, eb));
    p.idx = -1;
}

// One recompute window of the "out" phase (all lanes in natural labels):
//   alpha lane: steps [w0, w0+len) of [0, M): Z = running beta, X = alpha from its checkpoint
//   beta lane:  steps [w0, w0+len) of [M, N): Z = beta from its checkpoint, X = running alpha
// First beta is walked down through the window and parked in shared memory, then alpha is walked up with the
// a-posteriori maxima and the float32 epilogue (one step late).  TM: the window's records are in TMEM — column
// block (wa + u) for the alpha lane, block (wa + len-1-u) for the beta lane (the high records are stored reversed).
template <class AR, bool TM>
__device__ __forceinline__ void window(const Ctx &c, int wa, int w0, int len, typename AR::sf_t sf,
                                       float2 *LeOut, int nslot, int nw0, int nlen, Pend &pend)
{
    Buf B;
    auto issue = [&](int u) {
        if (TM) { tm_ld8(c.tq + 8u * (wa + u), B.a); tm_ld8(c.tq + 8u * (wa + len - 1 - u), B.b); }
        else    smem_get(c, w0 + u, B.a);
    };
    auto complete = [&](float (&g)[8]) {
        if (TM) { tm_wait_ld(B.a); tm_wait_ld(B.b); }
#pragma unroll
        for (int i = 0; i < 8; ++i) g[i] = (TM && c.isb) ? B.b[i] : B.a[i];
    };
    YQ nq;
    if (nlen) yq_load(c, nw0, nlen, nq);                            // next window's Y: a window of time to arrive
    float g[8];
    float4 *ws = c.wstore() + c.lane;
    {
        float Z[16];
        issue(len - 1);
        slot_get(c.slotZ(), c.lane, Z);
        complete(g);
        slot_put(ws + (len - 1) * 128, 0, Z);
        issue(len - 2);
        pend_flush<AR>(c, pend, sf, LeOut);
        AR::bwd_step(Z, g);
        complete(g);
        for (int u = len - 2; u >= 0; --u) {
            slot_put(ws + u * 128, 0, Z);                           // beta[k+1]
            issue(u > 0 ? u - 1 : 0);                               // u == 0: first record of the way up
            AR::bwd_step(Z, g);
            complete(g);
        }
        if (!c.isb) slot_put(c.slotZ(), c.lane, Z);                 // running beta of the alpha lane
    }
    float X[16];
    slot_get(c.slotX(), c.lane, X);
    if (nslot >= 0) issue_ckpt(c, nslot);
    cpa_commit();
    float yr[2], yn[2], uvp[4], zs[16];
    tm_ld2(c.tq + c.ycol, yr);
    issue(len > 1 ? 1 : 0);
    slot_get(ws, 0, zs);
    AR::app_maxima(X, zs, g, uvp);                                  // step 0 (its Y is not needed before the next step's epilogue)
    AR::pass_step(X, g, false);
    tm_wait_ld2(yr);
    complete(g);
    for (int u = 1; u < len; ++u) {
        tm_ld2(c.tq + c.ycol + 2u * u, yn);
        issue(u + 1 < len ? u + 1 : u);
        slot_get(ws + u * 128, 0, zs);
        float uv[4];
        AR::app_maxima(X, zs, g, uv);
        AR::pass_step(X, g, false);
        float ea, eb;                                               // epilogue of step u-1
        AR::make_extrinsic(uvp, yr[0], yr[1], sf, ea, eb);
        st_ws(LeOut + (w0 + u - 1) * 16 + c.f, make_float2(ea, eb));
        tm_wait_ld2(yn);
        complete(g);
#pragma unroll
        for (int i = 0; i < 4; ++i) uvp[i] = uv[i];
        yr[0] = yn[0]; yr[1] = yn[1];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) pend.uv[i] = uvp[i];
    pend.y[0] = yr[0]; pend.y[1] = yr[1];
    pend.idx = w0 + len - 1;
    if (c.isb) slot_put(c.slotX(), c.lane, X);                      // running alpha of the beta lane
    if (nlen) yq_park(c, nq, nw0, nlen, nslot - 1);
}

// ---- the "in" pass: records built on the fly (prep fused), checkpoints every kW steps -------------------------
// Channel LLRs live in the workspace as [j][32 lanes] float4: lanes 0-15 hold step k = j of frames 0-15, lanes
// 16-31 step k = N-1-j.
__device__ __forceinline__ int lpos(const Ctx &c, int k, int fr) { return k < c.M ? k * 32 + fr : (c.N - 1 - k) * 32 + 16 + fr; }

struct Idx { int a, b; };
__device__ __forceinline__ void idx_get(const Ctx &c, int jn, const int16_t *tbl, Idx &x)
{
    jn = min(jn, c.M - 2);
    const int k0 = c.isb ? c.N - 1 - jn : jn, k1 = c.isb ? k0 - 1 : k0 + 1;
    x.a = tbl[k0]; x.b = tbl[k1];
}
// Ring slot of a step pair: [x A][la A][x B][la B], 512 B each, lane-major 16-byte entries (conflict-free for the
// cp.async writes and the LDS reads).  The float32 a-priori pair of a frame is 8 bytes; cp.async only bypasses L1
// (.cg) for 16-byte copies, and L1 must be bypassed because the extrinsics are rewritten in L2 every half
// iteration: the lane copies the 16-byte chunk that holds its frame's pair (shared with the neighbouring frame)
// and reads its half.
__device__ __forceinline__ void prep_load_pair(const Ctx &c, unsigned char *slot, int jn, const float4 *Lsrc,
                                               const Idx &x, bool first, int si)
{
    jn = min(jn, c.M - 2);                                          // clamped at the end: harmless re-computation
    const unsigned d = s_addr(slot) * c.one;
    const float4 *src = Lsrc + jn * 32 + c.lane;
#ifdef NII_BULK_CHAN
    // the channel LLRs of a step pair are ONE contiguous kilobyte: a bulk copy issued by one lane (TMA unit) instead of
    // two LDGSTS warp-instructions through the LSU.  Slot layout [x A][x B][la A][la B].
    if (c.lane == 0) {
        mbar_expect_tx(c.rmbar + 8u * si, 1024u);
        bulk_g2s_stream(slot, Lsrc + jn * 32, 1024u, c.rmbar + 8u * si, c.pol);
    }
    if (!first) {
        cpa16_off<1024, 0>(d, reinterpret_cast<const float4 *>(c.Le + x.a * 16) + (c.f >> 1));
        cpa16_off<1536, 0>(d, reinterpret_cast<const float4 *>(c.Le + x.b * 16) + (c.f >> 1));
    }
    return;
#endif
    // (NII_ABL_*: timing-only ablation builds for profiles/r02_nii_ablation.txt; never defined in the shipped library)
#ifndef NII_ABL_NOCHAN
    cpa16_stream_off<0, 0>(d, src, c.pol);
    cpa16_stream_off<1024, 512>(d, src, c.pol);
#endif
#ifndef NII_ABL_NOGATHER
    // the a-priori pair of a frame is 8 bytes and a 16-byte chunk holds two neighbouring frames: only the EVEN lanes
    // copy, into chunk (lane / 2) of the la block, and both lanes of the pair read their half (the cost of the global
    // path is per byte, profiles/r02_nii_ablation.txt: 256 B per step instead of 512 B)
    if (!first && (c.lane & 1) == 0) {
        const unsigned dl = d - 8u * (unsigned)c.lane;              // slot base + (lane / 2) * 16
        cpa16_off<512, 0>(dl, reinterpret_cast<const float4 *>(c.Le + x.a * 16) + (c.f >> 1));
        cpa16_off<1536, 0>(dl, reinterpret_cast<const float4 *>(c.Le + x.b * 16) + (c.f >> 1));
    }
#endif
}
struct Raw { float4 xA, xB; float2 laA, laB; };
template <bool FIRST>
__device__ __forceinline__ void raw_get(const Ctx &c, const unsigned char *slot, Raw &r)
{
#ifdef NII_BULK_CHAN
    constexpr int oXB = 512, oLA = 1024;
#else
    constexpr int oXB = 1024, oLA = 512;
#endif
    r.xA = *reinterpret_cast<const float4 *>(slot);
    r.xB = *reinterpret_cast<const float4 *>(slot + oXB);
    r.laA = r.laB = make_float2(0.f, 0.f);
    if (!FIRST) {
#ifdef NII_BULK_CHAN
        r.laA = *reinterpret_cast<const float2 *>(slot + oLA + c.h8);
        r.laB = *reinterpret_cast<const float2 *>(slot + 1536 + c.h8);
#else
        const unsigned char *la = slot - 8 * c.lane;                // chunk (lane / 2), this lane's half (h8 = 8 * (lane & 1)): + 8 * lane in total
        r.laA = *reinterpret_cast<const float2 *>(la + oLA);
        r.laB = *reinterpret_cast<const float2 *>(la + 1536);
#endif
    }
}
struct PrepRec { float gA[8], gB[8]; };                      // records of two consecutive steps
template <class AR>
__device__ __forceinline__ void prep_pair(const Ctx &c, const Raw &r, int jn, PrepRec &out)
{
    jn = min(jn, c.M - 2);
    const float2 YA = make_float2(AR::add(r.xA.x, r.laA.x), AR::add(r.xA.y, r.laA.y));  // Lc + La
    const float2 YB = make_float2(AR::add(r.xB.x, r.laB.x), AR::add(r.xB.y, r.laB.y));
#ifndef NII_ABL_NOPREP
    AR::make_record(YA.x, YA.y, r.xA.z, r.xA.w, out.gA);
    AR::make_record(YB.x, YB.y, r.xB.z, r.xB.w, out.gB);
#else
#pragma unroll
    for (int i = 0; i < 8; ++i) { out.gA[i] = i & 1 ? YA.x : r.xA.z; out.gB[i] = i & 1 ? YB.y : r.xB.w; }
#endif
    const int ke = c.isb ? c.N - 2 - jn : jn;                       // the even (lower) k of the pair
#ifndef NII_ABL_NOY
    st_ws(c.Yb + (ke >> 1) * 16 + c.f, c.isb ? make_float4(YB.x, YB.y, YA.x, YA.y) : make_float4(YA.x, YA.y, YB.x, YB.y));
#endif
}
struct PrepState { PrepRec r; Raw raw; Idx ix; int ps; unsigned rph; };
// steps jj, jj+1 with the records in `in`; builds the records of steps jj+2, jj+3 (raw inputs `rin`) into `out` and
// pulls the raw inputs of steps jj+4, jj+5 out of the ring into `rout`.  CK: a checkpoint is due before step jj.
template <class AR, bool FIRST, bool TMST, bool CK>
__device__ __forceinline__ void in_pair(const Ctx &c, int jj, const float4 *Lsrc, const int16_t *tbl,
                                        int &ps, unsigned &rph, const PrepRec &in, PrepRec &out, const Raw &rin, Raw &rout,
                                        const Idx &xin, Idx &xout, float (&v)[16])
{
    const int N = c.N;
    unsigned char *slot = c.stage + c.lane * 16 + ps * 2048;
    cpa_wait<kRingPairs - 1>();
#ifdef NII_BULK_CHAN
    mbar_wait(c.rmbar + 8u * ps, (rph >> ps) & 1u);
    rph ^= 1u << ps;
    const int si = ps;
#else
    const int si = 0;
#endif
#ifndef NII_ABL_NORAW
    raw_get<FIRST>(c, slot, rout);
#else
    rout = rin;
#endif
#ifdef NII_BULK_CHAN
    __syncwarp();                                                   // every lane has issued its reads of this slot
#endif
    prep_load_pair(c, slot, jj + 4 + 2 * kRingPairs, Lsrc, xin, FIRST, si);   // (lane 0's slot address is the slot base)
    cpa_commit();
    if (!FIRST) idx_get(c, jj + 6 + 2 * kRingPairs, tbl, xout);
    ps = ps == kRingPairs - 1 ? 0 : ps + 1;
    prep_pair<AR>(c, rin, jj + 2, out);
#ifndef NII_ABL_NOCK
    if (CK) ck_store(c, (c.M - jj) / kW - 1, v);
#endif
    const int k0 = c.isb ? N - 1 - jj : jj, k1 = c.isb ? N - 2 - jj : jj + 1;
#ifndef NII_ABL_NOREC
    if (TMST) tm_st8(c.tq + 8u * jj, in.gA);
    else      smem_put(c, k0, in.gA);
#endif
    AR::pass_step(v, in.gA, c.isb);
#ifndef NII_ABL_NOREC
    if (TMST) tm_st8(c.tq + 8u * (jj + 1), in.gB);
    else      smem_put(c, k1, in.gB);
#endif
    AR::pass_step(v, in.gB, c.isb);
}
template <class AR, bool FIRST, bool TMST, bool CKA, bool CKB>
__device__ __forceinline__ void in_loop(const Ctx &c, int j0, int j1, const float4 *Lsrc, const int16_t *tbl,
                                        PrepState &P, float (&v)[16])
{
    PrepRec Q;
    Raw RQ;
    Idx XQ = P.ix;
    int jj = j0;
    for (; jj + 4 <= j1; jj += 4) {                                 // ping-pong: no register copies
        in_pair<AR, FIRST, TMST, CKA>(c, jj, Lsrc, tbl, P.ps, P.rph, P.r, Q, P.raw, RQ, P.ix, XQ, v);
        in_pair<AR, FIRST, TMST, CKB>(c, jj + 2, Lsrc, tbl, P.ps, P.rph, Q, P.r, RQ, P.raw, XQ, P.ix, v);
    }
    if (jj < j1) {
        in_pair<AR, FIRST, TMST, CKA>(c, jj, Lsrc, tbl, P.ps, P.rph, P.r, Q, P.raw, RQ, P.ix, XQ, v);
        P.r = Q;
        P.raw = RQ;
        P.ix = XQ;
    }
}
// steps [j0, j1) (even count): a checkpoint wherever (M - j) is a multiple of kW = 4, i.e. every second pair
template <class AR, bool FIRST, bool TMST>
__device__ __forceinline__ void in_range(const Ctx &c, int j0, int j1, const float4 *Lsrc, const int16_t *tbl,
                                         PrepState &P, float (&v)[16])
{
    static_assert(kW == 4, "checkpoints alternate between the step pairs of a four-step body");
    if (j0 >= j1) return;
    if (((c.M - j0) % kW) == 0) in_loop<AR, FIRST, TMST, true, false>(c, j0, j1, Lsrc, tbl, P, v);
    else                        in_loop<AR, FIRST, TMST, false, true>(c, j0, j1, Lsrc, tbl, P, v);
}

template <class AR, bool FIRST>
__device__ __forceinline__ void in_pass(const Ctx &c, bool second, float (&v)[16], unsigned &rph)
{
    const float4 *Lsrc = second ? c.L2A : c.L1A;
    const int16_t *tbl = second ? c.perm : c.inv;                   // La = Le[perm k] / Le[inv k]
    unsigned char *ring = c.stage + c.lane * 16;
    PrepState P;
    P.ix.a = P.ix.b = 0;
    P.rph = rph;                                                    // phase parities of the ring mbarriers persist across calls
#pragma unroll 1
    for (int p = 0; p < kRingPairs; ++p) {                          // ring of step pairs
        if (!FIRST) idx_get(c, 2 * p, tbl, P.ix);
        prep_load_pair(c, ring + p * 2048, 2 * p, Lsrc, P.ix, FIRST, p);
        cpa_commit();
    }
    if (!FIRST) idx_get(c, 2 * kRingPairs, tbl, P.ix);
    cpa_wait<kRingPairs - 1>();
#ifdef NII_BULK_CHAN
    mbar_wait(c.rmbar, P.rph & 1u); P.rph ^= 1u;
#endif
    raw_get<FIRST>(c, ring, P.raw);                                 // steps 0, 1
    prep_pair<AR>(c, P.raw, 0, P.r);
#ifdef NII_BULK_CHAN
    __syncwarp();
#endif
    prep_load_pair(c, ring, 2 * kRingPairs, Lsrc, P.ix, FIRST, 0);
    cpa_commit();
    if (!FIRST) idx_get(c, 2 * kRingPairs + 2, tbl, P.ix);
    cpa_wait<kRingPairs - 1>();
#ifdef NII_BULK_CHAN
    mbar_wait(c.rmbar + 8u, (P.rph >> 1) & 1u); P.rph ^= 2u;
#endif
    raw_get<FIRST>(c, ring + 2048, P.raw);                          // steps 2, 3
#ifdef NII_BULK_CHAN
    __syncwarp();
#endif
    prep_load_pair(c, ring + 2048, 2 * kRingPairs + 2, Lsrc, P.ix, FIRST, 1);
    cpa_commit();
    if (!FIRST) idx_get(c, 2 * kRingPairs + 4, tbl, P.ix);
    P.ps = 2 % kRingPairs;
    if ((c.M % kW) != 0) ck_store(c, c.M / kW, v);                  // the ragged last window starts at step 0
    in_range<AR, FIRST, true>(c, 0, c.T, Lsrc, tbl, P, v);
    in_range<AR, FIRST, false>(c, c.T, c.M, Lsrc, tbl, P, v);
    cpa_wait<0>();
#ifdef NII_BULK_CHAN
    // the ring runs kRingPairs (clamped) pairs ahead: one fill per slot is still outstanding.  It must land before the
    // staging area is reused for the windows' beta vectors, and its phase must be consumed to keep the parities in step.
#pragma unroll 1
    for (int i = 0; i < kRingPairs; ++i) { mbar_wait(c.rmbar + 8u * i, (P.rph >> i) & 1u); P.rph ^= 1u << i; }
#endif
    rph = P.rph;
}

// One SISO half-iteration for the 16 frames of this warp.
template <class AR, bool TIMED>
__device__ __forceinline__ void siso(const Ctx &c, bool second, bool first, bool last, bool first_iter, typename AR::sf_t sf, long long (&ph)[8], unsigned &rph)
{
    long long tA = TIMED ? clock64() : 0;
    const int N = c.N, M = c.M, T = c.T, lane = c.lane;
    float2 *LeOut = last ? c.LeF : c.Le;
    float4 *init = c.INIT + (second ? 128 : 0);
    float v[16];
    // ---- boundary metrics: alpha[0] / beta[N] = what this constituent decoder reached one iteration earlier ----
    if (first_iter) {
#pragma unroll
        for (int s = 0; s < 16; ++s) v[s] = 0.f;
    } else {
        float n[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 t = ld_ws4(init + q * 32 + lane);
            n[4 * q] = t.x; n[4 * q + 1] = t.y; n[4 * q + 2] = t.z; n[4 * q + 3] = t.w;
        }
#pragma unroll
        for (int s = 0; s < 16; ++s) v[s] = c.isb ? n[rho4(s)] : n[s];
    }
    if (TIMED) { const long long t = clock64(); ph[2] += t - tA; tA = t; }
    // ---- the "in" pass ------------------------------------------------------------------------------------------
    if (first) in_pass<AR, true>(c, second, v, rph);
    else       in_pass<AR, false>(c, second, v, rph);
    tm_wait_st();
    __syncwarp();
    if (!first && !last)                                            // old extrinsics are dead: every line is rewritten below
        for (int i = lane; i < N; i += 32) l2_discard(c.Le + i * 16);
    if (TIMED) { const long long t = clock64(); ph[1] += t - tA; tA = t; }
    const int nfull = M / kW, rag = M % kW, nwin = nfull + (rag ? 1 : 0);
    auto win_w0 = [&](int i) { return i < nfull ? (c.isb ? M + i * kW : M - (i + 1) * kW) : (c.isb ? N - rag : 0); };
    auto win_len = [&](int i) { return i < nfull ? kW : rag; };
    // ---- crossing: the half-warps swap chains (beta lanes back to natural labels): every lane drops its vector
    //      into the PARTNER's slot ----------------------------------------------------------------------------
    {
        float n[16];
#pragma unroll
        for (int s = 0; s < 16; ++s) n[s] = c.isb ? v[rho4(s)] : v[s];
        slot_put(c.isb ? c.slotZ() : c.slotX(), lane ^ 16, n);
    }
    {
        YQ q0;
        yq_load(c, win_w0(0), win_len(0), q0);
        issue_ckpt(c, 0);
        cpa_commit();
        yq_park(c, q0, win_w0(0), win_len(0), -1);
    }
    const int n_inner = (M - T) / kW;            // windows whose records are in shared memory
    if (TIMED) { const long long t = clock64(); ph[2] += t - tA; tA = t; }
    // ---- out phase: windows from the crossing point outwards ---------------------------------------------------
    Pend pend;
#pragma unroll
    for (int i = 0; i < 4; ++i) pend.uv[i] = 0.f;
    pend.y[0] = pend.y[1] = 0.f;
    pend.idx = -1;
    for (int i = 0; i < nwin; ++i) {
        cpa_wait<0>();
        __syncwarp();
        const int wa = i < nfull ? M - (i + 1) * kW : 0;
        const int nlen = i + 1 < nwin ? win_len(i + 1) : 0;
        const int nw0 = i + 1 < nwin ? win_w0(i + 1) : 0;
        if (i < n_inner) window<AR, false>(c, wa, win_w0(i), win_len(i), sf, LeOut, nlen ? i + 1 : -1, nw0, nlen, pend);
        else             window<AR, true>(c, wa, win_w0(i), win_len(i), sf, LeOut, nlen ? i + 1 : -1, nw0, nlen, pend);
        if (TIMED && i == n_inner - 1) { const long long t = clock64(); ph[4] += t - tA; tA = t; }
    }
    pend_flush<AR>(c, pend, sf, LeOut);
    cpa_wait<0>();
    __syncwarp();
    if (TIMED) { const long long t = clock64(); ph[5] += t - tA; tA = t; }
    // ---- boundary metrics for the next iteration: the alpha lane ended with beta[0] (its Z slot), the beta lane
    //      with alpha[N] (its X slot); each is what the PARTNER lane starts from -------------------------------
    if (!last) {
        const float4 *src = (c.isb ? c.slotX() : c.slotZ());
#pragma unroll
        for (int q = 0; q < 4; ++q) st_ws(init + q * 32 + (lane ^ 16), src[q * 32 + lane]);
    }
    if (TIMED) { const long long t = clock64(); ph[2] += t - tA; tA = t; }
}

template <class AR, bool TIMED, class LlrT>
__global__ void __launch_bounds__(kTpfWarps * 32, 1)
nii_kernel(const NiiArgs A)
{
    constexpr int kFpl = AR::kFpl;                                  // frames per lane
    constexpr int kTile = kTpfFrames * kFpl;                        // frames per warp tile: sub-frame i of lane f is frame 16 i + f
    const typename AR::sf_t sf_inner = kFpl == 2 ? (typename AR::sf_t)A.sf_inner_q : (typename AR::sf_t)A.sf_inner;
    const typename AR::sf_t sf_last = kFpl == 2 ? (typename AR::sf_t)A.sf_last_q : (typename AR::sf_t)A.sf_last;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const TpfGeom g = A.g;
    const int N = g.N;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int16_t *tab = reinterpret_cast<int16_t *>(smem_raw);
    const int tab_bytes = ((2 * N * 2 + 15) / 16) * 16;
    unsigned *tmem_slot = reinterpret_cast<unsigned *>(smem_raw + tab_bytes);
    float4 *srec_all = reinterpret_cast<float4 *>(smem_raw + tab_bytes + kHdrBytes);   // 32 B of slots + four 8-byte mbarriers (+ ring mbarriers)
    unsigned char *stage_all = reinterpret_cast<unsigned char *>(srec_all + (size_t)kTpfWarps * g.mid * 2 * 16);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"((unsigned)__cvta_generic_to_shared(tmem_slot)), "r"(g.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < 2 * N; i += blockDim.x) tab[i] = A.tab[i];
    const unsigned mbar = (unsigned)__cvta_generic_to_shared(smem_raw + tab_bytes + 32 + 8 * warp);   // this warp's mbarrier
    unsigned mphase = 0, rph = 0;
    if (lane == 0) {
        mbar_init(mbar, 1);
        for (int i = 0; i < kRingPairs; ++i) mbar_init((unsigned)__cvta_generic_to_shared(smem_raw + tab_bytes + 64 + 8 * (warp * kRingPairs + i)), 1);
        mbar_fence_init();
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem_base = *tmem_slot;

    Ctx c;
    c.N = N; c.M = g.M; c.T = g.T;
    c.f = lane & 15; c.isb = lane >> 4; c.lane = lane; c.h8 = (lane & 1) * 8;
    c.tq = tmem_base + (((unsigned)warp * 32u) << 16);
    c.ycol = 8u * g.T;
    c.srec = srec_all + (size_t)warp * g.mid * 2 * 16;
    {   // the staging base goes through memory (see cpa16: no [R+UR+imm] operand for LDGSTS)
        volatile unsigned *slots = reinterpret_cast<volatile unsigned *>(smem_raw + tab_bytes);
        if (lane == 0) { slots[4 + warp] = (unsigned)warp * kStageBytes; slots[1] = 1u; }
        __syncwarp();
        c.stage = stage_all + slots[4 + warp];
        c.one = slots[1];
        __syncwarp();
    }
    c.rmbar = (unsigned)__cvta_generic_to_shared(smem_raw + tab_bytes + 64 + 8 * warp * kRingPairs);
    c.perm = tab; c.inv = tab + N;
    const int wg = blockIdx.x * kTpfWarps + warp;
    unsigned char *ws = A.ws + (size_t)wg * g.ws_per_warp;
    c.L1A = reinterpret_cast<float4 *>(ws + g.off_l1);
    c.L2A = reinterpret_cast<float4 *>(ws + g.off_l2);
    c.Le = reinterpret_cast<float2 *>(ws + g.off_le);
    c.LeF = reinterpret_cast<float2 *>(ws + g.off_lef);
    c.Yb = reinterpret_cast<float4 *>(ws + g.off_y);
    c.CK = reinterpret_cast<float4 *>(ws + g.off_ck);
    c.INIT = reinterpret_cast<float4 *>(ws + g.off_init);
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(c.pol));
    const int16_t *g_off = A.tab + 2 * N;        // offA, offW1, offY1, offW2, offY2 (global, read-only)

    unsigned long long bit_err = 0, frm_err = 0, frames_done = 0;
    long long ph[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const long long t_begin = TIMED ? clock64() : 0;
    for (int tile = wg; tile < A.n_tiles; tile += gridDim.x * kTpfWarps) {
        const long long frame0 = (long long)tile * kTile;
        const long long t0 = TIMED ? clock64() : 0;
        const float sc = A.llr_scale;                               // int8 input only (llr_f32)
        // ---- de-puncture + transpose the 16 frames' LLRs into [j][lane] (as decode_tpf.cu) ------------------
        if (A.vec4) {
            const int nq = llr_row_q<LlrT>(A.n_llr);                // float4 per row (row pitch is a multiple of 16 B)
            const int pitch4 = ((nq + 6) & ~7) + 1;                 // row pitch = 4 (mod 32) words: rows land in different banks
            const int rec_bytes = g.mid * 2 * 16 * (int)sizeof(float4);
            const bool in_rec = rec_bytes > kStageBytes;
            float4 *rowbuf = in_rec ? c.srec : reinterpret_cast<float4 *>(c.stage);
            const int fit = (in_rec ? rec_bytes : kStageBytes - N * 16) / (pitch4 * 16);
            // G rows are staged at once: GL = G / kFpl lane-frames x kFpl sub-frames (row r < GL: frame g0 + r, row
            // GL + r: frame 16 + g0 + r).  Lane = (couple kq, lane-frame fr) with fr the minor index.
            const int lg = fit >= 8 ? 3 : fit >= 4 ? 2 : 1, G = 1 << lg;
            const int lgl = kFpl == 2 ? lg - 1 : lg, GL = 1 << lgl, KQ = 32 >> lgl;
            const int fr = lane & (GL - 1), kq = lane >> lgl;
            int4 *otab = reinterpret_cast<int4 *>(in_rec ? c.stage : c.stage + G * pitch4 * 16);
            for (int k = lane; k < N; k += 32) {
                const unsigned oa = (unsigned short)__ldg(g_off + k), op = (unsigned short)__ldg(g_off + c.perm[k]);
                const unsigned o0 = (unsigned short)__ldg(g_off + N + k), o1 = (unsigned short)__ldg(g_off + 2 * N + k);
                const unsigned o2 = (unsigned short)__ldg(g_off + 3 * N + k), o3 = (unsigned short)__ldg(g_off + 4 * N + k);
                otab[k] = make_int4((int)(oa | (op << 16)), (int)(o0 | (o1 << 16)), (int)(o2 | (o3 << 16)), 0);
            }
            // whole rows by bulk copy (cp.async.bulk: one instruction of one lane per 5 KB row, completed on this
            // warp's mbarrier) — the rows are the longest contiguous transfers of the kernel
            auto row_frame = [&](int g0, int r) { return frame0 + (r < GL ? g0 + r : kTpfFrames + g0 + r - GL); };
            auto pull = [&](int g0) {
                if (lane == 0) {
                    int live_rows = 0;
                    for (int r = 0; r < G; ++r) live_rows += row_frame(g0, r) < A.B;
                    fence_proxy_async();                            // the row buffer was read (or held records) before
                    mbar_expect_tx(mbar, (unsigned)(live_rows * nq * 16));
                    for (int r = 0; r < G; ++r)
                        if (row_frame(g0, r) < A.B)
                            bulk_g2s_stream(rowbuf + r * pitch4, static_cast<const LlrT *>(A.llr) + row_frame(g0, r) * A.llr_stride, (unsigned)(nq * 16), mbar, c.pol);
                }
            };
            pull(0);
            if (A.ref_bits) {                                       // the hard decision will want these rows in L2
                const int lines = (2 * N * kTile + 127) / 128;
                const long long nb = min((long long)kTile, A.B - frame0) * 2 * N;
                for (int i = lane; i < lines; i += 32)
                    if ((long long)i * 128 < nb) asm volatile("prefetch.global.L2 [%0];" ::"l"(A.ref_bits + frame0 * 2 * N + i * 128));
            }
            const LlrT *row = reinterpret_cast<const LlrT *>(rowbuf + fr * pitch4);
            const LlrT *rowh = reinterpret_cast<const LlrT *>(rowbuf + (GL + fr) * pitch4);   // sub-frame 1 (kFpl == 2)
            for (int g0 = 0; g0 < kTpfFrames; g0 += GL) {
                mbar_wait(mbar, mphase);
                mphase ^= 1u;
                const bool livef = frame0 + g0 + fr < A.B;
                const bool liveh = kFpl == 2 && frame0 + kTpfFrames + g0 + fr < A.B;
                auto val = [&](int o) { return AR::chan(livef ? llr_f32(row[o], sc) : 0.f, liveh ? llr_f32(rowh[o], sc) : 0.f); };
#pragma unroll 4
                for (int k0 = 0; k0 < N; k0 += KQ) {
                    const int k = k0 + kq;
                    const int4 e = otab[min(k, N - 1)];
                    const int oa = (short)(e.x & 0xffff), op = e.x >> 16, o0 = (short)(e.y & 0xffff), o1 = e.y >> 16;
                    const int o2 = (short)(e.z & 0xffff), o3 = e.z >> 16;
                    const float zero = AR::chan(0.f, 0.f);
                    float4 x1 = make_float4(zero, zero, zero, zero), x2 = x1;
                    x1.x = val(oa); x1.y = val(oa + 1); x2.x = val(op); x2.y = val(op + 1);
                    if (o0 >= 0) x1.z = val(o0);
                    if (o1 >= 0) x1.w = val(o1);
                    if (o2 >= 0) x2.z = val(o2);
                    if (o3 >= 0) x2.w = val(o3);
                    if (k < N) {
                        st_ws(c.L1A + lpos(c, k, g0 + fr), x1);
                        st_ws(c.L2A + lpos(c, k, g0 + fr), x2);
                    }
                }
                __syncwarp();
                if (g0 + GL < kTpfFrames) pull(g0 + GL);
            }
        } else
        for (int k = lane; k < N; k += 32) {
            const int oa = __ldg(g_off + k), op = __ldg(g_off + c.perm[k]);
            const int o0 = __ldg(g_off + N + k), o1 = __ldg(g_off + 2 * N + k);
            const int o2 = __ldg(g_off + 3 * N + k), o3 = __ldg(g_off + 4 * N + k);
            for (int fr = 0; fr < kTpfFrames; ++fr) {
                const long long fl_ = frame0 + fr, fh_ = frame0 + kTpfFrames + fr;
                const bool livef = fl_ < A.B, liveh = kFpl == 2 && fh_ < A.B;
                const LlrT *Lf = static_cast<const LlrT *>(A.llr) + (livef ? fl_ : 0) * A.llr_stride;
                const LlrT *Lh = static_cast<const LlrT *>(A.llr) + (liveh ? fh_ : 0) * A.llr_stride;
                auto val = [&](int o) { return AR::chan(livef ? llr_ldg(Lf + o, sc) : 0.f, liveh ? llr_ldg(Lh + o, sc) : 0.f); };
                const float zero = AR::chan(0.f, 0.f);
                float4 x1 = make_float4(zero, zero, zero, zero), x2 = x1;
                x1.x = val(oa); x1.y = val(oa + 1); x2.x = val(op); x2.y = val(op + 1);
                if (o0 >= 0) x1.z = val(o0);
                if (o1 >= 0) x1.w = val(o1);
                if (o2 >= 0) x2.z = val(o2);
                if (o3 >= 0) x2.w = val(o3);
                st_ws(c.L1A + lpos(c, k, fr), x1);
                st_ws(c.L2A + lpos(c, k, fr), x2);
            }
        }
        __syncwarp();
        if (TIMED) ph[0] += clock64() - t0;
        for (int h = 0; h < 2 * A.iterations; ++h) {
            const typename AR::sf_t sf = (h >> 1) < A.iterations - 1 ? sf_inner : sf_last;
            siso<AR, TIMED>(c, (h & 1) != 0, h == 0, h == 2 * A.iterations - 1, h < 2, sf, ph, rph);
        }
        const long long t6 = TIMED ? clock64() : 0;
        // ---- hard decision: (Lc + La) + Le1 < 0 in float32 + optional error counting ----------------------
        long long frame[kFpl];
        bool live[kFpl], cnt[kFpl];
        const uint8_t *refp[kFpl];
        int any_err[kFpl];
        unsigned word[kFpl];
#pragma unroll
        for (int i = 0; i < kFpl; ++i) {
            frame[i] = frame0 + kTpfFrames * i + c.f;
            live[i] = frame[i] < A.B;
            cnt[i] = live[i] && A.ref_bits != nullptr;
            refp[i] = cnt[i] ? A.ref_bits + (size_t)frame[i] * 2 * N : reinterpret_cast<const uint8_t *>(A.tab);
            any_err[i] = 0;
            word[i] = 0;
        }
        const int wpf = (2 * N + 31) / 32;
        constexpr int kHB = 3 * 8 * 32 * 16;                        // bytes of one staged batch: [array][t][lane] x 16 B
        const int rec_bytes_h = g.mid * 2 * 16 * (int)sizeof(float4);
        unsigned char *hbuf = rec_bytes_h >= kHB ? reinterpret_cast<unsigned char *>(c.srec) : c.stage;
        const int nst = rec_bytes_h >= 3 * kHB ? 3 : rec_bytes_h >= 2 * kHB ? 2 : 1;
        const int nwords = (N + 15) / 16;                           // == wpf
        const int nbu = 2 * ((nwords + 1) / 2);                     // batches of the alpha half (the beta half may idle through the last word)
        auto hissue = [&](int b, int st) {
            if (b < nbu) {
                const int kb = (c.isb + 2 * (b >> 1)) * 16 + 8 * (b & 1);
                const unsigned d = s_addr(hbuf + st * kHB + lane * 16) * c.one;
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    const int k = min(kb + t, N - 1);
                    const unsigned dt = d + t * 512;
                    cpa16_off<0, 0>(dt, c.L1A + lpos(c, k, c.f));
                    cpa16_off<4096, 0>(dt, reinterpret_cast<const float4 *>(c.LeF + c.inv[k] * 16) + (c.f >> 1));
                    cpa16_off<8192, 0>(dt, reinterpret_cast<const float4 *>(c.Le + k * 16) + (c.f >> 1));
                }
            }
            cpa_commit();
        };
        for (int b = 0; b < nst; ++b) hissue(b, b);
        for (int b = 0, st = 0; b < nbu; ++b) {
            if (nst == 3) cpa_wait<2>(); else if (nst == 2) cpa_wait<1>(); else cpa_wait<0>();
            const int kb = (c.isb + 2 * (b >> 1)) * 16 + 8 * (b & 1);
            const unsigned char *src = hbuf + st * kHB + lane * 16;
            unsigned short rb[kFpl][8];
#pragma unroll
            for (int i = 0; i < kFpl; ++i)
#pragma unroll
                for (int t = 0; t < 8; ++t) rb[i][t] = *reinterpret_cast<const unsigned short *>(refp[i] + 2 * min(kb + t, N - 1));
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const int k = kb + t;
                const float4 ab = *reinterpret_cast<const float4 *>(src + t * 512);
                const float2 la = *reinterpret_cast<const float2 *>(src + 4096 + t * 512 + c.h8);
                const float2 e1 = *reinterpret_cast<const float2 *>(src + 8192 + t * 512 + c.h8);
                const float LA = AR::add(AR::add(ab.x, la.x), e1.x);
                const float LB = AR::add(AR::add(ab.y, la.y), e1.y);
#pragma unroll
                for (int i = 0; i < kFpl; ++i) {
                    const int bA = AR::neg(LA, i), bB = AR::neg(LB, i);
                    if (k < N) {
                        word[i] |= (unsigned)(bA | (bB << 1)) << (2 * (8 * (b & 1) + t));
                        if (live[i] && A.bits)
                            *reinterpret_cast<int2 *>(A.bits + (size_t)frame[i] * 2 * N + 2 * k) = make_int2(bA, bB);
                        if (cnt[i]) {
                            const int errs = (bA != (rb[i][t] & 0xff)) + (bB != (rb[i][t] >> 8));
                            bit_err += errs;
                            any_err[i] |= errs;
                        }
                    }
                }
            }
            hissue(b + nst, st);                                    // refill the slot just read (same lane, same LSU queue: ordered)
            st = st + 1 == nst ? 0 : st + 1;
            if (b & 1) {
                const int w = c.isb + b - 1;
#pragma unroll
                for (int i = 0; i < kFpl; ++i) {
                    if (live[i] && A.packed && w < nwords) A.packed[(size_t)frame[i] * wpf + w] = word[i];
                    word[i] = 0;
                }
            }
        }
        cpa_wait<0>();
#pragma unroll
        for (int i = 0; i < kFpl; ++i) {
            any_err[i] |= __shfl_xor_sync(0xffffffffu, any_err[i], 16);
            if (live[i] && !c.isb) { frames_done += 1; frm_err += any_err[i] ? 1 : 0; }
        }
        __syncwarp();
        if (TIMED) ph[6] += clock64() - t6;
    }
    if (TIMED && lane == 0) {
        ph[7] = clock64() - t_begin;
        for (int i = 0; i < 8; ++i) atomicAdd(&g_nii_cycles[i], (unsigned long long)ph[i]);
    }
    if (A.counters) {
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
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(g.tmem_cols) : "memory");
}

}  // namespace

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
int nii_configure(Codec &c, size_t smem_optin)
{
    tpf_family_geometry(c.nii, c.N, 2 * kW, kHdrBytes, sizeof(float2), true, smem_optin);
    if (!c.nii.enabled) return B200DVB_OK;
    return for_each_llr_type([&](auto t) {
        using L = decltype(t);
        B2_CUDA(cudaFuncSetAttribute(nii_kernel<ArF32, false, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin));
        B2_CUDA(cudaFuncSetAttribute(nii_kernel<ArF32, true, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin));
        B2_CUDA(cudaFuncSetAttribute(nii_kernel<ArS16, false, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin));
        B2_CUDA(cudaFuncSetAttribute(nii_kernel<ArS16, true, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin));
        return B200DVB_OK;
    });
}

int nii_read_phase_cycles(double *out_h, int reset) { return read_phase_cycles(g_nii_cycles, out_h, reset); }

static int nii_tile(const Codec &c) { return c.opt_mode == B200DVB_MODE_NII16 ? 2 * kTpfFrames : kTpfFrames; }

size_t nii_workspace_bytes(const Codec &c, int B) { return tpf_family_workspace_bytes(c, c.nii, B, nii_tile(c)); }

int nii_launch_decode(const Codec &c, const DecodeIo &io)
{
    if (io.ws_bytes < nii_workspace_bytes(c, io.B)) return B200DVB_ENOMEM;
    NiiArgs A{};
    fill_decode_args(A, c, io);
    A.g = c.nii;
    const bool fixed = c.opt_mode == B200DVB_MODE_NII16;
    A.n_tiles = (io.B + nii_tile(c) - 1) / nii_tile(c);
    A.n_llr = c.n_llr;
    A.vec4 = tpf_family_row_staging(c, c.nii, io);
    A.sf_inner = (float)c.sf_inner; A.sf_last = (float)c.sf_last;
    A.sf_inner_q = (int)lrint(c.sf_inner * 64.0); A.sf_last_q = (int)lrint(c.sf_last * 64.0);   // Q6: 45 and 64 for 0.7 / 1.0
    A.ws = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(io.ws) + 255) & ~(uintptr_t)255);
    const int grid = tpf_family_grid(c, io.B, nii_tile(c));
    const size_t smem = c.nii.smem_bytes;
    const bool timed = c.opt_phase_timers != 0;
    with_llr_type(io.fmt, [&](auto t) {
        using L = decltype(t);
        if (fixed) {
            if (timed) nii_kernel<ArS16, true, L><<<grid, kTpfWarps * 32, smem, io.stream>>>(A);
            else       nii_kernel<ArS16, false, L><<<grid, kTpfWarps * 32, smem, io.stream>>>(A);
        } else {
            if (timed) nii_kernel<ArF32, true, L><<<grid, kTpfWarps * 32, smem, io.stream>>>(A);
            else       nii_kernel<ArF32, false, L><<<grid, kTpfWarps * 32, smem, io.stream>>>(A);
        }
    });
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

}  // namespace b200dvb
