// decode_tpf.cu — thread-per-frame ("TPF") max-log-MAP turbo decoder, bit-exact with the
// reference (dvb_rcs2_turbo.py:116-281 bcjr_max_log_map, :464-537 decode).
//
// Why (DESIGN.md §4.1): a thread that holds all 16 state metrics of one frame and one
// direction needs no shuffle and no shared-memory exchange — a trellis step is 32 adds +
// 16 FMNMX + 15 subtractions of straight-line code with 16-way instruction-level parallelism,
// issued as 24 packed FADD2 (two lanes per instruction, tpf_core.cuh) + 16 FMNMX, so ONE warp per
// SM sub-partition keeps the issue port busy (measured: 62.5 cycles per step, 77.6 unpacked).  What
// kept this mapping out of reach was storage: 32 B of branch metrics per step per frame,
// 64 frames per SM to feed four warps = 434 KB.  Here the SM's two on-chip memories are
// pooled: tensor memory (256 KB, otherwise idle — the decoder has no MMA) holds the records
// of the outer T steps of either frame end, shared memory the middle ones.
//
// Mapping:
//   * CTA = 4 warps, one per sub-partition / TMEM lane quadrant; a warp owns 16 frames for
//     the whole decode and never synchronises with the other warps.
//   * lane f (< 16) = forward (alpha) thread of frame f, lane 16 + f = backward (beta) thread
//     of the same frame.  During the two "in" passes the beta lanes work in bit-reversed
//     state labels, which gives their recursion the alpha wiring (tpf_core.cuh): one
//     instruction stream serves both half-warps.
//   * records [0, T) of frame f live in TMEM lane f (column 8k), records [N-T, N) in TMEM lane
//     16 + f in REVERSED order (column 8(N-1-k)): while alpha walks up and beta walks down,
//     both read "their" record with one tcgen05.ld.32x32b at the same column.  Where the
//     accesses cross (end of pass 1) tcgen05.ld.16x32bx2 lets thread f and thread 16 + f read
//     the same TMEM lane.
//   * prep (gather, a-priori add, float64 branch sums) is fused into the first half of pass
//     1: the alpha lane builds records 0.., the beta lane N-1.. exactly when it needs them.
//   * meet in the middle (M = N/2) with a checkpoint every 4 steps; after the crossing the
//     half-warps swap chains through their staging slots: the alpha lane walks beta down over
//     [0, M), the beta lane walks alpha up over [M, N), each re-computing the other direction 4
//     steps at a time from its OWN checkpoints (same operations, same order: exact).  The
//     extrinsic epilogue (float64) is fused into that walk; a-priori / extrinsic values live
//     in an L2-resident workspace laid out [step][frame] so every access is coalesced.
#include "common.cuh"
#include "tpf_core.cuh"
#include "tpf_dev.cuh"

namespace b200dvb {

namespace {

using namespace tpf;

constexpr int kW = kTpfWin;

// phase timers (SM cycles summed over warps): 0 transpose-in, 1 pass 1 first half (+prep), 2 pass 1
// second half, 3 pass 2 to the crossing, 4 out-phase windows in shared memory, 5 out-phase windows
// in tensor memory, 6 hard decision, 7 warp total
__device__ unsigned long long g_tpf_cycles[8];

struct TpfArgs {
    TpfGeom g;
    int B, iterations, n_tiles, n_llr, vec4;
    double sf_inner, sf_last;
    const int16_t *tab;
    const void *llr;                 // [B][llr_stride] elements of the kernel's LlrT (float32, binary16 or int8)
    long long llr_stride;
    int32_t *bits;
    uint32_t *packed;
    const uint8_t *ref_bits;
    unsigned long long *counters;
    unsigned char *ws;
    float llr_scale;                 // int8 element q is the LLR q * llr_scale (last: the other members keep their offsets)
    float *app;                      // [B][2N] a-posteriori LLRs (float2 per couple) or NULL; last, for the same reason
};

struct Ctx {
    int N, M, T;
    int f, isb, lane;                // frame within the tile, 0 = alpha lane / 1 = beta lane
    unsigned tq;                     // TMEM address of this warp's lane quadrant, column 0
    unsigned ycol;                   // first of the 4 kW spare TMEM columns that park the window's Y
    float4 *srec;                    // this warp's shared-memory records: [(k - T) * 2 + half][16 frames]
    unsigned char *stage;            // this warp's staging area (kStageBytes)
    const int16_t *perm, *inv;       // shared-memory copies of the interleaver tables
    float4 *L1A, *L2A;               // de-punctured channel LLRs [k][16]: (A,B,W1,Y1)[k] and (A,B)[perm k],(W2,Y2)[k]
    double2 *Le, *LeF, *Yb;          // extrinsics [k][16] (in place; last half-iteration -> LeF); Y = Lc + La, [k/2][16] x 32 B
    float4 *CK;                      // checkpoints [slot][4][32 lanes]
    unsigned long long pol;          // L2 evict-first policy for the channel LLRs
    unsigned one;                    // 1, opaque to the compiler (see cpa16)
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

// ---- record fetch during the "in" passes, split into issue / complete so that the load of
//      step j+1 is in flight while step j computes.  The alpha lane is at k = j, the beta lane
//      at k = N-1-j.  KIND 0: TMEM, same column for both half-warps; 1: shared memory;
//      2: TMEM crossed (alpha wants the partner's lane 16+f, beta lane f; same column). ----------
struct Buf { float a[8], b[8]; };
template <int KIND> __device__ __forceinline__ void pf_issue(const Ctx &c, int j, Buf &B)
{
    if (KIND == 0) tm_ld8(c.tq + 8u * j, B.a);
    if (KIND == 1) smem_get(c, c.isb ? c.N - 1 - j : j, B.a);
    if (KIND == 2) {
        const unsigned col = 8u * (c.N - 1 - j);
        tm_ld8_half(c.tq + col, B.b);                  // every thread <- lanes 0..15  (what the beta lanes want)
        tm_ld8_half(c.tq + (16u << 16) + col, B.a);    // every thread <- lanes 16..31 (what the alpha lanes want)
    }
}
template <int KIND> __device__ __forceinline__ void pf_complete(const Ctx &c, Buf &B, float (&g)[8])
{
    if (KIND == 0) tm_wait_ld(B.a);
    if (KIND == 2) { tm_wait_ld(B.a); tm_wait_ld(B.b); }
#pragma unroll
    for (int i = 0; i < 8; ++i) g[i] = (KIND == 2 && c.isb) ? B.b[i] : B.a[i];
}

// Vectors leave the registers in the order of the step that resumes them: beta vectors in natural state order, whose
// neighbours (z[2t], z[2t+1]) are the pairs of the packed bwd_step; alpha vectors in pair order, position p holding
// state apos(p) = (x0, x8, x1, x9, ...), the pairs (x[t], x[8+t]) of the packed forward steps.  Either way a 16-byte
// access moves two register pairs and the out phase needs no moves to rebuild them.
__device__ __forceinline__ constexpr int apos(int p) { return (p >> 1) | ((p & 1) << 3); }
// the vector of an "in" pass in its stored order: the beta lanes hold rho4 labels during the passes, and
// rho4(2t + 1) == rho4(2t) + 8, so both half-warps store the same kind of pair (v[t], v[8+t])
__device__ __forceinline__ void pass_out(const Ctx &c, const float (&v)[16], float (&n)[16])
{
#pragma unroll
    for (int p = 0; p < 16; ++p) n[p] = c.isb ? v[rho4(p)] : v[apos(p)];
}
__device__ __forceinline__ void ck_store(const Ctx &c, int slot, const float (&v)[16])
{
    float n[16];
    pass_out(c, v, n);
#pragma unroll
    for (int q = 0; q < 4; ++q)
        st_ws(c.CK + (slot * 4 + q) * 32 + c.lane, make_float4(n[4 * q], n[4 * q + 1], n[4 * q + 2], n[4 * q + 3]));
}

// steps [j0, j1) of an "in" pass (j1 - j0 even), records of storage class KIND; CKPT: store a
// checkpoint wherever (M - j) is a multiple of kW (pass 2 only; those j are even)
// steps j, j+1 of an "in" pass with the record of step j in g; leaves the record of step j+2 in g.  Loads past the
// end are clamped (a harmless re-read).  CK: a checkpoint is due before step j — a compile-time fact, so that the
// body stays ONE basic block (a branch around the store keeps the scheduler from interleaving across it)
template <int KIND, bool CK>
__device__ __forceinline__ void pass_two(const Ctx &c, int j, int j1, Buf &B0, Buf &B1, float (&g)[8], float (&v)[16])
{
    pf_issue<KIND>(c, j + 1, B1);
    if (CK) ck_store(c, (c.M - j) / kW - 1, v);
    pass_step(v, g, c.isb);
    pf_complete<KIND>(c, B1, g);
    pf_issue<KIND>(c, min(j + 2, j1 - 1), B0);
    pass_step(v, g, c.isb);
    pf_complete<KIND>(c, B0, g);
}
template <int KIND, bool CKA, bool CKB>
__device__ __forceinline__ void pass_loop(const Ctx &c, int j0, int j1, Buf &B0, Buf &B1, float (&g)[8], float (&v)[16])
{
    int j = j0;
    for (; j + 4 <= j1; j += 4) {                                   // four steps per iteration: loop overhead and the
        pass_two<KIND, CKA>(c, j, j1, B0, B1, g, v);                // instruction-fetch bubble of the back edge amortised
        pass_two<KIND, CKB>(c, j + 2, j1, B0, B1, g, v);
    }
    if (j < j1) pass_two<KIND, CKA>(c, j, j1, B0, B1, g, v);
}
// steps [j0, j1) of an "in" pass (j1 - j0 even), records of storage class KIND; CKPT (pass 2 only): a checkpoint
// wherever (M - j) is a multiple of kW = 4 — every second step pair, starting with the first pair of the range or
// with the second — plus the one of the ragged last window at j = 0
template <int KIND, bool CKPT>
__device__ __forceinline__ void run_pass(const Ctx &c, int j0, int j1, float (&v)[16])
{
    static_assert(kW == 4, "checkpoints alternate between the step pairs of a four-step body");
    if (j0 >= j1) return;
    Buf B0, B1;
    float g[8];
    pf_issue<KIND>(c, j0, B0);
    pf_complete<KIND>(c, B0, g);
    if (!CKPT) { pass_loop<KIND, false, false>(c, j0, j1, B0, B1, g, v); return; }
    if (j0 == 0 && (c.M % kW) != 0) ck_store(c, c.M / kW, v);
    if (((c.M - j0) % kW) == 0) pass_loop<KIND, CKPT, false>(c, j0, j1, B0, B1, g, v);
    else                        pass_loop<KIND, false, CKPT>(c, j0, j1, B0, B1, g, v);
}

__device__ __forceinline__ void issue_ckpt(const Ctx &c, int slot)
{   // alpha lanes need their alpha checkpoint as X, beta lanes their beta checkpoint as Z
    float4 *dst = (c.isb ? c.slotZ() : c.slotX()) + c.lane;
#pragma unroll
    for (int q = 0; q < 4; ++q) cpa16(dst + q * 32, c.CK + (slot * 4 + q) * 32 + c.lane, c.one);
}
// ALPHA: the slot holds an alpha vector (stored order apos), else a beta vector (natural order)
template <bool ALPHA = false>
__device__ __forceinline__ void slot_get(const float4 *slot, int lane, float (&v)[16])
{
    constexpr int P[4] = {ALPHA ? apos(0) : 0, ALPHA ? apos(1) : 1, ALPHA ? apos(2) : 2, ALPHA ? apos(3) : 3};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 t = slot[q * 32 + lane];
        const int b = ALPHA ? 2 * q : 4 * q;                        // apos(4q + i) == 2q + apos(i)
        v[b + P[0]] = t.x; v[b + P[1]] = t.y; v[b + P[2]] = t.z; v[b + P[3]] = t.w;
    }
}
template <bool ALPHA = false>
__device__ __forceinline__ void slot_put(float4 *slot, int lane, const float (&v)[16])
{
    constexpr int P[4] = {ALPHA ? apos(0) : 0, ALPHA ? apos(1) : 1, ALPHA ? apos(2) : 2, ALPHA ? apos(3) : 3};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int b = ALPHA ? 2 * q : 4 * q;
        slot[q * 32 + lane] = make_float4(v[b + P[0]], v[b + P[1]], v[b + P[2]], v[b + P[3]]);
    }
}

// Y = Lc + La travels in 32-byte entries: the two steps of a pair, in ascending k, per lane.  256-bit global
// accesses (sm_100: LDG/STG.E.ENL2.256): one instruction per pair instead of two.  Layout [k/2][16 frames].
__device__ __forceinline__ void st256_f64(void *p, double a, double b, double c, double d)
{
    asm volatile("st.global.cg.v4.f64 [%0], {%1,%2,%3,%4};" :: "l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}
__device__ __forceinline__ void ld256_f64(const void *p, double2 &lo, double2 &hi)
{
    asm volatile("ld.global.cg.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(lo.x), "=d"(lo.y), "=d"(hi.x), "=d"(hi.y) : "l"(p) : "memory");
}
__device__ __forceinline__ unsigned char *y_entry(const Ctx &c, int k_even)
{
    return reinterpret_cast<unsigned char *>(c.Yb) + ((size_t)(k_even >> 1) * 16 + c.f) * 32;
}
struct YQ { double2 y[kW]; };
__device__ __forceinline__ void yq_load(const Ctx &c, int w0, int len, YQ &q)
{   // global loads issued a whole window ahead of their use
    static_assert(kW == 4, "two 32-byte entries per window");
    ld256_f64(y_entry(c, w0), q.y[0], q.y[1]);                      // w0 is even for both half-warps
    ld256_f64(y_entry(c, len > 2 ? w0 + 2 : w0), q.y[2], q.y[3]);
}
__device__ __forceinline__ void yq_park(const Ctx &c, const YQ &q, int w0, int len, int ck_slot)
{

#pragma unroll
    for (int u = 0; u < kW; ++u)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};"
                     :: "r"(c.tq + c.ycol + 4u * u), "r"(__double2loint(q.y[u].x)), "r"(__double2hiint(q.y[u].x)),
                        "r"(__double2loint(q.y[u].y)), "r"(__double2hiint(q.y[u].y)) : "memory");
    tm_wait_st();
    // the values are in TMEM now.  ONE predicated discard instruction drops the dead scratch of this window:
    // lanes 0-15 the 2 x len x 2 lines of Y (lane = half-warp, step, half line), lanes 16-31 the 16 lines of
    // the checkpoint slot the window consumed
    const int dir = (c.lane >> 3) & 1, pr = (c.lane >> 2) & 1, l16 = c.lane & 15;
    const int w0d = __shfl_sync(0xffffffffu, w0, dir << 4);         // w0 of the alpha (lane 0) / beta (lane 16) half
    const void *line = c.lane < 16
        ? static_cast<const void *>(reinterpret_cast<const unsigned char *>(c.Yb) + ((size_t)((w0d >> 1) + pr) * 16) * 32 + (c.lane & 3) * 128)
        : static_cast<const void *>(c.CK + (ck_slot * 4 + (l16 >> 2)) * 32 + (l16 & 3) * 8);
    if (c.lane < 16 ? 2 * pr < len : ck_slot >= 0) l2_discard(line);
}

// One recompute window of the "out" phase (all lanes in natural labels):
//   alpha lane: steps [w0, w0+len) of [0, M): Z = running beta, X = alpha from its checkpoint
//   beta lane:  steps [w0, w0+len) of [M, N): Z = beta from its checkpoint, X = running alpha
// Both vectors arrive through the lane's staging slots (running ones written by the previous
// window, checkpoints by cp.async), so the two half-warps run identical code.  First beta is
// walked down through the window and parked in shared memory, then alpha is walked up with
// the extrinsic fused in; the float64 epilogue of step u runs one step late so that its
// dependent chain interleaves with the float32 work of step u+1.  Both loops are ROLLED and
// branch-free: with one warp per sub-partition nothing hides an instruction-cache miss or a
// dependency stall except the instruction scheduler.
// TM: the window's records are in TMEM — column block (wa + u) for the alpha lane, block
// (wa + len-1-u) for the beta lane (the high records are stored in reverse).
// the float64 epilogue of a window's LAST step, carried into the next window: there its dependent chain
// (~50 instructions) fills the load latencies of the window start instead of running alone at the window end
struct Pend { float uv[4], y[4]; int idx; };
__device__ __forceinline__ void pend_flush(const Ctx &c, Pend &p, double sf, double2 *LeOut)
{
    double ea, eb;
    make_extrinsic(p.uv, __hiloint2double(__float_as_int(p.y[1]), __float_as_int(p.y[0])),
                   __hiloint2double(__float_as_int(p.y[3]), __float_as_int(p.y[2])), sf, ea, eb);
    if (p.idx >= 0) st_ws(LeOut + p.idx * 16 + c.f, make_double2(ea, eb));
    p.idx = -1;
}
template <bool TM>
__device__ __forceinline__ void window(const Ctx &c, int wa, int w0, int len, double sf,
                                       double2 *LeOut, int nslot, int nw0, int nlen, Pend &pend)
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
        // first step of the way down peeled (len >= 2): the float64 epilogue chain of the previous window's last
        // step shares its basic block, so the scheduler interleaves the chain with the step's 64 independent FP32 ops
        slot_put(ws + (len - 1) * 128, 0, Z);
        issue(len - 2);
        pend_flush(c, pend, sf, LeOut);
        bwd_step(Z, g);
        complete(g);
        for (int u = len - 2; u >= 0; --u) {
            slot_put(ws + u * 128, 0, Z);                           // beta[k+1]
            issue(u > 0 ? u - 1 : 0);                               // u == 0: first record of the way up
            bwd_step(Z, g);
            complete(g);
        }
        if (!c.isb) slot_put(c.slotZ(), c.lane, Z);                 // running beta of the alpha lane
    }
    float X[16];
    slot_get<true>(c.slotX(), c.lane, X);
    if (nslot >= 0) issue_ckpt(c, nslot);
    cpa_commit();
    float yr[4], yn[4], uvp[4], zs[16];
    tm_ld4(c.tq + c.ycol, yr);
    issue(len > 1 ? 1 : 0);
    slot_get(ws, 0, zs);
    ext_step(X, zs, g, uvp);                                        // step 0 (its Y is not needed before the next step's epilogue)
    tm_wait_ld4(yr);
    complete(g);
    for (int u = 1; u < len; ++u) {
        tm_ld4(c.tq + c.ycol + 4u * u, yn);
        issue(u + 1 < len ? u + 1 : u);
        slot_get(ws + u * 128, 0, zs);
        float uv[4];
        ext_step(X, zs, g, uv);
        double ea, eb;                                              // epilogue of step u-1
        make_extrinsic(uvp, __hiloint2double(__float_as_int(yr[1]), __float_as_int(yr[0])),
                       __hiloint2double(__float_as_int(yr[3]), __float_as_int(yr[2])), sf, ea, eb);
        st_ws(LeOut + (w0 + u - 1) * 16 + c.f, make_double2(ea, eb));
        tm_wait_ld4(yn);
        complete(g);
#pragma unroll
        for (int i = 0; i < 4; ++i) { uvp[i] = uv[i]; yr[i] = yn[i]; }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) { pend.uv[i] = uvp[i]; pend.y[i] = yr[i]; }
    pend.idx = w0 + len - 1;
    if (c.isb) slot_put<true>(c.slotX(), c.lane, X);                // running alpha of the beta lane
    if (nlen) yq_park(c, nq, nw0, nlen, nslot - 1);
}

// pass 1, first half, steps [j0, j1) (even count): build this thread's records on the fly (prep
// fused).  Two steps per iteration: the float64 chains of steps j+2 and j+3 and the float32
// recursion of steps j and j+1 share one basic block, so the scheduler can interleave them.
// TMST: records go to TMEM (j < T) / shared memory.  PrepState: records and Lc+La of steps j0, j0+1.

// Channel LLRs live in the workspace as [j][32 lanes] float4: lanes 0-15 hold step k = j of frames 0-15, lanes
// 16-31 step k = N-1-j.  Pass 1a (the only streaming reader) fetches position j of ALL lanes from one 512-byte
// run, and the two steps of a pair are an immediate 512 bytes apart: one address register per pair.
__device__ __forceinline__ int lpos(const Ctx &c, int k, int fr) { return k < c.M ? k * 32 + fr : (c.N - 1 - k) * 32 + 16 + fr; }

// interleaver entries of this thread's positions of steps jn, jn+1 (jn even), looked up a whole pair before the
// gather that needs them: a shared-memory load issued behind the ring traffic takes 60-130 cycles to return
struct Idx { int a, b; };
__device__ __forceinline__ void idx_get(const Ctx &c, int jn, const int16_t *tbl, Idx &x)
{
    jn = min(jn, c.M - 2);
    const int k0 = c.isb ? c.N - 1 - jn : jn, k1 = c.isb ? k0 - 1 : k0 + 1;
    x.a = tbl[k0]; x.b = tbl[k1];
}
// loads for the prep of this thread's positions of steps jn, jn+1 (jn even) (:507-512, :523-524)
__device__ __forceinline__ void prep_load_pair(const Ctx &c, unsigned char *slot, int jn, const float4 *Lsrc,
                                               const Idx &x, bool first)
{
    jn = min(jn, c.M - 2);                                          // clamped at the end: harmless re-computation
    const unsigned d = s_addr(slot) * c.one;
    const float4 *src = Lsrc + jn * 32 + c.lane;
    cpa16_stream_off<0, 0>(d, src, c.pol);
    cpa16_stream_off<1024, 512>(d, src, c.pol);   // ring slot: [x A][la A][x B][la B], 512 B each, lane-major (conflict-free)
    if (!first) {
        cpa16_off<512, 0>(d, c.Le + x.a * 16 + c.f);
        cpa16_off<1536, 0>(d, c.Le + x.b * 16 + c.f);
    }
}
// raw inputs of a step pair, read out of the ring a whole pair before they are needed: a shared-memory load
// queued behind the ring traffic can take several times its nominal 29 cycles to return, and this warp has
// nothing else to run meanwhile.  Ring slot of a pair: [x A][la A][x B][la B], 512 B each, lane-major: both the
// cp.async writes and these LDS.128 are bank-conflict free (a [lane][x|la] slot cost 32 smem wavefronts per copy)
struct Raw { float4 xA, xB; double2 laA, laB; };
template <bool FIRST>
__device__ __forceinline__ void raw_get(const unsigned char *slot, Raw &r)
{
    r.xA = *reinterpret_cast<const float4 *>(slot);
    r.xB = *reinterpret_cast<const float4 *>(slot + 1024);
    r.laA = r.laB = make_double2(0.0, 0.0);
    if (!FIRST) {
        r.laA = *reinterpret_cast<const double2 *>(slot + 512);
        r.laB = *reinterpret_cast<const double2 *>(slot + 1536);
    }
}
// records of the step pair (jn, jn+1) from its raw inputs; Y = Lc + La of both steps goes to the workspace at once
// (one 256-bit store, ascending k: the beta lane walks k downwards, so its two steps swap) instead of riding along
// in registers until the pair is stepped
struct PrepRec { float gA[8], gB[8]; };                      // records of two consecutive steps
__device__ __forceinline__ void prep_pair(const Ctx &c, const Raw &r, int jn, PrepRec &out)
{
    jn = min(jn, c.M - 2);
    const double2 YA = make_double2(d_add((double)r.xA.x, r.laA.x), d_add((double)r.xA.y, r.laA.y));    // Lc + La (:135)
    const double2 YB = make_double2(d_add((double)r.xB.x, r.laB.x), d_add((double)r.xB.y, r.laB.y));
    make_record(YA.x, YA.y, r.xA.z, r.xA.w, out.gA);
    make_record(YB.x, YB.y, r.xB.z, r.xB.w, out.gB);
#ifndef TPF_ABL_NOY
    const int ke = c.isb ? c.N - 2 - jn : jn;                       // the even (lower) k of the pair
    st256_f64(y_entry(c, ke), c.isb ? YB.x : YA.x, c.isb ? YB.y : YA.y, c.isb ? YA.x : YB.x, c.isb ? YA.y : YB.y);
#endif
}
struct PrepState { PrepRec r; Raw raw; Idx ix; int ps; };
// steps jj, jj+1 with the records in `in`; builds the records of steps jj+2, jj+3 (raw inputs `rin`) into
// `out` and pulls the raw inputs of steps jj+4, jj+5 out of the ring into `rout`
// (TPF_ABL_* : timing-only ablation builds for profiles/r01_tpf_ablation.txt; never defined in the shipped library)
template <bool FIRST, bool TMST>
__device__ __forceinline__ void pass1a_pair(const Ctx &c, int jj, const float4 *Lsrc, const int16_t *tbl,
                                            int &ps, const PrepRec &in, PrepRec &out, const Raw &rin, Raw &rout,
                                            const Idx &xin, Idx &xout, float (&v)[16])
{
    const int N = c.N;
    unsigned char *slot = c.stage + c.lane * 16 + ps * 2048;
    cpa_wait<kRingPairs - 1>();
#ifndef TPF_ABL_NORAW
    raw_get<FIRST>(slot, rout);
#else
    rout = rin;
#endif
#ifndef TPF_ABL_NOCPA
    prep_load_pair(c, slot, jj + 4 + 2 * kRingPairs, Lsrc, xin, FIRST);
    cpa_commit();
    if (!FIRST) idx_get(c, jj + 6 + 2 * kRingPairs, tbl, xout);
#endif
    ps = ps == kRingPairs - 1 ? 0 : ps + 1;
#ifndef TPF_ABL_NOFP64
    prep_pair(c, rin, jj + 2, out);
#else
    out = in;
#endif
    const int k0 = c.isb ? N - 1 - jj : jj, k1 = c.isb ? N - 2 - jj : jj + 1;
#ifndef TPF_ABL_NOREC
    if (TMST) tm_st8(c.tq + 8u * jj, in.gA);
    else      smem_put(c, k0, in.gA);
#endif
    pass_step(v, in.gA, c.isb);
#ifndef TPF_ABL_NOREC
    if (TMST) tm_st8(c.tq + 8u * (jj + 1), in.gB);
    else      smem_put(c, k1, in.gB);
#endif
    pass_step(v, in.gB, c.isb);
}
template <bool FIRST, bool TMST>
__device__ __forceinline__ void pass1a_range(const Ctx &c, int j0, int j1, const float4 *Lsrc,
                                             const int16_t *tbl, PrepState &P, float (&v)[16])
{
    PrepRec Q;
    Raw RQ;
    Idx XQ = P.ix;
    int jj = j0;
    for (; jj + 4 <= j1; jj += 4) {                                 // ping-pong: no register copies
        pass1a_pair<FIRST, TMST>(c, jj, Lsrc, tbl, P.ps, P.r, Q, P.raw, RQ, P.ix, XQ, v);
        pass1a_pair<FIRST, TMST>(c, jj + 2, Lsrc, tbl, P.ps, Q, P.r, RQ, P.raw, XQ, P.ix, v);
    }
    if (jj < j1) {
        pass1a_pair<FIRST, TMST>(c, jj, Lsrc, tbl, P.ps, P.r, Q, P.raw, RQ, P.ix, XQ, v);
        P.r = Q;
        P.raw = RQ;
        P.ix = XQ;
    }
}

template <bool FIRST>
__device__ __forceinline__ void pass1a(const Ctx &c, bool second, float (&v)[16])
{
    const float4 *Lsrc = second ? c.L2A : c.L1A;
    const int16_t *tbl = second ? c.perm : c.inv;                   // La = Le[perm k] (:507-508) / Le[inv k] (:523-524)
    unsigned char *ring = c.stage + c.lane * 16;
    PrepState P;
    P.ix.a = P.ix.b = 0;
#pragma unroll 1
    for (int p = 0; p < kRingPairs; ++p) {                          // ring of step pairs
        if (!FIRST) idx_get(c, 2 * p, tbl, P.ix);
        prep_load_pair(c, ring + p * 2048, 2 * p, Lsrc, P.ix, FIRST);
        cpa_commit();
    }
    if (!FIRST) idx_get(c, 2 * kRingPairs, tbl, P.ix);
    cpa_wait<kRingPairs - 1>();
    raw_get<FIRST>(ring, P.raw);                                    // steps 0, 1
    prep_pair(c, P.raw, 0, P.r);
    prep_load_pair(c, ring, 2 * kRingPairs, Lsrc, P.ix, FIRST);
    cpa_commit();
    if (!FIRST) idx_get(c, 2 * kRingPairs + 2, tbl, P.ix);
    cpa_wait<kRingPairs - 1>();
    raw_get<FIRST>(ring + 2048, P.raw);                             // steps 2, 3
    prep_load_pair(c, ring + 2048, 2 * kRingPairs + 2, Lsrc, P.ix, FIRST);
    cpa_commit();
    if (!FIRST) idx_get(c, 2 * kRingPairs + 4, tbl, P.ix);
    P.ps = 2 % kRingPairs;
    pass1a_range<FIRST, true>(c, 0, c.T, Lsrc, tbl, P, v);
    pass1a_range<FIRST, false>(c, c.T, c.M, Lsrc, tbl, P, v);
    cpa_wait<0>();
}

// One SISO half-iteration for the 16 frames of this warp.
template <bool TIMED>
__device__ __forceinline__ void siso(const Ctx &c, bool second, bool first, bool last, double sf, long long (&ph)[8])
{
    long long tA = TIMED ? clock64() : 0;
    const int N = c.N, M = c.M, T = c.T, lane = c.lane;
    double2 *LeOut = last ? c.LeF : c.Le;
    float v[16];
#pragma unroll
    for (int s = 0; s < 16; ++s) v[s] = 0.f;
    // ---- pass 1, first half ------------------------------------------------------------------
    if (first) pass1a<true>(c, second, v);
    else       pass1a<false>(c, second, v);
    tm_wait_st();
    __syncwarp();
    if (!first && !last)                                            // old extrinsics are dead: every line is rewritten below
        for (int i = lane; i < N * 2; i += 32) l2_discard(c.Le + i * 8);
    if (TIMED) { const long long t = clock64(); ph[1] += t - tA; tA = t; }
    // ---- pass 1, second half: the records the partner lane built ---------------------------
    run_pass<1, false>(c, M, N - T, v);
    run_pass<2, false>(c, N - T, N, v);
    if (TIMED) { const long long t = clock64(); ph[2] += t - tA; tA = t; }
    // ---- pass 2 up to the crossing point, checkpoint every kW steps -------------------------
    const int nfull = M / kW, rag = M % kW, nwin = nfull + (rag ? 1 : 0);
    auto win_w0 = [&](int i) { return i < nfull ? (c.isb ? M + i * kW : M - (i + 1) * kW) : (c.isb ? N - rag : 0); };
    auto win_len = [&](int i) { return i < nfull ? kW : rag; };
    {
        YQ q0;
        yq_load(c, win_w0(0), win_len(0), q0);                      // Y of the first window: arrives during pass 2
        run_pass<0, true>(c, 0, T, v);
        run_pass<1, true>(c, T, M, v);
        yq_park(c, q0, win_w0(0), win_len(0), -1);
    }
    if (TIMED) { const long long t = clock64(); ph[3] += t - tA; tA = t; }
    // ---- crossing: the half-warps swap chains (beta lanes back to natural labels): every lane
    //      drops its vector into the PARTNER's slot -------------------------------------------
    {
        float n[16];
        pass_out(c, v, n);
        slot_put(c.isb ? c.slotZ() : c.slotX(), lane ^ 16, n);
    }
    const int n_inner = (M - T) / kW;            // windows whose records are in shared memory
    issue_ckpt(c, 0);
    cpa_commit();
    // ---- out phase: windows from the crossing point outwards ---------------------------------
    Pend pend;
#pragma unroll
    for (int i = 0; i < 4; ++i) pend.uv[i] = pend.y[i] = 0.f;
    pend.idx = -1;
    for (int i = 0; i < nwin; ++i) {
        cpa_wait<0>();
        __syncwarp();
        const int wa = i < nfull ? M - (i + 1) * kW : 0;
        const int nlen = i + 1 < nwin ? win_len(i + 1) : 0;
        const int nw0 = i + 1 < nwin ? win_w0(i + 1) : 0;
        if (i < n_inner) window<false>(c, wa, win_w0(i), win_len(i), sf, LeOut, nlen ? i + 1 : -1, nw0, nlen, pend);
        else             window<true>(c, wa, win_w0(i), win_len(i), sf, LeOut, nlen ? i + 1 : -1, nw0, nlen, pend);
        if (TIMED && i == n_inner - 1) { const long long t = clock64(); ph[4] += t - tA; tA = t; }
    }
    pend_flush(c, pend, sf, LeOut);
    cpa_wait<0>();
    __syncwarp();
    if (TIMED) { const long long t = clock64(); ph[5] += t - tA; tA = t; }
}

template <bool TIMED, class LlrT>
__global__ void __launch_bounds__(kTpfWarps * 32, 1)
tpf_kernel(const TpfArgs A)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const TpfGeom g = A.g;
    const int N = g.N;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int16_t *tab = reinterpret_cast<int16_t *>(smem_raw);
    const int tab_bytes = ((2 * N * 2 + 15) / 16) * 16;
    unsigned *tmem_slot = reinterpret_cast<unsigned *>(smem_raw + tab_bytes);
    float4 *srec_all = reinterpret_cast<float4 *>(smem_raw + tab_bytes + 64);   // 32 B of slots + four 8-byte mbarriers
    unsigned char *stage_all = reinterpret_cast<unsigned char *>(srec_all + (size_t)kTpfWarps * g.mid * 2 * 16);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"((unsigned)__cvta_generic_to_shared(tmem_slot)), "r"(g.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < 2 * N; i += blockDim.x) tab[i] = A.tab[i];
    const unsigned mbar = (unsigned)__cvta_generic_to_shared(smem_raw + tab_bytes + 32 + 8 * warp);   // this warp's mbarrier
    unsigned mphase = 0;
    if (lane == 0) { mbar_init(mbar, 1); mbar_fence_init(); }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem_base = *tmem_slot;

    Ctx c;
    c.N = N; c.M = g.M; c.T = g.T;
    c.f = lane & 15; c.isb = lane >> 4; c.lane = lane;
    c.tq = tmem_base + (((unsigned)warp * 32u) << 16);
    c.ycol = 8u * g.T;
    c.srec = srec_all + (size_t)warp * g.mid * 2 * 16;
    {   // ptxas folds a warp-uniform base into a [R+UR+imm] shared-memory operand; for LDGSTS (cp.async)
        // that form raises "illegal instruction" on sm_100a, so the staging base goes through memory
        volatile unsigned *slots = reinterpret_cast<volatile unsigned *>(smem_raw + tab_bytes);
        if (lane == 0) { slots[4 + warp] = (unsigned)warp * kStageBytes; slots[1] = 1u; }
        __syncwarp();
        c.stage = stage_all + slots[4 + warp];
        c.one = slots[1];
        __syncwarp();
    }
    c.perm = tab; c.inv = tab + N;
    const int wg = blockIdx.x * kTpfWarps + warp;
    unsigned char *ws = A.ws + (size_t)wg * g.ws_per_warp;
    c.L1A = reinterpret_cast<float4 *>(ws + g.off_l1);
    c.L2A = reinterpret_cast<float4 *>(ws + g.off_l2);
    c.Le = reinterpret_cast<double2 *>(ws + g.off_le);
    c.LeF = reinterpret_cast<double2 *>(ws + g.off_lef);
    c.Yb = reinterpret_cast<double2 *>(ws + g.off_y);
    c.CK = reinterpret_cast<float4 *>(ws + g.off_ck);
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(c.pol));
    const int16_t *g_off = A.tab + 2 * N;        // offA, offW1, offY1, offW2, offY2 (global, read-only)

    unsigned long long bit_err = 0, frm_err = 0, frames_done = 0;
    long long ph[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const long long t_begin = TIMED ? clock64() : 0;
    for (int tile = wg; tile < A.n_tiles; tile += gridDim.x * kTpfWarps) {
        const long long frame0 = (long long)tile * kTpfFrames;
        const long long t0 = TIMED ? clock64() : 0;
        const float sc = A.llr_scale;                               // int8 input only (llr_f32)
        // ---- de-puncture + transpose the 16 frames' LLRs into [k][frame] (:466-487, :507-512).
        //      Each frame's row is pulled into the staging area with coalesced 16-byte loads
        //      (every line of the input is read exactly once), two frames in flight; the lanes
        //      then pick their couples (and the permuted systematic pair) out of shared memory.
        if (A.vec4) {
            // rows of a GROUP of G frames (8 where they fit) are pulled at once into whichever of the warp's two
            // shared-memory areas is larger (the record area is dead between tiles).  Lane = (couple kq, frame fr)
            // with fr the minor index: one store instruction then writes 32/G couples x G frames x 16 B, i.e. FULL
            // 128-byte lines (G = 8) of the [j][lane] layout, instead of 32 partial lines.
            const int nq = llr_row_q<LlrT>(A.n_llr);                // float4 per row (row pitch is a multiple of 16 B)
            const int pitch4 = ((nq + 6) & ~7) + 1;                 // row pitch = 4 (mod 32) words: rows land in different banks
            const int rec_bytes = g.mid * 2 * 16 * (int)sizeof(float4);
            const bool in_rec = rec_bytes > kStageBytes;
            float4 *rowbuf = in_rec ? c.srec : reinterpret_cast<float4 *>(c.stage);
            const int fit = (in_rec ? rec_bytes : kStageBytes - N * 16) / (pitch4 * 16);
            const int lg = fit >= 8 ? 3 : fit >= 4 ? 2 : 1, G = 1 << lg, KQ = 32 >> lg;
            const int fr = lane & (G - 1), kq = lane >> lg;
            // stream offsets of every couple as one 16-byte shared-memory entry (offA, offA[perm], offW1, offY1,
            // offW2, offY2): the global tables are read once per tile, not once per couple and frame group
            int4 *otab = reinterpret_cast<int4 *>(in_rec ? c.stage : c.stage + G * pitch4 * 16);
            for (int k = lane; k < N; k += 32) {
                const unsigned oa = (unsigned short)__ldg(g_off + k), op = (unsigned short)__ldg(g_off + c.perm[k]);
                const unsigned o0 = (unsigned short)__ldg(g_off + N + k), o1 = (unsigned short)__ldg(g_off + 2 * N + k);
                const unsigned o2 = (unsigned short)__ldg(g_off + 3 * N + k), o3 = (unsigned short)__ldg(g_off + 4 * N + k);
                otab[k] = make_int4((int)(oa | (op << 16)), (int)(o0 | (o1 << 16)), (int)(o2 | (o3 << 16)), 0);
            }
            // whole rows by bulk copy (cp.async.bulk: one instruction of one lane per 5 KB row, completed on this
            // warp's mbarrier) — the rows are the longest contiguous transfers of the kernel
            auto pull = [&](int g0) {
                if (lane == 0) {
                    int live_rows = 0;
                    for (int r = 0; r < G; ++r) live_rows += frame0 + g0 + r < A.B;
                    fence_proxy_async();                            // the row buffer was read (or held records) before
                    mbar_expect_tx(mbar, (unsigned)(live_rows * nq * 16));
                    for (int r = 0; r < live_rows; ++r)
                        bulk_g2s_stream(rowbuf + r * pitch4, static_cast<const LlrT *>(A.llr) + (frame0 + g0 + r) * A.llr_stride, (unsigned)(nq * 16), mbar, c.pol);
                }
            };
            pull(0);
            if (A.ref_bits) {                                       // the hard decision will want these rows in L2
                const int lines = (2 * N * kTpfFrames + 127) / 128;
                const long long nb = min((long long)kTpfFrames, A.B - frame0) * 2 * N;
                for (int i = lane; i < lines; i += 32)
                    if ((long long)i * 128 < nb) asm volatile("prefetch.global.L2 [%0];" ::"l"(A.ref_bits + frame0 * 2 * N + i * 128));
            }
            const LlrT *row = reinterpret_cast<const LlrT *>(rowbuf + fr * pitch4);
            for (int g0 = 0; g0 < kTpfFrames; g0 += G) {
                mbar_wait(mbar, mphase);
                mphase ^= 1u;
                const bool livef = frame0 + g0 + fr < A.B;
#pragma unroll 4
                for (int k0 = 0; k0 < N; k0 += KQ) {
                    const int k = k0 + kq;
                    const int4 e = otab[min(k, N - 1)];
                    const int oa = (short)(e.x & 0xffff), op = e.x >> 16, o0 = (short)(e.y & 0xffff), o1 = e.y >> 16;
                    const int o2 = (short)(e.z & 0xffff), o3 = e.z >> 16;
                    float4 x1 = make_float4(0.f, 0.f, 0.f, 0.f), x2 = x1;
                    if (livef) {
                        x1.x = llr_f32(row[oa], sc); x1.y = llr_f32(row[oa + 1], sc); x2.x = llr_f32(row[op], sc); x2.y = llr_f32(row[op + 1], sc);
                        if (o0 >= 0) x1.z = llr_f32(row[o0], sc);
                        if (o1 >= 0) x1.w = llr_f32(row[o1], sc);
                        if (o2 >= 0) x2.z = llr_f32(row[o2], sc);
                        if (o3 >= 0) x2.w = llr_f32(row[o3], sc);
                    }
                    if (k < N) {
                        st_ws(c.L1A + lpos(c, k, g0 + fr), x1);
                        st_ws(c.L2A + lpos(c, k, g0 + fr), x2);
                    }
                }
                __syncwarp();
                if (g0 + G < kTpfFrames) pull(g0 + G);
            }
        } else
        for (int k = lane; k < N; k += 32) {
            const int oa = __ldg(g_off + k), op = __ldg(g_off + c.perm[k]);
            const int o0 = __ldg(g_off + N + k), o1 = __ldg(g_off + 2 * N + k);
            const int o2 = __ldg(g_off + 3 * N + k), o3 = __ldg(g_off + 4 * N + k);
#pragma unroll
            for (int f0 = 0; f0 < kTpfFrames; f0 += 8) {
                float4 x1[8], x2[8];
#pragma unroll
                for (int fr = 0; fr < 8; ++fr) {
                    const long long frame = frame0 + f0 + fr;
                    const LlrT *Lf = static_cast<const LlrT *>(A.llr) + frame * A.llr_stride;
                    x1[fr] = make_float4(0.f, 0.f, 0.f, 0.f); x2[fr] = x1[fr];
                    if (frame < A.B) {
                        x1[fr].x = llr_ldg(Lf + oa, sc); x1[fr].y = llr_ldg(Lf + oa + 1, sc);
                        x2[fr].x = llr_ldg(Lf + op, sc); x2[fr].y = llr_ldg(Lf + op + 1, sc);
                        if (o0 >= 0) x1[fr].z = llr_ldg(Lf + o0, sc);
                        if (o1 >= 0) x1[fr].w = llr_ldg(Lf + o1, sc);
                        if (o2 >= 0) x2[fr].z = llr_ldg(Lf + o2, sc);
                        if (o3 >= 0) x2[fr].w = llr_ldg(Lf + o3, sc);
                    }
                }
#pragma unroll
                for (int fr = 0; fr < 8; ++fr) {
                    st_ws(c.L1A + lpos(c, k, f0 + fr), x1[fr]);
                    st_ws(c.L2A + lpos(c, k, f0 + fr), x2[fr]);
                }
            }
        }
        __syncwarp();
        if (TIMED) ph[0] += clock64() - t0;
        for (int h = 0; h < 2 * A.iterations; ++h) {
            const double sf = (h >> 1) < A.iterations - 1 ? A.sf_inner : A.sf_last;
            siso<TIMED>(c, (h & 1) != 0, h == 0, h == 2 * A.iterations - 1, sf, ph);
        }
        const long long t6 = TIMED ? clock64() : 0;
        // ---- hard decision (dvb_rcs2_turbo.py:526-537) + optional error counting ------------
        const long long frame = frame0 + c.f;
        const bool live = frame < A.B;
        const int wpf = (2 * N + 31) / 32;
        // Batches of 8 couples per lane.  The phase is pure load latency and nothing else runs on this
        // sub-partition meanwhile, so the three workspace streams (Lc, La = Le2[inv], Le1) of up to three batches
        // ahead are kept in flight with cp.async into the record area, which is dead by now (registers cannot hold
        // that much).  Batch b of a lane covers couples (isb + 2 (b >> 1)) * 16 + 8 (b & 1) + [0, 8); slots are
        // lane-private, so no warp synchronisation is needed.
        const bool cnt = live && A.ref_bits != nullptr;
        const uint8_t *refp = cnt ? A.ref_bits + (size_t)frame * 2 * N : reinterpret_cast<const uint8_t *>(A.tab);
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
                    cpa16_off<4096, 0>(dt, c.LeF + c.inv[k] * 16 + c.f);
                    cpa16_off<8192, 0>(dt, c.Le + k * 16 + c.f);
                }
            }
            cpa_commit();
        };
        int any_err = 0;
        unsigned word = 0;
        for (int b = 0; b < nst; ++b) hissue(b, b);
        for (int b = 0, st = 0; b < nbu; ++b) {
            if (nst == 3) cpa_wait<2>(); else if (nst == 2) cpa_wait<1>(); else cpa_wait<0>();
            const int kb = (c.isb + 2 * (b >> 1)) * 16 + 8 * (b & 1);
            const unsigned char *src = hbuf + st * kHB + lane * 16;
            unsigned short rb[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) rb[t] = *reinterpret_cast<const unsigned short *>(refp + 2 * min(kb + t, N - 1));
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const int k = kb + t;
                const float4 ab = *reinterpret_cast<const float4 *>(src + t * 512);
                const double2 la = *reinterpret_cast<const double2 *>(src + 4096 + t * 512);
                const double2 e1 = *reinterpret_cast<const double2 *>(src + 8192 + t * 512);
                const double LA = d_add(d_add((double)ab.x, la.x), e1.x);
                const double LB = d_add(d_add((double)ab.y, la.y), e1.y);
                const int bA = LA < 0.0, bB = LB < 0.0;
                if (k < N) {
                    word |= (unsigned)(bA | (bB << 1)) << (2 * (8 * (b & 1) + t));
                    if (live && A.bits)
                        *reinterpret_cast<int2 *>(A.bits + (size_t)frame * 2 * N + 2 * k) = make_int2(bA, bB);
                    if (live && A.app)
                        *reinterpret_cast<float2 *>(A.app + (size_t)frame * 2 * N + 2 * k) =
                            make_float2(__double2float_rn(LA), __double2float_rn(LB));
                    if (cnt) {
                        const int errs = (bA != (rb[t] & 0xff)) + (bB != (rb[t] >> 8));
                        bit_err += errs;
                        any_err |= errs;
                    }
                }
            }
            hissue(b + nst, st);                                    // refill the slot just read (same lane, same LSU queue: ordered)
            st = st + 1 == nst ? 0 : st + 1;
            if (b & 1) {
                const int w = c.isb + b - 1;
                if (live && A.packed && w < nwords) A.packed[(size_t)frame * wpf + w] = word;
                word = 0;
            }
        }
        cpa_wait<0>();
        any_err |= __shfl_xor_sync(0xffffffffu, any_err, 16);
        if (live && !c.isb) { frames_done += 1; frm_err += any_err ? 1 : 0; }
        __syncwarp();
        if (TIMED) ph[6] += clock64() - t6;
    }
    if (TIMED && lane == 0) {
        ph[7] = clock64() - t_begin;
        for (int i = 0; i < 8; ++i) atomicAdd(&g_tpf_cycles[i], (unsigned long long)ph[i]);
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
// ---- shared with decode_nii.cu, whose kernel has this kernel's mapping, record pool and transposition ----
void tpf_family_geometry(TpfGeom &g, int N, int y_cols, size_t hdr_bytes, size_t ext_bytes, bool with_init, size_t smem_optin)
{
    g = TpfGeom{};
    if (N < 16 || (N % 4) != 0) return;
    const int M = N / 2;
    int T = M < 64 ? M : 64;
    while (T > 0 && (((M - T) % kW) != 0 || 8 * T + y_cols > 512)) --T;   // windows must not straddle TMEM / smem; Y columns
    if (T < kW) return;
    g.N = N; g.M = M; g.T = T; g.mid = N - 2 * T;
    g.nfull = M / kW; g.rag = M % kW; g.nslots = g.nfull + (g.rag ? 1 : 0);
    g.tmem_cols = 32;
    while (g.tmem_cols < 8 * T + y_cols) g.tmem_cols *= 2;        // records + the window's Y
    if (g.tmem_cols > 512) return;
    const size_t tab_bytes = ((size_t)2 * N * 2 + 15) / 16 * 16;
    g.smem_bytes = tab_bytes + hdr_bytes + (size_t)kTpfWarps * g.mid * 2 * 16 * sizeof(float4) + (size_t)kTpfWarps * kStageBytes;
    if (g.smem_bytes > smem_optin) return;                        // falls back to the quad kernel
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    g.off_l1 = take((size_t)N * 16 * sizeof(float4));
    g.off_l2 = take((size_t)N * 16 * sizeof(float4));
    g.off_le = take((size_t)N * 16 * ext_bytes);
    g.off_lef = take((size_t)N * 16 * ext_bytes);
    g.off_y = take((size_t)N * 16 * ext_bytes);
    g.off_ck = take((size_t)g.nslots * 4 * 32 * sizeof(float4));
    if (with_init) g.off_init = take((size_t)2 * 4 * 32 * sizeof(float4));
    g.ws_per_warp = off;
    g.enabled = 1;
}

int tpf_family_grid(const Codec &c, int B, int tile)
{
    const int tiles = (B + tile - 1) / tile;
    const int ctas = (tiles + kTpfWarps - 1) / kTpfWarps;
    return ctas < c.num_sms ? ctas : c.num_sms;
}

size_t tpf_family_workspace_bytes(const Codec &c, const TpfGeom &g, int B, int tile)
{
    return (size_t)tpf_family_grid(c, B, tile) * kTpfWarps * g.ws_per_warp + 256;
}

// whole rows by bulk copy: pitch and base 16-byte aligned, row fits half the staging area, and the group-staged
// transposition finds room for at least two padded rows (+ the offset table) in one of the warp's areas
int tpf_family_row_staging(const Codec &c, const TpfGeom &g, const DecodeIo &io)
{
    const int nq = llr_row_q(io.fmt, c.n_llr);
    if (c.N > 256 || (io.llr_stride * llr_bytes(io.fmt)) % 16 != 0 || (reinterpret_cast<uintptr_t>(io.llr) & 15) != 0 ||
        nq * 4 > kRowFloats || c.opt_no_row_staging)
        return 0;
    const int pitch4 = ((nq + 6) & ~7) + 1;
    const int rec_bytes = g.mid * 2 * 16 * (int)sizeof(float4);
    const int avail = rec_bytes > kStageBytes ? rec_bytes : kStageBytes - c.N * 16;
    return avail / (pitch4 * 16) >= 2;
}

// ---- the parity-mode kernel ----
int tpf_configure(Codec &c, size_t smem_optin)
{
    tpf_family_geometry(c.tpf, c.N, 4 * kW, 64, sizeof(double2), false, smem_optin);
    if (!c.tpf.enabled) return B200DVB_OK;
    // the device's maximum, not this codec's need: the attribute is per function and device, and codecs of several N coexist
    return for_each_llr_type([&](auto t) {
        using L = decltype(t);
        B2_CUDA(cudaFuncSetAttribute(tpf_kernel<false, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin));
        B2_CUDA(cudaFuncSetAttribute(tpf_kernel<true, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin));
        return B200DVB_OK;
    });
}

int tpf_read_phase_cycles(double *out_h, int reset) { return read_phase_cycles(g_tpf_cycles, out_h, reset); }

size_t tpf_workspace_bytes(const Codec &c, int B) { return tpf_family_workspace_bytes(c, c.tpf, B, kTpfFrames); }

int tpf_launch_decode(const Codec &c, const DecodeIo &io)
{
    if (io.ws_bytes < tpf_workspace_bytes(c, io.B)) return B200DVB_ENOMEM;
    TpfArgs A{};
    fill_decode_args(A, c, io);
    A.g = c.tpf;
    A.n_tiles = (io.B + kTpfFrames - 1) / kTpfFrames;
    A.n_llr = c.n_llr;
    A.vec4 = tpf_family_row_staging(c, c.tpf, io);
    A.ws = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(io.ws) + 255) & ~(uintptr_t)255);
    const int grid = tpf_family_grid(c, io.B, kTpfFrames);
    // B200DVB_OPT_PHASE_TIMERS (development): the instance with per-phase clock64() accounting, read by b200dvb_debug_tpf_cycles
    const bool timed = c.opt_phase_timers != 0;
    with_llr_type(io.fmt, [&](auto t) {
        using L = decltype(t);
        if (timed) tpf_kernel<true, L><<<grid, kTpfWarps * 32, c.tpf.smem_bytes, io.stream>>>(A);
        else       tpf_kernel<false, L><<<grid, kTpfWarps * 32, c.tpf.smem_bytes, io.stream>>>(A);
    });
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

}  // namespace b200dvb
