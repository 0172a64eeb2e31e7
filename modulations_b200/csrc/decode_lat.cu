// decode_lat.cu — the LOW-LATENCY decode path: one CTA per frame, bit-exact with the reference
// (dvb_rcs2_turbo.py:116-281 bcjr_max_log_map, :464-537 decode), for the reference's own call shape — one frame
// per decode() (turbo_test_suite.py:138-164, test.py:56-92).
//
// Why a third kernel.  A frame is 16 SISOs of strictly sequential recursions: the throughput kernels amortise that
// over 64 frames per SM, and a batch of ONE frame then costs what a full wave costs (thread-per-frame kernel: 0.99 ms
// at N=212; quad kernel: 0.65 ms; profiles/r02_measure_pack1.txt).  Here everything that is NOT sequential is spread
// over the 256 threads of a CTA, and the two recursions run on four warps with one state metric per lane (4 shuffles +
// 7 FP32 operations per step: ~80 cycles, against 120 for one thread holding all 16 states, whose 63 operations are
// issue-bound), their first lap cut into four speculative segments and the second lap ended where it has provably
// re-joined the first:
//   P0 (all threads, one trellis step each): a-priori gather, Y = Lc + La in float64, the merged branch-metric record;
//   P1 (four warps): `segmented_recursion` below — exact, ~N/4 + 48 + 50 sequential steps per SISO instead of 2 N;
//   P2 (all threads, one step each): the 64 a-posteriori sums of a step and the float64 extrinsic epilogue.
// The whole frame lives in shared memory (288 bytes per couple with conflict-free strides: 61 KB at N=212, 217 KB at
// N=752; 240 bytes per couple beyond N ~ 780: 204 KB at N=848), so the same kernel serves every N of the reference's
// table.  It is a latency path, not a throughput path: api.cu dispatches batches of up to min(6, N/50) passes of two
// CTAs per SM here (1 184 frames at N=212), larger ones to the wave kernels.
#include "common.cuh"
#include "tpf_core.cuh"

namespace b200dvb {

namespace {

using namespace tpf;

constexpr int kLatThreads = 256;
constexpr int kSegs = 4;            // lap-1 segments per direction: two warps, two segments per warp (one per half-warp)
// warm-up steps of a speculative segment (LatArgs.warm): 40 + N/16 within [48, 96] — measured optimum 48 at N=212, 80 - 96
// at N=752 (profiles/r02_lat_warmup.txt; every value gives the same bits); development override: B200DVB_DBG_LAT_WARM
static int lat_warm_for(int N) { const int w = 40 + N / 16; return w < 48 ? 48 : (w > 96 ? 96 : w); }

struct LatArgs {
    int N, B, iterations, n_llr, num_sms, warm;
    double sf_inner, sf_last;
    const int16_t *tab;             // [7][N]: perm, inv_perm, offA, offW1, offY1, offW2, offY2
    const void *llr;                 // [B][llr_stride] elements of the kernel's LlrT (float32, binary16 or int8)
    long long llr_stride;
    int32_t *bits;
    uint32_t *packed;
    const uint8_t *ref_bits;
    unsigned long long *counters;
    float llr_scale;                 // int8 element q is the LLR q * llr_scale (last: the other members keep their offsets)
    float *app;                      // [B][2N] a-posteriori LLRs (float2 per couple) or NULL; last, for the same reason
};

__device__ __forceinline__ void ld16(const float *p, float (&v)[16])
{
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 t = reinterpret_cast<const float4 *>(p)[q];
        v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
    }
}
__device__ __forceinline__ void st16(float *p, const float (&v)[16])
{
#pragma unroll
    for (int q = 0; q < 4; ++q) reinterpret_cast<float4 *>(p)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}
__device__ __forceinline__ void ld8(const float *p, float (&g)[8])
{
    const float4 a = reinterpret_cast<const float4 *>(p)[0], b = reinterpret_cast<const float4 *>(p)[1];
    g[0] = a.x; g[1] = a.y; g[2] = a.z; g[3] = a.w; g[4] = b.x; g[5] = b.y; g[6] = b.z; g[7] = b.w;
}


// ---- P1: one recursion (alpha, or beta in natural labels), SEGMENTED, one state metric per lane -----------------------
// The reference runs every recursion twice around the circular trellis: lap 1 from zeros, lap 2 from lap 1's end state
// (:167-183, :203-217); what it keeps is lap 2.  Two observations make that short here, both EXACT:
//  (1) the recursion is deterministic, so two runs over the same records that hold the same 16 metrics, bit for bit, at
//      one position hold the same metrics at every later position;
//  (2) runs started from different states re-join quickly (measured with the oracle: after 40 steps on average at N=212,
//      p99 108) because max-log survivors merge and the per-step normalisation removes the common offset.
// Phase A: kSegs runs of lap 1 proceed concurrently.  Segment 0 starts from zeros at position 0 — the reference's own
// lap 1; segment j > 0 starts from zeros kWarm steps before its first position, a GUESS that has usually re-joined the
// true lap 1 by the time the segment begins.  Each stores the metrics of its own positions and leaves its end state in
// shared memory.  All runs are equally long (L = (N + 3 kWarm) / 4 steps); two of them share a warp (one per half-warp:
// same direction, so both address streams advance by the same compile-time stride).
// Phase B: ONE warp carries the true trajectory.  It holds the true state at the start of segment 1 (the end state of
// segment 0); if that equals what segment 1 stored there, segment 1 and its end state are the true ones by (1) and the
// carrier jumps to the next boundary; if not, it recomputes and overwrites until its state equals the stored one (or
// the segment ends).  After the last segment it holds the true lap-1 end state and runs lap 2 from position 0 the same
// way: it stops where it has re-joined lap 1.  Every jump is taken on verified bitwise equality, so the stored metrics
// are exactly the reference's lap 2 whatever the guesses were; a frame whose runs never re-join costs two full laps.
// Sequential steps per SISO at N=212: ~101 (phase A) + ~50 (lap 2) + a few boundary checks, against 2 N = 424.
// Logical position i = 0 .. N-1 in recursion order: trellis step k = i (alpha) or N-1-i (beta).
// Per step: 4 shuffles -> 2 x (add, add, max) -> subtract: 77 - 80 cycles, of which 59 are the bare dependent chain
// (shuffle ~36 + add + max + subtract; timing-only builds), against ~120 issue cycles when one thread holds all 16
// states.  Measured slower: exchanging the metrics through shared memory (+10 %), hand-ordered schedules (+3 .. +14 %),
// alpha and beta of a segment on the two halves of one warp (per-lane stride: +45 % per step), eight warps in phase A
// (the SM's shuffle + shared-memory issue rate binds: 122 cycles per step).
template <bool BETA, int CS, int RS>   // CS / RS: floats between the metric cells / the records of consecutive steps
struct LaneRec {
    int N, la, lb, l0b, ps;
    bool swp;
    const float2 *rp, *r0;
    float *cells;                                                    // alpha: Al, beta: Be + 16; cell of step k at 16 k
    __device__ __forceinline__ void init(float *cells_, const float *rec, int N_, int tid)
    {
        const int s = tid & 15;
        // alpha: state s = 2t + b is fed by v[t], v[8+t]; beta: state s = 8 hi + t by z[2t], z[2t+1] (tpf_core.cuh)
        const int t = BETA ? (s & 7) : (s >> 1);
        N = N_; cells = cells_; ps = s;
        la = BETA ? 2 * t : t; lb = BETA ? 2 * t + 1 : 8 + t; l0b = BETA ? 1 : 8;
        swp = (((t >> 2) ^ (BETA ? (s >> 3) : s)) & 1) != 0;         // the metric added to the first operand is the odd entry
        rp = reinterpret_cast<const float2 *>(rec) + cls(t);
        r0 = reinterpret_cast<const float2 *>(rec);
    }
    __device__ __forceinline__ int kk(int i) const { return BETA ? N - 1 - i : i; }
    __device__ __forceinline__ float step(float v, float2 pc, float2 p0) const
    {
        const float a = __shfl_sync(0xffffffffu, v, la, 16), bq = __shfl_sync(0xffffffffu, v, lb, 16);
        const float v0 = __shfl_sync(0xffffffffu, v, 0, 16), v8 = __shfl_sync(0xffffffffu, v, l0b, 16);
        const float X = swp ? pc.y : pc.x, Yv = swp ? pc.x : pc.y;
        return f_sub(f_max(f_add(a, X), f_add(bq, Yv)), f_max(f_add(v0, p0.x), f_add(v8, p0.y)));
    }
    // phase A, TWO segments per warp (lanes 0-15 one, lanes 16-31 the next): from zeros at this lane's i0, `trips`
    // steps (warp-uniform), storing from step tstore on while i < i1.  Returns the state at i1.  (A short last segment
    // keeps stepping past i1 on records it does not use: the record array is padded and everything stays inside this
    // CTA's shared memory.)
    __device__ __forceinline__ float run2(int i0, int tstore, int i1, int trips) const
    {
        float v = 0.f, vend = 0.f;
        const float2 *q = rp + (RS / 2) * kk(i0), *q0 = r0 + (RS / 2) * kk(i0);
        float *cell = cells + CS * kk(i0) + ps;
        constexpr int D = BETA ? -1 : 1;
        float2 pc = q[0], p0 = q0[0];
        for (int t = 0; t < trips; ++t) {
            const float2 pn = q[(RS / 2) * D * (t + 1)], p0n = q0[(RS / 2) * D * (t + 1)];
            if (t >= tstore && i0 + t < i1) cell[CS * D * t] = v;
            v = step(v, pc, p0);
            vend = (i0 + t + 1 == i1) ? v : vend;
            pc = pn; p0 = p0n;
        }
        return vend;
    }
    // phase B: carry the true state v from position i0 towards i1, overwriting, until it equals the stored state.
    // Returns true when it re-joined (then the stored metrics from there to the end of the run they belong to are the
    // true ones); v is the true state at i1 otherwise.  (The upper half-warp mirrors the lower.)
    __device__ __forceinline__ bool carry(float &v, int i0, int i1) const
    {
        if (i0 >= i1) return false;
        float2 pc = rp[(RS / 2) * kk(i0)], p0 = r0[(RS / 2) * kk(i0)];
        bool joined = false;
        for (int i = i0; i < i1; ++i) {
            if (joined) return true;                                 // (tested one step late: the vote stays off the chain)
            const int kn = kk(i + 1 < i1 ? i + 1 : i);
            const float2 pn = rp[(RS / 2) * kn], p0n = r0[(RS / 2) * kn];
            float *cell = cells + CS * kk(i) + ps;
            joined = __all_sync(0xffffffffu, __float_as_uint(*cell) == __float_as_uint(v));
            *cell = v;
            v = step(v, pc, p0);
            pc = pn; p0 = p0n;
        }
        return joined;
    }
};

// segment boundaries: segment 0 is L steps long, segment j > 0 L - kWarm after kWarm warm-up steps: all runs take L steps
__device__ __forceinline__ int seg_len(int N, int kWarm) { return (N + (kSegs - 1) * kWarm + kSegs - 1) / kSegs; }
__device__ __forceinline__ int seg_start(int j, int N, int kWarm)
{
    if (j <= 0) return 0;
    if (j >= kSegs) return N;
    const int L = seg_len(N, kWarm);
    if (L <= kWarm) return N;                                        // short frames: segment 0 is the whole lap
    const int p = L + (j - 1) * (L - kWarm);
    return p < N ? p : N;
}

// warps 2 d and 2 d + 1 of the CTA serve direction d (0 alpha, 1 beta); wd = 0 / 1 is the warp's index in the direction
template <bool BETA, int CS, int RS>
__device__ __forceinline__ void segmented_recursion(float *cells, const float *rec, int N, int kWarm, int wd, int tid, float *es /* [kSegs][16] */)
{
    LaneRec<BETA, CS, RS> R;
    R.init(cells, rec, N, tid);
    // ---- phase A: segments 2 wd (lanes 0-15) and 2 wd + 1 (lanes 16-31) ----
    {
        const int j = 2 * wd + ((tid >> 4) & 1);
        const int p0 = seg_start(j, N, kWarm), p1 = seg_start(j + 1, N, kWarm);
        const int i0 = j == 0 ? 0 : (p0 > kWarm ? p0 - kWarm : 0);
        const int L = seg_len(N, kWarm);
        const int trips = L <= kWarm ? (wd == 0 ? N : 0) : L;       // (warp-uniform)
        // ONE call for the whole warp (it shuffles): a half-warp without a segment walks along segment 0 and stores nothing
        const bool has = p0 < p1;
        const float v = R.run2(has ? i0 : 0, has ? p0 - i0 : (1 << 30), has ? p1 : 0, trips);
        if (has) es[16 * j + R.ps] = v;
    }
    asm volatile("bar.sync %0, 64;" ::"r"(BETA ? 2 : 1) : "memory");   // the two warps of this direction
    if (wd != 0) return;
    // ---- phase B (first warp of the direction) ----
    float v = es[R.ps];                                              // true state at the end of segment 0
    for (int seg = 1; seg < kSegs; ++seg) {
        const int q0 = seg_start(seg, N, kWarm), q1 = seg_start(seg + 1, N, kWarm);
        if (q0 >= q1) continue;
        if (R.carry(v, q0, q1)) v = es[16 * seg + R.ps];             // re-joined: this segment's end state is the true one
    }
    R.carry(v, 0, N);                                                // lap 2 (:182-183 / :216-217)
}


// phase timers (SM cycles of thread 0, summed over CTAs): 0 tables + de-puncture, 1 P0, 2 P1, 3 P2, 4 hard decision, 5 total
__device__ unsigned long long g_lat_cycles[8];

// PAD: metric cells 20 instead of 16 floats apart and records 12 instead of 8, so that the position-parallel phases
// (thread k reads the 64-byte cell and the 32-byte record of step k with LDS.128) are free of bank conflicts: with
// strides of 16 / 8 words eight lanes hit two / four bank groups and P2 ran at 3 700 cycles per SISO instead of 1 500
// (ncu: its samples sit on the adds behind those loads).  Costs 48 bytes per couple: frames beyond N ~ 780 use PAD = false.
template <bool TIMED, bool PAD, class LlrT>
__global__ void __launch_bounds__(kLatThreads, 2)
lat_kernel(const LatArgs A)
{
    constexpr int CS = PAD ? 20 : 16, RS = PAD ? 12 : 8;
    long long ph[6] = {0, 0, 0, 0, 0, 0};
    const long long t_begin = TIMED ? clock64() : 0;
    extern __shared__ __align__(16) unsigned char sm[];
    const int N = A.N, tid = threadIdx.x;
    // shared-memory frame: [perm | inv] int16, then per couple: L1, L2 (float4), Le1, Le2, Y (double2), record (8 floats),
    // alpha (16 floats), beta (16 floats; index k holds beta[k], k = 1 .. N)
    int16_t *perm = reinterpret_cast<int16_t *>(sm);
    int16_t *inv = perm + N;
    unsigned char *p = sm + (((size_t)4 * N + 15) / 16) * 16;
    float4 *L1 = reinterpret_cast<float4 *>(p); p += (size_t)N * 16;
    float4 *L2 = reinterpret_cast<float4 *>(p); p += (size_t)N * 16;
    double2 *Le1 = reinterpret_cast<double2 *>(p); p += (size_t)N * 16;
    double2 *Le2 = reinterpret_cast<double2 *>(p); p += (size_t)N * 16;
    double2 *Y = reinterpret_cast<double2 *>(p); p += (size_t)N * 16;
    float *rec = reinterpret_cast<float *>(p) + RS; p += (size_t)(N + 2) * RS * 4;   // (one pad record on either side)
    float *Al = reinterpret_cast<float *>(p); p += (size_t)N * CS * 4;
    float *Be = reinterpret_cast<float *>(p); p += (size_t)(N + 1) * CS * 4;
    unsigned *words = reinterpret_cast<unsigned *>(p);              // packed hard decisions, ceil(2N/32) words
    __shared__ int s_err[2];
    __shared__ float s_es[2 * kSegs * 16];                          // end states of the lap-1 segments, per direction
    for (int frame = blockIdx.x; frame < A.B; frame += gridDim.x) {
        __syncthreads();
        long long tA = TIMED ? clock64() : 0;
        const LlrT *row = static_cast<const LlrT *>(A.llr) + (size_t)frame * A.llr_stride;
        for (int i = tid; i < 2 * N; i += kLatThreads) perm[i] = A.tab[i];
        if (tid < 2) s_err[tid] = 0;
        for (int i = tid; i < (2 * N + 31) / 32; i += kLatThreads) words[i] = 0u;
        __syncthreads();
        // ---- de-puncture (:466-487) and gather the interleaved systematic pair (:507-512) ----
        const int16_t *g_off = A.tab + 2 * N;
        for (int k = tid; k < N; k += kLatThreads) {
            const int oa = g_off[k], op = g_off[perm[k]];
            const int o0 = g_off[N + k], o1 = g_off[2 * N + k], o2 = g_off[3 * N + k], o3 = g_off[4 * N + k];
            const float sc = A.llr_scale;                           // int8 input only (llr_f32)
            L1[k] = make_float4(llr_ldg(row + oa, sc), llr_ldg(row + oa + 1, sc), o0 >= 0 ? llr_ldg(row + o0, sc) : 0.f, o1 >= 0 ? llr_ldg(row + o1, sc) : 0.f);
            L2[k] = make_float4(llr_ldg(row + op, sc), llr_ldg(row + op + 1, sc), o2 >= 0 ? llr_ldg(row + o2, sc) : 0.f, o3 >= 0 ? llr_ldg(row + o3, sc) : 0.f);
        }
        __syncthreads();
        if (TIMED) { const long long t = clock64(); ph[0] += t - tA; tA = t; }
        for (int h = 0; h < 2 * A.iterations; ++h) {
            const bool second = (h & 1) != 0, first = h == 0;
            const double sf = (h >> 1) < A.iterations - 1 ? A.sf_inner : A.sf_last;
            // ---- P0: a-priori gather, Y = Lc + La, branch-metric record (:131-160) ----
            for (int k = tid; k < N; k += kLatThreads) {
                const float4 x = second ? L2[k] : L1[k];
                double2 la = make_double2(0.0, 0.0);
                if (!first) la = second ? Le1[perm[k]] : Le2[inv[k]];
                const double YA = d_add((double)x.x, la.x), YB = d_add((double)x.y, la.y);
                float g[8];
                make_record(YA, YB, x.z, x.w, g);
                Y[k] = make_double2(YA, YB);
                reinterpret_cast<float4 *>(rec + RS * k)[0] = make_float4(g[0], g[1], g[2], g[3]);
                reinterpret_cast<float4 *>(rec + RS * k)[1] = make_float4(g[4], g[5], g[6], g[7]);
            }
            __syncthreads();
            if (TIMED) { const long long t = clock64(); ph[1] += t - tA; tA = t; }
            // ---- P1: the two recursions, twice around the circular trellis (:162-230): segmented_recursion above ----
            if (tid < 64) segmented_recursion<false, CS, RS>(Al, rec, N, A.warm, tid >> 5, tid, s_es);
            else if (tid < 128) segmented_recursion<true, CS, RS>(Be + CS, rec, N, A.warm, (tid >> 5) - 2, tid, s_es + kSegs * 16);
            __syncthreads();
            if (TIMED) { const long long t = clock64(); ph[2] += t - tA; tA = t; }
            // ---- P2: a-posteriori maxima and the float64 extrinsic (:232-281) ----
            double2 *LeOut = second ? Le2 : Le1;
            for (int k = tid; k < N; k += kLatThreads) {
                float x[16], zs[16], g[8], uv[4];
                ld16(Al + CS * k, x);
                ld16(Be + CS * (k + 1), zs);
                ld8(rec + RS * k, g);
                ext_step(x, zs, g, uv);
                const double2 y = Y[k];
                double ea, eb;
                make_extrinsic(uv, y.x, y.y, sf, ea, eb);
                LeOut[k] = make_double2(ea, eb);
            }
            __syncthreads();
            if (TIMED) { const long long t = clock64(); ph[3] += t - tA; tA = t; }
        }
        // ---- hard decision (:526-537) + optional error counting ----
        int my_err = 0;
        for (int k = tid; k < N; k += kLatThreads) {
            const float4 ab = L1[k];
            const double2 la = Le2[inv[k]], e1 = Le1[k];
            const double LA = d_add(d_add((double)ab.x, la.x), e1.x);
            const double LB = d_add(d_add((double)ab.y, la.y), e1.y);
            const int bA = LA < 0.0, bB = LB < 0.0;
            if (A.bits) *reinterpret_cast<int2 *>(A.bits + (size_t)frame * 2 * N + 2 * k) = make_int2(bA, bB);
            if (A.app)
                *reinterpret_cast<float2 *>(A.app + (size_t)frame * 2 * N + 2 * k) =
                    make_float2(__double2float_rn(LA), __double2float_rn(LB));
            atomicOr(&words[k >> 4], (unsigned)(bA | (bB << 1)) << (2 * (k & 15)));
            if (A.ref_bits) {
                const uint8_t *r = A.ref_bits + (size_t)frame * 2 * N + 2 * k;
                my_err += (bA != r[0]) + (bB != r[1]);
            }
        }
        if (my_err) atomicAdd(&s_err[0], my_err);
        __syncthreads();
        const int wpf = (2 * N + 31) / 32;
        if (A.packed)
            for (int i = tid; i < wpf; i += kLatThreads) A.packed[(size_t)frame * wpf + i] = words[i];
        if (tid == 0 && A.counters) {
            if (A.ref_bits) {
                if (s_err[0]) { atomicAdd(A.counters + 0, (unsigned long long)s_err[0]); atomicAdd(A.counters + 1, 1ull); }
            }
            atomicAdd(A.counters + 2, 1ull);
            atomicAdd(A.counters + 3, 2ull * N);
        }
        if (TIMED) { const long long t = clock64(); ph[4] += t - tA; tA = t; }
    }
    if (TIMED && tid == 0) {
        ph[5] = clock64() - t_begin;
        for (int i = 0; i < 6; ++i) atomicAdd(&g_lat_cycles[i], (unsigned long long)ph[i]);
    }
}

}  // namespace

int lat_read_phase_cycles(double *out_h, int reset) { return read_phase_cycles(g_lat_cycles, out_h, reset); }

static int g_lat_warm = 0;         // 0: lat_warm_for(N)
void set_lat_warm(int v) { g_lat_warm = v; }

static size_t lat_smem(int N, bool pad)
{
    const size_t cs = pad ? 20 : 16, rs = pad ? 12 : 8;
    return (((size_t)4 * N + 15) / 16) * 16 + (size_t)N * (16 + 16 + 16 + 16 + 16) + (size_t)(N + 2) * rs * 4 +
           (size_t)N * cs * 4 + (size_t)(N + 1) * cs * 4 + (size_t)((2 * N + 31) / 32) * 4 + 64;
}

static size_t lat_cap(size_t smem_optin)
{
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, lat_kernel<false, false, float>) != cudaSuccess) return 0;   // every instance has the same static words
    return smem_optin - fa.sharedSizeBytes;                        // the static words count against the limit
}

int lat_configure(Codec &c, size_t smem_optin)
{
    c.lat_enabled = 0;
    const size_t cap = lat_cap(smem_optin);
    if (lat_smem(c.N, false) > cap) return B200DVB_OK;
    c.lat_pad = lat_smem(c.N, true) <= cap;
    const size_t need = lat_smem(c.N, c.lat_pad != 0);
    B2_CHECK(for_each_llr_type([&](auto t) {
        using L = decltype(t);
        B2_CUDA(cudaFuncSetAttribute(lat_kernel<false, false, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap));
        B2_CUDA(cudaFuncSetAttribute(lat_kernel<true, false, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap));
        B2_CUDA(cudaFuncSetAttribute(lat_kernel<false, true, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap));
        B2_CUDA(cudaFuncSetAttribute(lat_kernel<true, true, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap));
        return B200DVB_OK;
    }));
    int occ = 0;
    if (c.lat_pad) B2_CHECK(occupancy_all_formats(&occ, [](auto t) { return lat_kernel<false, true, decltype(t)>; }, kLatThreads, need));
    else           B2_CHECK(occupancy_all_formats(&occ, [](auto t) { return lat_kernel<false, false, decltype(t)>; }, kLatThreads, need));
    if (occ < 1) return B200DVB_OK;
    c.lat_enabled = 1;
    c.lat_frames_per_wave = (occ < 2 ? occ : 2) * c.num_sms;     // at most two CTAs per SM
    return B200DVB_OK;
}

int lat_launch_decode(const Codec &c, const DecodeIo &io)
{
    LatArgs A{};
    fill_decode_args(A, c, io);
    A.N = c.N; A.n_llr = c.n_llr; A.num_sms = c.num_sms; A.warm = g_lat_warm > 0 ? g_lat_warm : lat_warm_for(c.N);
    const int grid = io.B < c.lat_frames_per_wave ? io.B : c.lat_frames_per_wave;
    const size_t smem = lat_smem(c.N, c.lat_pad != 0);
    const bool pad = c.lat_pad != 0, timed = c.opt_phase_timers != 0;
    with_llr_type(io.fmt, [&](auto t) {
        using L = decltype(t);
        if (pad) {
            if (timed) lat_kernel<true, true, L><<<grid, kLatThreads, smem, io.stream>>>(A);
            else       lat_kernel<false, true, L><<<grid, kLatThreads, smem, io.stream>>>(A);
        } else {
            if (timed) lat_kernel<true, false, L><<<grid, kLatThreads, smem, io.stream>>>(A);
            else       lat_kernel<false, false, L><<<grid, kLatThreads, smem, io.stream>>>(A);
        }
    });
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

}  // namespace b200dvb
