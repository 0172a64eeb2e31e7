// common.cuh — shared declarations for libb200dvb.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stddef.h>
#include <type_traits>
#include "../../include/b200dvb.h"

namespace b200dvb {

// ---- channel LLR element format ------------------------------------------------
// Channel LLRs arrive as float32 (b200dvb_decode), IEEE binary16 (b200dvb_decode_f16) or int8 with a float32 scale
// (b200dvb_decode_i8).  The decode kernels take the element type LlrT as a template parameter and read channel LLRs
// only through these helpers, which turn an element into its float32 value where the value is consumed: binary16 is
// widened exactly, int8 q becomes the IEEE product q * scale (the library builds with --fmad=false).  Everything after
// the load is the float32 kernel's, fed the same float32 values.  The float32 and binary16 overloads ignore the scale.
enum class LlrFormat { F32, F16, I8 };
// f(L{}) with L the element type of format fmt: the one place that maps a format to its type
template <class F> inline auto with_llr_type(LlrFormat fmt, F &&f)
{
    switch (fmt) {
    case LlrFormat::F16: return f(__half{});
    case LlrFormat::I8: return f(int8_t{});
    default: return f(float{});
    }
}
// f(L{}) for every element type, in turn while it returns B200DVB_OK; the first other code is the result
template <class F> inline int for_each_llr_type(F &&f)
{
    int rc = f(float{});
    if (rc == B200DVB_OK) rc = f(__half{});
    if (rc == B200DVB_OK) rc = f(int8_t{});
    return rc;
}
inline int llr_bytes(LlrFormat f) { return with_llr_type(f, [](auto t) { return (int)sizeof(t); }); }
__device__ __forceinline__ float llr_f32(float x, float) { return x; }
__device__ __forceinline__ float llr_f32(__half x, float) { return __half2float(x); }
__device__ __forceinline__ float llr_f32(int8_t x, float s) { return __fmul_rn((float)x, s); }
template <class L> __device__ __forceinline__ float llr_ldg(const L *p, float s) { return llr_f32(__ldg(p), s); }
// two adjacent elements; p is aligned to two elements
__device__ __forceinline__ float2 llr_ldg2(const float *p, float) { return __ldg(reinterpret_cast<const float2 *>(p)); }
__device__ __forceinline__ float2 llr_ldg2(const __half *p, float) { return __half22float2(__ldg(reinterpret_cast<const __half2 *>(p))); }
__device__ __forceinline__ float2 llr_ldg2(const int8_t *p, float s)
{
    const char2 v = __ldg(reinterpret_cast<const char2 *>(p));
    return make_float2(__fmul_rn((float)v.x, s), __fmul_rn((float)v.y, s));
}
// float4 (16-byte) units of an LLR row of n elements, as the bulk-copy transpositions stage it
template <class L> __host__ __device__ __forceinline__ int llr_row_q(int n)
{
    return sizeof(L) == 4 ? (n + 3) / 4 : sizeof(L) == 2 ? (n + 7) / 8 : (n + 15) / 16;
}
inline int llr_row_q(LlrFormat f, int n)
{
    return with_llr_type(f, [n](auto t) { return llr_row_q<decltype(t)>(n); });
}

// ---- error plumbing --------------------------------------------------------
void set_cuda_error(cudaError_t e, const char *where);
#define B2_CUDA(call)                                                     \
    do {                                                                  \
        cudaError_t e__ = (call);                                         \
        if (e__ != cudaSuccess) {                                         \
            ::b200dvb::set_cuda_error(e__, #call);                        \
            return B200DVB_ECUDA;                                         \
        }                                                                 \
    } while (0)
// a B200DVB_* code other than B200DVB_OK is returned to the caller as it is
#define B2_CHECK(call)                                                    \
    do {                                                                  \
        const int rc__ = (call);                                          \
        if (rc__ != B200DVB_OK) return rc__;                              \
    } while (0)

// CTAs per SM that every element-format instance of a kernel reaches (kernel_of(L{}) is the instance for element type
// L): one geometry (frames per wave, grid) serves float32, binary16 and int8 input, so it must fit the one with the
// largest footprint
template <class K> inline int occupancy_all_formats(int *occ, K kernel_of, int threads, size_t smem)
{
    *occ = 1 << 30;
    return for_each_llr_type([&](auto t) {
        int n = 0;
        B2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel_of(t), threads, smem));
        if (n < *occ) *occ = n;
        return B200DVB_OK;
    });
}

// a kernel's eight per-phase cycle counters (a __device__ unsigned long long[8]) -> out_h; reset: zero them
template <class Sym> int read_phase_cycles(const Sym &counters, double *out_h, int reset)
{
    unsigned long long h[8];
    B2_CUDA(cudaMemcpyFromSymbol(h, counters, sizeof h));
    for (int i = 0; i < 8; ++i) out_h[i] = (double)h[i];
    if (reset) {
        unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        B2_CUDA(cudaMemcpyToSymbol(counters, z, sizeof z));
    }
    return B200DVB_OK;
}

constexpr int kMaxN = 2048;

// ---- decoder geometry (decode_quad.cu) --------------------------------------
constexpr int kFramesPerCta = 8;    // one 4-lane "quad" per frame and direction
constexpr int kCtaThreads = 64;     // per group: one forward (alpha) warp + one backward (beta) warp
constexpr int kMaxGroups = 7;       // groups (of 8 frames) per CTA
constexpr int kMaxCtaThreads = 448; // 14 warps: 2 per group + helper warps for the data-parallel phases
constexpr int kWin = 8;             // checkpoint spacing / recompute window (steps)

struct QuadGeom {
    int N;            // couples per frame
    unsigned magic;   // floor(2^32 / N) + 1: flat position -> (frame, step) without a divide
    int M;            // crossing point: alpha warp owns [M,N), beta warp owns [0,M)
    int nckA;         // alpha checkpoints (alpha[0], alpha[8], ... alpha[M-8])
    int nckB;         // beta checkpoints, one per alpha-warp window end
    int rec_stride;   // floats between two frames' branch-metric records (8N + 8)
    int ck_stride;    // floats between two frames' checkpoint areas
    int groups;       // (alpha warp, beta warp) pairs per CTA
    int threads;      // CTA size: 64 * groups recursion threads + helper warps
    int use_tmem;     // recursion checkpoints live in tensor memory instead of shared memory
    int tmem_cols;    // TMEM columns allocated per CTA (power of two >= 32)
    int y_slots;      // > 0: Y = Lc + La is parked in TMEM, this many positions per thread
    int frames;       // frames per CTA (8 * groups, or 4/2/1 when even one group does not fit)
    int ctas_per_sm;
    int grec;         // branch-metric records live in the (L1/L2-cached) global workspace, not in shared memory
    size_t smem_bytes;
};

// ---- thread-per-frame decoder geometry (decode_tpf.cu) ----------------------
constexpr int kTpfFrames = 16;      // frames per warp: lanes 0-15 run alpha, lanes 16-31 beta of the same frames
constexpr int kTpfWarps = 4;        // one warp per SM sub-partition, each with its own TMEM lane quadrant
constexpr int kTpfWin = 4;          // checkpoint spacing / recompute window (steps)
constexpr int kRingPairs = 4;       // prefetch ring depth of the "in" pass in step pairs (2 KB each: the whole beta-vector area)
// per-warp staging area: [0, 8K) beta vectors of the current window, [kTpfWin][4][32] float4 (the prefetch ring of the
// "in" pass, 6 KB, aliases it); [8K, 10K) Z slot; [10K, 12K) X slot
constexpr int kStageBytes = 12288;
constexpr int kRowFloats = kStageBytes / 8;   // transposition: two frame rows of up to 1536 LLRs each share the staging area

struct TpfGeom {
    int enabled;      // this codec is decoded by the thread-per-frame kernel
    int N, M;         // couples per frame; crossing point M = N / 2
    int T;            // branch-metric records per frame end kept in tensor memory ([0,T) and [N-T,N))
    int mid;          // records per frame kept in shared memory ([T, N-T))
    int nfull, rag;   // full recompute windows per half and length of the ragged last one (M % kTpfWin)
    int nslots;       // checkpoints per lane
    int tmem_cols;    // TMEM columns allocated per CTA (power of two >= 8 T, >= 32)
    size_t smem_bytes;
    size_t off_l1, off_l2, off_le, off_lef, off_y, off_ck, off_init;   // byte offsets in a warp's workspace (off_init: nii mode only)
    size_t ws_per_warp;
};

struct Codec {
    int N = 0, period = 0, iterations = 0, n_llr = 0;
    double sf_inner = 0.7, sf_last = 1.0;
    QuadGeom geom{};
    QuadGeom geom_g{};            // long frames: the same kernel with its records in global memory (geom_g.grec = 1) or frames = 0
    TpfGeom tpf{};
    TpfGeom nii{};                // geometry of the non-parity "nii" mode (decode_nii.cu)
    int num_sms = 0;
    int vec_ab = 0, vec_wy = 0;   // (A,B) / (W,Y) LLR pairs are adjacent and even-aligned in the stream
    // development / test switches (b200dvb_codec_set_option); all 0 in production
    int opt_kernel = 0;           // 0: automatic choice per batch, 1: quad kernel, 2: thread-per-frame kernel, 3: low-latency kernel
    int opt_no_row_staging = 0;   // 1: thread-per-frame transposition without the cp.async row staging
    int opt_phase_timers = 0;     // 1: run the kernel instances that keep per-phase cycle counters
    int lat_pad = 0;              // low-latency kernel: conflict-free (padded) shared-memory strides fit for this N
    int lat_enabled = 0, lat_frames_per_wave = 0;   // low-latency kernel (decode_lat.cu): usable for this N; frames it takes at once
    int opt_mode = 0;             // decoder arithmetic: 0 = parity (the reference's), 1 = non-parity "nii" (B200DVB_MODE_NII)
    // device tables
    int16_t *d_tab = nullptr;     // [7][N] int16: perm, inv_perm, offA, offW1, offY1, offW2, offY2
    // host tables
    int32_t next_state[64], out_W[64], out_Y[64];
    int32_t circ_lut[16];
    int16_t *h_tab = nullptr;
};

struct Modem {
    int mod_id = 0, bps = 0, M = 0;
    int separable = 0;            // 1: first half of the label selects I, 2: selects Q, 0: not separable
    int half = 0, nlev = 0;       // bits / levels per axis when separable
    int pwl = 0;                  // piecewise-linear per-axis demapper usable (uniform PAM axes)
    int nseg = 0;                 // segments per axis (2*nlev - 2)
    float pwl_x0[2] = {0, 0}, pwl_invd[2] = {0, 0};   // per axis (0: first half of label, 1: second)
    double *d_table64 = nullptr;  // double2[M]
    float *d_table32 = nullptr;   // float2[M]
    float *d_pwl = nullptr;       // float2[2][half][nseg] (slope, intercept)
    double h_table[512];
};

// One decode call (b200dvb_decode / _f16 / _i8 / _app, B > 0): llr holds B rows of elements of format fmt, llr_stride
// elements apart; llr_scale multiplies int8 elements and is unused otherwise.  app (float32 [B][2N], 8-byte aligned:
// each couple's two values are stored as one float2), bits, packed, ref_bits and counters may be NULL.
struct DecodeIo {
    int B;
    const void *llr;
    LlrFormat fmt;
    float llr_scale;
    long long llr_stride;
    float *app;
    int32_t *bits;
    uint32_t *packed;
    const uint8_t *ref_bits;
    unsigned long long *counters;
    void *ws;
    size_t ws_bytes;
    cudaStream_t stream;
};

// the members every decode kernel's argument struct shares; sf_inner / sf_last where the struct keeps them in float64
template <class Args> inline void fill_decode_args(Args &A, const Codec &c, const DecodeIo &io)
{
    A.B = io.B; A.iterations = c.iterations; A.tab = c.d_tab;
    A.llr = io.llr; A.llr_stride = io.llr_stride; A.llr_scale = io.llr_scale;
    A.bits = io.bits; A.packed = io.packed; A.ref_bits = io.ref_bits; A.counters = io.counters; A.app = io.app;
    if constexpr (std::is_same<decltype(A.sf_inner), double>::value) { A.sf_inner = c.sf_inner; A.sf_last = c.sf_last; }
}

// launchers and configuration (each returns a B200DVB_* code).  *_configure: smem_optin is the device's
// sharedMemPerBlockOptin, and c.num_sms is set
int quad_configure(Codec &c, size_t smem_optin);
int quad_launch_decode(const Codec &c, const DecodeIo &io);
int launch_siso(const Codec &c, int B, const float *Lc_A, const float *Lc_B, const float *Lc_W,
                const float *Lc_Y, const double *La_A, const double *La_B, double sf,
                double *Le_A, double *Le_B, void *ws, size_t ws_bytes, cudaStream_t s);
size_t quad_workspace_bytes(const Codec &c, int B);
size_t siso_workspace_bytes(const Codec &c, int B);
int quad_read_phase_cycles(double *out_h, int reset);
int tpf_configure(Codec &c, size_t smem_optin);
int tpf_launch_decode(const Codec &c, const DecodeIo &io);
size_t tpf_workspace_bytes(const Codec &c, int B);
int tpf_read_phase_cycles(double *out_h, int reset);
int nii_configure(Codec &c, size_t smem_optin);
int nii_launch_decode(const Codec &c, const DecodeIo &io);
size_t nii_workspace_bytes(const Codec &c, int B);
int nii_read_phase_cycles(double *out_h, int reset);
int lat_configure(Codec &c, size_t smem_optin);
int lat_launch_decode(const Codec &c, const DecodeIo &io);
int lat_read_phase_cycles(double *out_h, int reset);

// host geometry of the thread-per-frame family (decode_tpf.cu: parity mode tpf; decode_nii.cu: nii / nii16)
// g for N couples, left disabled (g.enabled = 0) when N does not fit.  y_cols: spare TMEM columns per lane that park the
// window's Y; hdr_bytes: shared memory between the interleaver tables and the records; ext_bytes: bytes per frame and
// step of each of Le, LeF and Y in the workspace; with_init: the workspace also keeps the boundary metrics (nii)
void tpf_family_geometry(TpfGeom &g, int N, int y_cols, size_t hdr_bytes, size_t ext_bytes, bool with_init, size_t smem_optin);
int tpf_family_grid(const Codec &c, int B, int tile);   // CTAs for B frames, `tile` frames per warp
size_t tpf_family_workspace_bytes(const Codec &c, const TpfGeom &g, int B, int tile);
int tpf_family_row_staging(const Codec &c, const TpfGeom &g, const DecodeIo &io);   // the kernel's `vec4`

int launch_encode(const Codec &c, int B, const uint8_t *info, uint8_t *coded, uint8_t *circ,
                  cudaStream_t s);
int launch_mc_bpsk(const Codec &c, int B, float noise_var, unsigned long long seed,
                   unsigned long long frame_offset, uint8_t *info, uint8_t *coded, float *llr,
                   cudaStream_t s);

int launch_awgn_complex(size_t n, float sigma, unsigned long long seed, unsigned long long offset,
                        void *iq, cudaStream_t s);
int launch_fading_complex(size_t n, int block_len, float sigma, unsigned long long seed, unsigned long long offset,
                          void *iq, void *gain, cudaStream_t s);

int launch_map(const Modem &m, size_t n, const uint8_t *bits, void *iq, int out_f64, cudaStream_t s);
int launch_demap(const Modem &m, size_t n, const void *iq, float noise_var, float scale,
                 float *llr, cudaStream_t s);
int launch_demap_bf16(const Modem &m, size_t n, const void *iq, float noise_var, float scale,
                      float *llr, cudaStream_t s);
int launch_demap_csi(const Modem &m, size_t n, const void *iq, const void *gain, float noise_var, float scale,
                     float *llr, cudaStream_t s);
int launch_hard(const Modem &m, size_t n, const void *iq, int in_f64, uint8_t *bits, cudaStream_t s);

constexpr int kMaxFirTaps = 448;    // FIR taps travel in the kernel parameter space (constant bank): 8 B per tap of 4 KB
int launch_pulse_shape(size_t n_sym, const void *sym, const double *taps_h, int ntaps, int sps, void *out, cudaStream_t s);
int launch_matched_filter(size_t n, const void *x, const double *taps_h, int ntaps, int sps, long long start,
                          size_t n_out, void *out, cudaStream_t s);

void set_mf_variant(int v);
void set_lat_warm(int v);
void set_map_variant(int v);
int modem_build_pwl(Modem &m);
int run_microbench(double *results_h);
int run_microbench2(double *results16_h);
int run_tmem_selftest(int *result_h);

}  // namespace b200dvb
