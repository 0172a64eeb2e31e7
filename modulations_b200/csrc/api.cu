// api.cu — the extern "C" surface of libb200dvb.so (see include/b200dvb.h).
#include "common.cuh"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>

namespace b200dvb {

static thread_local char g_cuda_err[256] = "";

void set_cuda_error(cudaError_t e, const char *where)
{
    snprintf(g_cuda_err, sizeof g_cuda_err, "%s: %s (%s)", cudaGetErrorName(e),
             cudaGetErrorString(e), where);
}

// The decoder and encoder kernels are specialised for the reference trellis
// (dvb_rcs2_turbo.py:338-370): dk = A^B^s2^s3, ns = 2*(s&7) + dk,
// w = A^B^s0^s1^s2, y = A^B^s1.  Anything else is refused, not emulated.
static bool trellis_supported(const int32_t *ns, const int32_t *oW, const int32_t *oY)
{
    for (int s = 0; s < 16; ++s)
        for (int u = 0; u < 4; ++u) {
            const int ab = ((u >> 1) ^ u) & 1;
            const int s0 = s & 1, s1 = (s >> 1) & 1, s2 = (s >> 2) & 1, s3 = (s >> 3) & 1;
            const int dk = ab ^ s2 ^ s3;
            if (ns[s * 4 + u] != 2 * (s & 7) + dk) return false;
            if (oW[s * 4 + u] != (ab ^ s0 ^ s1 ^ s2)) return false;
            if (oY[s * 4 + u] != (ab ^ s1)) return false;
        }
    return true;
}

// GF(2) 4x4 matrices bit-packed one row per nibble-bit: row i = bits of m[i].
// x' = G x with x = (s0..s3) packed as an int (dvb_rcs2_turbo.py:372-383).
static inline int gf2_mat_vec(const int m[4], int x)
{
    int r = 0;
    for (int i = 0; i < 4; ++i) r |= (__builtin_popcount(m[i] & x) & 1) << i;
    return r;
}
static void gf2_mat_mul(const int a[4], const int b[4], int c[4])
{   // c = a*b ; column j of b is b applied to e_j
    int t[4] = {0, 0, 0, 0};
    for (int j = 0; j < 4; ++j) {
        const int col = gf2_mat_vec(a, gf2_mat_vec(b, 1 << j));
        for (int i = 0; i < 4; ++i) t[i] |= ((col >> i) & 1) << j;
    }
    memcpy(c, t, sizeof t);
}
// Sc = (I + G^N)^-1 Z for all 16 Z (mat_pow_gf2 + solve_circular_state_gf2,
// dvb_rcs2_turbo.py:50-114).  I + G^N is invertible for every N that is not a
// multiple of the LFSR period 15; if it is singular we reproduce the reference's
// Gaussian-elimination result instead of a true inverse.
static void circular_lut(const int32_t *ns, int N, int32_t lut[16])
{
    int G[4] = {0, 0, 0, 0};
    for (int j = 0; j < 4; ++j) {               // column j = zero-input response of e_j
        const int col = ns[(1 << j) * 4 + 0];
        for (int i = 0; i < 4; ++i) G[i] |= ((col >> i) & 1) << j;
    }
    int R[4] = {1, 2, 4, 8}, base[4];
    memcpy(base, G, sizeof base);
    for (long long p = N; p > 0; p >>= 1) {
        if (p & 1) gf2_mat_mul(R, base, R);
        gf2_mat_mul(base, base, base);
    }
    for (int z = 0; z < 16; ++z) {
        int M[4][5];
        for (int i = 0; i < 4; ++i) {
            for (int j = 0; j < 4; ++j) M[i][j] = ((i == j) + ((R[i] >> j) & 1)) & 1;
            M[i][4] = (z >> i) & 1;
        }
        for (int i = 0; i < 4; ++i) {
            if (M[i][i] == 0)
                for (int k = i + 1; k < 4; ++k)
                    if (M[k][i] == 1) {
                        for (int j = 0; j < 5; ++j) { int t = M[i][j]; M[i][j] = M[k][j]; M[k][j] = t; }
                        break;
                    }
            if (M[i][i] == 1)
                for (int k = i + 1; k < 4; ++k)
                    if (M[k][i] == 1)
                        for (int j = 0; j < 5; ++j) M[k][j] ^= M[i][j];
        }
        int x[4] = {0, 0, 0, 0}, st = 0;
        for (int i = 3; i >= 0; --i) {
            int sum = M[i][4];
            for (int j = i + 1; j < 4; ++j) sum ^= (M[i][j] & x[j]);
            x[i] = sum;
        }
        for (int i = 0; i < 4; ++i) if (x[i]) st |= 1 << i;
        lut[z] = st;
    }
}

}  // namespace b200dvb

using namespace b200dvb;

struct b200dvb_codec { Codec c; };
struct b200dvb_modem { Modem m; };

extern "C" {

int b200dvb_version(void) { return 100; }

const char *b200dvb_error_string(int code)
{
    switch (code) {
    case B200DVB_OK: return "ok";
    case B200DVB_EINVAL: return "invalid argument";
    case B200DVB_ENOSPEC: return "no kernel specialisation for these tables/sizes";
    case B200DVB_ECUDA: return "CUDA error";
    case B200DVB_ENOMEM: return "workspace too small or allocation failed";
    case B200DVB_EMOD: return "unknown modulation";
    default: return "unknown error";
    }
}

const char *b200dvb_last_cuda_error(void) { return g_cuda_err; }

int b200dvb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int b200dvb_codec_create(int N, const int32_t *next_state_h, const int32_t *out_W_h,
                         const int32_t *out_Y_h, const int32_t *perm_h, const int32_t *inv_perm_h,
                         const uint8_t *punct_h, int period, int iterations, double sf_inner,
                         double sf_last, b200dvb_codec_t *out)
{
    if (!out || !next_state_h || !out_W_h || !out_Y_h || !perm_h || !inv_perm_h || !punct_h)
        return B200DVB_EINVAL;
    if (period < 1 || period > 64 || iterations < 1 || N < 1) return B200DVB_EINVAL;
    if (!trellis_supported(next_state_h, out_W_h, out_Y_h)) return B200DVB_ENOSPEC;
    for (int i = 0; i < N; ++i)
        if (perm_h[i] < 0 || perm_h[i] >= N || inv_perm_h[i] < 0 || inv_perm_h[i] >= N)
            return B200DVB_EINVAL;
    b200dvb_codec *h = new (std::nothrow) b200dvb_codec();
    if (!h) return B200DVB_ENOMEM;
    Codec &c = h->c;
    c.N = N; c.period = period; c.iterations = iterations;
    c.sf_inner = sf_inner; c.sf_last = sf_last;
    memcpy(c.next_state, next_state_h, sizeof c.next_state);
    memcpy(c.out_W, out_W_h, sizeof c.out_W);
    memcpy(c.out_Y, out_Y_h, sizeof c.out_Y);
    circular_lut(next_state_h, N, c.circ_lut);
    // the device's SM count and shared-memory limit, read once for every decoder's geometry
    int dev = 0, smem_optin = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&c.num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) { set_cuda_error(e, "codec_create device attributes"); delete h; return B200DVB_ECUDA; }
    int rc = quad_configure(c, smem_optin);
    if (rc == B200DVB_OK) rc = tpf_configure(c, smem_optin);
    if (rc == B200DVB_OK) rc = nii_configure(c, smem_optin);
    if (rc == B200DVB_OK) rc = lat_configure(c, smem_optin);
    if (rc != B200DVB_OK) { delete h; return rc; }
    // stream offsets (depuncture order of dvb_rcs2_turbo.py:476-487)
    c.h_tab = (int16_t *)malloc(sizeof(int16_t) * 7 * N);
    if (!c.h_tab) { delete h; return B200DVB_ENOMEM; }
    int idx = 0;
    for (int i = 0; i < N; ++i) {
        const int p = i % period;
        c.h_tab[0 * N + i] = (int16_t)perm_h[i];
        c.h_tab[1 * N + i] = (int16_t)inv_perm_h[i];
        c.h_tab[2 * N + i] = (int16_t)idx; idx += 2;
        for (int j = 0; j < 4; ++j)
            c.h_tab[(3 + j) * N + i] = punct_h[j * period + p] ? (int16_t)idx++ : (int16_t)-1;
    }
    c.n_llr = idx;
    c.vec_ab = 1; c.vec_wy = 1;
    for (int i = 0; i < N; ++i) {
        if (c.h_tab[2 * N + i] & 1) c.vec_ab = 0;
        for (int e = 0; e < 2; ++e) {
            const int ow = c.h_tab[(3 + 2 * e) * N + i], oy = c.h_tab[(4 + 2 * e) * N + i];
            if (ow < 0 || oy != ow + 1 || (ow & 1)) c.vec_wy = 0;
        }
    }
    if (idx > 32767) { free(c.h_tab); delete h; return B200DVB_ENOSPEC; }
    e = cudaMalloc(&c.d_tab, sizeof(int16_t) * 7 * N);
    if (e == cudaSuccess)
        e = cudaMemcpy(c.d_tab, c.h_tab, sizeof(int16_t) * 7 * N, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        set_cuda_error(e, "codec_create tables");
        if (c.d_tab) cudaFree(c.d_tab);
        free(c.h_tab); delete h;
        return B200DVB_ECUDA;
    }
    *out = h;
    return B200DVB_OK;
}

int b200dvb_codec_destroy(b200dvb_codec_t codec)
{
    if (!codec) return B200DVB_EINVAL;
    if (codec->c.d_tab) cudaFree(codec->c.d_tab);
    free(codec->c.h_tab);
    delete codec;
    return B200DVB_OK;
}

int b200dvb_codec_n_llr(b200dvb_codec_t codec) { return codec ? codec->c.n_llr : B200DVB_EINVAL; }

int b200dvb_codec_frames_per_wave(b200dvb_codec_t codec)
{
    if (!codec) return B200DVB_EINVAL;
    const Codec &c = codec->c;
    if (c.opt_mode == B200DVB_MODE_NII16) return c.num_sms * kTpfWarps * kTpfFrames * 2;   // two frames per lane
    if (c.opt_mode == B200DVB_MODE_NII || c.tpf.enabled) return c.num_sms * kTpfWarps * kTpfFrames;
    if (c.geom_g.frames > 0) return c.num_sms * c.geom_g.ctas_per_sm * c.geom_g.frames;   // long frames, large batches
    return c.num_sms * c.geom.ctas_per_sm * c.geom.frames;
}

int b200dvb_codec_circular_lut(b200dvb_codec_t codec, int32_t *lut16_h)
{
    if (!codec || !lut16_h) return B200DVB_EINVAL;
    memcpy(lut16_h, codec->c.circ_lut, sizeof codec->c.circ_lut);
    return B200DVB_OK;
}

size_t b200dvb_siso_workspace_bytes(b200dvb_codec_t codec, int B)
{
    return (codec && B > 0) ? siso_workspace_bytes(codec->c, B) : 0;
}

int b200dvb_siso(b200dvb_codec_t codec, int B, const float *Lc_A, const float *Lc_B,
                 const float *Lc_W, const float *Lc_Y, const double *La_A, const double *La_B,
                 double scaling_factor, double *Le_A, double *Le_B, void *workspace,
                 size_t workspace_bytes, void *stream)
{
    if (!codec || B < 0 || !Lc_A || !Lc_B || !Lc_W || !Lc_Y || !Le_A || !Le_B || (B && !workspace))
        return B200DVB_EINVAL;
    return launch_siso(codec->c, B, Lc_A, Lc_B, Lc_W, Lc_Y, La_A, La_B, scaling_factor, Le_A, Le_B,
                       workspace, workspace_bytes, (cudaStream_t)stream);
}

// Which decode kernel serves a batch of B frames.  The thread-per-frame kernel has the higher throughput but a
// 16-frame tile takes as long as a full wave (64 frames per SM); the quad kernel finishes a wave of 32 frames per
// SM in 0.72x that time (profiles/r02_measure_pack1.txt: 0.75 ms against 1.05 ms at N=212), so batches that fit one
// quad wave go there.  A pure function of (codec, B): the workspace query and the launch agree.
// Small batches take the low-latency kernel (one CTA per frame, two CTAs per SM while the frame fits twice): a pass
// over up to lat_frames_per_wave frames takes 0.11 / 0.155 / 0.29 ms at N = 48 / 212 / 752, a quad-kernel wave 0.15 /
// 0.65 - 0.76 / 1.84 ms, so up to min(6, N / 50) passes of it beat one quad wave (profiles/r02_latency.txt).
static int lat_passes(const Codec &c) { const int p = c.N / 50; return p < 1 ? 1 : (p > 6 ? 6 : p); }
static bool use_lat(const Codec &c, int B)
{
    if (!c.lat_enabled) return false;
    if (c.opt_kernel == 3) return true;
    return c.opt_kernel == 0 && (long long)B <= (long long)lat_passes(c) * c.lat_frames_per_wave;
}

static bool use_tpf(const Codec &c, int B)
{
    if (!c.tpf.enabled || c.opt_kernel == 1) return false;
    if (c.opt_kernel == 2) return true;
    const long long quad_wave = (long long)c.num_sms * c.geom.ctas_per_sm * c.geom.frames;
    return !(c.geom.frames <= 32 && B <= quad_wave);
}

// The one decision of which kernel decodes a batch: both the workspace query and the launch switch on it.  The
// non-parity modes have one kernel.
enum class Decoder { NII, LAT, TPF, QUAD };
static Decoder decoder_for(const Codec &c, int B)
{
    if (c.opt_mode != B200DVB_MODE_PARITY) return Decoder::NII;
    if (use_lat(c, B)) return Decoder::LAT;
    return use_tpf(c, B) ? Decoder::TPF : Decoder::QUAD;
}

size_t b200dvb_decode_workspace_bytes(b200dvb_codec_t codec, int B)
{
    if (!codec || B <= 0) return 0;
    switch (decoder_for(codec->c, B)) {
    case Decoder::NII: return nii_workspace_bytes(codec->c, B);
    case Decoder::LAT: return 256;                                   // the whole frame lives in shared memory
    case Decoder::TPF: return tpf_workspace_bytes(codec->c, B);
    default: return quad_workspace_bytes(codec->c, B);
    }
}

int b200dvb_codec_set_option(b200dvb_codec_t codec, int option, int value)
{
    if (!codec) return B200DVB_EINVAL;
    Codec &c = codec->c;
    switch (option) {
    case B200DVB_OPT_KERNEL:
        if (value < 0 || value > 3) return B200DVB_EINVAL;
        if (value == 2 && !c.tpf.enabled) return B200DVB_ENOSPEC;
        if (value == 3 && !c.lat_enabled) return B200DVB_ENOSPEC;
        c.opt_kernel = value;
        return B200DVB_OK;
    case B200DVB_OPT_NO_ROW_STAGING: c.opt_no_row_staging = value != 0; return B200DVB_OK;
    case B200DVB_OPT_PHASE_TIMERS: c.opt_phase_timers = value != 0; return B200DVB_OK;
    case B200DVB_OPT_DECODER_MODE:
        if (value != B200DVB_MODE_PARITY && value != B200DVB_MODE_NII && value != B200DVB_MODE_NII16) return B200DVB_EINVAL;
        if (value != B200DVB_MODE_PARITY && !c.nii.enabled) return B200DVB_ENOSPEC;
        c.opt_mode = value;
        return B200DVB_OK;
    default: return B200DVB_EINVAL;
    }
}

// b200dvb_decode / _f16 / _i8 / _app: the kernel choice depends neither on the element format nor on the outputs
static int decode_any(b200dvb_codec_t codec, int B, const void *llr, LlrFormat fmt, float llr_scale, long long llr_stride,
                      float *app, int32_t *bits, uint32_t *packed, const uint8_t *ref_bits,
                      unsigned long long *counters, void *workspace, size_t workspace_bytes,
                      void *stream)
{
    if (!codec || B < 0 || !llr || (B && !workspace)) return B200DVB_EINVAL;
    if (llr_stride < codec->c.n_llr) return B200DVB_EINVAL;
    if (B == 0) return B200DVB_OK;
    const DecodeIo io{B, llr, fmt, llr_scale, llr_stride, app, bits, packed, ref_bits, counters, workspace,
                      workspace_bytes, (cudaStream_t)stream};
    switch (decoder_for(codec->c, B)) {
    case Decoder::NII: return nii_launch_decode(codec->c, io);
    case Decoder::LAT: return lat_launch_decode(codec->c, io);
    case Decoder::TPF: return tpf_launch_decode(codec->c, io);
    default: return quad_launch_decode(codec->c, io);
    }
}

int b200dvb_decode(b200dvb_codec_t codec, int B, const float *llr, long long llr_stride,
                   int32_t *bits, uint32_t *packed, const uint8_t *ref_bits,
                   unsigned long long *counters, void *workspace, size_t workspace_bytes,
                   void *stream)
{
    return decode_any(codec, B, llr, LlrFormat::F32, 1.f, llr_stride, nullptr, bits, packed, ref_bits, counters,
                      workspace, workspace_bytes, stream);
}

int b200dvb_decode_f16(b200dvb_codec_t codec, int B, const void *llr, long long llr_stride,
                       int32_t *bits, uint32_t *packed, const uint8_t *ref_bits,
                       unsigned long long *counters, void *workspace, size_t workspace_bytes,
                       void *stream)
{
    if (reinterpret_cast<uintptr_t>(llr) & 1) return B200DVB_EINVAL;
    return decode_any(codec, B, llr, LlrFormat::F16, 1.f, llr_stride, nullptr, bits, packed, ref_bits, counters,
                      workspace, workspace_bytes, stream);
}

int b200dvb_decode_i8(b200dvb_codec_t codec, int B, const void *llr, long long llr_stride, float scale,
                      int32_t *bits, uint32_t *packed, const uint8_t *ref_bits,
                      unsigned long long *counters, void *workspace, size_t workspace_bytes,
                      void *stream)
{
    if (!isfinite(scale) || scale == 0.f) return B200DVB_EINVAL;
    return decode_any(codec, B, llr, LlrFormat::I8, scale, llr_stride, nullptr, bits, packed, ref_bits, counters,
                      workspace, workspace_bytes, stream);
}

int b200dvb_decode_app(b200dvb_codec_t codec, int B, const void *llr, int llr_format, float llr_scale,
                       long long llr_stride, float *app, int32_t *bits, uint32_t *packed,
                       const uint8_t *ref_bits, unsigned long long *counters,
                       void *workspace, size_t workspace_bytes, void *stream)
{
    if (!app || (reinterpret_cast<uintptr_t>(app) & 7)) return B200DVB_EINVAL;   // one float2 store per couple
    LlrFormat fmt;
    switch (llr_format) {
    case B200DVB_LLR_F32: fmt = LlrFormat::F32; llr_scale = 1.f; break;
    case B200DVB_LLR_F16:
        if (reinterpret_cast<uintptr_t>(llr) & 1) return B200DVB_EINVAL;
        fmt = LlrFormat::F16; llr_scale = 1.f;
        break;
    case B200DVB_LLR_I8:
        if (!isfinite(llr_scale) || llr_scale == 0.f) return B200DVB_EINVAL;
        fmt = LlrFormat::I8;
        break;
    default: return B200DVB_EINVAL;
    }
    return decode_any(codec, B, llr, fmt, llr_scale, llr_stride, app, bits, packed, ref_bits, counters, workspace,
                      workspace_bytes, stream);
}

int b200dvb_encode(b200dvb_codec_t codec, int B, const uint8_t *info, uint8_t *coded,
                   uint8_t *circ, void *stream)
{
    if (!codec || B < 0 || !info || !coded) return B200DVB_EINVAL;
    return launch_encode(codec->c, B, info, coded, circ, (cudaStream_t)stream);
}

int b200dvb_mc_generate_bpsk(b200dvb_codec_t codec, int B, float noise_var,
                             unsigned long long seed, unsigned long long frame_offset,
                             uint8_t *info_out, uint8_t *coded_out, float *llr_out, void *stream)
{
    if (!codec || B < 0 || !info_out || !coded_out || !llr_out || !(noise_var > 0.f))
        return B200DVB_EINVAL;
    // the Philox counters advance in whole draws (16 info bits, 4 LLRs): a shard may only start on a draw boundary,
    // otherwise its streams would overlap the neighbouring shard's (montecarlo.ALIGN = 16 frames always satisfies this)
    if ((frame_offset * (unsigned long long)(2 * codec->c.N)) % 16ull != 0 ||
        (frame_offset * (unsigned long long)codec->c.n_llr) % 4ull != 0)
        return B200DVB_EINVAL;
    return launch_mc_bpsk(codec->c, B, noise_var, seed, frame_offset, info_out, coded_out, llr_out,
                          (cudaStream_t)stream);
}

int b200dvb_awgn_complex(size_t n_sym, float sigma, unsigned long long seed,
                         unsigned long long offset, void *iq, void *stream)
{
    if (!iq || !(sigma >= 0.f)) return B200DVB_EINVAL;
    return launch_awgn_complex(n_sym, sigma, seed, offset, iq, (cudaStream_t)stream);
}

int b200dvb_fading_complex(size_t n_sym, int block_len, float sigma, unsigned long long seed,
                           unsigned long long offset, void *iq, void *gain, void *stream)
{
    if (!iq || !(sigma >= 0.f) || block_len < 1 || (offset & 1ull)) return B200DVB_EINVAL;
    return launch_fading_complex(n_sym, block_len, sigma, seed, offset, iq, gain, (cudaStream_t)stream);
}

int b200dvb_pulse_shape(size_t n_sym, const void *sym, const double *taps_h, int ntaps, int sps, void *out, void *stream)
{
    if (!sym || !taps_h || !out || ntaps < 1 || ntaps > kMaxFirTaps || sps < 1 || sps > 64) return B200DVB_EINVAL;
    return launch_pulse_shape(n_sym, sym, taps_h, ntaps, sps, out, (cudaStream_t)stream);
}

int b200dvb_matched_filter(size_t n, const void *samples, const double *taps_h, int ntaps, int sps, long long start,
                           size_t n_out, void *out, void *stream)
{
    if (!samples || !taps_h || (!out && n_out) || ntaps < 1 || ntaps > kMaxFirTaps || sps < 1 || sps > 64 || start < 0)
        return B200DVB_EINVAL;
    return launch_matched_filter(n, samples, taps_h, ntaps, sps, start, n_out, out, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------
static const int kBps[6] = {1, 2, 3, 4, 6, 8};

int b200dvb_modem_create(int mod_id, const double *table_h, b200dvb_modem_t *out)
{
    if (!out || !table_h) return B200DVB_EINVAL;
    if (mod_id < 0 || mod_id > 5) return B200DVB_EMOD;
    b200dvb_modem *h = new (std::nothrow) b200dvb_modem();
    if (!h) return B200DVB_ENOMEM;
    Modem &m = h->m;
    m.mod_id = mod_id; m.bps = kBps[mod_id]; m.M = 1 << m.bps;
    memcpy(m.h_table, table_h, sizeof(double) * 2 * m.M);
    // separable square QAM?  label = (I-axis label | Q-axis label), either half first
    m.separable = 0;
    if ((m.bps % 2) == 0 && m.bps >= 2) {
        const int half = m.bps / 2, Lv = 1 << half;
        bool hi_is_I = true, hi_is_Q = true;
        for (int hi = 0; hi < Lv; ++hi)
            for (int lo = 0; lo < Lv; ++lo) {
                const double re = table_h[2 * (hi * Lv + lo)], im = table_h[2 * (hi * Lv + lo) + 1];
                if (re != table_h[2 * (hi * Lv)] || im != table_h[2 * lo + 1]) hi_is_I = false;
                if (im != table_h[2 * (hi * Lv) + 1] || re != table_h[2 * lo]) hi_is_Q = false;
            }
        if (hi_is_I) m.separable = 1;        // first half of the label selects I (SDRModem)
        else if (hi_is_Q) m.separable = 2;   // first half selects Q (Modulator meshgrid order)
        m.nlev = Lv; m.half = half;
    }
    float t32[512];
    for (int i = 0; i < 2 * m.M; ++i) t32[i] = (float)table_h[i];
    cudaError_t e = cudaMalloc(&m.d_table64, sizeof(double) * 2 * m.M);
    if (e == cudaSuccess) e = cudaMalloc(&m.d_table32, sizeof(float) * 2 * m.M);
    if (e == cudaSuccess) e = cudaMemcpy(m.d_table64, table_h, sizeof(double) * 2 * m.M, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(m.d_table32, t32, sizeof(float) * 2 * m.M, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        set_cuda_error(e, "modem_create");
        if (m.d_table64) cudaFree(m.d_table64);
        if (m.d_table32) cudaFree(m.d_table32);
        delete h;
        return B200DVB_ECUDA;
    }
    if (m.separable) {
        int rc = modem_build_pwl(m);
        if (rc != B200DVB_OK) { cudaFree(m.d_table64); cudaFree(m.d_table32); delete h; return rc; }
    }
    *out = h;
    return B200DVB_OK;
}

int b200dvb_modem_destroy(b200dvb_modem_t modem)
{
    if (!modem) return B200DVB_EINVAL;
    if (modem->m.d_table64) cudaFree(modem->m.d_table64);
    if (modem->m.d_table32) cudaFree(modem->m.d_table32);
    if (modem->m.d_pwl) cudaFree(modem->m.d_pwl);
    delete modem;
    return B200DVB_OK;
}

int b200dvb_map(b200dvb_modem_t modem, size_t n_sym, const uint8_t *bits, void *iq, int out_f64,
                void *stream)
{
    if (!modem || !bits || !iq) return B200DVB_EINVAL;
    return launch_map(modem->m, n_sym, bits, iq, out_f64, (cudaStream_t)stream);
}

int b200dvb_demap(b200dvb_modem_t modem, size_t n_sym, const void *iq, float noise_var,
                  float scale, float *llr, void *stream)
{
    if (!modem || !iq || !llr) return B200DVB_EINVAL;
    return launch_demap(modem->m, n_sym, iq, noise_var, scale, llr, (cudaStream_t)stream);
}

int b200dvb_demap_bf16(b200dvb_modem_t modem, size_t n_sym, const void *iq_bf16x2, float noise_var,
                       float scale, float *llr, void *stream)
{
    if (!modem || !iq_bf16x2 || !llr) return B200DVB_EINVAL;
    return launch_demap_bf16(modem->m, n_sym, iq_bf16x2, noise_var, scale, llr, (cudaStream_t)stream);
}

int b200dvb_demap_csi(b200dvb_modem_t modem, size_t n_sym, const void *iq, const void *gain, float noise_var,
                      float scale, float *llr, void *stream)
{
    if (!modem || !iq || !gain || !llr) return B200DVB_EINVAL;
    return launch_demap_csi(modem->m, n_sym, iq, gain, noise_var, scale, llr, (cudaStream_t)stream);
}

int b200dvb_hard_demod(b200dvb_modem_t modem, size_t n_sym, const void *iq, int in_f64,
                       uint8_t *bits, void *stream)
{
    if (!modem || !iq || !bits) return B200DVB_EINVAL;
    return launch_hard(modem->m, n_sym, iq, in_f64, bits, (cudaStream_t)stream);
}

int b200dvb_debug_phase_cycles(double *out8_h, int reset)
{
    if (!out8_h) return B200DVB_EINVAL;
    return quad_read_phase_cycles(out8_h, reset);
}

int b200dvb_debug_tpf_cycles(double *out8_h, int reset)
{
    if (!out8_h) return B200DVB_EINVAL;
    return tpf_read_phase_cycles(out8_h, reset);
}

int b200dvb_debug_nii_cycles(double *out8_h, int reset)
{
    if (!out8_h) return B200DVB_EINVAL;
    return nii_read_phase_cycles(out8_h, reset);
}

int b200dvb_debug_lat_cycles(double *out8_h, int reset)
{
    if (!out8_h) return B200DVB_EINVAL;
    return lat_read_phase_cycles(out8_h, reset);
}

int b200dvb_debug_set_option(int option, int value)
{
    switch (option) {
    case B200DVB_DBG_MF_VARIANT:
        if (value < 0 || value > 2) return B200DVB_EINVAL;
        set_mf_variant(value);
        return B200DVB_OK;
    case B200DVB_DBG_LAT_WARM:
        if (value < 0 || value > 1024) return B200DVB_EINVAL;
        set_lat_warm(value);
        return B200DVB_OK;
    case B200DVB_DBG_MAP_VARIANT:
        if (value < 0 || value > 2) return B200DVB_EINVAL;
        set_map_variant(value);
        return B200DVB_OK;
    default: return B200DVB_EINVAL;
    }
}

int b200dvb_tmem_selftest(int *errors_h)
{
    if (!errors_h) return B200DVB_EINVAL;
    return run_tmem_selftest(errors_h);
}

int b200dvb_microbench(double *results_h)
{
    if (!results_h) return B200DVB_EINVAL;
    return run_microbench(results_h);
}

int b200dvb_microbench2(double *results16_h)
{
    if (!results16_h) return B200DVB_EINVAL;
    return run_microbench2(results16_h);
}

}  // extern "C"
