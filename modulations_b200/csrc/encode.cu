// encode.cu — tail-biting duo-binary encoder + on-device Monte-Carlo source.
//
// Reference: DVBRCS2_Turbo.encode / _encode_component (dvb_rcs2_turbo.py:404-462)
// and the GF(2) circular-state solve (dvb_rcs2_turbo.py:50-114).  The solve
// Sc = (I + G^N)^-1 Z is linear over GF(2) in a 4-bit state, so for a given N it
// is a 16-entry nibble table; the host packs it into one 64-bit word
// (api.cu: circular_lut) and the kernel does `lut >> (4*Z) & 15`.
//
// Layout: a block stages `fpb` frames in shared memory (coalesced 16-byte
// copies in and out); one thread walks one frame's trellis four times (zero-state
// pass + circular pass for each constituent encoder).  Rows are padded to an odd
// number of 32-bit words so the 32 walking threads hit 32 different banks.
#include "common.cuh"

namespace b200dvb {

namespace {

__device__ __forceinline__ int trellis_next(int s, int ab)
{   // dk = A^B^s2^s3 ; ns = (s2,s1,s0,dk)   (dvb_rcs2_turbo.py:351,366)
    return ((s & 7) << 1) | (ab ^ ((s >> 2) & 1) ^ ((s >> 3) & 1));
}

__global__ void encode_kernel(int B, int N, int n_llr, int fpb, int in_stride, int out_stride,
                              const int16_t *__restrict__ tab, unsigned long long lut,
                              const uint8_t *__restrict__ info, uint8_t *__restrict__ coded,
                              uint8_t *__restrict__ circ)
{
    extern __shared__ __align__(16) unsigned char sm[];
    unsigned char *s_in = sm;                               // [fpb][in_stride]
    unsigned char *s_out = sm + (size_t)fpb * in_stride;    // [fpb][out_stride]
    int16_t *s_tab = reinterpret_cast<int16_t *>(s_out + (size_t)fpb * out_stride);   // [7][N]: the walkers' tables
    const int f0 = blockIdx.x * fpb;
    const int nf = min(fpb, B - f0);
    const int k2 = 2 * N;
    for (int i = threadIdx.x; i < 7 * N; i += blockDim.x) s_tab[i] = tab[i];
    // stage info bits.  The block's frames are ONE contiguous run of nf * 2N bytes in global memory: it is read with
    // 16-byte loads (several in flight per thread; a byte loop with a division per element spent 55 % of this kernel
    // waiting on one load at a time, profiles/r02_encode_ncu.txt) and scattered into the padded rows byte by byte.
    {
        const uint8_t *g = info + (size_t)f0 * k2;
        const int total = nf * k2;
        const int nv = (reinterpret_cast<uintptr_t>(g) & 15) == 0 ? total / 16 : 0;
        const uint4 *src = reinterpret_cast<const uint4 *>(g);
#pragma unroll 4
        for (int v = threadIdx.x; v < nv; v += blockDim.x) {
            const uint4 d = __ldg(src + v);
            const unsigned w[4] = {d.x, d.y, d.z, d.w};
            int f = (v * 16) / k2, j = v * 16 - f * k2;
            if ((k2 & 3) == 0) {                            // rows are whole words (N is a multiple of 4 everywhere in the table)
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    *reinterpret_cast<unsigned *>(s_in + f * in_stride + j) = w[t] & 0x01010101u;
                    j += 4;
                    if (j == k2) { j = 0; ++f; }
                }
            } else {
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    s_in[f * in_stride + j] = (w[t >> 2] >> (8 * (t & 3))) & 1u;
                    if (++j == k2) { j = 0; ++f; }
                }
            }
        }
        for (int i = nv * 16 + threadIdx.x; i < total; i += blockDim.x) {
            const int f = i / k2, j = i - f * k2;
            s_in[f * in_stride + j] = g[i] & 1;
        }
    }
    __syncthreads();
    // Two walkers per frame, one per constituent encoder (they only share the read-only info row): the walk is a
    // serial chain of shared-memory loads, so the kernel's speed is the number of chains in flight per SM.
    if (threadIdx.x < 2 * nf) {
        const int fr = threadIdx.x >> 1, e = threadIdx.x & 1;
        const unsigned char *in = s_in + fr * in_stride;
        unsigned char *out = s_out + fr * out_stride;
        const int16_t *perm = s_tab, *offA = s_tab + 2 * N;
        const int16_t *oW = s_tab + (3 + 2 * e) * N, *oY = s_tab + (4 + 2 * e) * N;
        int st = 0;                                         // zero-state response (:408-412)
#pragma unroll 4
        for (int i = 0; i < N; ++i) {
            const int j = e ? perm[i] : i;
            st = trellis_next(st, in[2 * j] ^ in[2 * j + 1]);
        }
        st = (int)((lut >> (4 * st)) & 15ull);              // circular start state (:416-417)
        if (circ) circ[(size_t)(f0 + fr) * 2 + e] = (uint8_t)st;
#pragma unroll 4
        for (int i = 0; i < N; ++i) {                       // :423-427
            const int j = e ? perm[i] : i;
            const int a = in[2 * j], b = in[2 * j + 1], ab = a ^ b;
            const int s0 = st & 1, s1 = (st >> 1) & 1, s2 = (st >> 2) & 1;
            if (e == 0) { const int oa = offA[i]; out[oa] = a; out[oa + 1] = b; }
            const int ow = oW[i], oy = oY[i];
            if (ow >= 0) out[ow] = ab ^ s0 ^ s1 ^ s2;       // :355
            if (oy >= 0) out[oy] = ab ^ s1;                 // :359
            st = trellis_next(st, ab);
        }
    }
    __syncthreads();
    {   // the block's code words are one contiguous run of nf * n_llr bytes: gathered 16 at a time, 16-byte stores
        uint8_t *g = coded + (size_t)f0 * n_llr;
        const int total = nf * n_llr;
        const int nv = (reinterpret_cast<uintptr_t>(g) & 15) == 0 ? total / 16 : 0;
        uint4 *dst = reinterpret_cast<uint4 *>(g);
        for (int v = threadIdx.x; v < nv; v += blockDim.x) {
            int f = (v * 16) / n_llr, j = v * 16 - f * n_llr;
            unsigned w[4] = {0u, 0u, 0u, 0u};
            if ((n_llr & 3) == 0) {                         // whole words per row: four 32-bit reads
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    w[t] = *reinterpret_cast<const unsigned *>(s_out + f * out_stride + j);
                    j += 4;
                    if (j == n_llr) { j = 0; ++f; }
                }
            } else {
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    w[t >> 2] |= (unsigned)s_out[f * out_stride + j] << (8 * (t & 3));
                    if (++j == n_llr) { j = 0; ++f; }
                }
            }
            dst[v] = make_uint4(w[0], w[1], w[2], w[3]);
        }
        for (int i = nv * 16 + threadIdx.x; i < total; i += blockDim.x) {
            const int f = i / n_llr, j = i - f * n_llr;
            g[i] = s_out[f * out_stride + j];
        }
    }
}

// Box-Muller pair from two uniforms in (0, 1): hardware approximations (MUFU.LG2 / RSQ / SIN / COS).  The source is
// statistical (Philox, not the reference's MT19937), so a 2^-21 error in a noise sample is immaterial; the library
// versions of logf / sincospif made the AWGN kernels compute-bound at a third of the HBM rate.
__device__ __forceinline__ void box_muller(float u1, float u2, float &n0, float &n1)
{
    const float rad = __fsqrt_rn(-2.0f * __logf(fminf(fmaxf(u1, 1e-12f), 1.0f)));
    float sn, cs;
    __sincosf(6.283185307179586f * u2 - 3.141592653589793f, &sn, &cs);   // argument in (-pi, pi): the fast path's accurate range
    n0 = -rad * cs; n1 = -rad * sn;                                      // cos(x - pi) = -cos x, sin(x - pi) = -sin x
}

// ---- Philox4x32-10 (Salmon et al., SC'11), counter-based ------------------------
struct Philox { unsigned c[4]; };
__device__ __forceinline__ Philox philox(unsigned long long counter, unsigned stream,
                                         unsigned long long seed)
{
    unsigned c0 = (unsigned)counter, c1 = (unsigned)(counter >> 32), c2 = stream, c3 = 0x5eed5eedu;
    unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return Philox{{c0, c1, c2, c3}};
}

__global__ void info_bits_kernel(size_t n16, unsigned long long seed, unsigned long long offset16,
                                 uint4 *__restrict__ out)
{   // 16 info bits (as 16 bytes) per thread
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n16) return;
    const Philox r = philox(offset16 + i, 1u, seed);
    const unsigned v = r.c[0];
    uint4 o;
    o.x = (v & 1u) | ((v >> 1 & 1u) << 8) | ((v >> 2 & 1u) << 16) | ((v >> 3 & 1u) << 24);
    o.y = (v >> 4 & 1u) | ((v >> 5 & 1u) << 8) | ((v >> 6 & 1u) << 16) | ((v >> 7 & 1u) << 24);
    o.z = (v >> 8 & 1u) | ((v >> 9 & 1u) << 8) | ((v >> 10 & 1u) << 16) | ((v >> 11 & 1u) << 24);
    o.w = (v >> 12 & 1u) | ((v >> 13 & 1u) << 8) | ((v >> 14 & 1u) << 16) | ((v >> 15 & 1u) << 24);
    out[i] = o;
}

// BPSK 0 -> +1 over AWGN, llr = 2y/sigma^2 clipped to +-50 (turbo_test_suite.py:147-161).
// Reads coded bytes, writes float LLRs; 4 elements per thread (one Philox call ->
// two Box-Muller pairs).
__global__ void awgn_bpsk_kernel(size_t n4, size_t n, float sigma, float two_over_var,
                                 unsigned long long seed, unsigned long long offset4,
                                 const uint8_t *__restrict__ coded, float *__restrict__ llr)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    const Philox r = philox(offset4 + i, 2u, seed);
    float nrm[4];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const float u1 = ((float)r.c[2 * h] + 0.5f) * 2.3283064365386963e-10f;
        const float u2 = ((float)r.c[2 * h + 1] + 0.5f) * 2.3283064365386963e-10f;
        box_muller(u1, u2, nrm[2 * h], nrm[2 * h + 1]);
    }
    const size_t e = 4 * i;
    if (e + 3 < n) {
        const uchar4 c = *reinterpret_cast<const uchar4 *>(coded + e);
        float4 o;
        o.x = fminf(fmaxf(((1.f - 2.f * c.x) + sigma * nrm[0]) * two_over_var, -50.f), 50.f);
        o.y = fminf(fmaxf(((1.f - 2.f * c.y) + sigma * nrm[1]) * two_over_var, -50.f), 50.f);
        o.z = fminf(fmaxf(((1.f - 2.f * c.z) + sigma * nrm[2]) * two_over_var, -50.f), 50.f);
        o.w = fminf(fmaxf(((1.f - 2.f * c.w) + sigma * nrm[3]) * two_over_var, -50.f), 50.f);
        *reinterpret_cast<float4 *>(llr + e) = o;
    } else {
        for (int t = 0; t < 4 && e + t < n; ++t)
            llr[e + t] = fminf(fmaxf(((1.f - 2.f * coded[e + t]) + sigma * nrm[t]) * two_over_var, -50.f), 50.f);
    }
}

// Complex AWGN added in place: iq[i] += sigma * (n_re + j n_im); 2 symbols per thread.
__global__ void awgn_complex_kernel(size_t n2, size_t n, float sigma, unsigned long long seed,
                                    unsigned long long offset2, float2 *__restrict__ iq)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n2) return;
    const Philox r = philox(offset2 + i, 3u, seed);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const size_t e = 2 * i + h;
        if (e >= n) break;
        const float u1 = ((float)r.c[2 * h] + 0.5f) * 2.3283064365386963e-10f;
        const float u2 = ((float)r.c[2 * h + 1] + 0.5f) * 2.3283064365386963e-10f;
        float g0, g1;
        box_muller(u1, u2, g0, g1);
        float2 v = iq[e];
        v.x += sigma * g0; v.y += sigma * g1;
        iq[e] = v;
    }
}

// Rayleigh block fading h[b] ~ CN(0, 1) of block b = (global symbol index) / block_len: one Philox draw of stream 4
// serves blocks 2d and 2d+1 (a Box-Muller pair each, scaled by sqrt(1/2) so that E|h|^2 = 1).
__device__ __forceinline__ float2 fading_gain(const Philox &r, unsigned long long b)
{
    const bool odd = b & 1ull;
    const float u1 = ((float)(odd ? r.c[2] : r.c[0]) + 0.5f) * 2.3283064365386963e-10f;
    const float u2 = ((float)(odd ? r.c[3] : r.c[1]) + 0.5f) * 2.3283064365386963e-10f;
    float n0, n1;
    box_muller(u1, u2, n0, n1);
    return make_float2(0.70710678118654752f * n0, 0.70710678118654752f * n1);
}

// iq[i] = h[b] iq[i] + sigma (n_re + j n_im) in place, 2 symbols per thread; the noise is awgn_complex_kernel's,
// draw for draw.  gain (nullable) receives the h of every symbol.
__global__ void fading_complex_kernel(size_t n2, size_t n, unsigned long long block_len, float sigma,
                                      unsigned long long seed, unsigned long long offset2, float2 *__restrict__ iq,
                                      float2 *__restrict__ gain)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n2) return;
    const Philox r = philox(offset2 + i, 3u, seed);
    // blocks of the thread's two symbols: b1 is b0 or b0 + 1
    const unsigned long long s0 = 2 * (offset2 + i);
    const unsigned long long b0 = block_len == 1 ? s0 : s0 / block_len;
    const unsigned long long b1 = block_len == 1 ? s0 + 1 : (s0 + 1) / block_len;
    const Philox q0 = philox(b0 >> 1, 4u, seed);
    const float2 h0 = fading_gain(q0, b0);
    const float2 h1 = b1 == b0 ? h0 : fading_gain((b1 >> 1) == (b0 >> 1) ? q0 : philox(b1 >> 1, 4u, seed), b1);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const size_t e = 2 * i + h;
        if (e >= n) break;
        const float u1 = ((float)r.c[2 * h] + 0.5f) * 2.3283064365386963e-10f;
        const float u2 = ((float)r.c[2 * h + 1] + 0.5f) * 2.3283064365386963e-10f;
        float g0, g1;
        box_muller(u1, u2, g0, g1);
        const float2 hb = h ? h1 : h0, v = iq[e];
        // + 0.f turns a faded -0 into +0: a zero input then gives awgn_complex_kernel's output bit for bit
        float2 o = make_float2((hb.x * v.x - hb.y * v.y) + 0.f, (hb.x * v.y + hb.y * v.x) + 0.f);
        o.x += sigma * g0; o.y += sigma * g1;
        iq[e] = o;
        if (gain) gain[e] = hb;
    }
}

int odd_words(int bytes)
{
    int w = (bytes + 3) / 4;
    if ((w & 1) == 0) ++w;
    return w * 4;
}

}  // namespace

int launch_encode(const Codec &c, int B, const uint8_t *info, uint8_t *coded, uint8_t *circ,
                  cudaStream_t s)
{
    if (B == 0) return B200DVB_OK;
    const int in_stride = odd_words(2 * c.N), out_stride = odd_words(c.n_llr);
    int fpb = 32;
    while (fpb > 1 && (size_t)fpb * (in_stride + out_stride) > 96 * 1024) fpb >>= 1;
    const size_t smem = (size_t)fpb * (in_stride + out_stride) + (size_t)7 * c.N * sizeof(int16_t);
    // a per-device attribute: set on every launch (cheap) rather than cached in a process-wide flag
    if (smem > 48 * 1024)
        B2_CUDA(cudaFuncSetAttribute(encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    unsigned long long lut = 0;
    for (int z = 0; z < 16; ++z) lut |= (unsigned long long)(c.circ_lut[z] & 15) << (4 * z);
    const int grid = (B + fpb - 1) / fpb;
    encode_kernel<<<grid, 128, smem, s>>>(B, c.N, c.n_llr, fpb, in_stride, out_stride, c.d_tab, lut,
                                          info, coded, circ);
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

int launch_mc_bpsk(const Codec &c, int B, float noise_var, unsigned long long seed,
                   unsigned long long frame_offset, uint8_t *info, uint8_t *coded, float *llr,
                   cudaStream_t s)
{
    if (B == 0) return B200DVB_OK;
    const size_t nbits = (size_t)B * 2 * c.N;
    if ((nbits % 16) != 0) return B200DVB_ENOSPEC;          // whole 16-bit Philox draws only
    const size_t n16 = nbits / 16;
    const unsigned long long off16 = frame_offset * (unsigned long long)(2 * c.N) / 16ull;
    info_bits_kernel<<<(unsigned)((n16 + 255) / 256), 256, 0, s>>>(n16, seed, off16,
                                                                   reinterpret_cast<uint4 *>(info));
    B2_CUDA(cudaGetLastError());
    int rc = launch_encode(c, B, info, coded, nullptr, s);
    if (rc != B200DVB_OK) return rc;
    const size_t n = (size_t)B * c.n_llr, n4 = (n + 3) / 4;
    awgn_bpsk_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, s>>>(
        n4, n, sqrtf(noise_var), 2.0f / noise_var, seed,
        frame_offset * (unsigned long long)c.n_llr / 4ull, coded, llr);
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

int launch_awgn_complex(size_t n, float sigma, unsigned long long seed, unsigned long long offset,
                        void *iq, cudaStream_t s)
{
    if (n == 0) return B200DVB_OK;
    const size_t n2 = (n + 1) / 2;
    awgn_complex_kernel<<<(unsigned)((n2 + 255) / 256), 256, 0, s>>>(n2, n, sigma, seed, offset / 2,
                                                                    reinterpret_cast<float2 *>(iq));
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

int launch_fading_complex(size_t n, int block_len, float sigma, unsigned long long seed, unsigned long long offset,
                          void *iq, void *gain, cudaStream_t s)
{
    if (n == 0) return B200DVB_OK;
    const size_t n2 = (n + 1) / 2;
    fading_complex_kernel<<<(unsigned)((n2 + 255) / 256), 256, 0, s>>>(
        n2, n, (unsigned long long)block_len, sigma, seed, offset / 2, reinterpret_cast<float2 *>(iq),
        reinterpret_cast<float2 *>(gain));
    B2_CUDA(cudaGetLastError());
    return B200DVB_OK;
}

}  // namespace b200dvb
