/*
 * b200dvb.h — C ABI of libb200dvb.so: the B200 (sm_100a) implementation of the
 * baseband decode hot path of poriya219/modulations.
 *
 * The reference has no FFI of its own (it is pure Python + numba); the boundary
 * is the set of Python callables listed in SURVEY.md §8(b).  Each entry point
 * below names the reference callable(s) it sits under (file:line in the
 * reference tree).  modulations_b200/ binds these with ctypes; INTEGRATION.md
 * shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer unless its name ends in _h (host).
 *  - All work is enqueued on `stream` (a cudaStream_t passed as void*; NULL =
 *    the legacy default stream).  No entry point synchronises the device.
 *  - The caller owns every buffer, including the workspaces whose sizes the
 *    *_workspace_bytes queries return.
 *  - Return value: 0 on success, a negative B200DVB_E* code otherwise.
 *    b200dvb_error_string() maps codes to text; B200DVB_ECUDA keeps the CUDA
 *    error retrievable with b200dvb_last_cuda_error().
 *  - There is no CPU fallback: without a CUDA device every compute entry point
 *    returns B200DVB_ECUDA.
 */
#ifndef B200DVB_H
#define B200DVB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200DVB_OK        0
#define B200DVB_EINVAL   -1   /* bad argument (NULL pointer, negative size, ...)            */
#define B200DVB_ENOSPEC  -2   /* tables/sizes this build has no kernel specialisation for   */
#define B200DVB_ECUDA    -3   /* a CUDA runtime call or launch failed                       */
#define B200DVB_ENOMEM   -4   /* workspace too small / allocation failed                    */
#define B200DVB_EMOD     -5   /* unknown modulation id  (reference: ValueError)             */

/* modulation ids: SDRModem.MODULATIONS, sdr_modem.py:29-36 */
#define B200DVB_BPSK    0
#define B200DVB_QPSK    1
#define B200DVB_8PSK    2
#define B200DVB_16QAM   3
#define B200DVB_64QAM   4
#define B200DVB_256QAM  5

int         b200dvb_version(void);
const char *b200dvb_error_string(int code);
const char *b200dvb_last_cuda_error(void);
int         b200dvb_device_count(void);

/* ------------------------------------------------------------------------
 * Turbo codec handle.  Replaces DVBRCS2_Turbo.__init__ (dvb_rcs2_turbo.py:
 * 287-309): the host computes the tables exactly as the reference does
 * (_init_interleaver :311-325, _init_trellis :327-396, PUNCTURE_PATTERNS :21-26)
 * and hands them over as opaque data — perm / inv_perm are NOT assumed to be
 * permutations (SURVEY §0 F2).
 *   next_state_h, out_W_h, out_Y_h : int32[16*4]   (:333-370)
 *   perm_h, inv_perm_h             : int32[N]      (:314-325)
 *   punct_h                        : uint8[4*period], rows W1,Y1,W2,Y2 (:21-26)
 *   sf_inner / sf_last             : extrinsic scaling 0.7 / 1.0 (:496)
 * Returns B200DVB_ENOSPEC if the trellis is not the 16-state butterfly the
 * kernels are specialised for, or if N is not a multiple of 4 in [12, 2048].
 * ---------------------------------------------------------------------- */
typedef struct b200dvb_codec *b200dvb_codec_t;

int b200dvb_codec_create(int N, const int32_t *next_state_h, const int32_t *out_W_h,
                         const int32_t *out_Y_h, const int32_t *perm_h,
                         const int32_t *inv_perm_h, const uint8_t *punct_h, int period,
                         int iterations, double sf_inner, double sf_last,
                         b200dvb_codec_t *out);
int b200dvb_codec_destroy(b200dvb_codec_t codec);
/* LLRs the depuncturer consumes per frame (= bits the encoder emits; differs
 * from the reference's n_coded when N % period != 0, dvb_rcs2_turbo.py:398-402) */
int b200dvb_codec_n_llr(b200dvb_codec_t codec);
/* Frames the decode kernel keeps resident at a time on this device (one "wave": SMs x frames per SM).
 * Batches and pipeline chunks that are multiples of it leave no SM idle in the last wave. */
int b200dvb_codec_frames_per_wave(b200dvb_codec_t codec);

/* Development / test switches of one codec handle (production code never needs them):
 *   B200DVB_OPT_KERNEL          0 = automatic (per batch size), 1 = quad kernel, 2 = thread-per-frame kernel,
 *                               3 = low-latency kernel (one CTA per frame; parity mode only)
 *                               (B200DVB_ENOSPEC when the codec's N has no geometry for the kernel asked for)
 *   B200DVB_OPT_NO_ROW_STAGING  1 = thread-per-frame transposition without the cp.async row staging
 *   B200DVB_OPT_PHASE_TIMERS    1 = launches add per-phase SM cycles to the b200dvb_debug_*_cycles counters */
#define B200DVB_OPT_KERNEL          1
#define B200DVB_OPT_NO_ROW_STAGING  2
#define B200DVB_OPT_PHASE_TIMERS    3
/* Decoder arithmetic of b200dvb_decode (NOT a development switch: an explicit, labelled choice of the caller):
 *   B200DVB_MODE_PARITY (default)  the reference's double-pass max-log-MAP, bit-exact with
 *                                  dvb_rcs2_turbo.py:116-281 / :464-537;
 *   B200DVB_MODE_NII               NON-PARITY: one pass per SISO, the circular boundary initialised from the
 *                                  previous iteration's metrics of the same constituent decoder, float32
 *                                  extrinsics, re-associated a-posteriori maxima (csrc/nii_core.cuh; SURVEY 8(f) N2,
 *                                  north_star "next-iteration circular-state initialisation").  Results differ from
 *                                  the reference's in isolated bits and are judged on BER/FER; B200DVB_ENOSPEC when N
 *                                  has no thread-per-frame geometry (N > 212).  b200dvb_siso is always parity. */
#define B200DVB_OPT_DECODER_MODE    4
#define B200DVB_MODE_PARITY         0
#define B200DVB_MODE_NII            1
/*   B200DVB_MODE_NII16             NON-PARITY: the nii decoder in 16-bit fixed point, two frames per 32-bit register,
 *                                  add-compare-select as one DPX instruction (VIADDMNMX.S16x2) per branch pair
 *                                  (csrc/nii16_core.cuh states the format: LLRs in 1/4 units clamped to +-31.75,
 *                                  extrinsics to +-63.75, scaling factors in Q6); checked bit for bit against
 *                                  oracle/nii16_model.c */
#define B200DVB_MODE_NII16          2
int b200dvb_codec_set_option(b200dvb_codec_t codec, int option, int value);

/* One SISO half-iteration for B independent frames.  Replaces bcjr_max_log_map
 * (dvb_rcs2_turbo.py:116-281; historic aliases bcjr_decode_circular /
 * max_log_map_decode).  Lc_* float32[B*N], La_* float64[B*N] (NULL = zeros),
 * Le_* float64[B*N].  Bit-exact with the reference's mixed fp64/fp32 arithmetic. */
size_t b200dvb_siso_workspace_bytes(b200dvb_codec_t codec, int B);
int b200dvb_siso(b200dvb_codec_t codec, int B, const float *Lc_A, const float *Lc_B,
                 const float *Lc_W, const float *Lc_Y, const double *La_A, const double *La_B,
                 double scaling_factor, double *Le_A, double *Le_B, void *workspace,
                 size_t workspace_bytes, void *stream);

/* Full decode of B frames: depuncture -> iterations x (SISO1, interleave, SISO2,
 * de-interleave) -> hard decision.  Replaces DVBRCS2_Turbo.decode
 * (dvb_rcs2_turbo.py:464-537).
 *   llr       float32[B][llr_stride], the first n_llr of each row are used
 *   bits      int32[B][2N]  (reference layout :532-535) or NULL
 *   packed    uint32[B][ceil(2N/32)], bit i of the frame at word i/32, bit i%32, or NULL
 *   ref_bits  uint8[B][2N] transmitted info bits for error counting, or NULL
 *   counters  uint64[4] += {bit errors, frame errors, frames, info bits}, or NULL
 *             (accumulated with atomicAdd; this is what the multi-GPU harness
 *             all-reduces) */
size_t b200dvb_decode_workspace_bytes(b200dvb_codec_t codec, int B);
int b200dvb_decode(b200dvb_codec_t codec, int B, const float *llr, long long llr_stride,
                   int32_t *bits, uint32_t *packed, const uint8_t *ref_bits,
                   unsigned long long *counters, void *workspace, size_t workspace_bytes,
                   void *stream);
/* b200dvb_decode with IEEE binary16 channel LLRs: llr = uint16 bit patterns [B][llr_stride] (elements), 2-byte aligned.
 * Every value is widened exactly to float32 and decoded as b200dvb_decode decodes it: for the same codec, options and
 * batch, the outputs (bits, packed, counters) equal b200dvb_decode's on the float32 widening, bit for bit, in every
 * decoder mode and for every kernel choice.  NaN / Inf inputs are undefined, as for float32.  Half the input bytes of
 * b200dvb_decode; the workspace is the same (b200dvb_decode_workspace_bytes). */
int b200dvb_decode_f16(b200dvb_codec_t codec, int B, const void *llr, long long llr_stride,
                       int32_t *bits, uint32_t *packed, const uint8_t *ref_bits,
                       unsigned long long *counters, void *workspace, size_t workspace_bytes, void *stream);
/* b200dvb_decode with 8-bit channel LLRs and a scale: llr = int8 [B][llr_stride] (elements = bytes), any alignment.
 * Element q (-128 ... 127) is decoded as the float32 value q * scale, rounded as IEEE float32 multiplication rounds it
 * (no FTZ, no fused multiply-add): for the same codec, options and batch, the outputs (bits, packed, counters) equal
 * b200dvb_decode's on the float32 array float32(q) * scale, bit for bit, in every decoder mode and for every kernel
 * choice.  scale must be finite and non-zero (else B200DVB_EINVAL); a negative scale flips the sign convention.
 * In B200DVB_MODE_NII16 (LLRs in 1/4 units), int8 q = clamp(rint(4 x), -127, 127) with scale 0.25 decodes exactly as
 * float32 x does: the mode's own quantisation of x is that q.  A quarter of the input bytes of b200dvb_decode; the
 * workspace is the same (b200dvb_decode_workspace_bytes). */
int b200dvb_decode_i8(b200dvb_codec_t codec, int B, const void *llr, long long llr_stride, float scale,
                      int32_t *bits, uint32_t *packed, const uint8_t *ref_bits,
                      unsigned long long *counters, void *workspace, size_t workspace_bytes, void *stream);
/* Soft-output decode: b200dvb_decode / _f16 / _i8 (llr_format B200DVB_LLR_F32 / _F16 / _I8, with the same argument rules:
 * F16 needs a 2-byte-aligned llr, I8 a finite non-zero llr_scale; llr_scale is ignored for F32 and F16) that also
 * writes the a-posteriori LLR of every info bit after the last iteration:
 *   app  float32[B][2N], required, 8-byte aligned (else B200DVB_EINVAL): app[f][2k] is bit A of couple k, app[f][2k+1]
 *        bit B, the layout of `bits`.  Positive means bit 0, the convention of the input LLRs.
 * The value is the one whose sign the hard decision takes (LA = (Lc + La) + Le1 of the final iteration):
 *   B200DVB_MODE_PARITY (every kernel)  (float)LA, LA the float64 sum, rounded to nearest: float32 of the oracle's
 *                                       Lfinal (dvb_rcs2_turbo.py:529-535), bit for bit
 *   B200DVB_MODE_NII                    the float32 sum LA itself, bit for bit
 *   B200DVB_MODE_NII16                  the int16 sum in 1/4-LLR units times 0.25f (exact: |LA| <= 637 units)
 * bits, packed, ref_bits and counters are optional and hold exactly what b200dvb_decode / _f16 / _i8 give for the same
 * input: the hard decisions are not derived from app.  fp16 and int8 input give the app of their float32 widening.
 * The kernel choice and the workspace (b200dvb_decode_workspace_bytes) are those of b200dvb_decode. */
#define B200DVB_LLR_F32 0
#define B200DVB_LLR_F16 1
#define B200DVB_LLR_I8  2
int b200dvb_decode_app(b200dvb_codec_t codec, int B, const void *llr, int llr_format, float llr_scale,
                       long long llr_stride, float *app, int32_t *bits, uint32_t *packed,
                       const uint8_t *ref_bits, unsigned long long *counters,
                       void *workspace, size_t workspace_bytes, void *stream);

/* Tail-biting encoder for B frames.  Replaces DVBRCS2_Turbo.encode
 * (dvb_rcs2_turbo.py:431-462) including _encode_component (:404-429) and the
 * GF(2) circular-state solve mat_pow_gf2 / solve_circular_state_gf2 (:50-114).
 *   info  uint8[B][2N] -> coded uint8[B][n_llr];  circ (nullable) uint8[B][2]
 *   receives the two circular start states. */
int b200dvb_encode(b200dvb_codec_t codec, int B, const uint8_t *info, uint8_t *coded,
                   uint8_t *circ, void *stream);
/* Sc = (I + G^N)^-1 Z for every Z in 0..15: the bit-packed GF(2) solve as a
 * host-visible table (solve_circular_state_gf2, dvb_rcs2_turbo.py:63-114). */
int b200dvb_codec_circular_lut(b200dvb_codec_t codec, int32_t *lut16_h);

/* ------------------------------------------------------------------------
 * Mapper / slicer / soft demapper.  `table` = constellation indexed by the
 * MSB-first bit label: double[2*M] (re,im) on the HOST, as produced by the
 * reference mapper on all labels (test_sdr_with_coding.py:207-208).
 * ---------------------------------------------------------------------- */
typedef struct b200dvb_modem *b200dvb_modem_t;
int b200dvb_modem_create(int mod_id, const double *table_h, b200dvb_modem_t *out);
int b200dvb_modem_destroy(b200dvb_modem_t modem);

/* bits uint8[n_sym*bps] (caller zero-pads, sdr_modem.py:122-124) -> symbols.
 * Replaces SDRModem.modulate (sdr_modem.py:222-243).  out_f64 = 0: float2
 * (complex64), 1: double2 (complex128, the dtype the reference returns for QPSK). */
int b200dvb_map(b200dvb_modem_t modem, size_t n_sym, const uint8_t *bits, void *iq,
                int out_f64, void *stream);
/* Max-log bit LLRs, clipped to +-30, positive = bit 1.  Replaces compute_llr
 * (test_sdr_with_coding.py:200-225).  iq float2[n_sym] -> llr float32[n_sym*bps];
 * noise_var is floored at 0.005 (:202); iq and llr must be 16-byte aligned.  `scale` multiplies the clipped LLR
 * (use -1 to feed the decoder, whose convention is positive = bit 0). */
int b200dvb_demap(b200dvb_modem_t modem, size_t n_sym, const void *iq, float noise_var,
                  float scale, float *llr, void *stream);
/* The same with bf16x2 symbols (4 bytes per symbol: bf16 I, then bf16 Q; BASELINE north_star "bf16x2 loads of I/Q"):
 * each component is widened exactly to float32 and goes through the arithmetic of b200dvb_demap, so
 * b200dvb_demap_bf16(x) == b200dvb_demap(float32(x)) bit for bit.  Reported separately in the bench line
 * (4 + 4 bps algorithmic bytes per symbol instead of 8 + 4 bps). */
int b200dvb_demap_bf16(b200dvb_modem_t modem, size_t n_sym, const void *iq_bf16x2, float noise_var,
                       float scale, float *llr, void *stream);
/* Max-log LLRs with perfect channel state: symbol i was received as y = h*c + noise with a known complex gain h.
 *   llr[i*bps+b] = clip((min_{c: b=0} |y - h c|^2 - min_{c: b=1} |y - h c|^2) / max(noise_var, 0.005), +-30) * scale
 * with the sign convention, floor, clip and scale of b200dvb_demap.  iq, gain float2[n_sym] and llr float32[n_sym*bps],
 * all 16-byte aligned; gain is required (else B200DVB_EINVAL).  Computed as the arithmetic of b200dvb_demap on the
 * equalised symbol z = y conj(h) / |h|^2 with 1/noise_var scaled by |h|^2, so a symbol with h = 1 gets exactly the
 * LLRs b200dvb_demap gives it (z is formed in float64, then rounded to float32).  h = 0 gives 0, and every finite y
 * and h give a finite LLR. */
int b200dvb_demap_csi(b200dvb_modem_t modem, size_t n_sym, const void *iq, const void *gain, float noise_var,
                      float scale, float *llr, void *stream);
/* Hard decisions.  Replaces SDRModem.demodulate (sdr_modem.py:245-266) and
 * Modulator._demod_qam_generic (modulators.py:165-171): nearest constellation
 * point, evaluated in float64.  in_f64 selects float2 / double2 input. */
int b200dvb_hard_demod(b200dvb_modem_t modem, size_t n_sym, const void *iq, int in_f64,
                       uint8_t *bits, void *stream);

/* ------------------------------------------------------------------------
 * Monte-Carlo source (harness shape of turbo_test_suite.py:121-199, test.py:
 * 34-103): Philox-seeded info bits, encode, BPSK/QPSK/.. map, AWGN, LLR — all on
 * device, written straight into the decoder's input layout.
 *   info_out uint8[B][2N]; coded_out uint8[B][n_llr]; llr_out float32[B][n_llr]
 *   (contiguous rows).  BPSK: llr = 2y/sigma^2 clipped to +-50
 *   (turbo_test_suite.py:158-161).  The streams are keyed by the GLOBAL frame index frame_offset + i;
 *   frame_offset must start on a whole Philox draw: frame_offset*2N a multiple of 16 and
 *   frame_offset*n_llr a multiple of 4 (any multiple of 16 frames), else B200DVB_EINVAL. */
int b200dvb_mc_generate_bpsk(b200dvb_codec_t codec, int B, float noise_var,
                             unsigned long long seed, unsigned long long frame_offset,
                             uint8_t *info_out, uint8_t *coded_out, float *llr_out,
                             void *stream);

/* Complex AWGN channel, in place: iq[i] += sigma*(n_re + j*n_im), Philox-keyed by
 * (seed, offset + i) so a sharded run draws the same noise as a single-GPU run
 * (channel model of test.py:66-68).  iq float2[n_sym]; offset must be even. */
int b200dvb_awgn_complex(size_t n_sym, float sigma, unsigned long long seed,
                         unsigned long long offset, void *iq, void *stream);
/* Rayleigh block-fading channel with AWGN, in place: iq[i] = h[b]*iq[i] + sigma*(n_re + j*n_im), b = (offset + i) /
 * block_len.  h[b] ~ CN(0, 1) (each component N(0, 1/2), E|h|^2 = 1) depends on (seed, b) only; block_len = 1 is fast
 * fading, and a block may straddle calls and frames.  The noise is keyed exactly as in b200dvb_awgn_complex: with iq
 * all zeros both write the same bits.  gain (nullable) float2[n_sym] receives the h applied to each symbol.
 * B200DVB_EINVAL for a NULL iq, sigma < 0 or NaN, block_len < 1 or an odd offset. */
int b200dvb_fading_complex(size_t n_sym, int block_len, float sigma, unsigned long long seed,
                           unsigned long long offset, void *iq, void *gain, void *stream);

/* Waveform stage next to the mapper / demapper (SURVEY 8(f) N4; float32 FMAs; taps_h = HOST float64[ntaps], the
 * reference's rrc_filter array, ntaps <= 448: they travel in the kernel's parameter space).
 * Pulse shaping = scipy.signal.upfirdn(taps, sym, up=sps) as modulators.py:85-100 calls it:
 *   out[i] = sum_k sym[k] * taps[i - k*sps],  out float2[(n_sym-1)*sps + ntaps]. */
int b200dvb_pulse_shape(size_t n_sym, const void *sym, const double *taps_h, int ntaps, int sps,
                        void *out, void *stream);
/* Matched filter + decimation = convolve(samples, taps, 'full')[start::sps] (modulators.py:102-117 with
 * start = 2*filter_delay; sdr_modem.py:558 is the same FIR):
 *   out[m] = sum_t taps[t] * samples[start + m*sps - t]  (samples outside [0, n) read as 0),  out float2[n_out]. */
int b200dvb_matched_filter(size_t n, const void *samples, const double *taps_h, int ntaps, int sps,
                           long long start, size_t n_out, void *out, void *stream);

/* Diagnostics: SM cycles the decoder CTAs spent per phase since the last reset, summed
 * over CTAs (synchronises the device).  out8_h: double[8] = {prep, recursion-in,
 * recursion-out + extrinsic, epilogue, hard decision, CTA total, 0, 0}. */
int b200dvb_debug_phase_cycles(double *out8_h, int reset);
/* Same for the thread-per-frame kernel (summed over warps): {transpose-in, pass 1 first half
 * incl. prep, pass 1 second half, pass 2 to the crossing, out-phase windows in shared memory,
 * out-phase windows in tensor memory, hard decision, warp total}.  Only launches of a codec with
 * B200DVB_OPT_PHASE_TIMERS set run the instance of the kernel that keeps these counters (the
 * production instance has no clock reads); tools/tpf_perf.py shows the use. */
int b200dvb_debug_tpf_cycles(double *out8_h, int reset);

/* Same for the non-parity "nii" kernel: {transpose-in, "in" pass incl. prep, boundary metrics + crossing, 0,
 * out-phase windows in shared memory, out-phase windows in tensor memory, hard decision, warp total}. */
int b200dvb_debug_nii_cycles(double *out8_h, int reset);

/* Same for the low-latency kernel (cycles of thread 0 of each CTA): {tables + de-puncture, P0 record build, P1 the two
 * recursions, P2 a-posteriori maxima + extrinsic, hard decision, CTA total, 0, 0}. */
int b200dvb_debug_lat_cycles(double *out8_h, int reset);

/* Process-wide development switches (never needed in production).
 *   B200DVB_DBG_MF_VARIANT  matched-filter kernel: 0 = default, 1 = double-buffered cp.async staging, 2 = round-1 kernel
 *   B200DVB_DBG_MAP_VARIANT complex64 mapper: 0 = per-order choice, 1 = one symbol per lane, 2 = four consecutive symbols per lane */
#define B200DVB_DBG_MF_VARIANT 1
#define B200DVB_DBG_MAP_VARIANT 2
#define B200DVB_DBG_LAT_WARM 3     /* low-latency kernel: warm-up steps of a speculative lap-1 segment (0 = default, 40 + N/16 within [48, 96]); any value is exact */
int b200dvb_debug_set_option(int option, int value);

/* Diagnostics: round trip through tensor memory (tcgen05.alloc/st/ld/dealloc) between the
 * two warps of a lane quadrant, as the decoder uses it; *errors_h = mismatching words. */
int b200dvb_tmem_selftest(int *errors_h);

/* Small device-throughput probes used by bench.py to state the ALU roofline
 * (FADD / FMNMX / SHFL lane-ops per clock per SM).  results_h: double[8]. */
int b200dvb_microbench(double *results_h);
/* Packed 16-bit / DPX probes for the non-parity decoder modes (lane-instructions per clock per SM;
 * layout in csrc/microbench.cu).  results16_h: double[16]. */
int b200dvb_microbench2(double *results16_h);

#ifdef __cplusplus
}
#endif
#endif /* B200DVB_H */
