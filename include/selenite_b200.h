/* selenite_b200.h — C ABI of the B200-native batched I/Q block-processing library.
 *
 * Drop-in boundary for the sample path of the Selenite Lite firmware (reference tree = /root/reference):
 * the functions of Core/Inc/dsp_if.h:42-51, (a) batched over independent channels with a context handle
 * prepended and the channel index as the slowest axis ([channels][size], `size` in the SAME unit as the
 * firmware function), and (b) as single-channel wrappers with the firmware's exact names and signatures so
 * a dsp_if.h consumer (USB_DEVICE/App/usbd_audio_if.c:179-202, the I2S callbacks dsp_if.c:50-67) links
 * unchanged. Plain pointers and sizes only; no CUDA or torch types appear in any signature (a CUDA stream is
 * passed as an opaque void*).
 *
 * Sample format everywhere: interleaved little-endian int16 I,Q (= L,R) frames, as on the I2S bus
 * (Core/Src/main.c:333-341) and the UAC1 endpoints (USB_DEVICE/Class/usbd_audio.c:329-334).
 *
 * There is no CPU fallback: every entry point that moves samples runs CUDA kernels on the context's device
 * and returns SLB_ERR_CUDA if that fails.
 */
#ifndef SELENITE_B200_H
#define SELENITE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLB_OK               0
#define SLB_ERR_ARG         (-1)   /* bad argument (null pointer, size not a whole number of blocks, ...) */
#define SLB_ERR_CUDA        (-2)   /* CUDA runtime error; text in slb_last_error() */
#define SLB_ERR_STATE       (-3)   /* call not valid in the current state */
#define SLB_ERR_UNSUPPORTED (-4)   /* parameter combination this build has no kernel for */

/* FT-817 mode bytes handed to DSP_Set_Mode (reference: Core/Inc/rxtx_if.h:33-43, call site rxtx_if.c:647) */
#define SLB_MODE_LSB 0x00
#define SLB_MODE_USB 0x01
#define SLB_MODE_CW  0x02
#define SLB_MODE_CWR 0x03
#define SLB_MODE_AM  0x04
#define SLB_MODE_FM  0x08
#define SLB_MODE_DIG 0x0A
#define SLB_MODE_PKT 0x0C

/* What sits between pbuf and the ring store inside DSP_In_Buff_Write (dsp_if.c:286-289) */
#define SLB_CHAIN_PASS        0    /* the firmware as shipped: bit-exact int16 copy */
#define SLB_CHAIN_RX_SSB_F32  1    /* unpack -> FFT overlap-save SSB demod -> biquad cascade -> AGC -> pack */
#define SLB_CHAIN_TX_SSB_F32  2    /* mic (L of L=R) -> FFT overlap-save SSB modulator (band-pass + Hilbert) -> ALC -> I/Q pack */

#define SLB_CHAIN_CHAN64_F32  3    /* wideband stream -> 64-branch polyphase FFT channelizer -> per-bin demod + AGC -> pack */

#define SLB_CHAIN_RX_SSB_Q15  4    /* all-integer phasing SSB demodulator: fir_q15 Hilbert pair -> add/sub -> q15 AGC (bit-exact) */

#define SLB_CHAIN_TX_F32      5    /* all-mode transmit: LSB, USB, CW, CW-R, DIG, PKT exactly as SLB_CHAIN_TX_SSB_F32; AM (carrier +
                                      envelope) and FM (integer-phase NCO) from the same band-limited mic (DESIGN.md §3.4) */

#define SLB_CHAIN_TX_SSB_Q15  6    /* all-integer phasing SSB modulator: mic (L of L=R) -> the fir_q15 Hilbert pair of RX-SSB-q15 -> rail
                                      order by sideband -> q15 ALC -> I/Q pack (bit-exact, DESIGN.md §3.7) */

#define SLB_CHAIN_RX_Q15      7    /* all-mode integer receiver: LSB, USB, CW, CW-R, DIG, PKT exactly as SLB_CHAIN_RX_SSB_Q15;
                                      AM by arm_cmplx_mag_q15, FM by an integer limiter-discriminator (DESIGN.md §3.8); bit-exact */

#define SLB_CHAIN_TX_Q15      8    /* all-mode integer transmitter: LSB, USB, CW, CW-R, DIG, PKT exactly as SLB_CHAIN_TX_SSB_Q15;
                                      AM (carrier + scaled audio) and FM (integer phase, table NCO) (DESIGN.md §3.9); bit-exact */

#define SLB_CHAIN_CHAN64_Q15  9    /* all-integer channelizer, 192 kHz only: 64-branch arm_fir_q15 polyphase bank -> arm_cfft_q15 (64) -> per-bin
                                      product or envelope detector -> q15 AGC -> pack (DESIGN.md §3.10); bit-exact */

#define SLB_MAX_STAGES 4
#define SLB_MAX_MASKS  8

typedef struct slb_ctx slb_ctx;

typedef struct
{
  uint32_t channels;     /* independent I/Q streams handled by this context (this GPU's shard) */
  uint32_t fs;           /* USBD_AUDIO_FREQ: 48000, 96000 or 192000 (usbd_audio.h:46, dsp_if.h:55-57) */
  int32_t  device;       /* CUDA device ordinal */
  uint32_t chain;        /* SLB_CHAIN_* */
} slb_config;

/* RX-SSB-f32 chain parameters (DESIGN.md §3). Oracle stage for each field in brackets. */
typedef struct
{
  uint32_t fft_len;                      /* overlap-save FFT length [arm_cfft_f32]; this build: 512 */
  uint32_t hop;                          /* new frames per FFT frame; this build: 384 (= DSP_BUFF_SIZE at 48 kHz) */
  uint32_t agc_block;                    /* AGC detector block = firmware block, fs/1000 frames; this build: 48 */
  uint32_t n_stages;                     /* audio biquad stages [arm_biquad_cascade_df2T_f32]; this build: 2 */
  float    biquad[5 * SLB_MAX_STAGES];   /* {b0,b1,b2,a1,a2} per stage, CMSIS sign (+a1,+a2 feedback) */
  float    agc_target, agc_decay, agc_floor, agc_gmax;
} slb_rx_f32_params;

/* TX-SSB-f32 chain parameters (DESIGN.md §3): the spectral masks are shared with RX (slb_set_mask). */
typedef struct
{
  uint32_t fft_len;                      /* this build: 512 */
  uint32_t hop;                          /* this build: 384 */
  uint32_t alc_block;                    /* ALC detector block [arm_cmplx_mag_f32 + arm_max_f32] = firmware block; this build: 48 */
  float    alc_target, alc_decay, alc_floor, alc_gmax;
} slb_tx_f32_params;

/* Modulator constants of SLB_CHAIN_TX_F32 (DESIGN.md §3.4). The ALC of slb_tx_f32_params measures max |Re z| per block for AM
 * and FM and holds it at am_depth (AM) or at 2 fm_deviation_hz / fs half-turns per sample (FM); alc_target is the SSB target. */
typedef struct
{
  float am_carrier;                      /* AM: I = am_carrier (1 + g Re z), Q = 0 [arm_offset_f32, arm_scale_f32]; (0, 1) */
  float am_depth;                        /* AM: peak modulation depth the ALC holds, (0, 1]: the envelope stays in carrier (1 +- depth) */
  float fm_deviation_hz;                 /* FM: peak deviation the ALC holds, (0, fs / 4] */
  float fm_level;                        /* FM: I + jQ = fm_level e^(j phi) [arm_cos_f32, arm_sin_f32, arm_scale_f32]; (0, 1) */
} slb_tx_mod_params;

/* CHAN-64-f32 chain parameters (DESIGN.md §3; BASELINE config 4). The context's `channels` are WIDEBAND streams; each
 * yields `bins` narrowband channels at fs/bins. Oracle stage for each field in brackets. */
#define SLB_CHAN_BINS 64
#define SLB_CHAN_TAPS 8
typedef struct
{
  uint32_t bins;                         /* branches = FFT length = decimation [arm_cfft_f32]; this build: 64 */
  uint32_t taps_per_branch;              /* [arm_fir_f32 numTaps per branch]; this build: 8 */
  uint32_t agc_block;                    /* narrowband samples per AGC block = one firmware block (1 ms); this build: 3 */
  uint32_t envelope;                     /* demodulator per bin: 0 = product detector (real part), 1 = envelope [arm_cmplx_mag_f32] */
  float    agc_target, agc_decay, agc_floor, agc_gmax;
  float    proto[SLB_CHAN_BINS * SLB_CHAN_TAPS];   /* prototype low-pass h[n]; branch r uses e_r[p] = h[bins*p + bins-1-r] */
} slb_chan_params;

/* Parameters of the integer chains, RX-SSB-q15 and TX-SSB-q15 (DESIGN.md §3, §3.7): the Hilbert pair and the gain law both directions
 * share. Every stage is an integer CMSIS-DSP routine, results are bit-exact. Oracle stage for each field in brackets. The sideband
 * follows the channel's mode (SLB_DSP_Set_Mode): RX: LSB / CW-R subtract the quadrature rail, every other SSB-style mode adds it;
 * TX: LSB / CW-R emit (I, Q) = (fi, fq), the others (fq, fi). On a TX context the agc_* fields are the ALC (its peak is the larger
 * of max |I| and max |Q| per block), and the chain runs on the tcgen05 kernel only: bq_stages != 0, a tap >= 32640 (one that does not
 * split into two signed bytes) or agc_window > 17 is refused with SLB_ERR_UNSUPPORTED and the parameters stay as they were.
 * Defaults: 48 kHz only. */
#define SLB_Q15_TAPS 64
#define SLB_Q15_WIN  32
typedef struct
{
  uint32_t ntaps;                        /* taps per rail [arm_fir_q15 numTaps, even]; this build: 64 */
  uint32_t agc_block;                    /* AGC detector block [arm_abs_q15 + arm_max_q15] = firmware block; this build: 48 */
  uint32_t agc_window;                   /* blocks of peak history the envelope sees (finite release), 1..SLB_Q15_WIN */
  int16_t  taps_i[SLB_Q15_TAPS];         /* b[0..ntaps-1] of the in-phase rail, q15, natural order */
  int16_t  taps_q[SLB_Q15_TAPS];         /* quadrature rail: same magnitude response, +90 degrees */
  int16_t  rel[SLB_Q15_WIN];             /* q15 release weight of a block peak by age in blocks; rel[0] unused */
  int16_t  agc_target, agc_floor;        /* q15 */
  uint32_t agc_gmax_q15;                 /* gain limit in Q15 (1.0 = 32768) [arm_scale_q15 scaleFract << shift] */
  /* optional audio filter between the mixer and the AGC detector (SURVEY Appendix B) [arm_biquad_cascade_df1_q15.c:62]: bq_stages = 0
   * (default) leaves it out and the chain runs as ONE fused tensor-core kernel; 1..4 stages run the chain as three kernels — fused FIR +
   * mixer, the integer biquad (one thread per channel: it truncates after every sample, so it cannot be evaluated time-parallel exactly),
   * AGC + scale — bit-exact all the same. Coefficients {b0, 0, b1, b2, a1, a2} per stage (arm_biquad_cascade_df1_init_q15). */
  uint32_t bq_stages; int32_t bq_postshift; int16_t bq_coeffs[6 * SLB_MAX_STAGES];
} slb_rx_q15_params;

/* The AM and FM detectors of SLB_CHAIN_RX_Q15 (DESIGN.md §3.8); slb_rx_q15_params keeps the SSB pair and the AGC, which all modes share.
 * Per channel and 48-frame block, a = arm_fir_q15 (I, taps), b = arm_fir_q15 (Q, taps) with the mode's taps on both rails, then
 *   AM: v = arm_cmplx_mag_q15 (a, b) (2.14: about |z| / 2; the carrier's DC stays in the audio)
 *   FM: m_n = arm_cmplx_mag_q15 (a_n, b_n), x_n = a_{n-1} b_n - b_{n-1} a_n (int64),
 *       v_n = sat16 (trunc (x_n 2^13 / max (m_{n-1} m_n, fm_floor))): q15 sin of the phase step, the sign of Im (z[n] conj z[n-1])
 * then the block peak [arm_abs_q15 + arm_max_q15], the gain law of slb_rx_q15_params and arm_scale_q15, written L = R. z[-1] of a call
 * is the current mode's FIR output at the frame before it (zero at a stream start); after a mode change between calls the FIRs and the
 * detector behave as if the channel had always been in the new mode, and the AGC's peak window carries over unchanged.
 * SLB_CHAIN_RX_Q15 runs on the tcgen05 kernel only: a tap >= 32640 here or in slb_rx_q15_params, fm_floor < 1, bq_stages != 0 or
 * agc_window > 17 is refused with SLB_ERR_UNSUPPORTED and the parameters stay as they were; tuning is refused too.
 * Defaults (48 kHz): 64-tap Kaiser (beta 6) low-passes of DC gain 1, -6 dB at 3 kHz (AM) and 6 kHz (FM); fm_floor = 2^18. */
typedef struct
{
  int16_t am_taps[SLB_Q15_TAPS];         /* b[0..63], q15, natural order */
  int16_t fm_taps[SLB_Q15_TAPS];
  int32_t fm_floor;                      /* >= 1; 2^18 = the f32 discriminator's 2^-10 soft squelch in these units */
} slb_rx_q15_mode_params;

/* The AM and FM modulators of SLB_CHAIN_TX_Q15 (DESIGN.md §3.9); slb_rx_q15_params keeps the SSB pair and the ALC constants, which all
 * modes share (agc_target is the SSB modes' target). Per channel and 48-frame block, mic = L of the L = R frames,
 *   a = arm_fir_q15 (mic, taps) -> block peak [arm_abs_q15 + arm_max_q15] -> the gain law of slb_rx_q15_params with the mode's target
 *   -> y = arm_scale_q15 (a, q >> s, s), then
 *   AM (target am_depth): I = arm_add_q15 (arm_scale_q15 (y, am_carrier, 0), am_carrier) (saturating), Q = 0
 *   FM (target fm_target): phi[n] = phi[n-1] + y[n] fm_inc mod 2^32 (a uint32 per channel, carried), (I, Q) = fm_level (cos, sin) of
 *       phi by the table NCO of SLB_CHAIN_TX_F32 (arm_cos_f32 / arm_sin_f32 -> arm_float_to_q15); a positive y moves the carrier up
 * written interleaved I, Q. The phase advances in FM blocks only; a direction switch and SLB_DSP_Init zero it, the checkpoint keeps it.
 * After a mode change between calls the FIR behaves as if the channel had always been in the new mode; the ALC's peak window carries over.
 * SLB_CHAIN_TX_Q15 runs on the tcgen05 kernel only: a tap >= 32640 here or in slb_rx_q15_params, bq_stages != 0, agc_window > 17,
 * am_carrier < 0, am_depth < 1, fm_target < 1 or |fm_inc| > 65535 is refused with SLB_ERR_UNSUPPORTED and the parameters stay as they
 * were; tuning is refused too.
 * Defaults (48 kHz): RX-Q15's AM low-pass (64-tap Kaiser, beta 6, DC gain 1, -6 dB at 3 kHz) for both modes, am_carrier 0.5,
 * am_depth 0.8, fm_target 0.25, fm_inc = llround (2500 2^32 / 48000 / 8192) (2.5 kHz peak deviation), fm_level 0.5. */
typedef struct
{
  int16_t am_taps[SLB_Q15_TAPS];         /* b[0..63], q15, natural order */
  int16_t fm_taps[SLB_Q15_TAPS];
  int16_t am_carrier;                    /* q15, >= 0 */
  int16_t am_depth;                      /* q15, >= 1: the AM ALC target */
  int16_t fm_target;                     /* q15, >= 1: the FM ALC target */
  int32_t fm_inc;                        /* 2^-32 turn per sample per LSB of y, |fm_inc| <= 65535 */
  float fm_level;                        /* NCO amplitude (full scale 1) */
} slb_tx_q15_mode_params;

/* CHAN-64-q15 chain parameters (DESIGN.md §3.10), the integer sibling of slb_chan_params. Per wideband stream and hop of 64 frames:
 *   branch r, rail I and rail Q separately: arm_fir_q15 with the 8 taps e_r[p] = proto[64 p + 63 - r] on the stride-64 commutated input
 *   -> arm_cfft_q15 (64, forward, the Cortex-M4 branch, natural order) of the 64 branch outputs: bin k in 7.9 format (X / 64)
 *   -> per bin: Re (product detector) or arm_cmplx_mag_q15 (envelope, 2.14) by SLB_DSP_Set_Mode (AM: envelope; FM is refused)
 *   -> per block of agc_block narrowband samples: peak [arm_abs_q15 + arm_max_q15], the finite-window gain law of slb_rx_q15_params,
 *      arm_scale_q15 -> int16 L = R in [stream][bin][hop][2], the layout of CHAN-64-f32.
 * Geometry other than 64 / 8 / 3 or agc_window > 17 is refused with SLB_ERR_UNSUPPORTED and the parameters stay as they were.
 * Defaults: CHAN-64-f32's Kaiser (beta 8) prototype scaled to DC gain 32 (llround to q15: no branch can saturate, an in-bin tone of
 * amplitude A leaves the FFT at A / 2), and the AGC of RX-SSB-q15 (window 16, rel[j] = e^(-j/6), target 8192, floor 16, gmax 64). */
typedef struct
{
  uint32_t bins;                         /* branches = FFT length = decimation [arm_cfft_q15]; this build: 64 */
  uint32_t taps_per_branch;              /* [arm_fir_q15 numTaps per branch]; this build: 8 */
  uint32_t agc_block;                    /* narrowband samples per AGC block (1 ms); this build: 3 */
  uint32_t envelope;                     /* 0 = product detector (real part), 1 = envelope [arm_cmplx_mag_q15] */
  int16_t  proto[SLB_CHAN_BINS * SLB_CHAN_TAPS];   /* prototype low-pass h[n], q15 */
  uint32_t agc_window;                   /* blocks of peak history the envelope sees (finite release), 1..17 */
  int16_t  rel[SLB_Q15_WIN];             /* q15 release weight of a block peak by age in blocks; rel[0] unused */
  int16_t  agc_target, agc_floor;        /* q15 */
  uint32_t agc_gmax_q15;                 /* gain limit in Q15 (1.0 = 32768) [arm_scale_q15 scaleFract << shift] */
} slb_chan_q15_params;

/* ---- life cycle ---- */
int  slb_create (const slb_config *cfg, slb_ctx **out);
void slb_destroy (slb_ctx *ctx);
const char *slb_last_error (const slb_ctx *ctx);           /* ctx may be NULL: last create() failure */
const char *slb_version (void);

/* ---- frozen default design (there are no taps or constants in the reference; SURVEY.md §0) ---- */
int slb_default_rx_f32_params (uint32_t fs, slb_rx_f32_params *out);
/* frequency response of the frozen 129-tap complex band-pass for `mode`, 2*fft_len floats re/im, UNSCALED */
int slb_default_mask (uint32_t fs, uint32_t fft_len, uint8_t mode, float *mask_out);
int slb_set_rx_f32_params (slb_ctx *ctx, const slb_rx_f32_params *p);
int slb_get_rx_f32_params (const slb_ctx *ctx, slb_rx_f32_params *p);
int slb_default_tx_f32_params (uint32_t fs, slb_tx_f32_params *out);
int slb_set_tx_f32_params (slb_ctx *ctx, const slb_tx_f32_params *p);
int slb_get_tx_f32_params (const slb_ctx *ctx, slb_tx_f32_params *p);
/* AM / FM modulator constants (SLB_CHAIN_TX_F32 contexts only; defaults: carrier 0.5, depth 0.8, deviation 2500 Hz, level 0.5) */
int slb_default_tx_mod_params (uint32_t fs, slb_tx_mod_params *out);
int slb_set_tx_mod_params (slb_ctx *ctx, const slb_tx_mod_params *p);
int slb_get_tx_mod_params (const slb_ctx *ctx, slb_tx_mod_params *p);
int slb_default_rx_q15_params (uint32_t fs, slb_rx_q15_params *out);
int slb_set_rx_q15_params (slb_ctx *ctx, const slb_rx_q15_params *p);
int slb_get_rx_q15_params (const slb_ctx *ctx, slb_rx_q15_params *p);
/* SLB_CHAIN_RX_Q15 contexts only (others: SLB_ERR_STATE) */
int slb_default_rx_q15_mode_params (uint32_t fs, slb_rx_q15_mode_params *out);
int slb_set_rx_q15_mode_params (slb_ctx *ctx, const slb_rx_q15_mode_params *p);
int slb_get_rx_q15_mode_params (const slb_ctx *ctx, slb_rx_q15_mode_params *p);
/* SLB_CHAIN_TX_Q15 contexts only (others: SLB_ERR_STATE) */
int slb_default_tx_q15_mode_params (uint32_t fs, slb_tx_q15_mode_params *out);
int slb_set_tx_q15_mode_params (slb_ctx *ctx, const slb_tx_q15_mode_params *p);
int slb_get_tx_q15_mode_params (const slb_ctx *ctx, slb_tx_q15_mode_params *p);
int slb_set_mask (slb_ctx *ctx, uint8_t mode, const float *mask);   /* host, 2*fft_len floats */
int slb_get_mask (const slb_ctx *ctx, uint8_t mode, float *mask);
/* which kernel serves the RX-SSB-f32 chain (DESIGN.md §4A): SLB_RX_PATH_AUTO = the tensor-core FIR kernel for every channel
 * whose mask is a 129-tap filter (all the default masks but AM), the FFT kernel for the rest; SLB_RX_PATH_FFT = the FFT
 * kernel for everything. Both carry the same state, so the path may change between calls. */
#define SLB_RX_PATH_AUTO 0
#define SLB_RX_PATH_FFT  1
int slb_set_rx_path (slb_ctx *ctx, int path);

/* ---- the firmware API, batched (reference: Core/Inc/dsp_if.h:42-51; bodies Core/Src/dsp_if.c) ----
 * pbuf is HOST memory laid out [channels][size]; `size` means what it means in the firmware. */
int SLB_DSP_Init (slb_ctx *ctx);                                                   /* dsp_if.c:377 */
int SLB_DSP_Set_RX (slb_ctx *ctx);                                                 /* dsp_if.c:347 */
int SLB_DSP_Set_TX (slb_ctx *ctx);                                                 /* dsp_if.c:357 */
int SLB_DSP_Set_Mode (slb_ctx *ctx, uint8_t mode);                                 /* dsp_if.c:367, all channels */
/* SLB_DSP_Set_RX / _TX act on a CHANGE of direction (as ptt_set_rx / ptt_set_tx do, rxtx_if.c:255-317): the codec's mute-reroute-unmute
 * (codec_if.c:230-345) becomes: the samples of both rings are flushed (pointers untouched, as DSP_Out_Buff_Mute) and the chain's carried
 * state is cleared, so nothing captured or queued under the old routing comes out under the new one. slb_get_direction: 0 = RX, 1 = TX. */
int slb_get_direction (const slb_ctx *ctx);
/* CW side-tone, mixed at the hook the firmware marks ("mix CW tone to speaker signal here", dsp_if.c:218): SLB_DSP_Out_Buff_Read[_Ch]
 * adds the tone to L and R of every keyed channel. Composition (ours) of reference stages: arm_sin_f32 (k 2 pi / fs) -> arm_scale_f32
 * (level) -> arm_float_to_q15 -> arm_add_q15 (saturating); the phase counter k = (k + freq) mod fs restarts at 0 with every key-down.
 * key_down: host [channels] bytes (NULL = all keys up). freq_hz = 0 switches the tone off. */
int SLB_DSP_Set_Sidetone (slb_ctx *ctx, uint32_t freq_hz, float level);
int SLB_DSP_Key (slb_ctx *ctx, const uint8_t *key_down);
int SLB_DSP_Set_Mode_Channel (slb_ctx *ctx, uint32_t channel, uint8_t mode);
int SLB_DSP_In_Buff_Write (slb_ctx *ctx, const uint16_t *pbuf, uint16_t size);     /* dsp_if.c:250, size = half-words */
int SLB_DSP_In_Buff_Read (slb_ctx *ctx, uint8_t *pbuf, uint32_t size);             /* dsp_if.c:310, size = bytes */
int SLB_DSP_Out_Buff_Write (slb_ctx *ctx, const uint8_t *pbuf, uint32_t size);     /* dsp_if.c:116, size = bytes */
int SLB_DSP_Out_Buff_Read (slb_ctx *ctx, uint16_t *pbuf, uint16_t size);           /* dsp_if.c:204, size = half-words */
int SLB_DSP_Out_Buff_Mute (slb_ctx *ctx);                                          /* dsp_if.c:188 */
/* ring introspection (tests): which 0 = RX ring (dsp_in_buff), 1 = TX ring (dsp_out_buff); out = {enable, rd, wr} */
int slb_ring_get_ptrs (const slb_ctx *ctx, int which, uint32_t out[3]);
/* ---- per-channel cadence (the ring's drift compensation as a batched primitive; dsp_if.c:136-179, :252-300) ----
 * `active` is a HOST array [channels] (NULL = all): a channel with active[c] == 0 is skipped by this call, exactly as if
 * its producer / consumer had not fired this millisecond. From the first such call on every channel carries its own
 * {enable, rd, wr} on the device, fill levels drift apart, and the firmware's own +-1 slip / repeat logic re-centres each
 * channel independently. A skipped channel's part of a read buffer is zero-filled. The producer side of the RX ring
 * accepts a mask with the PASS chain only (a chain's filter state has one cadence). */
int SLB_DSP_In_Buff_Write_Ch (slb_ctx *ctx, const uint16_t *pbuf, uint16_t size, const uint8_t *active);
int SLB_DSP_In_Buff_Read_Ch (slb_ctx *ctx, uint8_t *pbuf, uint32_t size, const uint8_t *active);
int SLB_DSP_Out_Buff_Write_Ch (slb_ctx *ctx, const uint8_t *pbuf, uint32_t size, const uint8_t *active);
int SLB_DSP_Out_Buff_Read_Ch (slb_ctx *ctx, uint16_t *pbuf, uint16_t size, const uint8_t *active);
int slb_ring_get_ptrs_channel (slb_ctx *ctx, int which, uint32_t channel, uint32_t out[3]);
/* copies the de-interleaved ring contents to host: i, q each [channels][DSP_BUFF_SIZE] */
int slb_ring_get_iq (slb_ctx *ctx, int which, int16_t *i, int16_t *q);

/* ---- bulk path: many firmware blocks per call, ring bypassed ----
 * in/out: [channels][frames][2] int16; frames must be a multiple of hop (PASS: any).
 * *_device: device pointers, asynchronous on `stream` (a cudaStream_t passed as void*, NULL = default stream).
 * *_host: host pointers; stages through pinned memory with chunked H2D / kernel / D2H overlap, synchronous. */
int slb_rx_process_device (slb_ctx *ctx, const int16_t *d_in, int16_t *d_out, uint32_t frames, void *stream);
int slb_rx_process_host (slb_ctx *ctx, const int16_t *h_in, int16_t *h_out, uint32_t frames);
/* TX direction (context created with SLB_CHAIN_TX_SSB_F32, SLB_CHAIN_TX_F32 or SLB_CHAIN_TX_SSB_Q15): in = mic frames (L = R as the
 * codec delivers them in TX, Core/Src/codec_if.c:304-306; L is used), out = modulated I/Q frames. Same shapes and rules as the RX calls
 * (SLB_CHAIN_TX_SSB_Q15: frames % 48 == 0, as RX-SSB-q15). With these chains SLB_DSP_In_Buff_Write runs the modulator at the 1 ms cadence
 * exactly as it runs the demodulator for RX (SLB_CHAIN_TX_SSB_Q15: in the call that delivers the block, no added latency). */
int slb_tx_process_device (slb_ctx *ctx, const int16_t *d_in, int16_t *d_out, uint32_t frames, void *stream);
int slb_tx_process_host (slb_ctx *ctx, const int16_t *h_in, int16_t *h_out, uint32_t frames);
/* Channelizer (context created with SLB_CHAIN_CHAN64_F32): in = wideband I/Q [streams][frames][2] int16, out =
 * demodulated narrowband audio, channel-major [streams][64 bins][frames/64][2] int16 (L = R). frames % 768 == 0
 * (4 firmware blocks of 192 frames). Debug taps (slb_rx_set_debug_taps): d_audio [streams][64][frames/64] f32 pre-AGC,
 * d_gain [streams][64][frames/192]. The firmware ring API is not offered for this chain (one ring holds one I/Q stream,
 * dsp_if.c:32-35); SLB_DSP_Set_Mode(AM) selects the envelope detector, any other mode the product detector. */
int slb_default_chan_params (uint32_t fs, slb_chan_params *out);
int slb_set_chan_params (slb_ctx *ctx, const slb_chan_params *p);
int slb_get_chan_params (const slb_ctx *ctx, slb_chan_params *p);
int slb_chan_process_device (slb_ctx *ctx, const int16_t *d_in, int16_t *d_out, uint32_t frames, void *stream);
int slb_chan_process_host (slb_ctx *ctx, const int16_t *h_in, int16_t *h_out, uint32_t frames);
/* CHAN-64-q15 (context created with SLB_CHAIN_CHAN64_Q15, fs 192000 only): slb_chan_process_* with the same shapes and rules; the debug
 * taps are slb_rx_q15_set_debug_taps: d_audio int16 [streams][64][frames/64] (the pre-AGC detector output), d_gain uint32
 * [streams][64][frames/192] (the Q15 gain word per block). Parameter calls on other contexts: SLB_ERR_STATE. */
int slb_default_chan_q15_params (uint32_t fs, slb_chan_q15_params *out);
int slb_set_chan_q15_params (slb_ctx *ctx, const slb_chan_q15_params *p);
int slb_get_chan_q15_params (const slb_ctx *ctx, slb_chan_q15_params *p);
/* optional float tap: post-biquad, pre-AGC audio [channels][frames] f32 and per-block gains [channels][frames/agc_block]
 * are written by the next slb_rx_process_device call(s) when non-NULL (device pointers). TX chain: d_audio receives
 * the pre-ALC complex baseband [channels][frames][2] f32. */
int slb_rx_set_debug_taps (slb_ctx *ctx, float *d_audio, float *d_gain);
/* SLB_CHAIN_TX_F32: the FM phase accumulator phi[n] (uint32, units of 2^-32 turn) after each sample, [channels][frames], device
 * pointer, written by the next slb_tx_process_device call(s) for FM channels when non-NULL (other channels' rows are left alone) */
int slb_tx_set_phase_tap (slb_ctx *ctx, uint32_t *d_phase);
/* RX-SSB-q15: pre-AGC q15 audio int16[channels][frames] and the per-block gain q (Q15) uint32[channels][frames/48].
 * RX-Q15: the same, the pre-AGC detector output of each channel's mode (AM: the 2.14 magnitude, FM: the discriminator).
 * TX-SSB-q15: d_audio receives the pre-ALC (I, Q) int16[channels][frames][2] (after the rail order), d_gain the same gain words.
 * TX-Q15: the same; AM and FM channels give (a, 0), the pre-ALC low-passed mic. */
int slb_rx_q15_set_debug_taps (slb_ctx *ctx, int16_t *d_audio, uint32_t *d_gain);

/* ---- per-channel tuning within the I/Q band (DESIGN.md §3.5): SLB_CHAIN_RX_SSB_F32, SLB_CHAIN_TX_SSB_F32, SLB_CHAIN_TX_F32 ----
 * A channel with offset f != 0 has its int16 I/Q mixed by a table NCO: in front of the RX chain (the chain then demodulates what sits
 * at +f Hz of the channel's input) and behind the TX chain (the signal leaves at +f Hz), so one offset pairs a TX and an RX context.
 * The NCO increment is inc = llround (f 2^32 / fs) (2^-32 turn per sample, computed in double); the realized offset is inc fs / 2^32,
 * and an offset is refused (SLB_ERR_ARG) unless |inc| <= 2^31 - 1, i.e. |f| < fs / 2. A rotated component that exceeds full scale
 * (|z| > 1) saturates. The phase is carried per channel in the context's state (a retune keeps it: phase-continuous), is zeroed by a
 * direction switch and SLB_DSP_Init, and is part of the checkpoint; the offsets are configuration that a direction switch keeps and
 * that the caller sets again on a context restored with slb_state_load, like chain parameters and masks. Calls and pushes issued
 * before a setter returns use the old offsets, those issued after it the new ones. A channel with offset 0 is passed unchanged and costs
 * nothing; its phase is kept (not advanced) until it is tuned again.
 * Other chains refuse with SLB_ERR_UNSUPPORTED. */
int slb_set_tune (slb_ctx *ctx, const double *offset_hz);                              /* host [channels] in Hz; NULL = all 0 */
int slb_set_tune_channel (slb_ctx *ctx, uint32_t ch, double offset_hz);
int slb_get_tune_channel (const slb_ctx *ctx, uint32_t ch, int32_t *inc, double *realized_hz);   /* either output may be NULL */

/* ---- carried state = the checkpoint (SURVEY.md §5): overlap tail, biquad d1/d2, AGC envelope, ring ---- */
int slb_state_size (const slb_ctx *ctx, size_t *bytes);
int slb_state_save (slb_ctx *ctx, void *host_buf, size_t bytes);
int slb_state_load (slb_ctx *ctx, const void *host_buf, size_t bytes);

/* ---- stage library: the CMSIS-DSP routines SURVEY.md §8(a) lists as stages of the path, batched, unfused ----
 * Array pointers are DEVICE pointers laid out [channels][n] (complex: interleaved re,im, n = complex count); coefficient
 * pointers are HOST pointers; `hist` / `state` are caller-owned DEVICE buffers that carry what the CMSIS instance would:
 * FIR hist = the first ntaps-1 state entries (interpolator: ntaps/L - 1) per channel; biquad state = the CMSIS layout
 * per channel (df2T 2/stage, stereo df2T 4/stage, df1 4/stage). `stream` is a cudaStream_t or NULL. Reference for each
 * name: Drivers/CMSIS/DSP/Source/<group>/arm_<name>.c. Integer routines are bit-exact; so are the sequential float ones. */
int slb_st_q15_to_float (slb_ctx *ctx, const int16_t *src, float *dst, uint32_t n, void *stream);
int slb_st_float_to_q15 (slb_ctx *ctx, const float *src, int16_t *dst, uint32_t n, void *stream);
int slb_st_scale_f32 (slb_ctx *ctx, const float *src, float scale, float *dst, uint32_t n, void *stream);
int slb_st_mult_f32 (slb_ctx *ctx, const float *a, const float *b, float *dst, uint32_t n, void *stream);
int slb_st_add_f32 (slb_ctx *ctx, const float *a, const float *b, float *dst, uint32_t n, void *stream);
int slb_st_sub_f32 (slb_ctx *ctx, const float *a, const float *b, float *dst, uint32_t n, void *stream);
int slb_st_abs_f32 (slb_ctx *ctx, const float *a, float *dst, uint32_t n, void *stream);
int slb_st_scale_q15 (slb_ctx *ctx, const int16_t *src, int16_t scale_fract, int32_t shift, int16_t *dst, uint32_t n, void *stream);
int slb_st_add_q15 (slb_ctx *ctx, const int16_t *a, const int16_t *b, int16_t *dst, uint32_t n, void *stream);
int slb_st_sub_q15 (slb_ctx *ctx, const int16_t *a, const int16_t *b, int16_t *dst, uint32_t n, void *stream);
int slb_st_abs_q15 (slb_ctx *ctx, const int16_t *a, int16_t *dst, uint32_t n, void *stream);
int slb_st_shift_q15 (slb_ctx *ctx, const int16_t *a, int32_t shift, int16_t *dst, uint32_t n, void *stream);
int slb_st_cmplx_mult_cmplx_f32 (slb_ctx *ctx, const float *a, const float *b, float *dst, uint32_t n, void *stream);
int slb_st_cmplx_mult_real_f32 (slb_ctx *ctx, const float *a, const float *r, float *dst, uint32_t n, void *stream);
int slb_st_cmplx_conj_f32 (slb_ctx *ctx, const float *a, float *dst, uint32_t n, void *stream);
int slb_st_cmplx_mag_f32 (slb_ctx *ctx, const float *a, float *dst, uint32_t n, void *stream);
int slb_st_cmplx_mag_squared_f32 (slb_ctx *ctx, const float *a, float *dst, uint32_t n, void *stream);
int slb_st_cmplx_mag_q15 (slb_ctx *ctx, const int16_t *a, int16_t *dst, uint32_t n, void *stream);
int slb_st_sin_f32 (slb_ctx *ctx, const float *x, float *dst, uint32_t n, void *stream);
int slb_st_cos_f32 (slb_ctx *ctx, const float *x, float *dst, uint32_t n, void *stream);
int slb_st_fir_f32 (slb_ctx *ctx, const float *coeffs, uint32_t ntaps, float *hist, const float *src, float *dst, uint32_t n, void *stream);
int slb_st_fir_q15 (slb_ctx *ctx, const int16_t *coeffs, uint32_t ntaps, int16_t *hist, const int16_t *src, int16_t *dst, uint32_t n, void *stream);
int slb_st_fir_fast_q15 (slb_ctx *ctx, const int16_t *coeffs, uint32_t ntaps, int16_t *hist, const int16_t *src, int16_t *dst, uint32_t n, void *stream);
int slb_st_fir_q31 (slb_ctx *ctx, const int32_t *coeffs, uint32_t ntaps, int32_t *hist, const int32_t *src, int32_t *dst, uint32_t n, void *stream);
int slb_st_fir_decimate_f32 (slb_ctx *ctx, const float *coeffs, uint32_t ntaps, uint32_t M, float *hist, const float *src, float *dst, uint32_t n, void *stream);
int slb_st_fir_decimate_q15 (slb_ctx *ctx, const int16_t *coeffs, uint32_t ntaps, uint32_t M, int16_t *hist, const int16_t *src, int16_t *dst, uint32_t n, void *stream);
int slb_st_fir_interpolate_f32 (slb_ctx *ctx, const float *coeffs, uint32_t ntaps, uint32_t L, float *hist, const float *src, float *dst, uint32_t n, void *stream);
int slb_st_fir_interpolate_q15 (slb_ctx *ctx, const int16_t *coeffs, uint32_t ntaps, uint32_t L, int16_t *hist, const int16_t *src, int16_t *dst, uint32_t n, void *stream);
int slb_st_fir_decimate_q31 (slb_ctx *ctx, const int32_t *coeffs, uint32_t ntaps, uint32_t M, int32_t *hist, const int32_t *src, int32_t *dst, uint32_t n, void *stream);      /* arm_fir_decimate_q31.c:60 */
int slb_st_fir_interpolate_q31 (slb_ctx *ctx, const int32_t *coeffs, uint32_t ntaps, uint32_t L, int32_t *hist, const int32_t *src, int32_t *dst, uint32_t n, void *stream);   /* arm_fir_interpolate_q31.c:62 */
/* normalised LMS adaptive FIR (arm_lms_norm_f32.c:161): noise reduction (out) / auto-notch (err) when src is a delayed copy of ref.
 * coeffs: device [channels][ntaps], state: device [channels][ntaps + 1] = ntaps - 1 previous samples, energy, x0; both updated in place. */
int slb_st_lms_norm_f32 (slb_ctx *ctx, float *coeffs, uint32_t ntaps, float mu, float *state, const float *src, const float *ref, float *out, float *err, uint32_t n, void *stream);
int slb_st_biquad_df2T_f32 (slb_ctx *ctx, const float *coeffs, uint32_t n_stages, float *state, const float *src, float *dst, uint32_t n, void *stream);
int slb_st_biquad_stereo_df2T_f32 (slb_ctx *ctx, const float *coeffs, uint32_t n_stages, float *state, const float *src, float *dst, uint32_t nframes, void *stream);
int slb_st_biquad_df1_f32 (slb_ctx *ctx, const float *coeffs, uint32_t n_stages, float *state, const float *src, float *dst, uint32_t n, void *stream);
int slb_st_biquad_df1_q15 (slb_ctx *ctx, const int16_t *coeffs, uint32_t n_stages, int32_t postshift, int16_t *state, const int16_t *src, int16_t *dst, uint32_t n, void *stream);
int slb_st_biquad_df1_q31 (slb_ctx *ctx, const int32_t *coeffs, uint32_t n_stages, int32_t postshift, int32_t *state, const int32_t *src, int32_t *dst, uint32_t n, void *stream);
/* per-block statistics: out is [channels][n / block]; idx (may be NULL) receives the position of the maximum */
int slb_st_max_f32 (slb_ctx *ctx, const float *src, uint32_t n, uint32_t block, float *out, uint32_t *idx, void *stream);
int slb_st_rms_f32 (slb_ctx *ctx, const float *src, uint32_t n, uint32_t block, float *out, void *stream);
int slb_st_power_f32 (slb_ctx *ctx, const float *src, uint32_t n, uint32_t block, float *out, void *stream);
int slb_st_mean_f32 (slb_ctx *ctx, const float *src, uint32_t n, uint32_t block, float *out, void *stream);
int slb_st_max_q15 (slb_ctx *ctx, const int16_t *src, uint32_t n, uint32_t block, int16_t *out, uint32_t *idx, void *stream);
int slb_st_rms_q15 (slb_ctx *ctx, const int16_t *src, uint32_t n, uint32_t block, int16_t *out, void *stream);
/* batched arm_cfft_f32 (bit-reversed output order is not offered): data [channels][count][2*N] floats, in place */
int slb_st_cfft_f32 (slb_ctx *ctx, float *data, uint32_t N, uint32_t count, int ifft, void *stream);
/* batched arm_cfft_q15 (arm_cfft_q15.c:77, in the ARM_MATH_DSP branch the firmware's ARM_MATH_CM4 build compiles) and arm_cfft_q31
 * (arm_cfft_q31.c:77): data [channels][count][2*N] q15 / q31, in place, N = 16..4096, natural output order, bit-exact; the output
 * scaling is the reference's (forward: 1/N for N = 4^m ... see arm_cfft_radix4_q15.c:94-104). slb_design_twiddle_*: the regenerated
 * twiddle tables (3 N / 4 (cos, sin) pairs), exported for the design check against arm_common_tables.c. */
int slb_st_cfft_q15 (slb_ctx *ctx, int16_t *data, uint32_t N, uint32_t count, int ifft, void *stream);
int slb_st_cfft_q31 (slb_ctx *ctx, int32_t *data, uint32_t N, uint32_t count, int ifft, void *stream);
int slb_design_twiddle_q15 (uint32_t N, int16_t *out);
int slb_design_twiddle_q31 (uint32_t N, int32_t *out);
/* batched arm_rfft_fast_f32 (arm_rfft_fast_f32.c:288): in / out [channels][count][N] floats, out of place, N = 32..4096;
 * forward output packed as the reference packs it: out[0] = X[0], out[1] = X[N/2], then (Re, Im) of X[1..N/2-1] */
int slb_st_rfft_fast_f32 (slb_ctx *ctx, const float *in, float *out, uint32_t N, uint32_t count, int ifft, void *stream);

/* ---- host stream feeder (SURVEY.md §8f.1): the stand-in for HAL DMA + UAC1 that replays the firmware's cadence ----
 * One tick = 1 ms = fs/1000 frames per channel, in this order (the I2S completion callback, dsp_if.c:50-67, then the two
 * USB class commands, usbd_audio_if.c:179-202):
 *     DSP_Out_Buff_Read (dac block t); DSP_In_Buff_Write (adc block t); DSP_Out_Buff_Write (usb_out packet t);
 *     DSP_In_Buff_Read (usb_in packet t)
 * slb_feeder_run() is equivalent to `ticks` rounds of those four batched calls, but moves whole streams: one H2D copy,
 * the context's chain over all ticks in one launch, the ring traffic of all ticks replayed by one kernel per ring (the
 * pointer evolution, including the start-up slips, is planned on the host with the firmware's own arithmetic), one
 * D2H copy. Buffers are HOST memory [channels][ticks * fs/1000][2]; a NULL pair skips that direction. With the
 * RX-SSB-f32 chain `ticks` must be a multiple of 8 (the 384-frame super-block). Not available while per-channel
 * cadence (SLB_DSP_*_Ch) is on. */
typedef struct
{
  const int16_t *adc;       /* RX in : what the codec ADC delivers on the I2S bus */
  int16_t *usb_in;          /* RX out: what AUDIO_CMD_RECORD hands to the USB IN endpoint */
  const int16_t *usb_out;   /* TX in : what AUDIO_CMD_PLAY receives from the USB OUT endpoint */
  int16_t *dac;             /* TX out: what the I2S TX half carries to the codec DAC */
} slb_feeder_io;
int slb_feeder_run (slb_ctx *ctx, const slb_feeder_io *io, uint32_t ticks);

/* ---- LIVE feeder: the same four calls per tick, as a pipeline over chunks of `ticks_per_chunk` ms (SURVEY.md §8f.1) ----
 * What replaces the double-buffered I2S DMA (dsp_if.c:50-67: one half is processed while the other fills) and the USB isochronous
 * endpoints (usbd_audio.c:707-745, :844-879) on a host: slb_live_push() takes the chunk that has just filled (host buffers, copied
 * into pinned staging), and returns at once; the chunk's host->device copy, its kernels (chain + ring replay) and its device->host
 * copy run on three streams, so chunk n is copied in while chunk n-1 computes and chunk n-2 is copied out. slb_live_pop() hands
 * out the oldest finished chunk (blocks until it is there; SLB_ERR_STATE when nothing is in flight). At most `depth` chunks
 * (2..8) are in flight; push with all slots taken returns SLB_ERR_STATE (pop first). Results are bit-identical to slb_feeder_run
 * and to the per-tick calls. latency_us (may be NULL) receives the time from the chunk's push to the moment its results were in
 * host memory. Directions as in slb_feeder_io: give adc to get usb_in, usb_out to get dac; which ones is fixed at open time. */
typedef struct slb_live slb_live;
int slb_live_open (slb_ctx *ctx, uint32_t ticks_per_chunk, uint32_t depth, int with_rx, int with_tx, slb_live **out);
int slb_live_push (slb_live *lv, const int16_t *adc, const int16_t *usb_out);
int slb_live_pop (slb_live *lv, int16_t *usb_in, int16_t *dac, float *latency_us);
int slb_live_in_flight (const slb_live *lv);
void slb_live_close (slb_live *lv);
/* USBD_AUDIO_ItfTypeDef.AudioCmd, batched (usbd_audio_if.c:179-202): cmd = 1 START (no-op), 2 PLAY -> DSP_Out_Buff_Write,
 * 3 STOP -> DSP_Out_Buff_Mute, 4 RECORD -> DSP_In_Buff_Read; pbuf is [channels][size] host memory, size in bytes */
int SLB_AUDIO_AudioCmd (slb_ctx *ctx, uint8_t *pbuf, uint32_t size, uint8_t cmd);

/* ---- host-only logic, callable without a GPU (unit tests of the index arithmetic and the scan tables) ----
 * One firmware ring's pointer logic, Core/Src/dsp_if.c:116-180, :204-219, :250-301, :310-340. state = {enable, rd, wr}
 * is updated in place; the return value is the ring slot of the first frame moved (a write stores frames+1 slots:
 * the block, then its last frame once more, dsp_if.c:291-300). */
uint32_t slb_ring_plan_write (uint32_t ring_frames, int is_out, uint32_t state[3], uint32_t frames);
uint32_t slb_ring_plan_read (uint32_t ring_frames, int is_out, uint32_t state[3], uint32_t frames);
/* tables of the time-parallel 2-stage df2T evaluation (DESIGN.md §4.3) for runs of 24 samples: Mpow[6][16] =
 * (A^24)^(2^k), Cresp[24][4] */
int slb_biquad_scan_tables (const float coef10[10], float *Mpow96, float *Cresp96);
/* the tensor-core form of the RX-SSB-f32 chain (DESIGN.md §4A). slb_design_tc_taps: the 129 complex taps whose DFT the mask
 * [512][2] is (SLB_ERR_UNSUPPORTED when the mask is no 129-tap filter: the FFT kernel then serves it).
 * slb_design_tc_block: builds the kernel's tcgen05 operand planes (taps composed with the zero-state response of the 2-stage
 * biquad, 24-bit digits) and evaluates them in integers on one raw window int16[176][2] = 128 frames of history + one
 * 48-frame block: out52[0..47] = the block's biquad output from a zero state, out52[48..51] = the biquad state after it. */
int slb_design_tc_taps (const float *mask_re_im, double taps_re[129], double taps_im[129]);
int slb_design_tc_block (const float *mask_re_im, const float coef10[10], const int16_t *window, double out52[52]);
/* the same for TX (sl_tx_ssb_tc.cu): window = int16[192] mic samples from 128 before the block, out = (I, Q) of its 48 samples */
int slb_design_tc_tx_block (const float *mask_re_im, const int16_t *window, double out_iq[96]);
/* and for the integer chain (sl_rx_q15_tc.cu): window = int16[112][2] I/Q frames from 64 before the block, out = the 48 arm_fir_q15
 * results of rail I, then of rail Q; SLB_ERR_UNSUPPORTED when a tap does not split into two signed bytes (|tap| >= 32640) */
int slb_design_q15_tc_block (const int16_t taps_i[64], const int16_t taps_q[64], const int16_t *window, int32_t out96[96]);
/* the TX planes of the same kernel (TX-SSB-q15): window = int16[112][2] L=R mic frames from 64 before the block, out = the 48 arm_fir_q15
 * results of L with taps_i (rail fi), then with taps_q (rail fq), before the rail order; R meets zero weight */
int slb_design_q15_tc_tx_block (const int16_t taps_i[64], const int16_t taps_q[64], const int16_t *window /* [112][2] L=R */, int32_t out96[96]);
/* the FM planes of the same kernel (RX-Q15): window = int16[112][2] I/Q frames from 64 before the block, out = the 49 arm_fir_q15 results
 * of rail I with taps at frames -1 .. 47 of the block, then the same of rail Q; SLB_ERR_UNSUPPORTED when a tap does not split */
int slb_design_q15_tc_fm_block (const int16_t taps[64], const int16_t *window, int32_t out98[98]);
int slb_design_mask (uint32_t fs, uint8_t mode, float *mask_re_im);
/* tables of the tensor-core kernel's time-parallel biquad for blocks of 48 samples: Mp[4][16] = A^(48 k), M192[16], Cresp[48][4] */
int slb_biquad_tc_tables (const float coef10[10], float *Mp64, float *M192, float *Cresp192);

/* ---- spectrum export (SURVEY.md §8f.4; the north-star's "gather spectra"): power spectrum of N frames per channel,
 * d_iq int16 [channels][N][2] -> d_power float [channels][N] (natural bin order, bin k = k fs / N, upper half = negative
 * frequencies), as arm_q15_to_float -> arm_cfft_f32 (N = 16..4096) -> arm_cmplx_mag_squared_f32. Device pointers, async;
 * gathering the shards' spectra over NCCL is selenite_lite_b200/shard.py::gather_spectra. */
int slb_rx_spectrum_device (slb_ctx *ctx, const int16_t *d_iq, float *d_power, uint32_t N, void *stream);

/* ---- accounting ---- */
uint64_t slb_kernel_launches (const slb_ctx *ctx);   /* kernels this context has launched since create */
int slb_sync (slb_ctx *ctx);

/* ---- single-channel drop-in with the firmware's own names and signatures (Core/Inc/dsp_if.h:42-51).
 * They drive one process-global 1-channel context on device 0 (env SELENITE_B200_DEVICE, SELENITE_B200_FS,
 * SELENITE_B200_CHAIN=pass|rx_ssb_f32|tx_ssb_f32|tx_f32|rx_ssb_q15|tx_ssb_q15|rx_q15|tx_q15; default pass at 48000 = the firmware's behaviour). Like the firmware
 * they return void; failures are reported through slb_dropin_status(). ---- */
void DSP_Init (void);
void DSP_Set_RX (void);
void DSP_Set_TX (void);
void DSP_Set_Mode (uint8_t mode);
void DSP_In_Buff_Write (uint16_t *pbuf, uint16_t size);
void DSP_In_Buff_Read (uint8_t *pbuf, uint32_t size);
void DSP_Out_Buff_Write (uint8_t *pbuf, uint32_t size);
void DSP_Out_Buff_Read (uint16_t *pbuf, uint16_t size);
void DSP_Out_Buff_Mute (void);
/* the rest of the firmware's sample-path surface, single channel: the I2S DMA double buffer and its two completion
 * callbacks (dsp_if.c:32, :50-67; hi2s is ignored) and the USB class dispatcher (usbd_audio_if.c:179-202) */
/* i2s_buff has the layout of the firmware's I2S_Buff_TypeDef (dsp_if.h:75-79): rx[I2S_BUFF_SIZE]; tx[I2S_BUFF_SIZE] with
 * I2S_BUFF_SIZE = 2 * (2 * USBD_AUDIO_FREQ / 1000) half-words (dsp_if.h:69-73) — 192 at 48 kHz, 384 at 96 kHz, 768 at 192 kHz. As in
 * the firmware the size is compile-time: build the consumer with the same -DUSBD_AUDIO_FREQ as dsp_if.h would see (default 48000,
 * dsp_if.h:55-57) and run the library with the same rate (SELENITE_B200_FS): the library places tx at
 * I2S_BUFF_SIZE of ITS rate. The object the
 * library exports is storage for the largest geometry, so every rate's struct is a prefix-compatible view of it. */
#ifndef USBD_AUDIO_FREQ
#define USBD_AUDIO_FREQ 48000U
#endif
#define SLB_I2S_BUFF_SIZE (2U * ((USBD_AUDIO_FREQ * 2U) / 1000U))
#ifdef SLB_BUILDING_LIBRARY
typedef struct { uint16_t words[2 * 768]; } SLB_I2S_Buff_TypeDef;                /* rx = words, tx = words + I2S_BUFF_SIZE of the run-time rate */
#else
typedef struct { uint16_t rx[SLB_I2S_BUFF_SIZE]; uint16_t tx[SLB_I2S_BUFF_SIZE]; } SLB_I2S_Buff_TypeDef;
#endif
extern SLB_I2S_Buff_TypeDef i2s_buff;
void HAL_I2SEx_TxRxHalfCpltCallback (void *hi2s);
void HAL_I2SEx_TxRxCpltCallback (void *hi2s);
int8_t AUDIO_AudioCmd_FS (uint8_t *pbuf, uint32_t size, uint8_t cmd);
int  slb_dropin_status (void);
slb_ctx *slb_dropin_ctx (void);

#ifdef __cplusplus
}
#endif
#endif /* SELENITE_B200_H */
