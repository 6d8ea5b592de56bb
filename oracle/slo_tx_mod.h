/* ORACLE / TEST INFRASTRUCTURE ONLY.
 *
 * The transmit AM and FM modulators of the all-mode TX chain (DESIGN.md §3.4), in the same two-implementation scheme as slo_api.h:
 * every box is a CMSIS-DSP V1.5.3 routine, the composition is ours. Kept beside slo_api.h (which it includes) so that the stages
 * and chains that header declares, and the digests recorded over their arguments, stay exactly as they are.
 */
#ifndef SLO_TX_MOD_H
#define SLO_TX_MOD_H
#include "slo_api.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- the three stages the modulators add (V1.5.3, plain-C branch, ARM_MATH_ROUNDING not defined) ----
 * offset_f32   BasicMathFunctions/arm_offset_f32.c      dst = src + offset
 * float_to_q31 SupportFunctions/arm_float_to_q31.c      dst = clip_q63_to_q31 ((q63_t) (src * 2147483648.0f))
 * q31_to_float SupportFunctions/arm_q31_to_float.c      dst = (float) src / 2147483648.0f */
void SLO (offset_f32) (const float *src, float offset, float *dst, uint32_t n);
void SLO (float_to_q31) (const float *src, int32_t *dst, uint32_t n);
void SLO (q31_to_float) (const int32_t *src, float *dst, uint32_t n);

/* TX-mod-f32: the front end of tx_ssb_f32 (mic = L -> q15_to_float -> overlap-save with the slot's mask, keep the last `hop`), then
 * on a[n] = Re z[n], per `alc_block`: peak = max_f32 (abs_f32 (a)), the ALC gain law of tx_ssb_f32 with the modulator's target, and
 *   AM  (modulator 1, target am_depth):  u = scale_f32 (a, g) -> offset_f32 (1) -> scale_f32 (am_carrier) -> float_to_q15 = I; Q = 0
 *   FM  (modulator 2, target T = 2 fm_deviation_hz / fs half-turns per sample):  inc = float_to_q31 (scale_f32 (a, g)),
 *       phi[n] = phi[n-1] + inc[n] mod 2^32 (uint32, carried), I/Q = tx_fm_nco (phi)
 * g |a| <= target, so the AM envelope stays in am_carrier (1 +- am_depth) and |inc| <= T 2^31. */
#define SLO_MOD_AM 1
#define SLO_MOD_FM 2
typedef struct
{
  uint32_t fft_len, hop, alc_block, fs;
  float alc_decay, alc_floor, alc_gmax;
  const float *mask;
  uint32_t modulator;                 /* SLO_MOD_AM or SLO_MOD_FM */
  float am_carrier, am_depth, fm_deviation_hz, fm_level;
} slo_tx_mod_params;

typedef struct
{
  int16_t ovl[SLO_MAX_FFT];           /* last (fft_len-hop) mic samples */
  float env;                          /* ALC envelope */
  uint32_t phase;                     /* FM phase accumulator, 2^-32 turn */
} slo_tx_mod_state;

/* frames % hop == 0. iq_dbg (optional): pre-ALC complex baseband [frames][2]; gain_dbg: per-block gain; phase_dbg (FM): phi[n]. */
void SLO (tx_mod_f32) (const slo_tx_mod_params *p, slo_tx_mod_state *st, const int16_t *in_lr, int16_t *out_iq,
                       float *iq_dbg, float *gain_dbg, uint32_t *phase_dbg, uint32_t frames);
/* The FM NCO alone: x = scale_f32 (q31_to_float ((int32) phase), 3.14159265f) -> I' = cos_f32 (x), Q' = sin_f32 (x)
 * -> scale_f32 (level) -> float_to_q15, written interleaved I, Q. */
void SLO (tx_fm_nco) (const uint32_t *phase, uint32_t n, float level, int16_t *out_iq);

#ifdef __cplusplus
}
#endif
#endif /* SLO_TX_MOD_H */
