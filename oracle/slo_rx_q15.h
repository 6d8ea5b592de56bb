/* ORACLE / TEST INFRASTRUCTURE ONLY.
 *
 * RX-Q15 (DESIGN.md §3.8): the all-mode integer receiver, in the same two-implementation scheme as slo_api.h. Every box is a CMSIS-DSP
 * V1.5.3 routine the port already restates and pins to the reference (fir_q15, cmplx_mag_q15 with its sqrt_q15, add_q15, sub_q15,
 * abs_q15, max_q15, scale_q15); the FM discriminator and the gain law are ours. Kept beside slo_api.h (which it includes) so that the
 * stages and chains that header declares, and the digests recorded over their arguments, stay exactly as they are.
 */
#ifndef SLO_RX_Q15_H
#define SLO_RX_Q15_H
#include "slo_api.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct
{
  slo_rx_q15_params q;                                   /* the SSB pair (lsb picks the sideband) and the AGC; bq_* unused */
  uint32_t kind;                                         /* the channel's detector: 0 SSB-style modes, 1 AM, 2 FM */
  int16_t am_taps[SLO_Q15_TAPS], fm_taps[SLO_Q15_TAPS];  /* b[0..ntaps-1], natural order */
  int32_t fm_floor;                                      /* >= 1 */
} slo_rx_q15m_params;

typedef struct
{
  int16_t raw_i[SLO_Q15_TAPS], raw_q[SLO_Q15_TAPS];      /* the last 64 input frames per rail, oldest first (z[-1] needs all 64) */
  int16_t peaks[SLO_Q15_WIN];                            /* peaks[j] = block peak j+1 blocks ago */
} slo_rx_q15m_state;

/* rx_q15: per `agc_block` (the firmware block) of 48 frames, with the window w = the 64 carried frames + the block's 48 per rail:
 * a = fir_q15 (w_I, taps), b = fir_q15 (w_Q, taps) at frames -1 .. 47 of the block (taps = taps_i / taps_q, am_taps or fm_taps by kind)
 * -> SSB: add_q15 (a, b) or, lsb = 1, sub_q15 (a, b)     [exactly rx_ssb_q15 without the biquad]
 *    AM:  v = cmplx_mag_q15 (a, b)                        [2.14]
 *    FM:  m = cmplx_mag_q15 (a, b) at frames -1 .. 47, x_n = a_{n-1} b_n - b_{n-1} a_n (int64),
 *         v_n = sat16 ((x_n * 2^13) / max (m_{n-1} m_n, fm_floor)) with C's truncating division
 * -> abs_q15 + max_q15 = block peak -> the finite-window gain law of rx_ssb_q15 -> scale_q15 -> written L = R.
 * The FIR state is the raw input, so a mode change between calls filters with the new taps as if the channel had always been in that
 * mode; the peak window carries over. frames % agc_block == 0. audio_dbg (optional): pre-AGC v [frames]; gain_dbg: q per block. */
void SLO (rx_q15) (const slo_rx_q15m_params *p, slo_rx_q15m_state *st, const int16_t *in_iq, int16_t *out_lr,
                   int16_t *audio_dbg, uint32_t *gain_dbg, uint32_t frames);

#ifdef __cplusplus
}
#endif
#endif /* SLO_RX_Q15_H */
