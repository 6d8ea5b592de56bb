/* ORACLE / TEST INFRASTRUCTURE ONLY.
 *
 * TX-Q15 (DESIGN.md §3.9): the all-mode integer transmitter, in the same two-implementation scheme as slo_api.h. Every box is a
 * CMSIS-DSP V1.5.3 routine the port already restates and pins to the reference (fir_q15, abs_q15, max_q15, scale_q15, add_q15, and the
 * table NCO tx_fm_nco of slo_tx_mod.h); the composition, the gain law and the phase accumulator are ours. Kept beside slo_api.h (which
 * it includes) so that the stages and chains that header declares, and the digests recorded over their arguments, stay exactly as they are.
 */
#ifndef SLO_TX_Q15_MOD_H
#define SLO_TX_Q15_MOD_H
#include "slo_api.h"
#include "slo_tx_mod.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct
{
  slo_rx_q15_params q;                                   /* the SSB pair (lsb picks the sideband) and the AGC; bq_* unused */
  uint32_t kind;                                         /* the channel's modulator: 0 SSB-style modes, 1 AM, 2 FM */
  int16_t am_taps[SLO_Q15_TAPS], fm_taps[SLO_Q15_TAPS];  /* b[0..ntaps-1], natural order */
  int16_t am_carrier, am_depth, fm_target;               /* q15; the ALC targets of AM and FM */
  int32_t fm_inc;                                        /* 2^-32 turn per LSB of y, |fm_inc| <= 65535 */
  float fm_level;                                        /* NCO amplitude (tx_fm_nco) */
} slo_tx_q15m_params;

typedef struct
{
  int16_t raw[SLO_Q15_TAPS];                             /* the last 64 mic samples, oldest first */
  int16_t peaks[SLO_Q15_WIN];                            /* peaks[j] = block peak j+1 blocks ago */
  uint32_t phase;                                        /* FM phase accumulator, 2^-32 turn; held in the other modes */
} slo_tx_q15m_state;

/* tx_q15: per `agc_block` (the firmware block) of 48 frames, mic = L of the L = R frames, w = the 64 carried mic samples + the block's 48:
 * SSB: fi = fir_q15 (w, taps_i), fq = fir_q15 (w, taps_q) -> exactly tx_ssb_q15 (rail order, peak over both rails, gain law, scale_q15
 *      on both rails)
 * AM / FM: a = fir_q15 (w, am_taps / fm_taps) -> block peak abs_q15 + max_q15 of a -> the finite-window gain law of rx_ssb_q15 with the
 *      modulator's target (am_depth / fm_target) -> y = scale_q15 (a, q >> s, s), then
 *   AM: I = add_q15 (scale_q15 (y, am_carrier, 0), am_carrier), Q = 0
 *   FM: inc[n] = y[n] fm_inc (int32), phase[n] = phase[n-1] + inc[n] mod 2^32 (carried), (I, Q) = tx_fm_nco (phase, fm_level)
 * written interleaved I, Q. The FIR state is the raw mic, so a mode change between calls filters with the new taps as if the channel had
 * always been in that mode; the peak window carries over, the phase advances in FM blocks only. frames % agc_block == 0.
 * iq_dbg (optional): the pre-ALC pair [frames][2] (SSB: after the rail order; AM / FM: (a, 0)); gain_dbg: q per block;
 * phase_dbg (optional): phase[n] after each sample (FM blocks; other blocks hold the carried phase). */
void SLO (tx_q15) (const slo_tx_q15m_params *p, slo_tx_q15m_state *st, const int16_t *in_lr, int16_t *out_iq,
                   int16_t *iq_dbg, uint32_t *gain_dbg, uint32_t *phase_dbg, uint32_t frames);

#ifdef __cplusplus
}
#endif
#endif /* SLO_TX_Q15_MOD_H */
