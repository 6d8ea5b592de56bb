/* ORACLE / TEST INFRASTRUCTURE ONLY.
 *
 * CHAN-64-q15 (DESIGN.md §3.10): the all-integer channelizer, in the same two-implementation scheme as slo_api.h. Every box is a
 * CMSIS-DSP V1.5.3 routine the port restates and pins (fir_q15, cfft_q15 in the Cortex-M4 branch, cmplx_mag_q15, abs_q15, max_q15,
 * scale_q15); the composition and the gain law are ours. Kept beside slo_api.h (which it includes) so that the stages and chains that
 * header declares, and the digests recorded over their arguments, stay exactly as they are. Built into the port only: the reference
 * build's cfft_q15 is the shift-based C branch, not the firmware's.
 */
#ifndef SLO_CHAN_Q15_H
#define SLO_CHAN_Q15_H
#include "slo_api.h"

#ifdef __cplusplus
extern "C" {
#endif

#define SLO_CHAN_BINS 64
#define SLO_CHAN_TAPS 8

/* the layout of slb_chan_q15_params (include/selenite_b200.h) */
typedef struct
{
  uint32_t bins, taps_per_branch, agc_block;             /* 64 / 8 / 3 */
  uint32_t envelope;                                     /* 0: Re (product detector), 1: cmplx_mag_q15 */
  int16_t proto[SLO_CHAN_BINS * SLO_CHAN_TAPS];          /* h[n], q15; branch r uses e_r[p] = h[bins p + bins-1-r] */
  uint32_t agc_window;                                   /* 1..SLO_Q15_WIN */
  int16_t rel[SLO_Q15_WIN];                              /* q15 release weight by block age; rel[0] unused */
  int16_t agc_target, agc_floor;
  uint32_t agc_gmax_q15;
} slo_chan_q15_params;

typedef struct
{
  int16_t fir_i[SLO_CHAN_BINS][SLO_CHAN_TAPS], fir_q[SLO_CHAN_BINS][SLO_CHAN_TAPS];   /* arm_fir_q15 pState per branch: the last 7 inputs, oldest first */
  int16_t peaks[SLO_CHAN_BINS][SLO_Q15_WIN];             /* per bin, peaks[j] = block peak j+1 blocks ago */
} slo_chan_q15_state;

/* chan_q15: one wideband stream in_iq int16 [frames][2], frames % bins == 0 and (frames / bins) % agc_block == 0.
 * Branch r, rails I and Q apart: fir_q15 (e_r time-reversed, numTaps 8) over the stride-bins commutated input x_r[m] = in[bins m + r]
 * -> per hop m: cfft_q15 (bins, forward, natural order) of the branch outputs -> Re or cmplx_mag_q15 per bin
 * -> per bin and block of agc_block hops: abs_q15 + max_q15 = block peak -> the finite-window gain law of rx_ssb_q15 -> scale_q15.
 * out_lr int16 [bins][hops][2] (L = R); audio_dbg (optional) int16 [bins][hops] pre-AGC; gain_dbg (optional) uint32 [bins][hops/agc_block]. */
void SLO (chan_q15) (const slo_chan_q15_params *p, slo_chan_q15_state *st, const int16_t *in_iq, int16_t *out_lr,
                     int16_t *audio_dbg, uint32_t *gain_dbg, uint32_t frames);

#ifdef __cplusplus
}
#endif
#endif /* SLO_CHAN_Q15_H */
