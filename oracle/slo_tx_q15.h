/* ORACLE / TEST INFRASTRUCTURE ONLY.
 *
 * TX-SSB-q15 (DESIGN.md §3.7, SURVEY.md Appendix B "the fully-integer variant", transmit side), in the same two-implementation scheme
 * as slo_api.h: every box is a CMSIS-DSP V1.5.3 routine the port already restates (fir_q15, abs_q15, max_q15, scale_q15), the
 * composition is ours. Kept beside slo_api.h (which it includes) so that the stages and chains that header declares, and the digests
 * recorded over their arguments, stay exactly as they are.
 */
#ifndef SLO_TX_Q15_H
#define SLO_TX_Q15_H
#include "slo_api.h"

#ifdef __cplusplus
extern "C" {
#endif

/* tx_ssb_q15: phasing-method SSB modulator with the parameters and state of rx_ssb_q15 (both FIR histories hold mic samples; bq_* unused).
 * Per `agc_block` (the firmware block):
 * mic = L of the L = R frames -> fi = fir_q15 (mic, taps_i), fq = fir_q15 (mic, taps_q)
 * -> rail order: lsb = 1 (LSB, CW-R) (I, Q) = (fi, fq); lsb = 0 (USB, CW, DIG, PKT) (I, Q) = (fq, fi)
 *    (with the frozen pair taps_i = a cos phi, taps_q = -a sin phi: fi + j fq = conj (c * mic) for the one-sided band-pass c, so the
 *    swap gives j (c * mic), the upper sideband: USB puts the mic tone at +f of I + jQ)
 * -> block peak p_b = max (max_q15 (abs_q15 (I)), max_q15 (abs_q15 (Q)))
 * -> the finite-window gain law of rx_ssb_q15 unchanged (q, s)
 * -> scale_q15 (I, q >> s, s), scale_q15 (Q, q >> s, s) -> written interleaved I, Q.
 * frames % agc_block == 0. iq_dbg (optional): the pre-ALC (I, Q) [frames][2] after the rail order; gain_dbg (optional): q per block. */
void SLO (tx_ssb_q15) (const slo_rx_q15_params *p, slo_rx_q15_state *st, const int16_t *in_lr, int16_t *out_iq,
                       int16_t *iq_dbg, uint32_t *gain_dbg, uint32_t frames);

#ifdef __cplusplus
}
#endif
#endif /* SLO_TX_Q15_H */
