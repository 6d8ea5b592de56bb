/* ORACLE / TEST INFRASTRUCTURE ONLY — never on the product path.
 *
 * The integer SSB modulator of slo_tx_q15.h, written with SLO(stage) calls like chains.inc.c so that each box is the CMSIS routine of
 * the library it is compiled into. THE COMPOSITION IS OURS (DESIGN.md §3.7); the reference firmware has no modulator.
 */
#include <string.h>
#include "slo_tx_q15.h"

void SLO (tx_ssb_q15) (const slo_rx_q15_params *p, slo_rx_q15_state *st, const int16_t *in_lr, int16_t *out_iq,
                       int16_t *iq_dbg, uint32_t *gain_dbg, uint32_t frames)
{
  const uint32_t T = p->ntaps, B = p->agc_block, K = p->agc_window;
  int16_t ci[SLO_Q15_TAPS], cq[SLO_Q15_TAPS];
  int16_t mic[SLO_Q15_MAX_BLOCK], fi[SLO_Q15_MAX_BLOCK], fq[SLO_Q15_MAX_BLOCK], ab[SLO_Q15_MAX_BLOCK];
  int16_t yi[SLO_Q15_MAX_BLOCK], yq[SLO_Q15_MAX_BLOCK];
  for (uint32_t k = 0; k < T; k++) { ci[k] = p->taps_i[T - 1 - k]; cq[k] = p->taps_q[T - 1 - k]; }   /* arm_fir_q15.c: pCoeffs time-reversed */

  for (uint32_t o = 0; o < frames; o += B)
  {
    for (uint32_t k = 0; k < B; k++) mic[k] = in_lr[2 * (size_t) (o + k)];                            /* L channel (codec_if.c:304-306) */
    SLO (fir_q15) (ci, T, st->fir_i, mic, fi, B, B);
    SLO (fir_q15) (cq, T, st->fir_q, mic, fq, B, B);
    const int16_t *I = p->lsb ? fi : fq, *Q = p->lsb ? fq : fi;                                      /* the sideband is the rail order */
    if (iq_dbg)
      for (uint32_t k = 0; k < B; k++) { iq_dbg[2 * (size_t) (o + k)] = I[k]; iq_dbg[2 * (size_t) (o + k) + 1] = Q[k]; }
    SLO (abs_q15) (I, ab, B);
    const int32_t pi = SLO (max_q15) (ab, B, 0);
    SLO (abs_q15) (Q, ab, B);
    const int32_t pq = SLO (max_q15) (ab, B, 0);
    const int32_t peak = pi > pq ? pi : pq;
    /* ALC law = the AGC law of rx_ssb_q15 (ours): finite-window peak hold with a q15 release table */
    int32_t env = peak;
    for (uint32_t j = 1; j < K; j++)
    {
      const int32_t v = ((int32_t) st->peaks[j - 1] * (int32_t) p->rel[j]) >> 15;
      if (v > env) env = v;
    }
    for (uint32_t j = SLO_Q15_WIN - 1; j > 0; j--) st->peaks[j] = st->peaks[j - 1];
    st->peaks[0] = (int16_t) peak;
    const uint32_t den = (uint32_t) (env > p->agc_floor ? env : p->agc_floor);
    uint32_t q = ((uint32_t) p->agc_target << 15) / den;
    if (q > p->agc_gmax_q15) q = p->agc_gmax_q15;
    uint32_t s = 0;
    while ((q >> s) > 32767u) s++;
    if (gain_dbg) gain_dbg[o / B] = q;
    SLO (scale_q15) (I, (int16_t) (q >> s), (int32_t) s, yi, B);
    SLO (scale_q15) (Q, (int16_t) (q >> s), (int32_t) s, yq, B);
    for (uint32_t k = 0; k < B; k++) { out_iq[2 * (size_t) (o + k)] = yi[k]; out_iq[2 * (size_t) (o + k) + 1] = yq[k]; }
  }
}
