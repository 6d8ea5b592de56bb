/* ORACLE / TEST INFRASTRUCTURE ONLY — never on the product path.
 *
 * The all-mode integer transmitter of slo_tx_q15_mod.h, written with SLO(stage) calls like chains.inc.c so that each box is the CMSIS
 * routine of the library it is compiled into. THE COMPOSITION IS OURS (DESIGN.md §3.9), as are the gain law and the phase accumulator;
 * the reference firmware has no modulator.
 */
#include <string.h>
#include "slo_tx_q15_mod.h"

#define SLO_TXQ_W (SLO_Q15_TAPS + 48)                    /* the window of one block: 64 carried mic samples + 48 */

void SLO (tx_q15) (const slo_tx_q15m_params *p, slo_tx_q15m_state *st, const int16_t *in_lr, int16_t *out_iq,
                   int16_t *iq_dbg, uint32_t *gain_dbg, uint32_t *phase_dbg, uint32_t frames)
{
  const uint32_t T = SLO_Q15_TAPS, B = p->q.agc_block, K = p->q.agc_window;
  const int ssb = p->kind == 0;
  const int16_t *ti = p->kind == 1 ? p->am_taps : (p->kind == 2 ? p->fm_taps : p->q.taps_i);
  const int16_t target = p->kind == 1 ? p->am_depth : (p->kind == 2 ? p->fm_target : p->q.agc_target);
  int16_t ci[SLO_Q15_TAPS], cq[SLO_Q15_TAPS];
  int16_t w[SLO_TXQ_W], fi[SLO_TXQ_W], fq[SLO_TXQ_W], zs[SLO_Q15_TAPS + SLO_TXQ_W];
  int16_t ab[48], yi[48], yq[48], car[48], zero[48];
  uint32_t phi[48];
  for (uint32_t k = 0; k < T; k++) { ci[k] = ti[T - 1 - k]; cq[k] = p->q.taps_q[T - 1 - k]; }   /* arm_fir_q15.c: pCoeffs time-reversed */
  for (uint32_t k = 0; k < B; k++) { car[k] = p->am_carrier; zero[k] = 0; }

  for (uint32_t o = 0; o < frames; o += B)
  {
    memcpy (w, st->raw, T * 2);
    for (uint32_t k = 0; k < B; k++) w[T + k] = in_lr[2 * (size_t) (o + k)];                    /* L channel (codec_if.c:304-306) */
    /* the FIR over the whole window from a zero state: outputs T .. T + B - 1 (frames 0 .. 47) see 64 frames each */
    memset (zs, 0, sizeof zs); SLO (fir_q15) (ci, T, zs, w, fi, T + B, T + B);
    if (ssb) { memset (zs, 0, sizeof zs); SLO (fir_q15) (cq, T, zs, w, fq, T + B, T + B); }
    /* SSB: the sideband is the rail order (tx_ssb_q15); AM / FM: one rail a, and Q = 0 before the modulator */
    const int16_t *I = ssb ? (p->q.lsb ? fi + T : fq + T) : fi + T, *Q = ssb ? (p->q.lsb ? fq + T : fi + T) : zero;
    if (iq_dbg)
      for (uint32_t k = 0; k < B; k++) { iq_dbg[2 * (size_t) (o + k)] = I[k]; iq_dbg[2 * (size_t) (o + k) + 1] = Q[k]; }
    SLO (abs_q15) (I, ab, B);
    int32_t peak = SLO (max_q15) (ab, B, 0);
    if (ssb)
    {
      SLO (abs_q15) (Q, ab, B);
      const int32_t pq = SLO (max_q15) (ab, B, 0);
      if (pq > peak) peak = pq;
    }
    /* ALC law = the AGC law of rx_ssb_q15 (ours) with the modulator's target: finite-window peak hold with a q15 release table */
    int32_t env = peak;
    for (uint32_t j = 1; j < K; j++)
    {
      const int32_t v = ((int32_t) st->peaks[j - 1] * (int32_t) p->q.rel[j]) >> 15;
      if (v > env) env = v;
    }
    for (uint32_t j = SLO_Q15_WIN - 1; j > 0; j--) st->peaks[j] = st->peaks[j - 1];
    st->peaks[0] = (int16_t) peak;
    const uint32_t den = (uint32_t) (env > p->q.agc_floor ? env : p->q.agc_floor);
    uint32_t q = ((uint32_t) target << 15) / den;
    if (q > p->q.agc_gmax_q15) q = p->q.agc_gmax_q15;
    uint32_t s = 0;
    while ((q >> s) > 32767u) s++;
    if (gain_dbg) gain_dbg[o / B] = q;
    SLO (scale_q15) (I, (int16_t) (q >> s), (int32_t) s, yi, B);
    if (ssb) SLO (scale_q15) (Q, (int16_t) (q >> s), (int32_t) s, yq, B);
    else if (p->kind == 1)
    {
      /* AM: the carrier plus y scaled by it, saturating; |y| <= am_depth keeps the envelope in am_carrier (1 +- am_depth) */
      SLO (scale_q15) (yi, p->am_carrier, 0, yq, B);
      SLO (add_q15) (yq, car, yi, B);
      memset (yq, 0, B * 2);
    }
    else
    {
      /* FM (ours): integer phase accumulator, wraps modulo one turn exactly; |y fm_inc| < 2^31 */
      for (uint32_t k = 0; k < B; k++) { st->phase += (uint32_t) ((int32_t) yi[k] * p->fm_inc); phi[k] = st->phase; }
      int16_t iq[2 * 48];
      SLO (tx_fm_nco) (phi, B, p->fm_level, iq);
      for (uint32_t k = 0; k < B; k++) { yi[k] = iq[2 * k]; yq[k] = iq[2 * k + 1]; }
    }
    if (phase_dbg)
      for (uint32_t k = 0; k < B; k++) phase_dbg[o + k] = p->kind == 2 ? phi[k] : st->phase;
    for (uint32_t k = 0; k < B; k++) { out_iq[2 * (size_t) (o + k)] = yi[k]; out_iq[2 * (size_t) (o + k) + 1] = yq[k]; }
    memcpy (st->raw, w + B, T * 2);                                                               /* the last 64 mic samples */
  }
}
