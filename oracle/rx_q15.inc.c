/* ORACLE / TEST INFRASTRUCTURE ONLY — never on the product path.
 *
 * The all-mode integer receiver of slo_rx_q15.h, written with SLO(stage) calls like chains.inc.c so that each box is the CMSIS routine of
 * the library it is compiled into. THE COMPOSITION IS OURS (DESIGN.md §3.8), as are the FM discriminator and the gain law.
 */
#include <string.h>
#include "slo_rx_q15.h"

#define SLO_RXQ_W (SLO_Q15_TAPS + 48)                    /* the window of one block: 64 carried frames + 48 */

void SLO (rx_q15) (const slo_rx_q15m_params *p, slo_rx_q15m_state *st, const int16_t *in_iq, int16_t *out_lr,
                   int16_t *audio_dbg, uint32_t *gain_dbg, uint32_t frames)
{
  const uint32_t T = SLO_Q15_TAPS, B = p->q.agc_block, K = p->q.agc_window;
  const int16_t *ti = p->kind == 1 ? p->am_taps : (p->kind == 2 ? p->fm_taps : p->q.taps_i);
  const int16_t *tq = p->kind == 1 ? p->am_taps : (p->kind == 2 ? p->fm_taps : p->q.taps_q);
  int16_t ci[SLO_Q15_TAPS], cq[SLO_Q15_TAPS];
  int16_t wi[SLO_RXQ_W], wq[SLO_RXQ_W], fi[SLO_RXQ_W], fq[SLO_RXQ_W], zs[SLO_Q15_TAPS + SLO_RXQ_W];
  int16_t ab[2 * SLO_RXQ_W], mag[SLO_RXQ_W], v[48], av[48], y[48];
  for (uint32_t k = 0; k < T; k++) { ci[k] = ti[T - 1 - k]; cq[k] = tq[T - 1 - k]; }   /* arm_fir_q15.c: pCoeffs time-reversed */

  for (uint32_t o = 0; o < frames; o += B)
  {
    memcpy (wi, st->raw_i, T * 2); memcpy (wq, st->raw_q, T * 2);
    for (uint32_t k = 0; k < B; k++) { wi[T + k] = in_iq[2 * (size_t) (o + k)]; wq[T + k] = in_iq[2 * (size_t) (o + k) + 1]; }
    /* the FIR over the whole window from a zero state: outputs T - 1 .. T + B - 1 (frames -1 .. 47) see 64 frames each */
    memset (zs, 0, sizeof zs); SLO (fir_q15) (ci, T, zs, wi, fi, T + B, T + B);
    memset (zs, 0, sizeof zs); SLO (fir_q15) (cq, T, zs, wq, fq, T + B, T + B);
    const int16_t *a = fi + T, *b = fq + T;                                                     /* a[-1], b[-1] exist */
    if (p->kind == 0)
    {
      if (p->q.lsb) SLO (sub_q15) (a, b, v, B); else SLO (add_q15) (a, b, v, B);
    }
    else
    {
      for (uint32_t k = 0; k <= B; k++) { ab[2 * k] = a[(int) k - 1]; ab[2 * k + 1] = b[(int) k - 1]; }
      SLO (cmplx_mag_q15) (ab, mag, B + 1);                                                    /* mag[k] = |z[k - 1]| (2.14) */
      for (uint32_t k = 0; k < B; k++)
      {
        if (p->kind == 1) { v[k] = mag[k + 1]; continue; }
        /* limiter-discriminator (ours): q15 sin of the phase step, sign of Im (z[n] conj z[n-1]) */
        const int64_t x = (int64_t) a[(int) k - 1] * b[k] - (int64_t) b[(int) k - 1] * a[k];
        int64_t den = (int64_t) mag[k] * mag[k + 1];
        if (den < p->fm_floor) den = p->fm_floor;
        const int64_t d = (x * 8192) / den;
        v[k] = (int16_t) (d > 32767 ? 32767 : (d < -32768 ? -32768 : d));
      }
    }
    if (audio_dbg) memcpy (audio_dbg + o, v, B * 2);
    SLO (abs_q15) (v, av, B);
    const int32_t peak = SLO (max_q15) (av, B, 0);
    /* AGC law of rx_ssb_q15 (ours): finite-window peak hold with a q15 release table */
    int32_t env = peak;
    for (uint32_t j = 1; j < K; j++)
    {
      const int32_t e = ((int32_t) st->peaks[j - 1] * (int32_t) p->q.rel[j]) >> 15;
      if (e > env) env = e;
    }
    for (uint32_t j = SLO_Q15_WIN - 1; j > 0; j--) st->peaks[j] = st->peaks[j - 1];
    st->peaks[0] = (int16_t) peak;
    const uint32_t den = (uint32_t) (env > p->q.agc_floor ? env : p->q.agc_floor);
    uint32_t q = ((uint32_t) p->q.agc_target << 15) / den;
    if (q > p->q.agc_gmax_q15) q = p->q.agc_gmax_q15;
    uint32_t s = 0;
    while ((q >> s) > 32767u) s++;
    if (gain_dbg) gain_dbg[o / B] = q;
    SLO (scale_q15) (v, (int16_t) (q >> s), (int32_t) s, y, B);
    for (uint32_t k = 0; k < B; k++) { out_lr[2 * (size_t) (o + k)] = y[k]; out_lr[2 * (size_t) (o + k) + 1] = y[k]; }
    memcpy (st->raw_i, wi + B, T * 2); memcpy (st->raw_q, wq + B, T * 2);                      /* the last 64 frames */
  }
}
