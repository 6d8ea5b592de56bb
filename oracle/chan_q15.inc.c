/* ORACLE / TEST INFRASTRUCTURE ONLY — never on the product path.
 *
 * The integer channelizer of slo_chan_q15.h, written with SLO(stage) calls like chains.inc.c (chan_f32 is its float twin, box for box).
 * THE COMPOSITION IS OURS (DESIGN.md §3.10), as is the gain law.
 */
#include <string.h>
#include <stdlib.h>
#include "slo_chan_q15.h"

void SLO (chan_q15) (const slo_chan_q15_params *p, slo_chan_q15_state *st, const int16_t *in_iq, int16_t *out_lr,
                     int16_t *audio_dbg, uint32_t *gain_dbg, uint32_t frames)
{
  const uint32_t M = p->bins, P = p->taps_per_branch, B = p->agc_block, K = p->agc_window, hops = frames / M;
  int16_t *bi = (int16_t *) malloc (sizeof (int16_t) * hops), *bq = (int16_t *) malloc (sizeof (int16_t) * hops);
  int16_t *vi = (int16_t *) malloc (sizeof (int16_t) * (size_t) M * hops), *vq = (int16_t *) malloc (sizeof (int16_t) * (size_t) M * hops);
  int16_t *fstate = (int16_t *) malloc (sizeof (int16_t) * (P + hops));
  int16_t coef[SLO_CHAN_TAPS], spec[2 * SLO_CHAN_BINS], magb[SLO_CHAN_BINS];
  int16_t *audio = (int16_t *) malloc (sizeof (int16_t) * (size_t) M * hops);
  int16_t absb[SLO_Q15_MAX_BLOCK], y[SLO_Q15_MAX_BLOCK];

  for (uint32_t r = 0; r < M; r++)
  {
    /* branch taps e_r[p] = h[M p + M-1-r], handed to CMSIS time-reversed (arm_fir_q15.c: pCoeffs) */
    for (uint32_t k = 0; k < P; k++) coef[k] = p->proto[M * (P - 1 - k) + (M - 1 - r)];
    for (uint32_t m = 0; m < hops; m++) { bi[m] = in_iq[2 * ((size_t) M * m + r)]; bq[m] = in_iq[2 * ((size_t) M * m + r) + 1]; }
    memset (fstate, 0, sizeof (int16_t) * (P + hops)); memcpy (fstate, st->fir_i[r], sizeof (int16_t) * (P - 1));
    SLO (fir_q15) (coef, P, fstate, bi, vi + (size_t) r * hops, hops, B);
    memcpy (st->fir_i[r], fstate, sizeof (int16_t) * (P - 1));
    memset (fstate, 0, sizeof (int16_t) * (P + hops)); memcpy (fstate, st->fir_q[r], sizeof (int16_t) * (P - 1));
    SLO (fir_q15) (coef, P, fstate, bq, vq + (size_t) r * hops, hops, B);
    memcpy (st->fir_q[r], fstate, sizeof (int16_t) * (P - 1));
  }
  for (uint32_t m = 0; m < hops; m++)
  {
    for (uint32_t r = 0; r < M; r++) { spec[2 * r] = vi[(size_t) r * hops + m]; spec[2 * r + 1] = vq[(size_t) r * hops + m]; }
    SLO (cfft_q15) (spec, M, 0, 1);
    if (p->envelope) { SLO (cmplx_mag_q15) (spec, magb, M); for (uint32_t k = 0; k < M; k++) audio[(size_t) k * hops + m] = magb[k]; }
    else for (uint32_t k = 0; k < M; k++) audio[(size_t) k * hops + m] = spec[2 * k];
  }
  if (audio_dbg) memcpy (audio_dbg, audio, sizeof (int16_t) * (size_t) M * hops);
  for (uint32_t k = 0; k < M; k++)
    for (uint32_t b = 0; b < hops; b += B)
    {
      const int16_t *a = audio + (size_t) k * hops + b;
      SLO (abs_q15) (a, absb, B);
      const int32_t peak = SLO (max_q15) (absb, B, 0);
      /* AGC law of rx_ssb_q15 (ours): finite-window peak hold with a q15 release table */
      int32_t env = peak;
      for (uint32_t j = 1; j < K; j++)
      {
        const int32_t v = ((int32_t) st->peaks[k][j - 1] * (int32_t) p->rel[j]) >> 15;
        if (v > env) env = v;
      }
      for (uint32_t j = SLO_Q15_WIN - 1; j > 0; j--) st->peaks[k][j] = st->peaks[k][j - 1];
      st->peaks[k][0] = (int16_t) peak;
      const uint32_t den = (uint32_t) (env > p->agc_floor ? env : p->agc_floor);
      uint32_t q = ((uint32_t) p->agc_target << 15) / den;
      if (q > p->agc_gmax_q15) q = p->agc_gmax_q15;
      uint32_t s = 0;
      while ((q >> s) > 32767u) s++;
      if (gain_dbg) gain_dbg[(size_t) k * (hops / B) + b / B] = q;
      SLO (scale_q15) (a, (int16_t) (q >> s), (int32_t) s, y, B);
      for (uint32_t i = 0; i < B; i++) { out_lr[2 * ((size_t) k * hops + b + i)] = y[i]; out_lr[2 * ((size_t) k * hops + b + i) + 1] = y[i]; }
    }
  free (bi); free (bq); free (vi); free (vq); free (fstate); free (audio);
}
