/* ORACLE / TEST INFRASTRUCTURE ONLY — never on the product path.
 *
 * The AM / FM transmit composition of slo_tx_mod.h, written with SLO(stage) calls like chains.inc.c so that each box is the CMSIS
 * routine of the library it is compiled into. THE COMPOSITION IS OURS (DESIGN.md §3.4); the reference firmware has no modulator.
 */
#include <string.h>
#include <stdlib.h>
#include "slo_tx_mod.h"

void SLO (tx_fm_nco) (const uint32_t *phase, uint32_t n, float level, int16_t *out_iq)
{
  float *x = (float *) malloc (sizeof (float) * n), *c = (float *) malloc (sizeof (float) * n), *s = (float *) malloc (sizeof (float) * n);
  int16_t *ci = (int16_t *) malloc (sizeof (int16_t) * n), *si = (int16_t *) malloc (sizeof (int16_t) * n);
  SLO (q31_to_float) ((const int32_t *) phase, x, n);                    /* phase as a signed fraction of half a turn */
  SLO (scale_f32) (x, 3.14159265f, x, n);
  SLO (cos_f32) (x, c, n);
  SLO (sin_f32) (x, s, n);
  SLO (scale_f32) (c, level, c, n);
  SLO (scale_f32) (s, level, s, n);
  SLO (float_to_q15) (c, ci, n);
  SLO (float_to_q15) (s, si, n);
  for (uint32_t k = 0; k < n; k++) { out_iq[2 * (size_t) k] = ci[k]; out_iq[2 * (size_t) k + 1] = si[k]; }
  free (x); free (c); free (s); free (ci); free (si);
}

void SLO (tx_mod_f32) (const slo_tx_mod_params *p, slo_tx_mod_state *st, const int16_t *in_lr, int16_t *out_iq,
                       float *iq_dbg, float *gain_dbg, uint32_t *phase_dbg, uint32_t frames)
{
  const uint32_t N = p->fft_len, hop = p->hop, ovl = N - hop, B = p->alc_block;
  const float target = (p->modulator == SLO_MOD_AM) ? p->am_depth : 2.0f * p->fm_deviation_hz / (float) p->fs;
  int16_t *raw = (int16_t *) malloc (sizeof (int16_t) * N);
  float *mic = (float *) malloc (sizeof (float) * N);
  float *frame = (float *) malloc (sizeof (float) * 2 * N);
  float *prod = (float *) malloc (sizeof (float) * 2 * N);
  float *a = (float *) malloc (sizeof (float) * hop), *u = (float *) malloc (sizeof (float) * hop);
  float *absb = (float *) malloc (sizeof (float) * B);
  int16_t *i16 = (int16_t *) malloc (sizeof (int16_t) * hop);
  int32_t *inc = (int32_t *) malloc (sizeof (int32_t) * hop);
  uint32_t *phi = (uint32_t *) malloc (sizeof (uint32_t) * hop);

  for (uint32_t o = 0; o < frames; o += hop)
  {
    /* front end: tx_ssb_f32's */
    memcpy (raw, st->ovl, sizeof (int16_t) * ovl);
    for (uint32_t k = 0; k < hop; k++) raw[ovl + k] = in_lr[2 * (size_t) (o + k)];   /* L channel */
    memcpy (st->ovl, raw + hop, sizeof (int16_t) * ovl);
    SLO (q15_to_float) (raw, mic, N);
    for (uint32_t k = 0; k < N; k++) { frame[2 * k] = mic[k]; frame[2 * k + 1] = 0.0f; }
    SLO (cfft_f32) (frame, N, 0, 1);
    SLO (cmplx_mult_cmplx_f32) (frame, p->mask, prod, N);
    SLO (cfft_f32) (prod, N, 1, 1);
    const float *iq = prod + 2 * ovl;                                      /* keep last hop */
    if (iq_dbg) memcpy (iq_dbg + 2 * (size_t) o, iq, sizeof (float) * 2 * hop);
    for (uint32_t k = 0; k < hop; k++) a[k] = iq[2 * k];                   /* the real part carries the (band-limited) audio */

    for (uint32_t b = 0; b < hop; b += B)
    {
      SLO (abs_f32) (a + b, absb, B);
      float peak = SLO (max_f32) (absb, B, 0);
      /* the ALC law of tx_ssb_f32 (ours) with the modulator's target */
      float rel = st->env * p->alc_decay;
      float env = peak > rel ? peak : rel;
      float den = env > p->alc_floor ? env : p->alc_floor;
      float g = target / den;
      if (g > p->alc_gmax) g = p->alc_gmax;
      st->env = env;
      if (gain_dbg) gain_dbg[(o + b) / B] = g;
      SLO (scale_f32) (a + b, g, u + b, B);
    }
    if (p->modulator == SLO_MOD_AM)
    {
      SLO (offset_f32) (u, 1.0f, u, hop);
      SLO (scale_f32) (u, p->am_carrier, u, hop);
      SLO (float_to_q15) (u, i16, hop);
      for (uint32_t k = 0; k < hop; k++) { out_iq[2 * (size_t) (o + k)] = i16[k]; out_iq[2 * (size_t) (o + k) + 1] = 0; }
    }
    else
    {
      /* integer phase accumulator: wraps modulo one turn exactly, and is associative (a parallel prefix sum reproduces it) */
      SLO (float_to_q31) (u, inc, hop);
      for (uint32_t k = 0; k < hop; k++) { st->phase += (uint32_t) inc[k]; phi[k] = st->phase; }
      if (phase_dbg) memcpy (phase_dbg + o, phi, sizeof (uint32_t) * hop);
      SLO (tx_fm_nco) (phi, hop, p->fm_level, out_iq + 2 * (size_t) o);
    }
  }
  free (raw); free (mic); free (frame); free (prod); free (a); free (u); free (absb); free (i16); free (inc); free (phi);
}
