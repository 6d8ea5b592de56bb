/* ORACLE / TEST INFRASTRUCTURE ONLY — never on the product path.
 *
 * The tuner of slo_tune.h, written with SLO(stage) calls like chains.inc.c so that each box is the CMSIS routine of the library it is
 * compiled into. THE COMPOSITION IS OURS (DESIGN.md §3.5).
 */
#include <stdlib.h>
#include "slo_tune.h"

void SLO (tune_q15) (const int16_t *in, int16_t *out, uint32_t frames, int32_t inc, uint32_t *phase, int up)
{
  const size_t n = frames;
  int32_t *ph = (int32_t *) malloc (sizeof (int32_t) * (n ? n : 1));
  float *x = (float *) malloc (sizeof (float) * (n ? n : 1)), *c = (float *) malloc (sizeof (float) * (n ? n : 1)), *s = (float *) malloc (sizeof (float) * (n ? n : 1));
  float *w = (float *) malloc (sizeof (float) * 2 * (n ? n : 1)), *z = (float *) malloc (sizeof (float) * 2 * (n ? n : 1));
  const uint32_t phi0 = *phase;
  for (size_t k = 0; k < n; k++) ph[k] = (int32_t) (phi0 + (uint32_t) k * (uint32_t) inc);   /* integer phase: exact, wraps modulo one turn */
  SLO (q31_to_float) (ph, x, frames);                                                       /* phase as a signed fraction of half a turn */
  SLO (scale_f32) (x, 3.14159265f, x, frames);
  SLO (cos_f32) (x, c, frames);
  SLO (sin_f32) (x, s, frames);
  for (size_t k = 0; k < n; k++) { w[2 * k] = c[k]; w[2 * k + 1] = s[k]; }
  if (!up) SLO (cmplx_conj_f32) (w, w, frames);
  SLO (q15_to_float) (in, z, 2 * frames);
  SLO (cmplx_mult_cmplx_f32) (z, w, z, frames);
  SLO (float_to_q15) (z, out, 2 * frames);
  *phase = phi0 + frames * (uint32_t) inc;
  free (ph); free (x); free (c); free (s); free (w); free (z);
}
