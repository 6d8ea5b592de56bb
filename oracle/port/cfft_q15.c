/* ORACLE / TEST INFRASTRUCTURE ONLY. arm_cfft_q15 (Source/TransformFunctions/arm_cfft_q15.c:77) in the ARM_MATH_DSP branch the firmware's
 * Cortex-M4 build compiles (arm_cfft_radix4_q15.c:156-560, arm_cfft_q15.c:134-236): the branch of ref_cfft_q15_cm4
 * (../ref_glue/cm4_fft_q15.c) and of tests/fft_fixed_model.py, NOT the shift-based C branch that ref_cfft_q15 compiles. With it the port
 * is no longer without a q15 FFT (fft.c keeps the float transforms); pinned bit for bit to tests/golden/cfft_fixed.npz and to that model
 * by tests/test_chan64_q15_oracle.py. Twiddles are regenerated (floor (v 2^15) clipped to q15, the rule of arm_common_tables.c). */
#include "port_common.h"

/* ---- arm_cfft_q15, ARM_MATH_DSP branch. A q15 complex word is a pair of lanes (x = real, y = imaginary): saturating (__QADD16,
 * __QSUB16, __QASX, __QSAX) and halving (__SHADD16, __SHSUB16, __SHASX, __SHSAX) lane adds; twiddle products keep the high half-word
 * of a wrapping 32-bit sum of two 16 x 16 products (__SMUAD, __SMUSDX forward; __SMUSD, __SMUADX inverse). */
typedef struct { int32_t x, y; } slo_c16;
static inline slo_c16 c16_qadd (slo_c16 a, slo_c16 b) { slo_c16 r = { slo_ssat16 (a.x + b.x), slo_ssat16 (a.y + b.y) }; return r; }
static inline slo_c16 c16_qsub (slo_c16 a, slo_c16 b) { slo_c16 r = { slo_ssat16 (a.x - b.x), slo_ssat16 (a.y - b.y) }; return r; }
static inline slo_c16 c16_hadd (slo_c16 a, slo_c16 b) { slo_c16 r = { (a.x + b.x) >> 1, (a.y + b.y) >> 1 }; return r; }
static inline slo_c16 c16_hsub (slo_c16 a, slo_c16 b) { slo_c16 r = { (a.x - b.x) >> 1, (a.y - b.y) >> 1 }; return r; }
static inline slo_c16 c16_qasx (slo_c16 a, slo_c16 b) { slo_c16 r = { slo_ssat16 (a.x - b.y), slo_ssat16 (a.y + b.x) }; return r; }
static inline slo_c16 c16_qsax (slo_c16 a, slo_c16 b) { slo_c16 r = { slo_ssat16 (a.x + b.y), slo_ssat16 (a.y - b.x) }; return r; }
static inline slo_c16 c16_hasx (slo_c16 a, slo_c16 b) { slo_c16 r = { (a.x - b.y) >> 1, (a.y + b.x) >> 1 }; return r; }
static inline slo_c16 c16_hsax (slo_c16 a, slo_c16 b) { slo_c16 r = { (a.x + b.y) >> 1, (a.y - b.x) >> 1 }; return r; }
static inline slo_c16 c16_shr (slo_c16 a, int s) { slo_c16 r = { a.x >> s, a.y >> s }; return r; }
static inline int32_t slo_wrap32 (int64_t v) { return (int32_t) (uint32_t) (uint64_t) v; }
static inline slo_c16 c16_twid (slo_c16 c, slo_c16 v, int inv)
{
  const int32_t re = slo_wrap32 (inv ? (int64_t) c.x * v.x - (int64_t) c.y * v.y : (int64_t) c.x * v.x + (int64_t) c.y * v.y);
  const int32_t im = slo_wrap32 (inv ? (int64_t) c.x * v.y + (int64_t) c.y * v.x : (int64_t) c.x * v.y - (int64_t) c.y * v.x);
  slo_c16 r = { (int16_t) (re >> 16), im >> 16 }; return r;
}

/* arm_radix4_butterfly_{,inverse_}q15 on z[0..L), twiddle index step `mod` on the table of the full length (tw: (cos, sin) pairs) */
static void slo_radix4_q15 (slo_c16 *z, uint32_t L, uint32_t mod, const slo_c16 *tw, int inv)
{
  uint32_t n2 = L >> 2, ic = 0;
  for (uint32_t i0 = 0; i0 < n2; i0++, ic += mod)                      /* first stage: inputs >> 2, saturating sums */
  {
    slo_c16 *p0 = z + i0, *p1 = p0 + n2, *p2 = p1 + n2, *p3 = p2 + n2;
    const slo_c16 a = c16_shr (*p0, 2), b = c16_shr (*p1, 2), c = c16_shr (*p2, 2), d = c16_shr (*p3, 2);
    const slo_c16 R = c16_qadd (a, c), S = c16_qsub (a, c), T = c16_qadd (b, d), T2 = c16_qsub (b, d);
    *p0 = c16_hadd (R, T);
    *p1 = c16_twid (tw[2 * ic], c16_qsub (R, T), inv);
    *p2 = c16_twid (tw[ic], inv ? c16_qasx (S, T2) : c16_qsax (S, T2), inv);
    *p3 = c16_twid (tw[3 * ic], inv ? c16_qsax (S, T2) : c16_qasx (S, T2), inv);
  }
  mod <<= 2;
  for (uint32_t k = L >> 2; k > 4; k >>= 2, mod <<= 2)                 /* middle stages: every output halved twice */
  {
    const uint32_t n1 = n2;
    n2 >>= 2;
    for (uint32_t j = 0; j < n2; j++)
      for (uint32_t i0 = j; i0 < L; i0 += n1)
      {
        const uint32_t icj = j * mod;
        slo_c16 *p0 = z + i0, *p1 = p0 + n2, *p2 = p1 + n2, *p3 = p2 + n2;
        const slo_c16 a = *p0, b = *p1, c = *p2, d = *p3;
        const slo_c16 R = c16_qadd (a, c), S = c16_qsub (a, c), T = c16_qadd (b, d), T2 = c16_qsub (b, d);
        *p0 = c16_shr (c16_hadd (R, T), 1);
        *p1 = c16_twid (tw[2 * icj], c16_hsub (R, T), inv);
        *p2 = c16_twid (tw[icj], inv ? c16_hasx (S, T2) : c16_hsax (S, T2), inv);
        *p3 = c16_twid (tw[3 * icj], inv ? c16_hsax (S, T2) : c16_hasx (S, T2), inv);
      }
  }
  for (uint32_t i0 = 0; i0 < L; i0 += 4)                               /* last stage: four neighbours, no twiddles */
  {
    slo_c16 *p = z + i0;
    const slo_c16 R = c16_qadd (p[0], p[2]), T = c16_qadd (p[1], p[3]), S = c16_qsub (p[0], p[2]), U = c16_qsub (p[1], p[3]);
    p[0] = c16_hadd (R, T); p[1] = c16_hsub (R, T);
    p[2] = inv ? c16_hasx (S, U) : c16_hsax (S, U);
    p[3] = inv ? c16_hsax (S, U) : c16_hasx (S, U);
  }
}

void port_cfft_q15 (int16_t *d, uint32_t N, int ifft, int bitrev)
{
  slo_c16 *z = (slo_c16 *) malloc (sizeof (slo_c16) * N), *tw = (slo_c16 *) malloc (sizeof (slo_c16) * (3 * N / 4));
  for (uint32_t k = 0; k < 3 * N / 4; k++)                             /* twiddleCoef_N_q15: floor (v 2^15) clipped to q15 */
  {
    const double a = 2.0 * M_PI * (double) k / (double) N, cs = floor (cos (a) * 32768.0), sn = floor (sin (a) * 32768.0);
    tw[k].x = (int32_t) (cs > 32767.0 ? 32767.0 : cs); tw[k].y = (int32_t) (sn > 32767.0 ? 32767.0 : sn);
  }
  for (uint32_t i = 0; i < N; i++) { z[i].x = d[2 * i]; z[i].y = d[2 * i + 1]; }
  uint32_t log2n = 0;
  while ((1u << log2n) < N) log2n++;
  if ((log2n & 1) == 0) slo_radix4_q15 (z, N, 1, tw, ifft);
  else
  {
    /* arm_cfft_radix4by2_{,inverse_}q15: halve both halves, saturating difference times W^i, two half-length transforms on the same
     * table with step 2, then p <<= 1 stored back into a q15_t (wraps) */
    const uint32_t n2 = N >> 1;
    for (uint32_t i = 0; i < n2; i++)
    {
      const slo_c16 T = c16_shr (z[i], 1), S = c16_shr (z[i + n2], 1);
      z[i] = c16_hadd (T, S);
      z[i + n2] = c16_twid (tw[i], c16_qsub (T, S), ifft);
    }
    slo_radix4_q15 (z, n2, 2, tw, ifft);
    slo_radix4_q15 (z + n2, n2, 2, tw, ifft);
    for (uint32_t i = 0; i < N; i++) { z[i].x = (int16_t) (z[i].x << 1); z[i].y = (int16_t) (z[i].y << 1); }
  }
  for (uint32_t i = 0; i < N; i++)                                     /* arm_bitreversal_16: natural order */
  {
    uint32_t j = 0;
    for (uint32_t b = 0; b < log2n; b++) j |= ((i >> b) & 1u) << (log2n - 1 - b);
    const uint32_t src = bitrev ? j : i;
    d[2 * i] = (int16_t) z[src].x; d[2 * i + 1] = (int16_t) z[src].y;
  }
  free (z); free (tw);
}
