/* ORACLE / TEST INFRASTRUCTURE ONLY. The stages the transmit modulators add, restated, and the port_ instantiation of
 * ../tx_mod.inc.c. Paths are relative to Drivers/CMSIS/DSP/ of the reference tree (CMSIS-DSP V1.5.3). */
#include "port_common.h"
#include "../slo_tx_mod.h"

/* Source/BasicMathFunctions/arm_offset_f32.c (plain-C loop) : *pDst++ = (*pSrc++) + offset */
void port_offset_f32 (const float *s, float offset, float *d, uint32_t n) { for (uint32_t i = 0; i < n; i++) d[i] = s[i] + offset; }

/* Source/SupportFunctions/arm_float_to_q31.c, ARM_MATH_ROUNDING not defined: clip_q63_to_q31 ((q63_t) (*pIn++ * 2147483648.0f)).
 * The product is exact (power of two); the cast truncates toward zero; clip_q63_to_q31 is Include/arm_math.h's. */
void port_float_to_q31 (const float *s, int32_t *d, uint32_t n)
{ for (uint32_t i = 0; i < n; i++) d[i] = slo_clip_q63_to_q31 ((int64_t) (s[i] * 2147483648.0f)); }

/* Source/SupportFunctions/arm_q31_to_float.c : *pDst++ = ((float32_t) *pIn++ / 2147483648.0f) */
void port_q31_to_float (const int32_t *s, float *d, uint32_t n) { for (uint32_t i = 0; i < n; i++) d[i] = (float) s[i] / 2147483648.0f; }

#include "../tx_mod.inc.c"
