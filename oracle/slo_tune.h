/* ORACLE / TEST INFRASTRUCTURE ONLY.
 *
 * The per-channel tuner of the f32 RX and TX chains (DESIGN.md §3.5), in the same two-implementation scheme as slo_api.h: every box
 * is a CMSIS-DSP V1.5.3 routine the port already restates, the composition is ours. Kept beside slo_api.h and slo_tx_mod.h (which it
 * includes for q31_to_float) so that those headers, and the digests recorded over their arguments, stay exactly as they are.
 */
#ifndef SLO_TUNE_H
#define SLO_TUNE_H
#include "slo_tx_mod.h"

#ifdef __cplusplus
extern "C" {
#endif

/* tune_q15: a q15 -> q15 complex mixer with an integer-phase NCO. For sample n of the call (phi0 = *phase on entry):
 *   phi[n] = phi0 + n inc (mod 2^32)
 *   x      = scale_f32 (q31_to_float ((int32) phi[n]), 3.14159265f)          (the x of tx_fm_nco)
 *   w      = cos_f32 (x) + j sin_f32 (x);  up == 0 (RX): w = cmplx_conj_f32 (w)
 *   out    = float_to_q15 (cmplx_mult_cmplx_f32 (q15_to_float (in), w))
 * and *phase = phi0 + frames inc on return. inc is in units of 2^-32 turn per sample; up = 1 moves the signal UP by inc (TX), up = 0
 * moves what sits at +inc down to 0 (RX). float_to_q15 saturates a component that exceeds full scale (|z| > 1 rotated). in / out are
 * interleaved I, Q [frames][2]; they may be the same array. The chains apply it only to channels with inc != 0: a channel with offset 0
 * passes unchanged and keeps its phase (tune_q15 with inc = 0 would rotate by the carried phase). */
void SLO (tune_q15) (const int16_t *in, int16_t *out, uint32_t frames, int32_t inc, uint32_t *phase, int up);

#ifdef __cplusplus
}
#endif
#endif /* SLO_TUNE_H */
