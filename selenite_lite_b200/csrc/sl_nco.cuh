// Device helpers shared by the kernels that write I/Q or evaluate the table NCO: the FFT chain kernel (sl_rx_ssb_f32.cu), the TX
// tensor-core kernel (sl_tx_ssb_tc.cu), the tuner (sl_tune.cu) and the q15 tensor-core kernel (sl_rx_q15_tc.cu, TX-Q15 FM).
// Included inside each translation unit's anonymous namespace.
#pragma once

// arm_float_to_q15.c:147 per component: truncation toward zero, then saturation; interleaved I,Q as on the I2S bus (main.c:333-341).
// The caller has already multiplied by 32768 (a power of two, folded into its gain).
__device__ __forceinline__ uint32_t pack_iq (float i_times_32768, float q_times_32768)
{
  short a, b;
  asm ("cvt.rzi.sat.s16.f32 %0, %1;" : "=h"(a) : "f"(i_times_32768));
  asm ("cvt.rzi.sat.s16.f32 %0, %1;" : "=h"(b) : "f"(q_times_32768));
  return (uint32_t) (uint16_t) a | ((uint32_t) (uint16_t) b << 16);
}

// arm_sin_f32.c:72-119 / arm_cos_f32.c, op for op (sl_stages.cu OpSinCosF32): table lookup + linear interpolation
__device__ __forceinline__ float arm_sincos (float v, const float *tab, bool is_cos)
{
  float in; int n;
  if (!is_cos)
  {
    if (v < 0.0f && v >= -1.9e-7f) return v;
    in = __fmul_rn (v, 0.159154943092f); n = (int) in; if (v < 0.0f) n--;
  }
  else { in = __fadd_rn (__fmul_rn (v, 0.159154943092f), 0.25f); n = (int) in; if (in < 0.0f) n--; }
  in = __fsub_rn (in, (float) n);
  const float findex = __fmul_rn (512.0f, in);
  const unsigned idx = ((unsigned) (uint16_t) (int) findex) & 0x1ffu;
  const float fract = __fsub_rn (findex, (float) idx);
  return __fadd_rn (__fmul_rn (__fsub_rn (1.0f, fract), tab[idx]), __fmul_rn (fract, tab[idx + 1]));
}

// the NCO argument of a uint32 phase (2^-32 turn): arm_q31_to_float ((int32) phi) -> arm_scale_f32 (3.14159265f). The 1/2^31 of
// arm_q31_to_float is a power of two, folded into the constant (exact)
__device__ __forceinline__ float nco_arg (uint32_t phi) { return __fmul_rn (__int2float_rn ((int) phi), 3.14159265f / 2147483648.0f); }

// FM NCO of one sample (oracle tx_fm_nco): arm_q31_to_float ((int32) phi) -> arm_scale_f32 (pi) -> arm_cos_f32 / arm_sin_f32 ->
// arm_scale_f32 (level) -> arm_float_to_q15. The 1/2^31 of arm_q31_to_float and the x32768 are powers of two, folded into the constants.
__device__ __forceinline__ uint32_t fm_nco (uint32_t phi, const float *tab, float level15)
{
  const float x = nco_arg (phi);
  return pack_iq (__fmul_rn (arm_sincos (x, tab, true), level15), __fmul_rn (arm_sincos (x, tab, false), level15));
}
