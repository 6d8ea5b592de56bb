// q15 integer arithmetic shared by the kernels that restate CMSIS-DSP's q15 routines bit for bit: the dual 16-bit lane operations of
// arm_cfft_q15's ARM_MATH_DSP branch (sl_fft_fixed.cu, sl_chan64_q15.cu) and arm_sqrt_q15 / arm_cmplx_mag_q15 (sl_rx_q15_tc.cu,
// sl_chan64_q15.cu). Included inside each translation unit's anonymous namespace; every function is inlined where it is used.
#pragma once
#include <cstdint>

__device__ __forceinline__ int sat16 (int v) { return max (-32768, min (32767, v)); }

// ------------------------------------------------------------------ q15 lane arithmetic ------------------------------------------------------------------
struct C16 { int x, y; };                                                   // one complex q15 sample, lanes sign-extended
__device__ __forceinline__ C16 unpack16 (uint32_t w) { return C16{ (int) (int16_t) (w & 0xFFFFu), (int) (int16_t) (w >> 16) }; }
__device__ __forceinline__ uint32_t pack16 (C16 v) { return ((uint32_t) v.x & 0xFFFFu) | ((uint32_t) v.y << 16); }
__device__ __forceinline__ C16 shr (C16 a, int s) { return C16{ a.x >> s, a.y >> s }; }
__device__ __forceinline__ C16 qadd (C16 a, C16 b) { return C16{ sat16 (a.x + b.x), sat16 (a.y + b.y) }; }            // __QADD16
__device__ __forceinline__ C16 qsub (C16 a, C16 b) { return C16{ sat16 (a.x - b.x), sat16 (a.y - b.y) }; }            // __QSUB16
__device__ __forceinline__ C16 hadd (C16 a, C16 b) { return C16{ (a.x + b.x) >> 1, (a.y + b.y) >> 1 }; }              // __SHADD16
__device__ __forceinline__ C16 hsub (C16 a, C16 b) { return C16{ (a.x - b.x) >> 1, (a.y - b.y) >> 1 }; }              // __SHSUB16
// a - j b and a + j b on the lanes: __QASX (re - im', im + re'), __QSAX (re + im', im - re'), and their halving forms
__device__ __forceinline__ C16 qasx (C16 a, C16 b) { return C16{ sat16 (a.x - b.y), sat16 (a.y + b.x) }; }
__device__ __forceinline__ C16 qsax (C16 a, C16 b) { return C16{ sat16 (a.x + b.y), sat16 (a.y - b.x) }; }
__device__ __forceinline__ C16 hasx (C16 a, C16 b) { return C16{ (a.x - b.y) >> 1, (a.y + b.x) >> 1 }; }
__device__ __forceinline__ C16 hsax (C16 a, C16 b) { return C16{ (a.x + b.y) >> 1, (a.y - b.x) >> 1 }; }
// twiddle product, truncated to the high half-word of the wrapping 32-bit sums: forward v * (co - j si) = __SMUAD >> 16 | __SMUSDX,
// inverse v * (co + j si) = __SMUSD >> 16 | __SMUADX
template <bool INV> __device__ __forceinline__ C16 twid (C16 c, C16 v)
{
  const uint32_t xx = (uint32_t) (c.x * v.x), yy = (uint32_t) (c.y * v.y), xy = (uint32_t) (c.x * v.y), yx = (uint32_t) (c.y * v.x);
  const int re = (int) (INV ? xx - yy : xx + yy), im = (int) (INV ? xy + yx : xy - yx);
  return C16{ re >> 16, im >> 16 };
}

// ------------------------------------------------------------------ magnitude ------------------------------------------------------------------
// arm_sqrt_q15 (FastMathFunctions/arm_sqrt_q15.c) as oracle/port/stats_cmplx.c restates it, every cast included: normalise by an even
// shift, a float seed (a power-of-two multiply, the 0x5f3759df bit trick), three q15 Newton steps, multiply back, undo half the shift
__device__ __forceinline__ int sqrt_q15 (int number)
{
  if (number <= 0) return 0;
  const int sh = (__clz (number) - 17) & ~1;                                      // signBits1, or signBits1 - 1 when it is odd
  number = (int) (int16_t) (number << sh);
  const int half = number >> 1, temp1 = number;
  const float tf = __int_as_float (0x5f3759df - (__float_as_int ((float) number * 3.051757812500000e-005f) >> 1));
  int var1 = (int) (int16_t) (int) (tf * 16384.0f);
#pragma unroll
  for (int it = 0; it < 3; it++)
  {
    const int sq = (int) (int16_t) ((var1 * var1) >> 15);
    const int hs = (int) (int16_t) ((sq * half) >> 15);
    var1 = (int) (int16_t) ((int) (int16_t) ((var1 * (0x3000 - hs)) >> 15) << 2);
  }
  var1 = (int) (int16_t) ((int) (int16_t) ((temp1 * var1) >> 15) << 1);
  return var1 >> (sh / 2);
}
// arm_cmplx_mag_q15 (arm_cmplx_mag_q15.c): sqrt_q15 ((re^2 + im^2) >> 17), 2.14 format
__device__ __forceinline__ int cmag_q15 (int re, int im) { return sqrt_q15 ((int) (((unsigned) (re * re) + (unsigned) (im * im)) >> 17)); }
