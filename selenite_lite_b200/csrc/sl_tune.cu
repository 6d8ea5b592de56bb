// Per-channel tuning (DESIGN.md §3.5): a q15 -> q15 complex mixer with an integer-phase NCO, in front of the RX chains (on the int16
// I/Q input) and behind the TX chains (on the int16 I/Q output), so that every chain kernel serves tuned channels unchanged.
//
//   oracle (oracle/tune.inc.c tune_q15), per sample n of a call, phi0 = the phase carried in word 7 of the channel's state record:
//     phi[n] = phi0 + n inc (mod 2^32)
//     x      = arm_scale_f32 (arm_q31_to_float ((int32) phi[n]), 3.14159265f)         (the x of the TX FM NCO)
//     w      = arm_cos_f32 (x) + j arm_sin_f32 (x);  RX: w = arm_cmplx_conj_f32 (w)
//     out    = arm_float_to_q15 (arm_cmplx_mult_cmplx_f32 (arm_q15_to_float (in), w))
//   The 1/32768 of arm_q15_to_float and the x32768 of arm_float_to_q15 are powers of two that scale every product and sum exactly,
//   so the kernel works on the integer-valued samples; the complex product keeps the CMSIS order (ac - bd, ad + bc) with no FMA
//   contraction, and the pack truncates and saturates like arm_float_to_q15 (a rotated |z| > 1 component saturates).
//
// The phase of every sample is computed directly from phi0 (integer arithmetic, no scan), so CTAs of one channel are independent.
// They only read phi0; a second launch advances it by frames * inc after every CTA has read it.
#include <cuda_runtime.h>
#include <cstdint>
#include "sl_internal.h"

namespace sl {

namespace {
#include "sl_nco.cuh"

constexpr int kThreads = 256;
constexpr int kBatch = 4;                                     // 16-byte loads a thread has in flight before it computes
constexpr uint32_t kChunkVecs = 8u * kThreads;                // 4-frame vectors of one CTA: 8192 frames
constexpr uint32_t kMaxGridY = 65535u;

__device__ __forceinline__ uint32_t mix_frame (uint32_t v, uint32_t phi, const float *tab, bool up)
{
  const float x = nco_arg (phi);
  const float c = arm_sincos (x, tab, true);
  const float s = up ? arm_sincos (x, tab, false) : -arm_sincos (x, tab, false);   // arm_cmplx_conj_f32 for RX
  const float a = (float) (int16_t) (v & 0xFFFFu), b = (float) (int16_t) (v >> 16);
  return pack_iq (__fsub_rn (__fmul_rn (a, c), __fmul_rn (b, s)), __fadd_rn (__fmul_rn (a, s), __fmul_rn (b, c)));
}

// grid: x = 8192-frame chunks of a row, y = entries of the list. in and out may be the same rows; an entry with inc = 0 (an untuned
// row of a staged, out-of-place pass) is copied.
template <bool kUp>
__global__ void __launch_bounds__ (kThreads) tune_mix_kernel (const uint4 *in, uint4 *out, const uint32_t *list, const uint32_t *state,
                                                              uint32_t frames, uint32_t n_list, const float *sin513)
{
  __shared__ float tab[516];
  for (int k = threadIdx.x; k < 513; k += kThreads) tab[k] = sin513[k];
  __syncthreads ();
  const uint32_t vecs = frames / 4u;
  const uint32_t v0 = blockIdx.x * kChunkVecs, v1 = min (vecs, v0 + kChunkVecs);
  for (uint32_t e = blockIdx.y; e < n_list; e += gridDim.y)
  {
    const uint32_t row = list[2 * e], inc = list[2 * e + 1];
    const uint32_t phi0 = state[(size_t) row * 8 + 7];
    const uint4 *src = in + (size_t) row * vecs;
    uint4 *dst = out + (size_t) row * vecs;
    if (inc == 0)
    {
      for (uint32_t k = v0 + threadIdx.x; k < v1; k += kThreads) dst[k] = src[k];
      continue;
    }
    for (uint32_t base = v0 + threadIdx.x; base < v1; base += kBatch * kThreads)
    {
      uint4 w[kBatch];
#pragma unroll
      for (int j = 0; j < kBatch; j++) { const uint32_t k = base + j * kThreads; if (k < v1) w[j] = src[k]; }
#pragma unroll
      for (int j = 0; j < kBatch; j++)
      {
        const uint32_t k = base + j * kThreads;
        if (k >= v1) break;
        const uint32_t phi = phi0 + 4u * k * inc;
        dst[k] = make_uint4 (mix_frame (w[j].x, phi, tab, kUp), mix_frame (w[j].y, phi + inc, tab, kUp), mix_frame (w[j].z, phi + 2u * inc, tab, kUp),
                             mix_frame (w[j].w, phi + 3u * inc, tab, kUp));
      }
    }
  }
}

__global__ void tune_advance_kernel (const uint32_t *list, uint32_t *state, uint32_t frames, uint32_t n_list)
{
  const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n_list) state[(size_t) list[2 * e] * 8 + 7] += frames * list[2 * e + 1];
}
}  // namespace

int launch_tune (const int16_t *d_in, int16_t *d_out, const uint32_t *d_list, uint32_t n_list, uint32_t n_tuned, float *state, uint32_t frames,
                 bool up, const float *sin513, void *stream_)
{
  if (n_list == 0 || frames == 0) return (int) cudaSuccess;
  if (frames % 4u != 0) return (int) cudaErrorInvalidValue;
  // 16-byte loads and stores: a caller's row that is not 16-byte aligned is refused here, before the mixer touches it
  if ((reinterpret_cast<uintptr_t> (d_in) | reinterpret_cast<uintptr_t> (d_out)) & 15u) return (int) cudaErrorMisalignedAddress;
  cudaStream_t stream = (cudaStream_t) stream_;
  const uint32_t vecs = frames / 4u;
  const dim3 grid ((vecs + kChunkVecs - 1) / kChunkVecs, n_list < kMaxGridY ? n_list : kMaxGridY);
  const uint4 *in = reinterpret_cast<const uint4 *> (d_in);
  uint4 *out = reinterpret_cast<uint4 *> (d_out);
  uint32_t *st = reinterpret_cast<uint32_t *> (state);
  if (up) tune_mix_kernel<true><<<grid, kThreads, 0, stream>>> (in, out, d_list, st, frames, n_list, sin513);
  else tune_mix_kernel<false><<<grid, kThreads, 0, stream>>> (in, out, d_list, st, frames, n_list, sin513);
  cudaError_t e = cudaGetLastError ();
  if (e != cudaSuccess) return (int) e;
  tune_advance_kernel<<<(n_tuned + 255) / 256, 256, 0, stream>>> (d_list, st, frames, n_tuned);
  return (int) cudaGetLastError ();
}

}  // namespace sl
