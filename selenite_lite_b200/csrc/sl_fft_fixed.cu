// Fixed-point complex FFTs of the stage library: arm_cfft_q15 (TransformFunctions/arm_cfft_q15.c:77) and arm_cfft_q31
// (arm_cfft_q31.c:77), batched, bit-exact, one CTA per transform with the data in shared memory.
//
// Both reference routines are decimation-in-frequency, in place: N = 4^m runs m radix-4 stages, N = 2 * 4^m one radix-2
// stage, the two half-length radix-4 transforms, and a final doubling (arm_cfft_radix4by2_*); the first radix-4 stage scales its
// inputs (q15: >> 2, q31: >> 4), the middle stages scale their outputs, the last stage has no twiddles; every stage puts the
// W^2 output in the second quarter and the W^1 output in the third, so the result is in BIT-reversed order and a bit reversal
// (arm_bitreversal_16 / _32, Cortex-M assembly in the reference) brings it to natural order — here it is the index the store uses.
//
// q15 follows the branch the FIRMWARE compiles (ARM_MATH_CM4 -> ARM_MATH_DSP, .cproject:44): the dual-16-bit butterflies of
// arm_cfft_radix4_q15.c:156-560 and arm_cfft_q15.c:134-236 (saturating / halving lane adds, products truncated to their high
// half-word). It differs by a few LSB from the shift-based C branch of the same file (SURVEY.md §8c.3); the oracle builds that
// branch from the reference sources (oracle/ref_glue/cm4_fft_q15.c). The lane operations are written out below as plain integer
// arithmetic on (re, im) pairs; q31 (arm_cfft_radix4_q31.c:142 ff., path-independent) uses 32-bit wrapping sums and the high
// word of 64-bit products exactly as the reference does.
//
// Twiddles are not copied from the reference tables: they are regenerated (q15: floor (cos * 2^15), q31: floor (cos * 2^31 + 0.05),
// both clipped at +1.0 — the rules that reproduce arm_common_tables.c entry for entry, checked by tests/test_fft_fixed_tables.py).
#include <cuda_runtime.h>
#include <cmath>
#include <cstdint>
#include <map>
#include <mutex>
#include <vector>
#include "sl_internal.h"

namespace sl {

namespace {

#include "sl_q15.cuh"

// one radix-4 transform of length L at s[0..L), twiddle index step m0 (1: own table, 2: half of a radix-4-by-2 transform)
template <bool INV> __device__ void radix4_q15 (uint32_t *s, int L, int m0, const uint32_t *__restrict__ tw, int b0, int nb, int tid, int nthreads)
{
  int stages = 0; for (int t = L; t > 1; t >>= 2) stages++;
  for (int st = 0; st < stages; st++)
  {
    const int n1 = L >> (2 * st), n2 = n1 >> 2, mod = m0 << (2 * st);
    for (int b = b0 + tid; b < b0 + nb; b += nthreads)
    {
      const int bb = b - b0;
      if (st == stages - 1)
      {
        // last stage: four neighbours, no twiddles (arm_cfft_radix4_q15.c:520-560)
        uint32_t *p = s + 4 * bb;
        const C16 a = unpack16 (p[0]), bq = unpack16 (p[1]), c = unpack16 (p[2]), d = unpack16 (p[3]);
        const C16 R = qadd (a, c), T = qadd (bq, d), S = qsub (a, c), U = qsub (bq, d);
        p[0] = pack16 (hadd (R, T)); p[1] = pack16 (hsub (R, T));
        p[2] = pack16 (INV ? hasx (S, U) : hsax (S, U)); p[3] = pack16 (INV ? hsax (S, U) : hasx (S, U));
        continue;
      }
      const int j = bb % n2, i0 = (bb / n2) * n1 + j, ic = j * mod;
      uint32_t *p0 = s + i0, *p1 = p0 + n2, *p2 = p1 + n2, *p3 = p2 + n2;
      C16 a = unpack16 (*p0), bq = unpack16 (*p1), c = unpack16 (*p2), d = unpack16 (*p3);
      const C16 c1 = unpack16 (tw[ic]), c2 = unpack16 (tw[2 * ic]), c3 = unpack16 (tw[3 * ic]);
      if (st == 0)
      {
        // first stage: inputs >> 2 (two halving adds with zero), saturating sums (arm_cfft_radix4_q15.c:186-330)
        a = shr (a, 2); bq = shr (bq, 2); c = shr (c, 2); d = shr (d, 2);
        const C16 R = qadd (a, c), S = qsub (a, c), T = qadd (bq, d);
        *p0 = pack16 (hadd (R, T));
        *p1 = pack16 (twid<INV> (c2, qsub (R, T)));
        const C16 T2 = qsub (bq, d);
        const C16 Rr = INV ? qsax (S, T2) : qasx (S, T2), Ss = INV ? qasx (S, T2) : qsax (S, T2);
        *p2 = pack16 (twid<INV> (c1, Ss));
        *p3 = pack16 (twid<INV> (c3, Rr));
      }
      else
      {
        // middle stages: outputs halved (arm_cfft_radix4_q15.c:340-505)
        const C16 R = qadd (a, c), S = qsub (a, c), T = qadd (bq, d);
        *p0 = pack16 (shr (hadd (R, T), 1));
        *p1 = pack16 (twid<INV> (c2, hsub (R, T)));
        const C16 T2 = qsub (bq, d);
        const C16 Rr = INV ? hsax (S, T2) : hasx (S, T2), Ss = INV ? hasx (S, T2) : hsax (S, T2);
        *p2 = pack16 (twid<INV> (c1, Ss));
        *p3 = pack16 (twid<INV> (c3, Rr));
      }
    }
    __syncthreads ();
  }
}

template <bool INV> __global__ void cfft_q15_kernel (uint32_t *__restrict__ data, int N, int log2n, const uint32_t *__restrict__ tw)
{
  extern __shared__ uint32_t fx_smem[];
  uint32_t *s = fx_smem;
  uint32_t *g = data + (size_t) blockIdx.x * N;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int i = tid; i < N; i += nt) s[i] = g[i];
  __syncthreads ();
  const bool by2 = (log2n & 1) != 0;
  if (by2)
  {
    // radix-2 stage of arm_cfft_radix4by2_q15 (arm_cfft_q15.c:155-188 / :262-295): halve, saturating difference, twiddle
    const int n2 = N >> 1;
    for (int i = tid; i < n2; i += nt)
    {
      const C16 T = shr (unpack16 (s[i]), 1), S = shr (unpack16 (s[i + n2]), 1);
      s[i] = pack16 (hadd (T, S));
      s[i + n2] = pack16 (twid<INV> (unpack16 (tw[i]), qsub (T, S)));
    }
    __syncthreads ();
    // the two half-length transforms, twiddle step 2 on the same table (arm_cfft_q15.c:218-220)
    radix4_q15<INV> (s, n2, 2, tw, 0, n2 / 4, tid, nt);
    radix4_q15<INV> (s + n2, n2, 2, tw, 0, n2 / 4, tid, nt);
    for (int i = tid; i < N; i += nt)
    {
      const C16 v = unpack16 (s[i]);                                          // p <<= 1 on q15_t (arm_cfft_q15.c:222-236)
      s[i] = pack16 (C16{ (int) (int16_t) (v.x << 1), (int) (int16_t) (v.y << 1) });
    }
    __syncthreads ();
  }
  else radix4_q15<INV> (s, N, 1, tw, 0, N / 4, tid, nt);
  for (int i = tid; i < N; i += nt) g[__brev ((unsigned) i) >> (32 - log2n)] = s[i];          // arm_bitreversal_16: natural order
}

// ------------------------------------------------------------------ q31 ------------------------------------------------------------------
__device__ __forceinline__ int wadd (int a, int b) { return (int) ((uint32_t) a + (uint32_t) b); }
__device__ __forceinline__ int wsub (int a, int b) { return (int) ((uint32_t) a - (uint32_t) b); }
__device__ __forceinline__ int wshl (int a, int s) { return (int) ((uint32_t) a << s); }
__device__ __forceinline__ int mulhi (int a, int b) { return __mulhi (a, b); }                                            // (q63) a * b >> 32
template <bool INV> __device__ __forceinline__ int2 twid31 (int co, int si, int r, int s_)
{
  return INV ? make_int2 (wsub (mulhi (r, co), mulhi (s_, si)), wadd (mulhi (s_, co), mulhi (r, si)))
             : make_int2 (wadd (mulhi (r, co), mulhi (s_, si)), wsub (mulhi (s_, co), mulhi (r, si)));
}

template <bool INV> __device__ void radix4_q31 (int2 *s, int L, int m0, const int2 *__restrict__ tw, int tid, int nthreads)
{
  int stages = 0; for (int t = L; t > 1; t >>= 2) stages++;
  for (int st = 0; st < stages; st++)
  {
    const int n1 = L >> (2 * st), n2 = n1 >> 2, mod = m0 << (2 * st);
    for (int bb = tid; bb < L / 4; bb += nthreads)
    {
      if (st == stages - 1)
      {
        // last stage (arm_cfft_radix4_q31.c:640-745 / inverse :1280-1385)
        int2 *p = s + 4 * bb;
        const int2 a = p[0], b = p[1], c = p[2], d = p[3];
        p[0] = make_int2 (wadd (wadd (a.x, b.x), wadd (c.x, d.x)), wadd (wadd (a.y, b.y), wadd (c.y, d.y)));
        p[1] = make_int2 (wsub (wadd (wsub (a.x, b.x), c.x), d.x), wsub (wadd (wsub (a.y, b.y), c.y), d.y));
        const int2 plus = make_int2 (wsub (wsub (wadd (a.x, b.y), c.x), d.y), wadd (wsub (wsub (a.y, b.x), c.y), d.x));     // (xa + yb - xc - yd, ya - xb - yc + xd)
        const int2 minus = make_int2 (wadd (wsub (wsub (a.x, b.y), c.x), d.y), wsub (wsub (wadd (a.y, b.x), c.y), d.x));    // (xa - yb - xc + yd, ya + xb - yc - xd)
        p[2] = INV ? minus : plus; p[3] = INV ? plus : minus;
        continue;
      }
      const int j = bb % n2, i0 = (bb / n2) * n1 + j, ia = j * mod;
      int2 *p0 = s + i0, *p1 = p0 + n2, *p2 = p1 + n2, *p3 = p2 + n2;
      int2 a = *p0, b = *p1, c = *p2, d = *p3;
      const int2 w1 = tw[ia], w2 = tw[2 * ia], w3 = tw[3 * ia];
      const bool first = st == 0;
      if (first) { a.x >>= 4; a.y >>= 4; b.x >>= 4; b.y >>= 4; c.x >>= 4; c.y >>= 4; d.x >>= 4; d.y >>= 4; }               // arm_cfft_radix4_q31.c:395-400
      int r1 = wadd (a.x, c.x), r2 = wsub (a.x, c.x), t1 = wadd (b.x, d.x), s1 = wadd (a.y, c.y), s2 = wsub (a.y, c.y);
      const int o0x = wadd (r1, t1);
      r1 = wsub (r1, t1);
      int t2 = wadd (b.y, d.y);
      const int o0y = wadd (s1, t2);
      s1 = wsub (s1, t2);
      t1 = wsub (b.y, d.y); t2 = wsub (b.x, d.x);
      *p0 = first ? make_int2 (o0x, o0y) : make_int2 (o0x >> 2, o0y >> 2);
      int2 o1 = twid31<INV> (w2.x, w2.y, r1, s1);
      if (INV) { r1 = wsub (r2, t1); r2 = wadd (r2, t1); s1 = wadd (s2, t2); s2 = wsub (s2, t2); }
      else { r1 = wadd (r2, t1); r2 = wsub (r2, t1); s1 = wsub (s2, t2); s2 = wadd (s2, t2); }
      int2 o2 = twid31<INV> (w1.x, w1.y, r1, s1), o3 = twid31<INV> (w3.x, w3.y, r2, s2);
      if (first) { o1 = make_int2 (wshl (o1.x, 1), wshl (o1.y, 1)); o2 = make_int2 (wshl (o2.x, 1), wshl (o2.y, 1)); o3 = make_int2 (wshl (o3.x, 1), wshl (o3.y, 1)); }
      else { o1 = make_int2 (o1.x >> 1, o1.y >> 1); o2 = make_int2 (o2.x >> 1, o2.y >> 1); o3 = make_int2 (o3.x >> 1, o3.y >> 1); }
      *p1 = o1; *p2 = o2; *p3 = o3;
    }
    __syncthreads ();
  }
}

template <bool INV> __global__ void cfft_q31_kernel (int2 *__restrict__ data, int N, int log2n, const int2 *__restrict__ tw)
{
  extern __shared__ uint32_t fx_smem[];
  int2 *s = reinterpret_cast<int2 *> (fx_smem);
  int2 *g = data + (size_t) blockIdx.x * N;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int i = tid; i < N; i += nt) s[i] = g[i];
  __syncthreads ();
  if (log2n & 1)
  {
    // radix-2 stage of arm_cfft_radix4by2_q31 (arm_cfft_q31.c:134-168 / inverse :190-228): inputs >> 2, rounded high-word products
    const int n2 = N >> 1;
    for (int i = tid; i < n2; i += nt)
    {
      const int2 u = s[i], v = s[i + n2], w = tw[i];
      const int xt = wsub (u.x >> 2, v.x >> 2), yt = wsub (u.y >> 2, v.y >> 2);
      s[i] = make_int2 (wadd (u.x >> 2, v.x >> 2), wadd (v.y >> 2, u.y >> 2));
      // mult_32x32_keep32_R, then multAcc_ / multSub_32x32_keep32_R (arm_math.h:7023-7032): 64-bit sums, rounded, high word kept
      const unsigned long long half = 0x80000000ULL;
      const int p0a = (int) ((long long) ((unsigned long long) ((long long) xt * w.x) + half) >> 32), p1a = (int) ((long long) ((unsigned long long) ((long long) yt * w.x) + half) >> 32);
      const unsigned long long ys = (unsigned long long) ((long long) yt * w.y), xs = (unsigned long long) ((long long) xt * w.y);
      const unsigned long long b0 = (unsigned long long) (long long) p0a << 32, b1 = (unsigned long long) (long long) p1a << 32;
      const int p0 = (int) ((long long) (INV ? b0 - ys + half : b0 + ys + half) >> 32);
      const int p1 = (int) ((long long) (INV ? b1 + xs + half : b1 - xs + half) >> 32);
      s[i + n2] = make_int2 (wshl (p0, 1), wshl (p1, 1));
    }
    __syncthreads ();
    radix4_q31<INV> (s, n2, 2, tw, tid, nt);
    radix4_q31<INV> (s + n2, n2, 2, tw, tid, nt);
    for (int i = tid; i < N; i += nt) s[i] = make_int2 (wshl (s[i].x, 1), wshl (s[i].y, 1));
    __syncthreads ();
  }
  else radix4_q31<INV> (s, N, 1, tw, tid, nt);
  for (int i = tid; i < N; i += nt) g[__brev ((unsigned) i) >> (32 - log2n)] = s[i];          // arm_bitreversal_32: natural order
}

// ------------------------------------------------------------------ twiddle tables ------------------------------------------------------------------
std::mutex g_tw_mu;
std::map<uint32_t, std::vector<int16_t>> g_tw15;
std::map<uint32_t, std::vector<int32_t>> g_tw31;

int log2_of (uint32_t N) { int l = 0; while ((1u << l) < N) l++; return ((1u << l) == N) ? l : -1; }

}  // namespace

// twiddleCoef_N_q15 / twiddleCoef_N_q31 (CommonTables/arm_common_tables.c): 3 N / 4 pairs (cos, sin) of 2 pi k / N
const int16_t *fft_twiddle_q15 (uint32_t N)
{
  std::lock_guard<std::mutex> lk (g_tw_mu);
  auto &t = g_tw15[N];
  if (t.empty ())
  {
    t.resize (3 * N / 4 * 2);
    for (uint32_t k = 0; k < 3 * N / 4; k++)
    {
      const double a = 2.0 * 3.14159265358979323846 * (double) k / (double) N;
      const double v[2] = { std::cos (a), std::sin (a) };
      for (int i = 0; i < 2; i++) { double q = std::floor (v[i] * 32768.0); if (q > 32767.0) q = 32767.0; if (q < -32768.0) q = -32768.0; t[2 * k + i] = (int16_t) q; }
    }
  }
  return t.data ();
}
const int32_t *fft_twiddle_q31 (uint32_t N)
{
  std::lock_guard<std::mutex> lk (g_tw_mu);
  auto &t = g_tw31[N];
  if (t.empty ())
  {
    t.resize (3 * N / 4 * 2);
    for (uint32_t k = 0; k < 3 * N / 4; k++)
    {
      const double a = 2.0 * 3.14159265358979323846 * (double) k / (double) N;
      const double v[2] = { std::cos (a), std::sin (a) };
      for (int i = 0; i < 2; i++)
      {
        double q = std::floor (v[i] * 2147483648.0 + 0.05);
        if (q > 2147483647.0) q = 2147483647.0; if (q < -2147483648.0) q = -2147483648.0;
        t[2 * k + i] = (int32_t) q;
      }
    }
  }
  return t.data ();
}

int launch_cfft_q15 (int16_t *d_data, uint32_t N, size_t transforms, int ifft, const int16_t *d_tw, void *stream)
{
  const int l2 = log2_of (N);
  if (l2 < 4 || l2 > 12) return (int) cudaErrorInvalidValue;
  const unsigned nt = N / 4 < 256 ? (N / 4 < 32 ? 32 : N / 4) : 256;
  const size_t smem = (size_t) N * 4;
  if (ifft) cfft_q15_kernel<true><<<(unsigned) transforms, nt, smem, (cudaStream_t) stream>>> (reinterpret_cast<uint32_t *> (d_data), (int) N, l2, reinterpret_cast<const uint32_t *> (d_tw));
  else cfft_q15_kernel<false><<<(unsigned) transforms, nt, smem, (cudaStream_t) stream>>> (reinterpret_cast<uint32_t *> (d_data), (int) N, l2, reinterpret_cast<const uint32_t *> (d_tw));
  return (int) cudaGetLastError ();
}
int launch_cfft_q31 (int32_t *d_data, uint32_t N, size_t transforms, int ifft, const int32_t *d_tw, void *stream)
{
  const int l2 = log2_of (N);
  if (l2 < 4 || l2 > 12) return (int) cudaErrorInvalidValue;
  const unsigned nt = N / 4 < 256 ? (N / 4 < 32 ? 32 : N / 4) : 256;
  const size_t smem = (size_t) N * 8;
  if (ifft) cfft_q31_kernel<true><<<(unsigned) transforms, nt, smem, (cudaStream_t) stream>>> (reinterpret_cast<int2 *> (d_data), (int) N, l2, reinterpret_cast<const int2 *> (d_tw));
  else cfft_q31_kernel<false><<<(unsigned) transforms, nt, smem, (cudaStream_t) stream>>> (reinterpret_cast<int2 *> (d_data), (int) N, l2, reinterpret_cast<const int2 *> (d_tw));
  return (int) cudaGetLastError ();
}

}  // namespace sl
