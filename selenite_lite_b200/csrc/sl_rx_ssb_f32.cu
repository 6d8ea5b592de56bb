// RX-SSB-f32: the fused receive chain, one kernel, every sample crosses HBM once (4 B in, 4 B out).
//
//   int16 I/Q  --unpack-->  overlap-save FFT filter (512-pt, hop 384)  --Re-->  2-stage df2T biquad  -->  per-48-frame AGC  -->  int16 L=R
//   oracle stage per box (reference = /root/reference/Drivers/CMSIS/DSP/Source/...):
//     unpack   SupportFunctions/arm_q15_to_float.c:65            FFT/IFFT  TransformFunctions/arm_cfft_f32.c:562 (len 512)
//     mask     ComplexMathFunctions/arm_cmplx_mult_cmplx_f32.c:72  biquad   FilteringFunctions/arm_biquad_cascade_df2T_f32.c:142
//     AGC      BasicMathFunctions/arm_abs_f32.c:63, StatisticsFunctions/arm_max_f32.c:58, arm_scale_f32.c:77 (+ our gain law)
//     pack     SupportFunctions/arm_float_to_q15.c:64 (truncating)
//   and it sits where the firmware would call it: between pbuf and the ring store in DSP_In_Buff_Write (Core/Src/dsp_if.c:286-289).
//
// Structure (DESIGN.md §4). The chain is bound by the FP32 pipe, not by HBM (~130 FP32 lane-ops per complex sample
// for two 512-point FFTs per 384 samples), so the kernel is organised around instruction count and issue slots:
//   * warp-specialised CTA of 5 warps. Warps 0..3 each own one overlap-save frame of a 4-frame tile: load, unpack,
//     forward FFT, mask, inverse FFT — entirely warp-local (private shared-memory scratch, __syncwarp only, no CTA
//     barrier). Warp 4 runs the time recurrences (biquad cascade, AGC) of the PREVIOUS tile, packs and stores it.
//     The two sides meet through a double-buffered audio tile in shared memory and four named barriers.
//   * every FFT lane carries TWO radix-8 butterflies and evaluates them together with packed FP32x2 instructions
//     (FADD2 / FMUL2 / FFMA2, new on sm_100): half the FP32 issue slots of scalar code.
//   * the biquad recurrence is evaluated time-parallel: lane k filters the two 24-sample runs of its 48-sample AGC block
//     from a zero state (both runs at once, packed FP32x2), block end states are chained with a 5-step warp scan over
//     4x4 transition matrices, and the true start states are added back through the cascade's zero-input response
//     (tables from sl_design.cpp).
//   * a CTA owns (channel, segment of 8 tiles); segments of one channel are chained through 5 floats in global memory
//     with a release/acquire flag. Items are dealt round-robin in segment-major order, so the flag is already set
//     whenever at least as many channels as resident CTAs are in flight.
#include <cuda_runtime.h>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include "sl_internal.h"

namespace sl {

namespace {
#include "sl_stress.cuh"

constexpr int kN = 512;                          // FFT length
constexpr int kHop = 384;                        // new frames per FFT frame
constexpr int kOvl = kN - kHop;                  // 128 carried frames
#ifndef SL_RX_FFTWARPS
#define SL_RX_FFTWARPS 4
#endif
constexpr int kFftWarps = SL_RX_FFTWARPS;        // = frames per tile
constexpr int kTile = kHop * kFftWarps;          // 1536 frames
constexpr int kThreads = 32 * (kFftWarps + 1);   // + the recurrence warp
constexpr int kBlocksPerTile = kTile / kAgcBlock; // 32 AGC blocks of 48 samples = one per recurrence lane
constexpr int kBlkStride = 50;                   // words per block in the audio tile: 8-byte aligned, conflict-free for
                                                 // the lane-per-block 64-bit reads (18 l mod 32 hits 16 distinct even banks)
constexpr int kTxBlkStride = 100;                // TX tile: 48 complex per block + pad; 16-byte aligned, the lane-per-block
                                                 // 128-bit reads (100 l mod 32 = 4 l) cover all banks once per 8 lanes
constexpr int kTilesPerItem = 16;                // tiles a CTA processes with the recurrence state in registers
constexpr int kPlane = kN;                       // floats per re / im scratch plane (XOR swizzle: no padding)
constexpr int kRawWords = kTile + kOvl;          // raw frames (one u32 each) a tile needs: its 1536 + the 128 before it
#ifndef SL_RX_RAWBUFS
#define SL_RX_RAWBUFS 2
#endif
#ifndef SL_RX_AUDIOBUFS
#define SL_RX_AUDIOBUFS 3
#endif
#ifndef SL_RX_CTAS
#define SL_RX_CTAS 4
#endif
constexpr int kRawBufs = SL_RX_RAWBUFS;          // raw staging: filled by bulk asynchronous copies kRawBufs tiles ahead

// dynamic shared memory layout (bytes). RX keeps three audio tiles in flight so that the FFT warps and the recurrence
// warp only meet when one side is a whole tile late; the TX tile is twice as large (complex) and stays double-buffered.
template <bool kTx, bool kMod = false> struct Smem
{
  static constexpr int kAudioBufs = kTx ? 2 : SL_RX_AUDIOBUFS;
  static constexpr int kAudioWords = kBlocksPerTile * (kTx ? kTxBlkStride : kBlkStride);
  static constexpr size_t scratch = 0;
  static constexpr size_t audio = scratch + (size_t) kFftWarps * 2 * kPlane * 4;
  static constexpr size_t raw = audio + (size_t) kAudioBufs * kAudioWords * 4;
  static constexpr size_t tw = raw + (size_t) kRawBufs * kRawWords * 4;
  static constexpr size_t bars = tw + 6 * 32 * 16;
  static constexpr size_t sin = bars + (2 * kRawBufs + 2 * kAudioBufs) * 8;
  static constexpr size_t bytes = sin + (kMod ? 516 * 4 : 0);   // TX all-mode: arm_sin_f32's 513-entry table
};

// shared-memory index of FFT point i inside a plane. The LSU data pipe is the busiest unit of this kernel (ncu:
// l1tex__data_pipe_lsu_wavefronts 84 % before this swizzle, half of all store wavefronts were bank conflicts), so the
// layout is chosen to make every access pattern of the three passes conflict-free with 64-bit accesses: bits [4:1]
// of the word index are XORed with bits [7:4]. Pairs (2k, 2k+1) stay adjacent and 8-byte aligned. (DESIGN.md §4.2)
[[maybe_unused]] __device__ __forceinline__ int phys (int i) { return i ^ (((i >> 4) & 15) << 1); }   // (the definition of record: call sites fold it)

// ---- packed FP32x2: one 64-bit register pair holds the same quantity for butterfly A (lo) and butterfly B (hi) ----
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk (float lo, float hi) { u64 r; asm ("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ float lo_of (u64 a) { float x; [[maybe_unused]] float y; asm ("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(a)); return x; }
__device__ __forceinline__ float hi_of (u64 a) { [[maybe_unused]] float x; float y; asm ("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(a)); return y; }
__device__ __forceinline__ u64 pair_lo (u64 a, u64 b) { return pk (lo_of (a), lo_of (b)); }   // 2x2 transpose helpers
__device__ __forceinline__ u64 pair_hi (u64 a, u64 b) { return pk (hi_of (a), hi_of (b)); }
__device__ __forceinline__ u64 add2 (u64 a, u64 b) { u64 r; asm ("add.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 sub2 (u64 a, u64 b) { u64 r; asm ("sub.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 mul2 (u64 a, u64 b) { u64 r; asm ("mul.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 fma2 (u64 a, u64 b, u64 c) { u64 r; asm ("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

// 8-point forward DFT of two butterflies at once, natural order in and out; re[] / im[] are packed (A,B).
// 52 packed instructions (26 per butterfly): the W8 rotations are folded into FMAs with +-1/sqrt2.
__device__ __forceinline__ void dft8x2 (u64 *re, u64 *im)
{
  const u64 H = pk (0.70710678118654752f, 0.70710678118654752f), NH = pk (-0.70710678118654752f, -0.70710678118654752f);
  const u64 a0r = add2 (re[0], re[4]), a0i = add2 (im[0], im[4]), t0r = sub2 (re[0], re[4]), t0i = sub2 (im[0], im[4]);
  const u64 a1r = add2 (re[1], re[5]), a1i = add2 (im[1], im[5]), t1r = sub2 (re[1], re[5]), t1i = sub2 (im[1], im[5]);
  const u64 a2r = add2 (re[2], re[6]), a2i = add2 (im[2], im[6]), t2r = sub2 (re[2], re[6]), t2i = sub2 (im[2], im[6]);
  const u64 a3r = add2 (re[3], re[7]), a3i = add2 (im[3], im[7]), t3r = sub2 (re[3], re[7]), t3i = sub2 (im[3], im[7]);
  // even outputs: DFT4 of a
  {
    const u64 s0r = add2 (a0r, a2r), s0i = add2 (a0i, a2i), s1r = sub2 (a0r, a2r), s1i = sub2 (a0i, a2i);
    const u64 s2r = add2 (a1r, a3r), s2i = add2 (a1i, a3i), dr = sub2 (a1r, a3r), di = sub2 (a1i, a3i);
    re[0] = add2 (s0r, s2r); im[0] = add2 (s0i, s2i);
    re[4] = sub2 (s0r, s2r); im[4] = sub2 (s0i, s2i);
    re[2] = add2 (s1r, di); im[2] = sub2 (s1i, dr);        // s1 + (-i) d
    re[6] = sub2 (s1r, di); im[6] = add2 (s1i, dr);        // s1 - (-i) d
  }
  // odd outputs: DFT4 of b, b0 = t0, b1 = t1 W8, b2 = -i t2, b3 = t3 W8^3
  {
    const u64 s0r = add2 (t0r, t2i), s0i = sub2 (t0i, t2r), s1r = sub2 (t0r, t2i), s1i = add2 (t0i, t2r);
    const u64 p = add2 (t1r, t1i), q = sub2 (t1i, t1r), u = sub2 (t3i, t3r), v = add2 (t3r, t3i);
    const u64 pu = add2 (p, u), qv = sub2 (q, v), pmu = sub2 (p, u), qpv = add2 (q, v);   // s2 = h (pu, qv), d = h (pmu, qpv)
    re[1] = fma2 (H, pu, s0r); im[1] = fma2 (H, qv, s0i);
    re[5] = fma2 (NH, pu, s0r); im[5] = fma2 (NH, qv, s0i);
    re[3] = fma2 (H, qpv, s1r); im[3] = fma2 (NH, pmu, s1i);
    re[7] = fma2 (NH, qpv, s1r); im[7] = fma2 (H, pmu, s1i);
  }
}

struct KParams
{
  const uint32_t *in; uint32_t *out;            // one u32 = one I/Q (or L/R) frame
  float *audio_dbg; float *gain_dbg;
  const uint32_t *ovl_in; uint32_t *ovl_out;
  float *state; unsigned *flag;
  const float4 *masks;                          // [slot][r][lane] = (HrA, HrB, HiA, HiB) * 1/(512*32768)
  const uint8_t *mask_slot;
  const float4 *twiddle;                        // [pass 1|2][w, w^2, w^4][lane] = (WrA, WrB, WiA, WiB)
  unsigned flag_base;
  uint32_t channels, frames, tiles_per_channel, items_per_channel;
  float agc_target, agc_decay, agc_floor, agc_gmax;
  BiquadScanTables tab;
  float am_depth, am_carrier15, fm_target, fm_level15;   // TX all-mode (x15: the final x32768 of arm_float_to_q15 folded in)
  uint32_t *phase_dbg;
  const float *sin513;
};

__device__ __forceinline__ unsigned ld_acquire (const unsigned *p)
{
  unsigned v;
  asm volatile ("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// polling load for the hand-over spin: coherent at GPU scope but WITHOUT acquire semantics, so the loop does not
// invalidate the SM's L1 on every iteration (ld.acquire compiles to LDG.STRONG + CCTL.IVALL); one acquire follows.
// watchdog of the inter-CTA hand-over polls: a tile's predecessor is published within microseconds (the grid is launched cooperatively,
// so it is resident); 2^23 polls of >= 32 ns + an L2 round trip are several seconds
constexpr unsigned kSpinLimit = 1u << 23;
__device__ __forceinline__ unsigned ld_relaxed (const unsigned *p)
{
  unsigned v;
  asm volatile ("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release (unsigned *p, unsigned v)
{
  asm volatile ("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// output stores that do not allocate in L1: the lanes of a warp store to 32 different lines, which would evict what the
// shared-memory / L1 data pipe is needed for (measured on the tensor-core RX kernel: 366 -> 408 Gsamples/s)
__device__ __forceinline__ void st_na (uint4 *p, uint4 v)
{
  asm volatile ("st.global.L1::no_allocate.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint32_t pack_lr (float x_times_32768)
{
  // arm_float_to_q15.c:147 : (q15_t) __SSAT((q31_t)(x * 32768.0f), 16) — the cast truncates toward zero, then saturates.
  // F2I.S16.TRUNC does both; the caller has already multiplied by 32768 (a power of two, folded into the gain).
  short v;
  asm ("cvt.rzi.sat.s16.f32 %0, %1;" : "=h"(v) : "f"(x_times_32768));
  return __byte_perm ((uint32_t) (uint16_t) v, 0u, 0x1010);   // stereo endpoint, L = R
}

__device__ __forceinline__ uint32_t pack_iq (float i_times_32768, float q_times_32768)
{
  short a, b;
  asm ("cvt.rzi.sat.s16.f32 %0, %1;" : "=h"(a) : "f"(i_times_32768));
  asm ("cvt.rzi.sat.s16.f32 %0, %1;" : "=h"(b) : "f"(q_times_32768));
  return (uint32_t) (uint16_t) a | ((uint32_t) (uint16_t) b << 16);              // interleaved I,Q as on the I2S bus (main.c:333-341)
}

// arm_float_to_q31.c (V1.5.3, ARM_MATH_ROUNDING not defined): clip_q63_to_q31 ((q63_t) (x * 2147483648.0f)). The product is exact
// (power of two); F2I.S32.TRUNC.SAT truncates toward zero and saturates like the cast + clip for every finite x
__device__ __forceinline__ int32_t f2q31 (float x)
{
  int32_t v;
  asm ("cvt.rzi.sat.s32.f32 %0, %1;" : "=r"(v) : "f"(x * 2147483648.0f));
  return v;
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
// FM NCO of one sample (oracle tx_fm_nco): arm_q31_to_float ((int32) phi) -> arm_scale_f32 (pi) -> arm_cos_f32 / arm_sin_f32 ->
// arm_scale_f32 (level) -> arm_float_to_q15. The 1/2^31 of arm_q31_to_float and the x32768 are powers of two, folded into the constants.
__device__ __forceinline__ uint32_t fm_nco (uint32_t phi, const float *tab, float level15)
{
  const float x = __fmul_rn (__int2float_rn ((int) phi), 3.14159265f / 2147483648.0f);
  return pack_iq (__fmul_rn (arm_sincos (x, tab, true), level15), __fmul_rn (arm_sincos (x, tab, false), level15));
}

// ---- bulk asynchronous copy (TMA engine, SASS UBLKCP) + mbarrier: raw tiles are staged global -> shared without
// passing through registers, two tiles ahead of the FFTs ----
__device__ __forceinline__ uint32_t smem_u32 (const void *p) { return (uint32_t) __cvta_generic_to_shared (p); }
__device__ __forceinline__ void mbar_init (uint64_t *bar, unsigned count)
{
  asm volatile ("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32 (bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx (uint64_t *bar, unsigned bytes)
{
  asm volatile ("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32 (bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive (uint64_t *bar)
{
  sl_jitter ();
  asm volatile ("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32 (bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait (uint64_t *bar, unsigned parity)
{
  sl_jitter ();
  asm volatile (
#ifdef SL_RX_WAIT_HINT
      // the time hint lets the hardware park the warp until the phase flips instead of spinning through issue slots
      "{\n .reg .pred p;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}\n"
      ::"r"(smem_u32 (bar)), "r"(parity), "r"(SL_RX_WAIT_HINT) : "memory");
#else
      "{\n .reg .pred p;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}\n"
      ::"r"(smem_u32 (bar)), "r"(parity) : "memory");
#endif
}
__device__ __forceinline__ void bulk_g2s (void *dst, const void *src, unsigned bytes, uint64_t *bar)
{
  asm volatile ("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                ::"r"(smem_u32 (dst)), "l"(src), "r"(bytes), "r"(smem_u32 (bar)) : "memory");
}

// work-list walk shared by all roles: CTA b takes items b, b + grid, ... (segment-major), each item = up to
// kTilesPerItem consecutive tiles of one channel
struct TileIter
{
  unsigned item;
  uint32_t c, tile, tiles_left;                   // channel, tile index inside the channel, tiles left in the item (incl. this)
  __device__ __forceinline__ bool valid () const { return tiles_left != 0; }
  __device__ __forceinline__ void set_item (const KParams &P)
  {
    if (item >= P.channels * P.items_per_channel) { tiles_left = 0; return; }
    const uint32_t seg = item / P.channels;
    c = item - seg * P.channels;
    tile = seg * kTilesPerItem;
    tiles_left = min ((uint32_t) kTilesPerItem, P.tiles_per_channel - tile);
  }
  __device__ __forceinline__ void start (const KParams &P) { item = blockIdx.x; set_item (P); }
  __device__ __forceinline__ void next (const KParams &P)
  {
    tile++;
    if (--tiles_left != 0) return;
    item += gridDim.x; set_item (P);
  }
  __device__ __forceinline__ uint32_t t0 () const { return tile * kTile; }
  __device__ __forceinline__ int hops (const KParams &P) const { return (int) min ((uint32_t) kFftWarps, (P.frames - tile * kTile) / kHop); }
  __device__ __forceinline__ bool first_of_item () const { return tile % kTilesPerItem == 0; }
  __device__ __forceinline__ bool last_of_item () const { return tiles_left == 1; }
  __device__ __forceinline__ uint32_t seg () const { return tile / kTilesPerItem; }
};

// stage the raw frames of tile `it` (its hops * 384 frames and the 128 before them) into `dst`; one thread
__device__ __forceinline__ void issue_raw_tile (const KParams &P, const TileIter &it, uint32_t *dst, uint64_t *bar)
{
  const uint32_t t0 = it.t0 ();
  const unsigned body = (unsigned) it.hops (P) * kHop * 4u;
  const uint32_t *in_c = P.in + (size_t) it.c * P.frames;
  mbar_expect_tx (bar, body + kOvl * 4u);
  if (t0 == 0)
  {
    // the stream starts here: the 128 frames before it are the carried tail of the previous call
    bulk_g2s (dst, P.ovl_in + (size_t) it.c * kOvl, kOvl * 4u, bar);
    bulk_g2s (dst + kOvl, in_c, body, bar);
  }
  else
    bulk_g2s (dst, in_c + t0 - kOvl, body + kOvl * 4u, bar);
}

// exact parallel form of the oracle's release walk env_k = max(peak_k, fl(env_{k-1} * decay)) over the 32 blocks of a tile
// (lane = block). Because x -> fl(x * decay) is monotonic, fl(max(a, b) * decay) = max(fl(a * decay), fl(b * decay)):
// a Kogge-Stone max-scan whose step of distance d applies the rounded multiply d times gives bit-for-bit the value
// the sequential walk produces (31 dependent multiplies per lane instead of 32 round trips through shared memory).
__device__ __forceinline__ float env_scan (float peak, float carry, float decay, int lane)
{
  float v = (lane == 0) ? fmaxf (peak, carry * decay) : peak;
#pragma unroll
  for (int s = 0; s < 5; s++)
  {
    float w = v;
#pragma unroll
    for (int i = 0; i < (1 << s); i++) w = w * decay;
    w = __shfl_up_sync (0xffffffffu, w, 1 << s);
    if (lane >= (1 << s)) v = fmaxf (v, w);
  }
  return v;
}

// ---------------------------------------------------------------------------------------------------------------
// FFT warp: one overlap-save frame. re/im planes are this warp's private scratch.
// ---------------------------------------------------------------------------------------------------------------
// complex multiply of packed pairs, 4 packed instructions (ptxas folds the subtraction into an FFMA2 with a negated addend)
__device__ __forceinline__ void cmul2 (u64 ar, u64 ai, u64 br, u64 bi, u64 &cr, u64 &ci)
{
  cr = sub2 (mul2 (ar, br), mul2 (ai, bi));
  ci = fma2 (ar, bi, mul2 (ai, br));
}

// twiddle x[r] *= w^r, r = 1..7, from the three table entries w, w^2, w^4 (3 x 16-byte loads instead of 7: the
// shared-memory pipe is the scarce resource, the FP32 pipe has room for the 4 extra complex products)
__device__ __forceinline__ void twiddle8x2 (u64 *xr, u64 *xi, const float4 *tw3, int lane)
{
  const float4 t1 = tw3[lane], t2 = tw3[32 + lane], t4 = tw3[64 + lane];
  const u64 w1r = pk (t1.x, t1.y), w1i = pk (t1.z, t1.w), w2r = pk (t2.x, t2.y), w2i = pk (t2.z, t2.w);
  const u64 w4r = pk (t4.x, t4.y), w4i = pk (t4.z, t4.w);
  u64 w3r, w3i, w5r, w5i, w6r, w6i, w7r, w7i;
  cmul2 (w1r, w1i, w2r, w2i, w3r, w3i);
  cmul2 (w1r, w1i, w4r, w4i, w5r, w5i);
  cmul2 (w2r, w2i, w4r, w4i, w6r, w6i);
  cmul2 (w3r, w3i, w4r, w4i, w7r, w7i);
  cmul2 (xr[1], xi[1], w1r, w1i, xr[1], xi[1]);
  cmul2 (xr[2], xi[2], w2r, w2i, xr[2], xi[2]);
  cmul2 (xr[3], xi[3], w3r, w3i, xr[3], xi[3]);
  cmul2 (xr[4], xi[4], w4r, w4i, xr[4], xi[4]);
  cmul2 (xr[5], xi[5], w5r, w5i, xr[5], xi[5]);
  cmul2 (xr[6], xi[6], w6r, w6i, xr[6], xi[6]);
  cmul2 (xr[7], xi[7], w7r, w7i, xr[7], xi[7]);
}

// One 512-point forward transform of the lane's 16 points (two radix-8 butterflies per pass, packed), Stockham
// autosort, three radix-8 passes. Entry: xr/xi[r] = x[j + 64 r] for j = 2*lane (lo) and 2*lane+1 (hi); exit: the same
// indexing of the spectrum. The passes run through ONE copy of the butterfly / twiddle / gather code (rolled loop): the
// kernel is sensitive to its instruction footprint (see the note at the call site). The XOR swizzle `phys` is folded
// into per-lane bases so that every access is base-register + immediate (gathers) or one LOP3 away from it (scatters).
__device__ __forceinline__ void fft512x2 (u64 *xr, u64 *xi, float *sre, const float4 *tw, int lane)
{
  // gather x[2 lane + 64 r]: phys = ((2 lane ^ 2 (lane >> 3)) ^ 8 (r & 3)) + 64 r
  const int gl = (2 * lane) ^ (2 * (lane >> 3));
  // pass-0 scatter, Ns = 1: idx = 8 j + r, outputs r, r+1 of ONE butterfly are neighbours (transposed 2x2 in registers
  // and stored 64 bits at a time): phys (16 lane + r + 8 h) = (16 lane ^ 2 (lane & 15)) ^ (r + 8 h)
  const int sa = (16 * lane) ^ (2 * (lane & 15));
  // pass-1 scatter, Ns = 8: idx = (j / 8) * 64 + (j & 7) + 8 r: phys = (base ^ (8 (r & 3) + 2 (r >> 1))) + 32 (r >> 2)
  const int sc = 64 * (lane >> 2) + 8 * ((lane >> 2) & 3) + 2 * (lane & 3);
#pragma unroll 1
  for (int p = 0; p < 3; p++)
  {
    if (p != 0)
    {
      if (p == 1)
      {
#pragma unroll
        for (int r = 0; r < 8; r += 2)
        {
          float *qa = sre + (sa ^ r), *qb = sre + (sa ^ (r + 8));
          *reinterpret_cast<u64 *> (qa) = pair_lo (xr[r], xr[r + 1]); *reinterpret_cast<u64 *> (qa + kPlane) = pair_lo (xi[r], xi[r + 1]);
          *reinterpret_cast<u64 *> (qb) = pair_hi (xr[r], xr[r + 1]); *reinterpret_cast<u64 *> (qb + kPlane) = pair_hi (xi[r], xi[r + 1]);
        }
      }
      else
      {
#pragma unroll
        for (int r = 0; r < 8; r++)
        {
          float *q = sre + (sc ^ (8 * (r & 3) + 2 * (r >> 1))) + 32 * (r >> 2);
          *reinterpret_cast<u64 *> (q) = xr[r]; *reinterpret_cast<u64 *> (q + kPlane) = xi[r];
        }
      }
      __syncwarp ();
#pragma unroll
      for (int r = 0; r < 8; r++)
      {
        const float *q = sre + (gl ^ (8 * (r & 3))) + 64 * r;
        xr[r] = *reinterpret_cast<const u64 *> (q); xi[r] = *reinterpret_cast<const u64 *> (q + kPlane);
      }
      // twiddles: pass 1 W_64^{r (j & 7)}, pass 2 W_512^{r j}
      twiddle8x2 (xr, xi, tw + 96 * (p - 1), lane);
    }
    dft8x2 (xr, xi);
    __syncwarp ();
  }
}

// kTx = false: RX-SSB-f32 (complex I/Q in, real audio out through biquad + AGC, written L = R).
// kTx = true : TX-SSB-f32 (mic audio = L of the L = R frames in, complex I/Q out through the ALC): same overlap-save
//              filter with the mode's one-sided mask acting as band-pass + Hilbert pair, no biquad; the post warp measures
//              |I + jQ| per firmware block (arm_cmplx_mag_f32 + arm_max_f32) and applies the same gain law.
// kMod (TX only, SLB_CHAIN_TX_F32): channels on the AM and FM slots are modulated as DESIGN.md §3.4 describes; the other slots run the
//              TX-SSB code unchanged.
template <bool kTx, bool kMod = false>
#ifdef SL_RX_MAXNREG
__global__ void __maxnreg__ (SL_RX_MAXNREG) ssb_f32_kernel
#else
__global__ void __launch_bounds__ (kThreads, SL_RX_CTAS) ssb_f32_kernel
#endif
 (const __grid_constant__ KParams P)
{
  typedef Smem<kTx, kMod> S;
  constexpr int kAB = S::kAudioBufs;
  extern __shared__ __align__ (128) unsigned char smem[];
  float *sScratch = reinterpret_cast<float *> (smem + S::scratch);
  float *sAudio = reinterpret_cast<float *> (smem + S::audio);
  uint32_t *sRaw = reinterpret_cast<uint32_t *> (smem + S::raw);
  float4 *sTw = reinterpret_cast<float4 *> (smem + S::tw);
  uint64_t *sFull = reinterpret_cast<uint64_t *> (smem + S::bars), *sEmpty = sFull + kRawBufs;
  // audio tiles: aFull[b] completes when the four FFT warps have each stored their frame, aEmpty[b] when the recurrence
  // warp has taken the tile into registers. mbarriers, not named barriers: a named barrier would also make the four FFT
  // warps rendezvous with EACH OTHER once per tile (ncu: 23 % of their time), although they only depend on the consumer.
  uint64_t *aFull = sEmpty + kRawBufs, *aEmpty = aFull + kAB;

  const int tid = threadIdx.x, lane = tid & 31;
  // Warp w of a CTA runs on scheduler (SMSP) w % 4, so a fixed "warp 4 = recurrence warp" would stack the recurrence
  // warps of all resident CTAs on SMSP 0 (measured: that scheduler became the bottleneck). The role rotates with the
  // CTA index instead; `warp` below is the FFT frame index (0..3) or kFftWarps for the recurrence role.
  const int hw_warp = tid >> 5, rec_warp = (blockIdx.x + blockIdx.x / 148u) % (kFftWarps + 1);
  const int warp = (hw_warp == rec_warp) ? kFftWarps : (hw_warp < rec_warp ? hw_warp : hw_warp - 1);
  for (int i = tid; i < 6 * 32; i += kThreads) sTw[i] = P.twiddle[i];
  float *sSin = reinterpret_cast<float *> (smem + S::sin);
  if constexpr (kMod)
    for (int i = tid; i < 513; i += kThreads) sSin[i] = P.sin513[i];
  if (tid == 0)
  {
#pragma unroll
    for (int b = 0; b < kRawBufs; b++) { mbar_init (sFull + b, 1); mbar_init (sEmpty + b, kFftWarps); }
#pragma unroll
    for (int b = 0; b < kAB; b++) { mbar_init (aFull + b, kFftWarps); mbar_init (aEmpty + b, 1); }
    asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads ();

  unsigned tile_seq = 0;                          // tiles this CTA has pushed through the audio buffers
  int abuf = 0;                                   // = tile_seq % kAB
  unsigned ause = 0;                              // = tile_seq / kAB: how often audio buffer `abuf` has been used before

  if (warp < kFftWarps)
  {
    // =========================================== FFT warps ===========================================
    float *sre = sScratch + warp * 2 * kPlane;              // re plane; the im plane follows it
    const u64 NB = pk (-8421376.0f, -8421376.0f);
    TileIter it; it.start (P);
    TileIter itl = it;                            // warp 0 is also the loader: its second iterator runs kRawBufs tiles ahead
    if (warp == 0)
    {
#pragma unroll
      for (int b = 0; b < kRawBufs; b++)
        if (itl.valid ())
        {
          if (lane == 0) issue_raw_tile (P, itl, sRaw + b * kRawWords, sFull + b);
          itl.next (P);
        }
    }
    for (; it.valid (); tile_seq++)
    {
      const int rbuf = (kRawBufs == 1) ? 0 : (int) (tile_seq & 1);
      const unsigned rpar = (kRawBufs == 1) ? (tile_seq & 1) : ((tile_seq >> 1) & 1);
      const bool mine = warp < it.hops (P);
      const uint32_t c = it.c, t0 = it.t0 ();
      u64 xr[8], xi[8];
      mbar_wait (sFull + rbuf, rpar);                                              // the raw tile has landed
      if (mine)
      {
        // ---- unpack (arm_q15_to_float): the frame covers stream samples [ts, ts + 512), ts = t0 + 384 w - 128; the lane
        // takes the adjacent pair 2*lane, 2*lane+1 of every 64-sample row. int16 -> float exactly through the mantissa of
        // 2^23 (no conversion pipe); the 1/32768 of arm_q15_to_float is a power of two and is folded into the mask.
        const uint2 *rawp = reinterpret_cast<const uint2 *> (sRaw + rbuf * kRawWords + warp * kHop) + lane;
        uint2 tail6 = make_uint2 (0u, 0u), tail7 = tail6;
#pragma unroll
        for (int r = 0; r < 8; r++)
        {
          const uint2 v = rawp[32 * r];
          if (r == 6) tail6 = v;
          if (r == 7) tail7 = v;
          const uint32_t a = v.x ^ 0x80008000u, b = v.y ^ 0x80008000u;
          xr[r] = add2 (pk (__uint_as_float (__byte_perm (a, 0x4B000000u, 0x7610)), __uint_as_float (__byte_perm (b, 0x4B000000u, 0x7610))), NB);
          // TX: the mic is the L half of an L = R frame
          xi[r] = kTx ? 0ull : add2 (pk (__uint_as_float (__byte_perm (a, 0x4B000000u, 0x7632)), __uint_as_float (__byte_perm (b, 0x4B000000u, 0x7632))), NB);
        }
        // carry the raw tail of the stream for the next call (this launch reads ovl_in and writes ovl_out)
        if (t0 + (warp + 1) * kHop == P.frames)
        {
          uint2 *dst = reinterpret_cast<uint2 *> (P.ovl_out + (size_t) c * kOvl);
          dst[lane] = tail6; dst[lane + 32] = tail7;                              // rows 6, 7 = the last 128 frames
        }
      }
      __syncwarp ();
      if (lane == 0) mbar_arrive (sEmpty + rbuf);                                  // this warp no longer needs raw[rbuf]
      const int slot = P.mask_slot[c];
      const float4 *mask = P.masks + (size_t) slot * 256;
      const bool envelope = !kTx && slot == kAmMaskSlot;                           // AM: |z| instead of Re z
      it.next (P);
      // ---- forward FFT (arm_cfft_f32 forward; pass 0 needs no twiddles), spectral mask (arm_cmplx_mult_cmplx_f32), then
      // the inverse transform as a forward transform of the re/im-swapped spectrum: N ifft(Y) = swap(fft(swap(Y))), so
      // Re ifft(Y) = Im fft(swap Y) / N (1/N is in the mask). Both transforms run through ONE copy of the FFT code (a
      // rolled two-trip loop): the unrolled kernel was bound by instruction fetch, not by any execution pipe (ncu:
      // gcc__cache_requests_type_instruction at 93 % of peak with a 64 KB body against the 32 KB L1.5 instruction cache).
#pragma unroll 1
      for (int dir = 0; dir < 2; dir++)
      {
        if (mine)
        {
#ifndef SL_RX_ABLATE_FFT                                                            // (profiling aid: time the recurrence side alone)
          fft512x2 (xr, xi, sre, sTw, lane);
#endif
        }
        if (dir == 0)
        {
          if (warp == 0 && itl.valid ())
          {
            // ---- refill raw[rbuf] with a later tile, as soon as the four warps have unpacked the current one
            if (lane == 0)
            {
              mbar_wait (sEmpty + rbuf, rpar);
              asm volatile ("fence.proxy.async.shared::cta;" ::: "memory");
              issue_raw_tile (P, itl, sRaw + rbuf * kRawWords, sFull + rbuf);
            }
            itl.next (P);
            __syncwarp ();
          }
          if (mine)
          {
#pragma unroll
            for (int r = 0; r < 8; r++)
            {
              const float4 h = __ldg (mask + r * 32 + lane);
              const u64 hr = pk (h.x, h.y), hi = pk (h.z, h.w);
              const u64 yr = sub2 (mul2 (xr[r], hr), mul2 (xi[r], hi));
              const u64 yi = fma2 (xr[r], hi, mul2 (xi[r], hr));
              xr[r] = yi; xi[r] = yr;                                              // swap
            }
          }
        }
      }
      // ---- hand the audio of this frame to the recurrence warp: keep the last 384 outputs (rows r >= 2)
      if (ause != 0) mbar_wait (aEmpty + abuf, (ause - 1) & 1);                    // wait until the buffer was drained
      if (mine)
      {
        float *a = sAudio + abuf * S::kAudioWords;
#pragma unroll
        for (int r = 2; r < 8; r++)
        {
          const int n = warp * kHop + 2 * lane + 64 * (r - 2);                     // even: n and n+1 share run and block
          const int blk = n / kAgcBlock, i = n - blk * kAgcBlock;
          // (xr, xi) hold fft(swap Y) = swap(N ifft(Y)): real part of the inverse transform in xi, imaginary part in xr
          if (kTx)
            *reinterpret_cast<float4 *> (a + blk * kTxBlkStride + 2 * i) = make_float4 (lo_of (xi[r]), lo_of (xr[r]), hi_of (xi[r]), hi_of (xr[r]));
          else
          {
            const int half = i / kRun, k = i - half * kRun;
            const int pos = blk * kBlkStride + 2 * k + half;                       // runs A/B of a block are interleaved
            float v0 = lo_of (xi[r]), v1 = hi_of (xi[r]);
            if (envelope)
            {
              // arm_cmplx_mag_f32.c:72: sqrt (re * re + im * im), each product rounded (the oracle build does not contract)
              const float u0 = lo_of (xr[r]), u1 = hi_of (xr[r]);
              v0 = __fsqrt_rn (__fadd_rn (__fmul_rn (v0, v0), __fmul_rn (u0, u0)));
              v1 = __fsqrt_rn (__fadd_rn (__fmul_rn (v1, v1), __fmul_rn (u1, u1)));
            }
            a[pos] = v0; a[pos + 2] = v1;
          }
        }
      }
      __syncwarp ();
      if (lane == 0) mbar_arrive (aFull + abuf);
      if (++abuf == kAB) { abuf = 0; ause++; }
    }
  }
  else if constexpr (kTx)
  {
    // ===================================== TX post warp: ALC =====================================
    // Lane l owns firmware block l of the tile (48 complex samples = 192 output bytes). Pass 1 finds the block peak of
    // |I + jQ|, the envelope walk is the AGC's, pass 2 re-reads the tile, scales, packs and stores.
    // kMod, AM / FM channels: the peak is max |Re z| (arm_abs_f32 + arm_max_f32) and pass 2 runs the modulator of the channel's slot.
    const float decay = P.agc_decay;
    float env = 0.f;
    uint32_t phase = 0;                                                            // FM phase accumulator (kMod), carried like env
    TileIter it; it.start (P);
    for (; it.valid (); it.next (P), tile_seq++)
    {
      const uint32_t c = it.c, t0 = it.t0 ();
      const int nblk = it.hops (P) * (kHop / kAgcBlock);
      const float4 *blk = reinterpret_cast<const float4 *> (sAudio + abuf * S::kAudioWords + lane * kTxBlkStride);
      // 0: SSB-style, 1: AM, 2: FM (uniform across the warp: one channel per tile)
      int mod = 0;
      if constexpr (kMod) { const int slot = P.mask_slot[c]; mod = slot == kAmMaskSlot ? 1 : slot == kFmMaskSlot ? 2 : 0; }
      mbar_wait (aFull + abuf, ause & 1);                                          // I/Q tile is complete
      // arm_cmplx_mag_f32.c:72 : sqrt(re*re + im*im), each product rounded (no contraction in the oracle build);
      // arm_max_f32 over the block. sqrt is monotonic and correctly rounded, so max(sqrt) = sqrt(max).
      float m2 = 0.f;
      if (mod == 0)
      {
#pragma unroll
        for (int k = 0; k < kAgcBlock / 2; k++)
        {
          const float4 v = blk[k];
          m2 = fmaxf (m2, fmaxf (__fadd_rn (__fmul_rn (v.x, v.x), __fmul_rn (v.y, v.y)), __fadd_rn (__fmul_rn (v.z, v.z), __fmul_rn (v.w, v.w))));
        }
      }
      else
      {
#pragma unroll
        for (int k = 0; k < kAgcBlock / 2; k++)
        {
          const float4 v = blk[k];
          m2 = fmaxf (m2, fmaxf (fabsf (v.x), fabsf (v.z)));
        }
      }
      if (it.first_of_item ())
      {
        if (lane == 0)
        {
          const unsigned want = P.flag_base + it.seg ();
          for (unsigned spins = 0; ld_relaxed (P.flag + c) != want; __nanosleep (32))
            if (++spins > kSpinLimit) __trap ();                                   // (seconds: the predecessor tile never arrived — an error, not a hung GPU)
          (void) ld_acquire (P.flag + c);
        }
        __syncwarp ();
        env = __ldcg (P.state + (size_t) c * 8 + 4);
        if constexpr (kMod) phase = __ldcg (reinterpret_cast<const unsigned *> (P.state) + (size_t) c * 8 + 5);
      }
      const float e = env_scan (mod == 0 ? __fsqrt_rn (m2) : m2, env, decay, lane);
      env = __shfl_sync (0xffffffffu, e, nblk - 1);
      const float target = mod == 0 ? P.agc_target : mod == 1 ? P.am_depth : P.fm_target;
      const float g = fminf (__fdiv_rn (target, fmaxf (e, P.agc_floor)), P.agc_gmax);
      uint32_t phi = 0;                                                            // FM: phase before the lane's first sample
      if (kMod && mod == 2)
      {
        // phi[n] = phi[n-1] + inc[n] mod 2^32 is an integer prefix sum, so it is associative: each lane sums its block's increments,
        // a warp exclusive scan over the blocks plus the carried phase gives every block's start phase, bit for bit the sequential walk
        uint32_t sum = 0;
#pragma unroll
        for (int k = 0; k < kAgcBlock / 2; k++)
        {
          const float4 v = blk[k];
          sum += (uint32_t) f2q31 (__fmul_rn (v.x, g)) + (uint32_t) f2q31 (__fmul_rn (v.z, g));
        }
        uint32_t incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1)
        {
          const uint32_t o = __shfl_up_sync (0xffffffffu, incl, d);
          if (lane >= d) incl += o;
        }
        phi = phase + incl - sum;
        phase += __shfl_sync (0xffffffffu, incl, nblk - 1);
      }
      if (lane < nblk)
      {
        if (P.audio_dbg)
        {
          float4 *adbg = reinterpret_cast<float4 *> (P.audio_dbg + 2 * ((size_t) c * P.frames + t0 + lane * kAgcBlock));
#pragma unroll
          for (int k = 0; k < kAgcBlock / 2; k++) adbg[k] = blk[k];
        }
        if (P.gain_dbg) P.gain_dbg[(size_t) c * (P.frames / kAgcBlock) + t0 / kAgcBlock + lane] = g;
        uint4 *dst = reinterpret_cast<uint4 *> (P.out + (size_t) c * P.frames + t0 + lane * kAgcBlock);
        if (mod == 0)
        {
          const float g15 = g * 32768.0f;                                         // arm_scale_f32 then arm_float_to_q15: exact fold
#pragma unroll
          for (int k = 0; k < kAgcBlock / 4; k++)
          {
            const float4 u = blk[2 * k], v = blk[2 * k + 1];
            st_na (dst + k, make_uint4 (pack_iq (u.x * g15, u.y * g15), pack_iq (u.z * g15, u.w * g15), pack_iq (v.x * g15, v.y * g15), pack_iq (v.z * g15, v.w * g15)));
          }
        }
        else if (kMod && mod == 1)
        {
          // AM: arm_scale_f32 (g) -> arm_offset_f32 (1) -> arm_scale_f32 (carrier) -> arm_float_to_q15 as I, Q = 0; each op rounded in
          // the oracle's order (only the x32768 is folded, into the carrier)
          const float c15 = P.am_carrier15;
#pragma unroll
          for (int k = 0; k < kAgcBlock / 4; k++)
          {
            const float4 u = blk[2 * k], v = blk[2 * k + 1];
            st_na (dst + k, make_uint4 (pack_iq (__fmul_rn (__fadd_rn (__fmul_rn (u.x, g), 1.0f), c15), 0.f), pack_iq (__fmul_rn (__fadd_rn (__fmul_rn (u.z, g), 1.0f), c15), 0.f),
                                        pack_iq (__fmul_rn (__fadd_rn (__fmul_rn (v.x, g), 1.0f), c15), 0.f), pack_iq (__fmul_rn (__fadd_rn (__fmul_rn (v.z, g), 1.0f), c15), 0.f)));
          }
        }
        else if (kMod)
        {
          // FM: arm_scale_f32 (g) -> arm_float_to_q31 = the phase increment; the accumulator walks the block from its start phase
          const float l15 = P.fm_level15;
          uint4 *pdbg = P.phase_dbg ? reinterpret_cast<uint4 *> (P.phase_dbg + (size_t) c * P.frames + t0 + lane * kAgcBlock) : nullptr;
#pragma unroll 2
          for (int k = 0; k < kAgcBlock / 4; k++)
          {
            const float4 u = blk[2 * k], v = blk[2 * k + 1];
            const uint32_t p0 = phi + (uint32_t) f2q31 (__fmul_rn (u.x, g));
            const uint32_t p1 = p0 + (uint32_t) f2q31 (__fmul_rn (u.z, g));
            const uint32_t p2 = p1 + (uint32_t) f2q31 (__fmul_rn (v.x, g));
            const uint32_t p3 = p2 + (uint32_t) f2q31 (__fmul_rn (v.z, g));
            phi = p3;
            if (pdbg) pdbg[k] = make_uint4 (p0, p1, p2, p3);
            st_na (dst + k, make_uint4 (fm_nco (p0, sSin, l15), fm_nco (p1, sSin, l15), fm_nco (p2, sSin, l15), fm_nco (p3, sSin, l15)));
          }
        }
      }
      __syncwarp ();
      if (lane == 0) mbar_arrive (aEmpty + abuf);                                  // the tile has been consumed
      if (++abuf == kAB) { abuf = 0; ause++; }
      if (it.last_of_item () && lane == 0)
      {
        __stcg (P.state + (size_t) c * 8 + 4, env);
        if constexpr (kMod) __stcg (reinterpret_cast<unsigned *> (P.state) + (size_t) c * 8 + 5, phase);
        __threadfence ();
        st_release (P.flag + c, P.flag_base + it.seg () + 1u);
      }
    }
  }
  else
  {
    // ======================================= recurrence warp =======================================
    // Lane l owns AGC block l of the tile (48 samples) as TWO runs of 24 evaluated together in packed FP32x2:
    // lo = run A (samples 0..23 of the block), hi = run B (24..47).
    const float *cf = P.tab.coef;
    u64 c2[10];
#pragma unroll
    for (int i = 0; i < 10; i++) c2[i] = pk (cf[i], cf[i]);
    const float decay = P.agc_decay;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, env = 0.f;                       // carried state (uniform across lanes)
    TileIter it; it.start (P);
    for (; it.valid (); it.next (P), tile_seq++)
    {
      const uint32_t c = it.c, t0 = it.t0 ();
      const int nblk = it.hops (P) * (kHop / kAgcBlock);
      const float *blk = sAudio + abuf * S::kAudioWords + lane * kBlkStride;
      mbar_wait (aFull + abuf, ause & 1);                                          // audio tile is complete

      // zero-state response of the cascade over both runs; per-sample recurrences as
      // arm_biquad_cascade_df2T_f32.c:551-562:  y = b0 x + d1;  d1 = (b1 x + a1 y) + d2;  d2 = b2 x + a2 y
      // ((b1 x + d2) is formed before y is known, so each stage costs two dependent FMAs per sample)
      u64 y[kRun];
      u64 d1a = 0ull, d2a = 0ull, d1b = 0ull, d2b = 0ull;
#pragma unroll
      for (int k = 0; k < kRun; k++)
      {
        const u64 x = *reinterpret_cast<const u64 *> (blk + 2 * k);
        const u64 y0 = fma2 (c2[0], x, d1a);
        d1a = fma2 (c2[3], y0, fma2 (c2[1], x, d2a));
        d2a = fma2 (c2[4], y0, mul2 (c2[2], x));
        const u64 y1 = fma2 (c2[5], y0, d1b);
        d1b = fma2 (c2[8], y1, fma2 (c2[6], y0, d2b));
        d2b = fma2 (c2[9], y1, mul2 (c2[7], y0));
        y[k] = y1;
      }
      __syncwarp ();
      if (lane == 0) mbar_arrive (aEmpty + abuf);                                  // the audio tile now lives in registers
      if (++abuf == kAB) { abuf = 0; ause++; }
      if (it.first_of_item ())
      {
        // state of the previous segment of this channel (segment-major dealing makes the wait a formality)
        if (lane == 0)
        {
          const unsigned want = P.flag_base + it.seg ();
          for (unsigned spins = 0; ld_relaxed (P.flag + c) != want; __nanosleep (32))
            if (++spins > kSpinLimit) __trap ();                                   // (seconds: the predecessor tile never arrived — an error, not a hung GPU)
          (void) ld_acquire (P.flag + c);
        }
        __syncwarp ();
        const float *stc = P.state + (size_t) c * 8;
        s0 = __ldcg (stc + 0); s1 = __ldcg (stc + 1); s2 = __ldcg (stc + 2); s3 = __ldcg (stc + 3); env = __ldcg (stc + 4);
      }
      // zero-start end state of the whole block: zB + M24 zA
      const float a0 = lo_of (d1a), a1 = lo_of (d2a), a2 = lo_of (d1b), a3 = lo_of (d2b);
      float z0, z1, z2, z3;
      {
        const float *M = P.tab.Mpow[0];
        z0 = hi_of (d1a) + (M[0] * a0 + M[1] * a1 + M[2] * a2 + M[3] * a3);
        z1 = hi_of (d2a) + (M[4] * a0 + M[5] * a1 + M[6] * a2 + M[7] * a3);
        z2 = hi_of (d1b) + (M[8] * a0 + M[9] * a1 + M[10] * a2 + M[11] * a3);
        z3 = hi_of (d2b) + (M[12] * a0 + M[13] * a1 + M[14] * a2 + M[15] * a3);
      }
      // end state of block l given all earlier blocks: z_l = zs_l + M48 z_{l-1}; lane 0 folds the carried state in
      if (lane == 0)
      {
        const float *M = P.tab.Mpow[1];
        z0 += M[0] * s0 + M[1] * s1 + M[2] * s2 + M[3] * s3;
        z1 += M[4] * s0 + M[5] * s1 + M[6] * s2 + M[7] * s3;
        z2 += M[8] * s0 + M[9] * s1 + M[10] * s2 + M[11] * s3;
        z3 += M[12] * s0 + M[13] * s1 + M[14] * s2 + M[15] * s3;
      }
#pragma unroll
      for (int k = 0; k < 5; k++)
      {
        const int d = 1 << k;
        const float *M = P.tab.Mpow[k + 1];
        const float p0 = __shfl_up_sync (0xffffffffu, z0, d), p1 = __shfl_up_sync (0xffffffffu, z1, d);
        const float p2 = __shfl_up_sync (0xffffffffu, z2, d), p3 = __shfl_up_sync (0xffffffffu, z3, d);
        if (lane >= d)
        {
          z0 += M[0] * p0 + M[1] * p1 + M[2] * p2 + M[3] * p3;
          z1 += M[4] * p0 + M[5] * p1 + M[6] * p2 + M[7] * p3;
          z2 += M[8] * p0 + M[9] * p1 + M[10] * p2 + M[11] * p3;
          z3 += M[12] * p0 + M[13] * p1 + M[14] * p2 + M[15] * p3;
        }
      }
      // start state of run A = end state of the previous block; of run B = zA + M24 (start of A)
      float b0 = __shfl_up_sync (0xffffffffu, z0, 1), b1 = __shfl_up_sync (0xffffffffu, z1, 1);
      float b2 = __shfl_up_sync (0xffffffffu, z2, 1), b3 = __shfl_up_sync (0xffffffffu, z3, 1);
      if (lane == 0) { b0 = s0; b1 = s1; b2 = s2; b3 = s3; }
      u64 q0, q1, q2, q3;
      {
        const float *M = P.tab.Mpow[0];
        q0 = pk (b0, a0 + (M[0] * b0 + M[1] * b1 + M[2] * b2 + M[3] * b3));
        q1 = pk (b1, a1 + (M[4] * b0 + M[5] * b1 + M[6] * b2 + M[7] * b3));
        q2 = pk (b2, a2 + (M[8] * b0 + M[9] * b1 + M[10] * b2 + M[11] * b3));
        q3 = pk (b3, a3 + (M[12] * b0 + M[13] * b1 + M[14] * b2 + M[15] * b3));
      }
      // carried state for the next tile = end state of the last block
      s0 = __shfl_sync (0xffffffffu, z0, nblk - 1); s1 = __shfl_sync (0xffffffffu, z1, nblk - 1);
      s2 = __shfl_sync (0xffffffffu, z2, nblk - 1); s3 = __shfl_sync (0xffffffffu, z3, nblk - 1);

      // add the zero-input response of the true start states; block peak (arm_abs_f32 + arm_max_f32)
      float pk0 = 0.f, pk1 = 0.f;
#pragma unroll
      for (int k = 0; k < kRun; k++)
      {
        const float *C = P.tab.Cresp[k];
        y[k] = fma2 (pk (C[0], C[0]), q0, fma2 (pk (C[1], C[1]), q1, fma2 (pk (C[2], C[2]), q2, fma2 (pk (C[3], C[3]), q3, y[k]))));
        pk0 = fmaxf (pk0, fabsf (lo_of (y[k]))); pk1 = fmaxf (pk1, fabsf (hi_of (y[k])));
      }
      // AGC envelope: the oracle's sequential walk over the blocks, evaluated as an exact max-scan (env_scan above)
      const float e = env_scan (fmaxf (pk0, pk1), env, decay, lane);
      env = __shfl_sync (0xffffffffu, e, nblk - 1);
      const float g = fminf (__fdiv_rn (P.agc_target, fmaxf (e, P.agc_floor)), P.agc_gmax);
      if (lane < nblk)
      {
        if (P.audio_dbg)
        {
          float *adbg = P.audio_dbg + (size_t) c * P.frames + t0 + lane * kAgcBlock;
#pragma unroll
          for (int k = 0; k < kRun; k++) { adbg[k] = lo_of (y[k]); adbg[kRun + k] = hi_of (y[k]); }
        }
        if (P.gain_dbg) P.gain_dbg[(size_t) c * (P.frames / kAgcBlock) + t0 / kAgcBlock + lane] = g;
        // gain (arm_scale_f32), pack (arm_float_to_q15) and store: the lane's block is 192 contiguous bytes
        const float g15 = g * 32768.0f;                                           // exact: power of two
        uint4 *dst = reinterpret_cast<uint4 *> (P.out + (size_t) c * P.frames + t0 + lane * kAgcBlock);
#pragma unroll
        for (int k = 0; k < kRun; k += 4)
        {
          st_na (dst + k / 4, make_uint4 (pack_lr (lo_of (y[k]) * g15), pack_lr (lo_of (y[k + 1]) * g15), pack_lr (lo_of (y[k + 2]) * g15), pack_lr (lo_of (y[k + 3]) * g15)));
          st_na (dst + (kRun + k) / 4, make_uint4 (pack_lr (hi_of (y[k]) * g15), pack_lr (hi_of (y[k + 1]) * g15), pack_lr (hi_of (y[k + 2]) * g15), pack_lr (hi_of (y[k + 3]) * g15)));
        }
      }
      if (it.last_of_item () && lane == 0)
      {
        float *stw = P.state + (size_t) c * 8;
        __stcg (stw + 0, s0); __stcg (stw + 1, s1); __stcg (stw + 2, s2); __stcg (stw + 3, s3); __stcg (stw + 4, env);
        __threadfence ();
        st_release (P.flag + c, P.flag_base + it.seg () + 1u);
      }
    }
  }
}

}  // namespace

uint32_t rx_ssb_f32_launches_per_call () { return 1u; }
// the per-channel flag advances by one per segment (= kTilesPerItem tiles)
uint32_t rx_ssb_f32_tiles (uint32_t frames)
{
  const uint32_t tiles = (frames + kTile - 1) / kTile;
  return (tiles + kTilesPerItem - 1) / kTilesPerItem;
}

// twiddles in the per-lane packed layout the kernel reads with one 16-byte load: [pass][e][lane] = (WrA, WrB, WiA, WiB)
// for the lane's butterflies jA = 2 lane, jB = 2 lane + 1 and the powers w^1, w^2, w^4 (e = 0, 1, 2) of the
// butterfly's base twiddle; pass 1: w = W_64^{j & 7}, pass 2: w = W_512^{j}
void rx_ssb_f32_pack_twiddles (float *out /* kTwiddleFloats */)
{
  const double two_pi = 6.283185307179586476925286766559;
  for (int pass = 0; pass < 2; pass++)
    for (int e = 0; e < 3; e++)
      for (int lane = 0; lane < 32; lane++)
      {
        float *o = out + ((pass * 3 + e) * 32 + lane) * 4;
        for (int b = 0; b < 2; b++)
        {
          const int j = 2 * lane + b, r = 1 << e;
          const int ex = (pass == 0) ? (r * (j & 7) * 8) % kN : (r * j) % kN;
          const double a = -two_pi * (double) ex / (double) kN;
          o[b] = (float) std::cos (a); o[2 + b] = (float) std::sin (a);
        }
      }
}
// mask (already scaled by the caller) in the packed layout: [r][lane] = (HrA, HrB, HiA, HiB), k = 2 lane + b + 64 r
void rx_ssb_f32_pack_mask (const float *mask_re_im /* 2*512 */, float scale, float *out /* 8*32*4 */)
{
  for (int r = 0; r < 8; r++)
    for (int lane = 0; lane < 32; lane++)
      for (int b = 0; b < 2; b++)
      {
        const int k = 2 * lane + b + 64 * r;
        out[(r * 32 + lane) * 4 + b] = mask_re_im[2 * k] * scale;
        out[(r * 32 + lane) * 4 + 2 + b] = mask_re_im[2 * k + 1] * scale;
      }
}

int launch_rx_ssb_f32 (const RxF32Launch &L, int sm_count, void *stream_)
{
  cudaStream_t stream = (cudaStream_t) stream_;
  if (L.frames % kHop != 0 || L.frames == 0 || L.channels == 0) return (int) cudaErrorInvalidValue;
  KParams P;
  P.in = reinterpret_cast<const uint32_t *> (L.in); P.out = reinterpret_cast<uint32_t *> (L.out);
  P.audio_dbg = L.audio_dbg; P.gain_dbg = L.gain_dbg;
  P.ovl_in = reinterpret_cast<const uint32_t *> (L.ovl_in); P.ovl_out = reinterpret_cast<uint32_t *> (L.ovl_out);
  P.state = L.state; P.flag = L.flag;
  P.masks = reinterpret_cast<const float4 *> (L.masks); P.mask_slot = L.mask_slot;
  P.twiddle = reinterpret_cast<const float4 *> (L.twiddle);
  P.flag_base = L.flag_base; P.channels = L.channels; P.frames = L.frames;
  P.tiles_per_channel = (L.frames + kTile - 1) / kTile;
  P.items_per_channel = (P.tiles_per_channel + kTilesPerItem - 1) / kTilesPerItem;
  P.agc_target = L.agc_target; P.agc_decay = L.agc_decay; P.agc_floor = L.agc_floor; P.agc_gmax = L.agc_gmax;
  P.am_depth = L.am_depth; P.am_carrier15 = L.am_carrier * 32768.0f; P.fm_target = L.fm_target; P.fm_level15 = L.fm_level * 32768.0f;
  P.phase_dbg = L.phase_dbg; P.sin513 = L.sin513;
  P.tab = *L.tables;

  // the bulk copies need 16-byte aligned sources: frames % 384 == 0 keeps every channel row and every tile start aligned
  if ((reinterpret_cast<uintptr_t> (L.in) | reinterpret_cast<uintptr_t> (L.ovl_in)) & 15u) return (int) cudaErrorMisalignedAddress;
  if (L.tx_mod && (!L.tx || !L.sin513)) return (int) cudaErrorInvalidValue;
  const size_t smem = L.tx_mod ? Smem<true, true>::bytes : L.tx ? Smem<true>::bytes : Smem<false>::bytes;
  const void *fn = L.tx_mod ? (const void *) ssb_f32_kernel<true, true> : L.tx ? (const void *) ssb_f32_kernel<true> : (const void *) ssb_f32_kernel<false>;
  cudaError_t e = cudaFuncSetAttribute (fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
  if (e != cudaSuccess) return (int) e;
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor (&per_sm, fn, kThreads, smem);
  if (e != cudaSuccess) return (int) e;
  if (per_sm < 1) per_sm = 1;
  const uint64_t items = (uint64_t) L.channels * P.items_per_channel;
  uint64_t grid = (uint64_t) sm_count * per_sm;      // all CTAs co-resident: the segment hand-over may spin
  if (grid > items) grid = items;
  // (Measured, profiles/r01_summary.md: throughput is proportional to the number of resident CTAs — 592: 155, 512: 132,
  // 448: 117 Gsamples/s — i.e. every CTA is an internally latency-bound pipeline; shrinking the grid to make the segment
  // hand-over trivially satisfied costs more than the polling it removes.)
  if (const char *g = std::getenv ("SELENITE_B200_RX_GRID")) { const long v = std::atol (g); if (v > 0 && (uint64_t) v <= (uint64_t) sm_count * per_sm) grid = (uint64_t) v; }   // profiling aid
  // Cooperative launch: consecutive segments of a channel hand over through a flag the successor polls, so every CTA of the
  // grid must be resident at once. The cooperative attribute makes the driver schedule the grid as a gang — next to other
  // work on the device (a second stream of this library, another context, MPS) the launch waits for room or fails with
  // cudaErrorCooperativeLaunchTooLarge, where a plain launch could leave resident CTAs spinning on one that never starts.
  cudaLaunchConfig_t lc{};
  lc.gridDim = dim3 ((unsigned) grid); lc.blockDim = dim3 (kThreads); lc.dynamicSmemBytes = smem; lc.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeCooperative; at[0].val.cooperative = 1;
  lc.attrs = at; lc.numAttrs = 1;
  e = L.tx_mod ? cudaLaunchKernelEx (&lc, ssb_f32_kernel<true, true>, P)
      : L.tx ? cudaLaunchKernelEx (&lc, ssb_f32_kernel<true>, P) : cudaLaunchKernelEx (&lc, ssb_f32_kernel<false>, P);
  return (int) (e != cudaSuccess ? e : cudaGetLastError ());
}

}  // namespace sl
