// RX-SSB-f32 on the 5th-generation tensor cores (tcgen05 + TMEM), one kernel, every sample crosses HBM once.
//
// The oracle chain filters by overlap-save: arm_q15_to_float -> arm_cfft_f32(512) -> arm_cmplx_mult_cmplx_f32 with the
// mode's mask -> arm_cfft_f32 inverse -> keep 384 (DESIGN.md §3.2), then arm_biquad_cascade_df2T_f32. The mask is the DFT
// of a 129-tap complex filter, so the first part IS the linear convolution
//   Re y[n] = sum_{d=0..128} hr[d] I[n-d] - hi[d] Q[n-d]
// of int16 samples with fixed taps, and the biquad is linear: inside one firmware block of 48 samples its output is
// (zero-state response to the block's y) + (zero-input response of the state at the block start). Everything up to and
// including the zero-state response, and the block's end state from a zero start, is ONE fixed linear map of the 176-frame
// raw window — a dense contraction, the case the north-star reserves the tensor cores for. It is evaluated in integers:
// x = 256 xh + xl (signed high byte, unsigned low byte), map entries quantised to 24 bits as three balanced base-256
// digits, all six digit products by tcgen05.mma kind::i8 into four int32 TMEM accumulators by weight (2^24, 2^16, 2^8, 1).
// No product is dropped: the only deviation from infinite precision is the 2^-24 quantisation of the map, of the order
// of one float32 epsilon of the INPUT level like the oracle's own FFT noise (tolerances: DESIGN.md §3.6).
//
//   MMA shape: M = 128 rows = 8 channels (the 8 rows of a core matrix) x 16 consecutive firmware blocks (row groups),
//   N = 208 (high data byte: 52 outputs of a block = 48 audio + 4 end-state, x 4 map digits) or 160 (low data byte: the top 3 digits + 4 rows), K = 32 bytes = 16 frames (I, Q bytes) per
//   instruction, 11 K-steps cover the 128 + 48 frame window. The A operand is the byte plane of the channel group's samples,
//   ONCE: row group q is the same plane 48 frames (6 sixteen-byte chunks) further on, so the descriptor's row-group stride
//   (SBO = 768 B) makes the 16 row groups alias one contiguous buffer — no Toeplitz expansion of the data, only of the
//   (constant) map. An SS-mode MMA is bound by its operand fetch ((4 KB of A + 32 N bytes of B) at ~74 B/clk, measured): N = 160
//   instead of 144 costs 8 clocks per MMA and takes the whole per-sample recurrence off the CUDA cores.
//
//   Roles (warps): 2 x 4 epilogue warps (TMEM lane = (block q, channel j): int32 -> float, chain the 16 block end states,
//   add the zero-input response, AGC envelope walk, gain, float -> q15, 192-byte stores), 2 converter warps (raw int16 ->
//   byte planes, PRMT only), 1 MMA issuer (one elected lane, 22 tcgen05.mma per supertile), 1 bulk-copy producer.
//   mbarrier pipelines: raw stages, A planes (2), TMEM accumulators (2), biquad / envelope carry between supertiles.
//
// Oracle stage per box as in sl_rx_ssb_f32.cu; the chain sits where the firmware would call it (Core/Src/dsp_if.c:286-289).
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdlib>
#include "sl_internal.h"

namespace sl {

namespace {

constexpr int kJ = kTcChannels;          // 8 channels per group
constexpr int kQ = 16;                   // firmware blocks per supertile = row groups of one MMA
constexpr int kBlk = 48;                 // frames per firmware block (48 kHz)
constexpr int kSuper = kQ * kBlk;        // 768 frames
constexpr int kHist = kTcTaps - 1;       // 128 frames of history
constexpr int kChunkBytes = kJ * 16;     // one K-chunk (8 frames x {I,Q} bytes) of all 8 channels = one core matrix
constexpr int kChunksHist = kHist / 8;   // 16
constexpr int kChunksNew = kSuper / 8;   // 96
constexpr int kPlaneBytes = (kChunksHist + kChunksNew) * kChunkBytes;   // 14336
constexpr int kKSteps = 11;              // (128 + 48) frames * 2 bytes / 32
constexpr int kBStep = kTcRowGroups * 256; // B bytes per K-step: 26 row groups (4 digits x 52 rows: 48 audio + 4 state) x 2 chunks x 128 B
constexpr int kDig = kTcDigit;           // accumulator columns per digit weight (52)
constexpr int kNhi = kTcRowGroups * 8;   // 208 = N of the xh MMAs: the high data byte meets all four digits of the 32-bit map
constexpr int kN = 160;                  // N of the xl MMAs: the low data byte meets the top three digits (3 x 52 rows + 4: a multiple of 16; the
                                         // four extra rows are the first rows of the lowest digit and land in columns 208..211, which nobody reads)
constexpr int kRawRow = kSuper * 4 + 16; // raw stage row (one channel), padded: conflict-free 16-byte reads across channels
constexpr int kHistRow = kHist * 4 + 16;
// Epilogue warps per TMEM lane quadrant and set: 1. Splitting a block's 48 samples between two warps (16 epilogue warps of 80
// registers instead of 8 of 168) measured equal (416 vs 423 Gsamples/s at 1024 channels, 461 vs 460 at 8192): the kernel is bound
// by the L1 / shared-memory data pipe (tensor-core operand reads + LSU wavefronts), not by the latency of an epilogue set.
// Two-CTA clusters (tcgen05.mma.cta_group::2, M = 256, each CTA fetching half of the map operand) measured slower: 315 vs 403 Gsamples/s
// at 1024 channels, 370 vs 445 at 8192.
constexpr int kMmaUnroll = 1;
constexpr int kSets = 2;                         // epilogue warp sets (warpgroups), taking supertiles in turn
constexpr int kRawStages = 3;                    // raw stages: a bulk copy takes ~4400 clocks to land (measured), a supertile ~3000
constexpr int kEpiWarps = 4 * kSets;
constexpr int kConvWarps = 2;                    // the converters' shared-memory accesses queue behind the tensor core's operand reads (latency-bound role)
constexpr int kGroups = kChunksNew / 4;            // groups of 4 chunks (32 frames) of a supertile: 24; warp cw converts the groups t = cw (mod kConvWarps)
static_assert ((kGroups / 2) % kConvWarps == 0, "a half supertile splits evenly too");
constexpr int kMmaWarp = kEpiWarps + kConvWarps, kProdWarp = kMmaWarp + 1;
constexpr int kThreads = 32 * (kProdWarp + 1);   // 12 warps: 2 epilogue sets + {2 converters, MMA issuer, producer}
constexpr int kTmemCols = 512;           // two accumulator buffers of 256 columns

struct Smem
{
  static constexpr size_t a = 0;                                        // [2 buffers][hi plane | lo plane]
  static constexpr size_t b = a + 2 * 2 * kPlaneBytes;                  // tap planes of the current mask
  static constexpr size_t raw = b + kTcPlaneBytes;                      // [stages][8 rows]
  static constexpr size_t hist = raw + kRawStages * kJ * kRawRow;       // [stages][8 rows] carried tail of the previous call
  static constexpr size_t wsum = hist + kRawStages * kJ * kHistRow;     // [sets][4 warps][8][4] floats
  static constexpr size_t pk = wsum + kSets * 4 * kJ * 4 * 4;           // [sets][16][8] floats
  static constexpr size_t carry_s = pk + kSets * kQ * kJ * 4;           // [2][8][4] floats
  static constexpr size_t carry_e = carry_s + 2 * kJ * 4 * 4;           // [2][8] floats
  static constexpr size_t mp = carry_e + 2 * kJ * 4;                    // [4][20] floats: A^(48 a), rows padded to 20 (bank spread)
  static constexpr size_t bars = mp + 4 * 20 * 4;
  static constexpr int n_bars = 28;                                     // 22 in use
  static constexpr size_t tmem_ptr = bars + n_bars * 8;
  static constexpr size_t bytes = tmem_ptr + 16;
};

struct KParams
{
  const uint32_t *in; uint32_t *out;            // one u32 = one I/Q (or L/R) frame
  float *audio_dbg; float *gain_dbg;
  const uint32_t *ovl_in; uint32_t *ovl_out;
  float *state; unsigned *flag;
  const uint32_t *chan; const uint32_t *gstart; const uint32_t *ginfo;
  const uint8_t *planes;
  float s0[SLB_MAX_MASKS], sz[SLB_MAX_MASKS];
  unsigned flag_final;
  uint32_t n_groups, frames, supers;
  float agc_target, agc_decay, agc_floor, agc_gmax;
  TcBiquadTables tab;
};

#include "sl_tc_common.cuh"

__device__ __forceinline__ uint32_t pack_lr (float x_times_32768)
{
  // arm_float_to_q15.c:147 : (q15_t) __SSAT((q31_t)(x * 32768.0f), 16): truncation toward zero, then saturation.
  // (An exact form without the conversion pipe, 7 instructions instead of 2, measured slower: 266 vs 291 Gsamples/s; the
  // epilogue is bound by instruction count, not by the F2I rate.)
  short v;
  asm ("cvt.rzi.sat.s16.f32 %0, %1;" : "=h"(v) : "f"(x_times_32768));
  return __byte_perm ((uint32_t) (uint16_t) v, 0u, 0x1010);   // stereo endpoint, L = R (usbd_audio.c:399-404)
}

// y = M x (4x4 row-major, uniform M) + add
__device__ __forceinline__ void matvec4 (const float *M, const float *x, const float *add, float *y)
{
#pragma unroll
  for (int r = 0; r < 4; r++) y[r] = add[r] + (M[4 * r] * x[0] + M[4 * r + 1] * x[1] + M[4 * r + 2] * x[2] + M[4 * r + 3] * x[3]);
}

__global__ void __launch_bounds__ (kThreads, 1) rx_ssb_tc_kernel (const __grid_constant__ KParams P)
{
  extern __shared__ __align__ (1024) unsigned char smem[];
  unsigned char *sA = smem + Smem::a, *sB = smem + Smem::b, *sRaw = smem + Smem::raw, *sHist = smem + Smem::hist;
  float *sW = reinterpret_cast<float *> (smem + Smem::wsum), *sPk = reinterpret_cast<float *> (smem + Smem::pk);
  float *sCarryS = reinterpret_cast<float *> (smem + Smem::carry_s), *sCarryE = reinterpret_cast<float *> (smem + Smem::carry_e);
  float *sMp = reinterpret_cast<float *> (smem + Smem::mp);
  uint64_t *bars = reinterpret_cast<uint64_t *> (smem + Smem::bars);
  uint64_t *raw_full = bars, *raw_empty = bars + 3, *a_full = bars + 6, *a_empty = bars + 8, *t_empty = bars + 10;
  uint64_t *s_bar = bars + 12, *e_bar = bars + 14, *b_full = bars + 16, *drain = bars + 17, *t_full = bars + 18;
  // t_full has FOUR slots although there are two accumulator buffers: an epilogue set may start waiting for supertile
  // kk + 2 while kk is still in flight, and on a two-slot barrier that wait would alias the phase before kk's and pass at once
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *> (smem + Smem::tmem_ptr);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t g0 = blockIdx.x, gstride = gridDim.x;   // this CTA's groups: g0, g0 + gstride, ...
  if (tid == 0)
  {
    for (int i = 0; i < kRawStages; i++) { mbar_init (raw_full + i, 1); mbar_init (raw_empty + i, kConvWarps); }
    for (int i = 0; i < 2; i++)
    {
      mbar_init (a_full + i, kConvWarps); mbar_init (a_empty + i, 1);
      mbar_init (t_full + i, 1); mbar_init (t_full + 2 + i, 1); mbar_init (t_empty + i, 4); mbar_init (s_bar + i, kJ); mbar_init (e_bar + i, kJ);
    }
    mbar_init (b_full, 1); mbar_init (drain, 1);
    asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 64) sMp[(tid >> 4) * 20 + (tid & 15)] = P.tab.Mp[tid >> 4][tid & 15];
  if (warp == kMmaWarp)
  {
    asm volatile ("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32 (tmem_ptr)), "n"(kTmemCols) : "memory");
    asm volatile ("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before ();
  __syncthreads ();
  tc_fence_after ();
  const uint32_t tmem = *tmem_ptr;
  const uint32_t supers = P.supers;
  // Columns [0,52) of both accumulator buffers start at zero: the xh MMAs accumulate into them (see the MMA issuer); afterwards
  // the epilogue set that drains a buffer zeroes them again.
  if (warp < 8) tmem_zero<kDig> (tmem + (uint32_t) (warp >> 2) * 256u + ((uint32_t) (32 * (warp & 3)) << 16));
  tc_fence_before ();
  __syncthreads ();
  tc_fence_after ();

  if (warp == kProdWarp)
  {
    // ======================================= bulk-copy producer =======================================
    // Lane j < 8 owns row j of the group: it reads its channel index ONCE per group and issues that row's bulk copy for
    // every supertile. (Until round 2 one lane walked the eight rows and read the index from global memory for every row of every
    // supertile — eight dependent L2 round trips of ~400 clocks under load: the producer, not the epilogue or the MMAs, set the
    // kernel's pace of ~3500 clocks per supertile, which is why no epilogue or MMA variant ever moved it.)
    {
      unsigned kk = 0;
      for (uint32_t g = g0; g < P.n_groups; g += gstride)
      {
        const uint32_t gs = P.gstart[g], nv = P.ginfo[g] >> 8;
        const uint32_t c = P.chan[gs + min ((uint32_t) (lane & 7), nv - 1u)];    // short groups repeat their last channel (rows computed, never stored)
        const uint32_t *src = P.in + (size_t) c * P.frames;
        for (uint32_t k = 0; k < supers; k++, kk++)
        {
          const int rb = kk % kRawStages;
          const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper);
          if (lane == 0)
          {
            mbar_wait_guarded (raw_empty + rb, ((kk / kRawStages) & 1) ^ 1);
            mbar_expect_tx (raw_full + rb, kJ * nfr * 4u + (k == 0 ? kJ * kHist * 4u : 0u));
          }
          __syncwarp ();
          if (lane < kJ)
          {
            bulk_g2s (sRaw + (rb * kJ + lane) * kRawRow, src + (size_t) k * kSuper, nfr * 4u, raw_full + rb);
            if (k == 0) bulk_g2s (sHist + (rb * kJ + lane) * kHistRow, P.ovl_in + (size_t) c * kHist, kHist * 4u, raw_full + rb);
          }
          __syncwarp ();
        }
      }
    }
  }
  else if (warp >= kEpiWarps && warp < kEpiWarps + kConvWarps)
  {
    // ========================================== converters ==========================================
    // int16 I/Q frames -> the two byte planes of the A operand: chunk = 8 frames, 16 bytes (I, Q) per channel,
    // 8 channels contiguous (one core matrix). Two PRMTs per pair of frames and plane; no arithmetic. A lane keeps its
    // channel (lane & 7) and walks the chunks lane >> 3, + 4, + 8, ...: constant strides, three chunks in flight (the role runs on 56 registers).
    const int cw = warp - kEpiWarps, j = lane & 7, c4 = lane >> 3;
    unsigned kk = 0;
    for (uint32_t g = g0; g < P.n_groups; g += gstride)
    {
      const uint32_t nvalid = P.ginfo[g] >> 8, gs = P.gstart[g];
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        const int rb = kk % kRawStages, ab = kk & 1;
        const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper);
        unsigned char *Ahi = sA + ab * 2 * kPlaneBytes;
        mbar_wait (raw_full + rb, (kk / kRawStages) & 1);
        mbar_wait (a_empty + ab, ((kk >> 1) & 1) ^ 1);                              // the MMAs of supertile kk - 2 have read this buffer
        if (cw == 0 && k == 0)
        {
          // history = the carried raw tail of the previous call (this launch reads ovl_in and writes ovl_out)
          const unsigned char *src = sHist + (rb * kJ + j) * kHistRow + c4 * 32;
          unsigned char *dst = Ahi + c4 * kChunkBytes + j * 16;
#pragma unroll
          for (int t = 0; t < kChunksHist / 4; t++)
          {
            const uint4 v0 = *reinterpret_cast<const uint4 *> (src + t * 128), v1 = *reinterpret_cast<const uint4 *> (src + t * 128 + 16);
            *reinterpret_cast<uint4 *> (dst + t * 4 * kChunkBytes) =
                make_uint4 (__byte_perm (v0.x, v0.y, 0x7531), __byte_perm (v0.z, v0.w, 0x7531), __byte_perm (v1.x, v1.y, 0x7531), __byte_perm (v1.z, v1.w, 0x7531));
            *reinterpret_cast<uint4 *> (dst + kPlaneBytes + t * 4 * kChunkBytes) =
                make_uint4 (__byte_perm (v0.x, v0.y, 0x6420), __byte_perm (v0.z, v0.w, 0x6420), __byte_perm (v1.x, v1.y, 0x6420), __byte_perm (v1.z, v1.w, 0x6420));
          }
        }
        if (k != 0)
        {
          // history = the last 16 chunks of the previous supertile's planes (the other buffer). Every warp moves the groups it
          // wrote itself (program order is all the synchronisation that takes): group kGroups - 4 + hg -> history group hg
#pragma unroll
          for (int hg = 0; hg < 4; hg++)
            if ((kGroups - 4 + hg) % kConvWarps == cw)
            {
              const unsigned char *prev = sA + (ab ^ 1) * 2 * kPlaneBytes + (kChunksNew + 4 * hg) * kChunkBytes + lane * 16;
              unsigned char *cur = Ahi + 4 * hg * kChunkBytes + lane * 16;
              const uint4 v0 = *reinterpret_cast<const uint4 *> (prev), v1 = *reinterpret_cast<const uint4 *> (prev + kPlaneBytes);
              *reinterpret_cast<uint4 *> (cur) = v0; *reinterpret_cast<uint4 *> (cur + kPlaneBytes) = v1;
            }
        }
        {
          // this warp's share of the new chunks: groups t = cw + kConvWarps * i, chunk = c4 + 4 t
          const int per = (int) (nfr / 32) / kConvWarps;                          // groups per warp (half of it for the half supertile at the end of a stream)
          const unsigned char *src = sRaw + (rb * kJ + j) * kRawRow + (c4 + 4 * cw) * 32;
          unsigned char *dst = Ahi + (kChunksHist + c4 + 4 * cw) * kChunkBytes + j * 16;
          constexpr int kB = kGroups / 2 / kConvWarps;                            // groups in flight
          constexpr int kS = kConvWarps * 128, kD = kConvWarps * 4 * kChunkBytes;  // strides from one of the warp's groups to the next
          for (int t0 = 0; t0 < per; t0 += kB)
          {
            uint4 v[2 * kB];
#pragma unroll
            for (int t = 0; t < kB; t++) { v[2 * t] = *reinterpret_cast<const uint4 *> (src + (t0 + t) * kS); v[2 * t + 1] = *reinterpret_cast<const uint4 *> (src + (t0 + t) * kS + 16); }
#pragma unroll
            for (int t = 0; t < kB; t++)
            {
              const uint4 v0 = v[2 * t], v1 = v[2 * t + 1];
              *reinterpret_cast<uint4 *> (dst + (t0 + t) * kD) =
                  make_uint4 (__byte_perm (v0.x, v0.y, 0x7531), __byte_perm (v0.z, v0.w, 0x7531), __byte_perm (v1.x, v1.y, 0x7531), __byte_perm (v1.z, v1.w, 0x7531));
              *reinterpret_cast<uint4 *> (dst + kPlaneBytes + (t0 + t) * kD) =
                  make_uint4 (__byte_perm (v0.x, v0.y, 0x6420), __byte_perm (v0.z, v0.w, 0x6420), __byte_perm (v1.x, v1.y, 0x6420), __byte_perm (v1.z, v1.w, 0x6420));
            }
          }
        }
        if (cw == 0 && k + 1 == supers)
        {
          // carry the raw tail of the stream for the next call: the last 128 frames of every valid channel
          for (int i = lane; i < kJ * (kHist / 4); i += 32)
          {
            const int jj = i >> 5, o = i & 31;
            if ((uint32_t) jj < nvalid)
            {
              const uint32_t c = P.chan[gs + jj];
              reinterpret_cast<uint4 *> (P.ovl_out + (size_t) c * kHist)[o] =
                  *reinterpret_cast<const uint4 *> (sRaw + (rb * kJ + jj) * kRawRow + (nfr - kHist) * 4 + o * 16);
            }
          }
        }
        asm volatile ("fence.proxy.async.shared::cta;" ::: "memory");        // generic-proxy stores -> visible to the tensor core's reads
        __syncwarp ();
        if (lane == 0) { mbar_arrive (a_full + ab); mbar_arrive (raw_empty + rb); }
      }
    }
  }
  else if (warp == kMmaWarp)
  {
    // ========================================== MMA issuer ==========================================
    // The whole warp walks the loop converged and ONE elected lane issues: with `if (lane == 0)` around the loop the
    // compiler cannot keep descriptors in uniform registers and wraps every tcgen05.mma in a vote / broadcast loop —
    // measured 128 clocks of issue per MMA against 116 of execution (N = 144).
    constexpr uint32_t id_ss = umma_idesc (kNhi, 1, 1), id_us = umma_idesc (kN, 0, 1);
    const uint32_t aBase = smem_u32 (sA), bBase = smem_u32 (sB);
    // constant upper halves of the descriptors: LBO = 128 (A and B), SBO = 768 (A, aliased row groups) / 256 (B), version 1
    constexpr uint64_t kDescA = ((uint64_t) (kChunkBytes >> 4) << 16) | ((uint64_t) ((6 * kChunkBytes) >> 4) << 32) | (1ull << 46);
    constexpr uint64_t kDescB = ((uint64_t) (128 >> 4) << 16) | ((uint64_t) (256 >> 4) << 32) | (1ull << 46);
    unsigned kk = 0, b_loads = 0, drains = 0;
    int cur_slot = -1;
    for (uint32_t g = g0; g < P.n_groups; g += gstride)
    {
      const int slot = (int) (P.ginfo[g] & 0xFFu);
      if (slot != cur_slot)
      {
        // (re)load the tap planes of this mask; earlier MMAs may still be reading the old ones
        if (kk != 0)
        {
          if (elect_one ()) umma_commit (drain);
          __syncwarp ();
          mbar_wait (drain, drains & 1); drains++;
        }
        if (elect_one ())
        {
          mbar_expect_tx (b_full, (unsigned) kTcPlaneBytes);
          bulk_g2s (sB, P.planes + (size_t) slot * kTcPlaneBytes, (unsigned) kTcPlaneBytes, b_full);
        }
        __syncwarp ();
        mbar_wait (b_full, b_loads & 1);
        b_loads++;
        cur_slot = slot;
      }
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        const int ab = kk & 1, tb = kk & 1;
        mbar_wait_guarded (a_full + ab, (kk >> 1) & 1);
        // the epilogue has drained this accumulator buffer and zeroed its columns [0,52)
        mbar_wait_guarded (t_empty + tb, ((kk >> 1) & 1) ^ 1);
        tc_fence_after ();
        const uint32_t d = tmem + (uint32_t) tb * 256u;
        const uint32_t aHi = (aBase + ab * 2 * kPlaneBytes) >> 4, aLo = aHi + (kPlaneBytes >> 4), b0 = bBase >> 4;
        if (elect_one ())
        {
          // the map is 32 bits wide, h = h3 2^24 + h2 2^16 + h1 2^8 + h0 (balanced digits). Accumulator columns, in units of the 2^8 class:
          // [0,52) weight 2^24 = xh h3, [52,104) 2^16 = xh h2 + xl h3, [104,156) 2^8 = xh h1 + xl h2, [156,208) 1 = xh h0 + xl h1; the class
          // below (xl h0, 2^-32 of full scale) is not computed. (Round 1's 24-bit map missed the 1e-5 bar by 1.1 .. 2.0 x on outputs dominated by a
          // REJECTED tone, for every mode: its quantisation error scales with the input. The fourth digit for the high data byte costs 24 clocks
          // per xh MMA and removes the special bar that case needed.)
          // inside each group of 52: 48 audio outputs, 4 end-state outputs. Both planes meet the SAME operand [h3|h2|h1|h0] (xh: N = 208, xl: the first 160 rows,
          // rows 156..159 zero), xl one digit to the right of xh. The first xl MMA starts columns [52,212) afresh; columns [0,52)
          // were zeroed by the epilogue set that drained the buffer (N must be a multiple of 16: there is no MMA that could
          // start exactly these 52 columns), so every xh MMA accumulates.
          // (Tried: two independent chains, xh * [h2|h1|h0] and xl * [h2|h1|h0] in disjoint columns, added in the epilogue. No faster,
          // and it costs the second accumulator buffer.)
#pragma unroll kMmaUnroll
          for (int ks = 0; ks < kKSteps; ks++)
          {
            const uint32_t ao = (uint32_t) (ks * 2 * kChunkBytes) >> 4, bo = (uint32_t) (ks * kBStep) >> 4;
            umma_i8 (d + kDig, kDescA | (aLo + ao), kDescB | (b0 + bo), id_us, ks ? 1u : 0u);
            umma_i8 (d, kDescA | (aHi + ao), kDescB | (b0 + bo), id_ss, 1u);
          }
          // accumulators complete -> epilogue; planes read -> converter may overwrite them
          umma_commit (t_full + (kk & 3)); umma_commit (a_empty + ab);
        }
        __syncwarp ();
      }
    }
  }
  else
  {
    // ========================================== epilogue ==========================================
    // TMEM lane = 32 w + lane = 8 q + j: thread (q, j) owns firmware block q of channel j of the supertile.
    const int es = warp >> 2, w = warp & 3, a = lane >> 3, j = lane & 7, q = 4 * w + a;
    float *myW = sW + es * (4 * kJ * 4), *myPk = sPk + es * (kQ * kJ);
    const float decay = P.agc_decay;
    unsigned kk = 0;
    for (uint32_t g = g0; g < P.n_groups; g += gstride)
    {
      const uint32_t gi = P.ginfo[g];
      const bool jvalid = (uint32_t) j < (gi >> 8);
      const uint32_t c = P.chan[P.gstart[g] + min ((uint32_t) j, (gi >> 8) - 1u)];
      const float s0 = P.s0[gi & 0xFFu], s8 = s0 * 256.0f, s16 = s0 * 65536.0f, s24 = s0 * 16777216.0f, z0s = P.sz[gi & 0xFFu];
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        if ((int) (kk % kSets) != es) continue;
        const int tb = kk & 1;
        const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper);
        const int nblk = (int) (nfr / kBlk);
        const bool last_q = q == nblk - 1;
        mbar_wait (t_full + (kk & 3), (kk >> 2) & 1);
        tc_fence_after ();
        // ---- accumulators -> float: y = (D24 2^24 + D16 2^16 + D8 2^8 + D0) * unit (arm_q15_to_float's 1/32768 folded in)
        float y[kBlk];
        const uint32_t taddr = tmem + (uint32_t) tb * 256u + ((uint32_t) (32 * w) << 16);
        constexpr int kW = 16;                                                     // accumulator columns per tcgen05.ld
#pragma unroll
        for (int i = 0; i < kBlk / kW; i++)
        {
          uint32_t v0[kW], v1[kW], v2[kW], v3[kW];
          tmem_ld16 (taddr + kW * i, v0); tmem_ld16 (taddr + kDig + kW * i, v1); tmem_ld16 (taddr + 2 * kDig + kW * i, v2); tmem_ld16 (taddr + 3 * kDig + kW * i, v3);
          tmem_ld_wait ();
#pragma unroll
          for (int n = 0; n < kW; n++)
            y[kW * i + n] = fmaf (__int2float_rn ((int) v0[n]), s24, fmaf (__int2float_rn ((int) v1[n]), s16, fmaf (__int2float_rn ((int) v2[n]), s8, __int2float_rn ((int) v3[n]) * s0)));
        }
        float z[4];
        {
          uint32_t v0[4], v1[4], v2[4], v3[4];
          tmem_ld4 (taddr + 48, v0); tmem_ld4 (taddr + kDig + 48, v1); tmem_ld4 (taddr + 2 * kDig + 48, v2); tmem_ld4 (taddr + 3 * kDig + 48, v3);
          tmem_ld_wait ();
          const float z8 = z0s * 256.0f, z16 = z0s * 65536.0f, z24 = z0s * 16777216.0f;
#pragma unroll
          for (int r = 0; r < 4; r++)
            z[r] = fmaf (__int2float_rn ((int) v0[r]), z24, fmaf (__int2float_rn ((int) v1[r]), z16, fmaf (__int2float_rn ((int) v2[r]), z8, __int2float_rn ((int) v3[r]) * z0s)));
        }
        tmem_zero<kDig> (taddr);                                                   // the next supertile's xh MMAs accumulate into these columns
        tc_fence_before ();
        __syncwarp ();
        if (lane == 0) mbar_arrive (t_empty + tb);                                 // the accumulator buffer now lives in registers

        // (y[] already IS the zero-state response of the biquad cascade over the block — the operand planes hold the FIR
        //  composed with it — and columns 48..51 of each digit group hold the cascade's end state from a zero start)
        // ---- level 1: start state of the block inside the warp (zero at the warp's first block): P_{a+1} = M48 P_a + z_a
        float Pst[4] = { 0.f, 0.f, 0.f, 0.f };
#pragma unroll
        for (int kq = 0; kq < 3; kq++)
        {
          float t[4], nx[4];
#pragma unroll
          for (int r = 0; r < 4; r++) t[r] = __shfl_sync (0xffffffffu, z[r], kq * 8 + j);
          matvec4 (P.tab.Mp[1], Pst, t, nx);
          if (kq < a) { Pst[0] = nx[0]; Pst[1] = nx[1]; Pst[2] = nx[2]; Pst[3] = nx[3]; }
        }
        if (a == 3)
        {
          float We[4];
          matvec4 (P.tab.Mp[1], Pst, z, We);                                      // the warp's four blocks from a zero start
          *reinterpret_cast<float4 *> (myW + (w * kJ + j) * 4) = make_float4 (We[0], We[1], We[2], We[3]);
        }
        // ---- carried state of the channel: from the previous call (first supertile) or the previous supertile
        // (every supertile but the CTA's first waits for its predecessor's hand-over, also across groups where the value is
        // not used: no phase of the two-slot carry barriers is ever skipped, so a parity can never be mistaken for an older one)
        float S[4], envc;
        if (kk != 0) mbar_wait (s_bar + ((kk - 1) & 1), ((kk - 1) >> 1) & 1);
        if (k == 0)
        {
          const float *stc = P.state + (size_t) c * 8;
          S[0] = __ldcg (stc + 0); S[1] = __ldcg (stc + 1); S[2] = __ldcg (stc + 2); S[3] = __ldcg (stc + 3);
        }
        else
        {
          const float4 v = *reinterpret_cast<const float4 *> (sCarryS + (((kk - 1) & 1) * kJ + j) * 4);
          S[0] = v.x; S[1] = v.y; S[2] = v.z; S[3] = v.w;
        }
        named_bar (1 + 3 * es, 128);
        // ---- level 2: state at the warp's first block, then at this block
#pragma unroll
        for (int ww = 0; ww < 3; ww++)
          if (ww < w)
          {
            const float4 v = *reinterpret_cast<const float4 *> (myW + (ww * kJ + j) * 4);
            const float add[4] = { v.x, v.y, v.z, v.w };
            float nx[4];
            matvec4 (P.tab.M192, S, add, nx);
            S[0] = nx[0]; S[1] = nx[1]; S[2] = nx[2]; S[3] = nx[3];
          }
        float st[4];
        {
          const float4 m0 = *reinterpret_cast<const float4 *> (sMp + a * 20), m1 = *reinterpret_cast<const float4 *> (sMp + a * 20 + 4);
          const float4 m2 = *reinterpret_cast<const float4 *> (sMp + a * 20 + 8), m3 = *reinterpret_cast<const float4 *> (sMp + a * 20 + 12);
          st[0] = Pst[0] + (m0.x * S[0] + m0.y * S[1] + m0.z * S[2] + m0.w * S[3]);
          st[1] = Pst[1] + (m1.x * S[0] + m1.y * S[1] + m1.z * S[2] + m1.w * S[3]);
          st[2] = Pst[2] + (m2.x * S[0] + m2.y * S[1] + m2.z * S[2] + m2.w * S[3]);
          st[3] = Pst[3] + (m3.x * S[0] + m3.y * S[1] + m3.z * S[2] + m3.w * S[3]);
        }
        if (last_q)
        {
          // end state of the last block = carried state of the next supertile / the next call
          float en[4];
          matvec4 (P.tab.Mp[1], st, z, en);
          *reinterpret_cast<float4 *> (sCarryS + ((kk & 1) * kJ + j) * 4) = make_float4 (en[0], en[1], en[2], en[3]);
          if (k + 1 == supers && jvalid)
          {
            float *stw = P.state + (size_t) c * 8;
            __stcg (stw + 0, en[0]); __stcg (stw + 1, en[1]); __stcg (stw + 2, en[2]); __stcg (stw + 3, en[3]);
          }
          mbar_arrive (s_bar + (kk & 1));
        }
        // ---- add the zero-input response of the true start state; block peak (arm_abs_f32 + arm_max_f32)
        float peak = 0.f;
#pragma unroll
        for (int n = 0; n < kBlk; n++)
        {
          const float *C = P.tab.Cresp[n];
          y[n] = fmaf (C[0], st[0], fmaf (C[1], st[1], fmaf (C[2], st[2], fmaf (C[3], st[3], y[n]))));
          peak = fmaxf (peak, fabsf (y[n]));
        }
        myPk[q * kJ + j] = peak;
        if (kk != 0) mbar_wait (e_bar + ((kk - 1) & 1), ((kk - 1) >> 1) & 1);
        envc = (k == 0) ? __ldcg (P.state + (size_t) c * 8 + 4) : sCarryE[((kk - 1) & 1) * kJ + j];
        named_bar (2 + 3 * es, 128);
        // ---- AGC envelope: the oracle's sequential walk env_b = max(peak_b, fl(env_{b-1} * decay)) over the blocks before and including this one
        float e = envc;
#pragma unroll
        for (int qq = 0; qq < kQ; qq++)
        {
          const float p = myPk[qq * kJ + j];
          if (qq <= q) e = fmaxf (p, e * decay);
        }
        if (last_q)
        {
          sCarryE[(kk & 1) * kJ + j] = e;
          if (k + 1 == supers && jvalid)
          {
            __stcg (P.state + (size_t) c * 8 + 4, e);
            P.flag[c] = P.flag_final;                                              // the FFT kernel's hand-over counter stays consistent
          }
          mbar_arrive (e_bar + (kk & 1));
        }
        const float gain = fminf (__fdiv_rn (P.agc_target, fmaxf (e, P.agc_floor)), P.agc_gmax);
        if (q < nblk && jvalid)
        {
          const size_t t0 = (size_t) k * kSuper + (size_t) q * kBlk;
          if (P.audio_dbg)
          {
            float4 *adbg = reinterpret_cast<float4 *> (P.audio_dbg + (size_t) c * P.frames + t0);
#pragma unroll
            for (int n = 0; n < kBlk; n += 4) adbg[n / 4] = make_float4 (y[n], y[n + 1], y[n + 2], y[n + 3]);
          }
          if (P.gain_dbg) P.gain_dbg[(size_t) c * (P.frames / kBlk) + t0 / kBlk] = gain;
        }
        // ---- gain (arm_scale_f32), pack (arm_float_to_q15) and store: the block is 192 contiguous bytes
        if (q < nblk && jvalid)
        {
          const float g15 = gain * 32768.0f;                                       // exact: power of two
          uint4 *dst = reinterpret_cast<uint4 *> (P.out + (size_t) c * P.frames + (size_t) k * kSuper + (size_t) q * kBlk);
#pragma unroll
          for (int n = 0; n < kBlk; n += 8)
          {
            // 256-bit stores (sm_100: STG.E.256): the 32 lanes of a store hit 32 different lines whatever its width, so the
            // L1 wavefronts per block halve; and the lines must not allocate in L1 — the shared-memory / L1 data pipe is what the
            // tensor core fetches its operands through, and the MMAs are the critical path (measured: plain 366, .cg 371, .cs 376,
            // .L1::no_allocate 408 Gsamples/s)
            asm volatile ("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst + n / 4),
                          "r"(pack_lr (y[n] * g15)), "r"(pack_lr (y[n + 1] * g15)), "r"(pack_lr (y[n + 2] * g15)), "r"(pack_lr (y[n + 3] * g15)),
                          "r"(pack_lr (y[n + 4] * g15)), "r"(pack_lr (y[n + 5] * g15)), "r"(pack_lr (y[n + 6] * g15)), "r"(pack_lr (y[n + 7] * g15)) : "memory");
          }
        }
      }
    }
  }

  tc_fence_before ();
  __syncthreads ();
  if (warp == kMmaWarp)
  {
    tc_fence_after ();
    asm volatile ("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kTmemCols) : "memory");
  }
}

}  // namespace

int launch_rx_ssb_tc (const RxTcLaunch &L, int sm_count, void *stream_)
{
  cudaStream_t stream = (cudaStream_t) stream_;
  if (L.frames % 384u != 0 || L.frames == 0 || L.n_groups == 0) return (int) cudaErrorInvalidValue;
  if ((reinterpret_cast<uintptr_t> (L.in) | reinterpret_cast<uintptr_t> (L.ovl_in) | reinterpret_cast<uintptr_t> (L.ovl_out) | reinterpret_cast<uintptr_t> (L.out) |
       reinterpret_cast<uintptr_t> (L.planes)) & 15u)
    return (int) cudaErrorMisalignedAddress;
  KParams P;
  P.in = reinterpret_cast<const uint32_t *> (L.in); P.out = reinterpret_cast<uint32_t *> (L.out);
  P.audio_dbg = L.audio_dbg; P.gain_dbg = L.gain_dbg;
  P.ovl_in = reinterpret_cast<const uint32_t *> (L.ovl_in); P.ovl_out = reinterpret_cast<uint32_t *> (L.ovl_out);
  P.state = L.state; P.flag = L.flag; P.chan = L.chan; P.gstart = L.gstart; P.ginfo = L.ginfo; P.planes = L.planes;
  for (int i = 0; i < SLB_MAX_MASKS; i++) { P.s0[i] = L.s0[i]; P.sz[i] = L.sz[i]; }
  P.flag_final = L.flag_final; P.n_groups = L.n_groups; P.frames = L.frames; P.supers = (L.frames + kSuper - 1) / kSuper;
  P.agc_target = L.agc_target; P.agc_decay = L.agc_decay; P.agc_floor = L.agc_floor; P.agc_gmax = L.agc_gmax;
  P.tab = *L.tables;
  static_assert (sizeof (KParams) <= 4000, "kernel parameter block");
  cudaError_t e = cudaFuncSetAttribute (rx_ssb_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) Smem::bytes);
  if (e != cudaSuccess) return (int) e;
  // one CTA per SM, in clusters of one
  uint32_t grid = (uint32_t) sm_count;
  if (grid > P.n_groups) grid = P.n_groups;
  if (const char *gs = std::getenv ("SELENITE_B200_TC_GRID")) { const long v = std::atol (gs); if (v > 0 && (uint32_t) v <= grid) grid = (uint32_t) v; }   // profiling aid
  cudaLaunchConfig_t lc{};
  lc.gridDim = dim3 (grid); lc.blockDim = dim3 (kThreads); lc.dynamicSmemBytes = Smem::bytes; lc.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = 1; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  lc.attrs = at; lc.numAttrs = 1;
  e = cudaLaunchKernelEx (&lc, rx_ssb_tc_kernel, P);
  return (int) (e != cudaSuccess ? e : cudaGetLastError ());
}

}  // namespace sl
