// TX-SSB-f32 on the 5th-generation tensor cores (tcgen05 + TMEM): BASELINE config 3, one kernel, every sample crosses HBM once.
//
// The oracle chain (oracle/chains.inc.c tx_ssb_f32): mic = L of every L = R frame (codec_if.c:304-306) -> arm_q15_to_float ->
// overlap-save with the mode's one-sided mask (arm_cfft_f32 512 / arm_cmplx_mult_cmplx_f32 / inverse, keep 384) -> per
// 48-frame block arm_cmplx_mag_f32 + arm_max_f32 -> ALC gain law -> arm_scale_f32 -> arm_float_to_q15, written I,Q.
// The mask is the DFT of a 129-tap complex filter, so the filter is the linear convolution of the REAL int16 mic samples
// with fixed complex taps,  I[n] = sum_d hr[d] m[n-d],  Q[n] = sum_d hi[d] m[n-d]: two dense contractions with Toeplitz
// matrices of taps, evaluated exactly in integers like sl_rx_ssb_tc.cu (m = 256 mh + ml, 24-bit taps as three balanced
// base-256 digits, tcgen05.mma kind::i8, int32 TMEM accumulators by weight).
//
//   Differences to the RX kernel: the A operand holds mic bytes only (one byte per sample and plane: a 16-byte chunk is 16
//   samples, a block is 3 chunks further on: SBO = 384 B), so 6 K-steps of 32 samples cover the 128 + 48 window; there are
//   two output rails (I, Q), each N = 3 digits x 48 = 144 columns with its own tap planes: 26 MMAs per supertile into
//   2 x 192 accumulator columns — one accumulator buffer, the MMAs of a supertile start when the epilogue has read the
//   previous one; no biquad, so the only carry between supertiles is the ALC envelope.
//
// Roles, pipelines and the row mapping (TMEM lane = 8 q + j: block q of channel j) are those of sl_rx_ssb_tc.cu.
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include "sl_internal.h"

namespace sl {

namespace {

constexpr int kJ = kTcChannels;          // 8 channels per group
constexpr int kQ = 16;                   // firmware blocks per supertile
constexpr int kBlk = 48;
constexpr int kSuper = kQ * kBlk;        // 768 frames
constexpr int kHist = kTcTaps - 1;       // 128 samples of history
constexpr int kChunkBytes = kJ * 16;     // one K-chunk (16 mic samples x 1 byte) of all 8 channels = one core matrix
constexpr int kChunksHist = kHist / 16;  // 8
constexpr int kChunksNew = kSuper / 16;  // 48
constexpr int kChunks = kChunksHist + kChunksNew + 1;   // + one chunk the last block's sixth K-step reaches into (zero taps there)
constexpr int kPlaneBytes = kChunks * kChunkBytes;      // 7296
constexpr int kKSteps = 6;               // ceil ((128 + 48) / 32)
constexpr int kBStep = 18 * 256;         // B bytes per K-step and rail: 18 row groups (3 digits x 48) x 2 chunks x 128 B
constexpr int kRawRow = kSuper * 4 + 16;
constexpr int kHistRow = kHist * 4 + 16;
constexpr int kMmaUnroll = 1, kRailUnroll = 1;  // rolled MMA loops: the kernel's instruction fetch sat at 88 % of the GPC cache's request rate (icc hit 84.6 %)
constexpr int kSets = 2, kEpiWarps = 4 * kSets, kConvWarps = 2, kRawStages = 4;   // raw stages: a bulk copy lands ~4000 clocks after it is issued
constexpr int kGroups = kChunksNew / 4;  // groups of 4 chunks (64 samples) of a supertile: 12; converter warp cw takes the groups t = cw (mod kConvWarps)
constexpr int kMmaWarp = kEpiWarps + kConvWarps, kProdWarp = kMmaWarp + 1;
constexpr int kThreads = 32 * (kProdWarp + 1);
constexpr int kTmemCols = 512;           // I accumulators in columns [0,192), Q in [192,384)

struct Smem
{
  static constexpr size_t a = 0;                                        // [2 buffers][hi plane | lo plane]
  static constexpr size_t b = a + 2 * 2 * kPlaneBytes;                  // tap planes of the current mask: [rail][K-step]
  static constexpr size_t raw = b + kTcTxPlaneBytes;
  static constexpr size_t hist = raw + kRawStages * kJ * kRawRow;
  static constexpr size_t pk = hist + kRawStages * kJ * kHistRow;       // [sets][16][8] floats
  static constexpr size_t carry_e = pk + kSets * kQ * kJ * 4;           // [2][8] floats
  static constexpr size_t bars = carry_e + 2 * kJ * 4;
  static constexpr int n_bars = 24;
  static constexpr size_t tmem_ptr = bars + n_bars * 8;
  static constexpr size_t bytes = tmem_ptr + 16;
};

struct KParams
{
  const uint32_t *in; uint32_t *out;            // one u32 = one L/R (in) or I/Q (out) frame
  float *iq_dbg; float *gain_dbg;
  const uint32_t *ovl_in; uint32_t *ovl_out;
  float *state; unsigned *flag;
  const uint32_t *chan; const uint32_t *gstart; const uint32_t *ginfo;
  const uint8_t *planes;
  float unit[SLB_MAX_MASKS];
  unsigned flag_final;
  uint32_t n_groups, frames, supers;
  float alc_target, alc_decay, alc_floor, alc_gmax;
};

#include "sl_tc_common.cuh"
#include "sl_nco.cuh"

// bytes 1 (hi) or 0 (lo) of four consecutive frames' L halves
__device__ __forceinline__ uint32_t hi4 (uint4 v) { return __byte_perm (__byte_perm (v.x, v.y, 0x0051), __byte_perm (v.z, v.w, 0x0051), 0x5410); }
__device__ __forceinline__ uint32_t lo4 (uint4 v) { return __byte_perm (__byte_perm (v.x, v.y, 0x0040), __byte_perm (v.z, v.w, 0x0040), 0x5410); }

__global__ void __launch_bounds__ (kThreads, 1) tx_ssb_tc_kernel (const __grid_constant__ KParams P)
{
  extern __shared__ __align__ (1024) unsigned char smem[];
  unsigned char *sA = smem + Smem::a, *sB = smem + Smem::b, *sRaw = smem + Smem::raw, *sHist = smem + Smem::hist;
  float *sPk = reinterpret_cast<float *> (smem + Smem::pk), *sCarryE = reinterpret_cast<float *> (smem + Smem::carry_e);
  uint64_t *bars = reinterpret_cast<uint64_t *> (smem + Smem::bars);
  uint64_t *raw_full = bars, *raw_empty = bars + 4, *a_full = bars + 8, *a_empty = bars + 10, *t_empty = bars + 12;
  uint64_t *e_bar = bars + 13, *b_full = bars + 15, *drain = bars + 16, *t_full = bars + 17;      // t_full: two slots (one accumulator buffer)
  // the two rails have their own hand-over (rail Q: t_full_q / t_empty_q): the epilogue frees the I columns while the Q MMAs still
  // run, so the next supertile's I MMAs start at once and the tensor pipe never waits for a whole accumulator drain
  uint64_t *t_full_q = bars + 19, *t_empty_q = bars + 21;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *> (smem + Smem::tmem_ptr);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0)
  {
    static_assert (kRawStages >= 2 && kRawStages <= 4, "barrier layout");
    for (int i = 0; i < kRawStages; i++) { mbar_init (raw_full + i, 1); mbar_init (raw_empty + i, kConvWarps); }
    for (int i = 0; i < 2; i++)
    {
      mbar_init (a_full + i, kConvWarps); mbar_init (a_empty + i, 1);
      mbar_init (e_bar + i, kJ); mbar_init (t_full + i, 1);
    }
    mbar_init (t_empty, 4); mbar_init (b_full, 1); mbar_init (drain, 1);
    mbar_init (t_full_q, 1); mbar_init (t_full_q + 1, 1); mbar_init (t_empty_q, 4);
    asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // the pad chunk of every plane is read (times zero taps) but never written by the converters: keep it finite
  for (int i = tid; i < 4 * kChunkBytes / 16; i += kThreads)
    reinterpret_cast<uint4 *> (sA + (i / (kChunkBytes / 16)) * kPlaneBytes + (kChunks - 1) * kChunkBytes)[i % (kChunkBytes / 16)] = make_uint4 (0, 0, 0, 0);
  asm volatile ("fence.proxy.async.shared::cta;" ::: "memory");
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

  if (warp == kProdWarp)
  {
    // ======================================= bulk-copy producer =======================================
    // lane j < 8 owns row j of the group: its channel index is read once per group, its bulk copy issued per supertile (as sl_rx_ssb_tc.cu)
    {
      unsigned kk = 0;
      for (uint32_t g = blockIdx.x; g < P.n_groups; g += gridDim.x)
      {
        const uint32_t gs = P.gstart[g], nv = P.ginfo[g] >> 8;
        const uint32_t c = P.chan[gs + min ((uint32_t) (lane & 7), nv - 1u)];
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
    // L halves of the frames -> the two byte planes of the A operand: chunk = 16 samples = 16 bytes per channel
    const int cw = warp - kEpiWarps, j = lane & 7, c4 = lane >> 3;
    unsigned kk = 0;
    for (uint32_t g = blockIdx.x; g < P.n_groups; g += gridDim.x)
    {
      const uint32_t nvalid = P.ginfo[g] >> 8, gs = P.gstart[g];
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        const int rb = kk % kRawStages, ab = kk & 1;
        const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper);
        unsigned char *Ahi = sA + ab * 2 * kPlaneBytes;
        mbar_wait (raw_full + rb, (kk / kRawStages) & 1);
        mbar_wait (a_empty + ab, ((kk >> 1) & 1) ^ 1);
        if (cw == 0 && k == 0)
        {
          // history = the carried raw tail of the previous call: 8 chunks x 8 channels = 2 per lane
          const unsigned char *src = sHist + (rb * kJ + j) * kHistRow + c4 * 64;
          unsigned char *dst = Ahi + c4 * kChunkBytes + j * 16;
#pragma unroll
          for (int t = 0; t < kChunksHist / 4; t++)
          {
            const uint4 *s = reinterpret_cast<const uint4 *> (src + t * 256);
            const uint4 v0 = s[0], v1 = s[1], v2 = s[2], v3 = s[3];
            *reinterpret_cast<uint4 *> (dst + t * 4 * kChunkBytes) = make_uint4 (hi4 (v0), hi4 (v1), hi4 (v2), hi4 (v3));
            *reinterpret_cast<uint4 *> (dst + kPlaneBytes + t * 4 * kChunkBytes) = make_uint4 (lo4 (v0), lo4 (v1), lo4 (v2), lo4 (v3));
          }
        }
        if (k != 0)
        {
          // history = the last 8 chunks of the previous supertile's planes (the other buffer): every warp moves the group it wrote itself
#pragma unroll
          for (int hg = 0; hg < kChunksHist / 4; hg++)
            if ((kGroups - kChunksHist / 4 + hg) % kConvWarps == cw)
            {
              const unsigned char *prev = sA + (ab ^ 1) * 2 * kPlaneBytes + (kChunksNew + 4 * hg) * kChunkBytes + lane * 16;
              unsigned char *cur = Ahi + 4 * hg * kChunkBytes + lane * 16;
              const uint4 v0 = *reinterpret_cast<const uint4 *> (prev), v1 = *reinterpret_cast<const uint4 *> (prev + kPlaneBytes);
              *reinterpret_cast<uint4 *> (cur) = v0; *reinterpret_cast<uint4 *> (cur + kPlaneBytes) = v1;
            }
        }
        {
          // this warp's share of the new chunks: groups t = cw + kConvWarps i (4 chunks = 64 samples each), chunk = c4 + 4 t
          const int per = (int) (nfr / 64) / kConvWarps;                          // 6 (3 for the half supertile at the end of a stream)
          const unsigned char *src = sRaw + (rb * kJ + j) * kRawRow + (c4 + 4 * cw) * 64;
          unsigned char *dst = Ahi + (kChunksHist + c4 + 4 * cw) * kChunkBytes + j * 16;
          constexpr int kS = kConvWarps * 256, kD = kConvWarps * 4 * kChunkBytes;
          for (int t0 = 0; t0 < per; t0 += 3)
          {
            uint4 v[12];
#pragma unroll
            for (int t = 0; t < 3; t++)
#pragma unroll
              for (int u = 0; u < 4; u++) v[4 * t + u] = *reinterpret_cast<const uint4 *> (src + (t0 + t) * kS + u * 16);
#pragma unroll
            for (int t = 0; t < 3; t++)
            {
              *reinterpret_cast<uint4 *> (dst + (t0 + t) * kD) = make_uint4 (hi4 (v[4 * t]), hi4 (v[4 * t + 1]), hi4 (v[4 * t + 2]), hi4 (v[4 * t + 3]));
              *reinterpret_cast<uint4 *> (dst + kPlaneBytes + (t0 + t) * kD) = make_uint4 (lo4 (v[4 * t]), lo4 (v[4 * t + 1]), lo4 (v[4 * t + 2]), lo4 (v[4 * t + 3]));
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
              reinterpret_cast<uint4 *> (P.ovl_out + (size_t) P.chan[gs + jj] * kHist)[o] =
                  *reinterpret_cast<const uint4 *> (sRaw + (rb * kJ + jj) * kRawRow + (nfr - kHist) * 4 + o * 16);
          }
        }
        asm volatile ("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp ();
        if (lane == 0) { mbar_arrive (a_full + ab); mbar_arrive (raw_empty + rb); }
      }
    }
  }
  else if (warp == kMmaWarp)
  {
    // ========================================== MMA issuer ==========================================
    constexpr uint32_t id_ss48 = umma_idesc (48, 1, 1), id_ss96 = umma_idesc (96, 1, 1), id_ss144 = umma_idesc (144, 1, 1), id_us144 = umma_idesc (144, 0, 1);
    const uint32_t aBase = smem_u32 (sA), bBase = smem_u32 (sB);
    // descriptors: LBO = 128 (A and B), SBO = 384 (A: a block is 3 chunks further on, aliased row groups) / 256 (B), version 1
    constexpr uint64_t kDescA = ((uint64_t) (kChunkBytes >> 4) << 16) | ((uint64_t) ((3 * kChunkBytes) >> 4) << 32) | (1ull << 46);
    constexpr uint64_t kDescB = ((uint64_t) (128 >> 4) << 16) | ((uint64_t) (256 >> 4) << 32) | (1ull << 46);
    unsigned kk = 0, b_loads = 0, drains = 0;
    int cur_slot = -1;
    for (uint32_t g = blockIdx.x; g < P.n_groups; g += gridDim.x)
    {
      const int slot = (int) (P.ginfo[g] & 0xFFu);
      if (slot != cur_slot)
      {
        if (kk != 0) { if (elect_one ()) umma_commit (drain); __syncwarp (); mbar_wait (drain, drains & 1); drains++; }
        if (elect_one ())
        {
          mbar_expect_tx (b_full, (unsigned) kTcTxPlaneBytes);
          bulk_g2s (sB, P.planes + (size_t) slot * kTcTxPlaneBytes, (unsigned) kTcTxPlaneBytes, b_full);
        }
        __syncwarp ();
        mbar_wait (b_full, b_loads & 1); b_loads++;
        cur_slot = slot;
      }
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        const int ab = kk & 1;
        mbar_wait_guarded (a_full + ab, (kk >> 1) & 1);
        const uint32_t aHi = (aBase + ab * 2 * kPlaneBytes) >> 4, aLo = aHi + (kPlaneBytes >> 4);
#pragma unroll kRailUnroll
        for (int rail = 0; rail < 2; rail++)
        {
          mbar_wait_guarded (rail ? t_empty_q : t_empty, (kk & 1) ^ 1);                // the epilogue has read this rail's accumulators of supertile kk - 1
          tc_fence_after ();
          if (elect_one ())
          {
            // per rail: columns [0,48) weight 2^24 = mh h2, [48,96) 2^16 = mh h1 + ml h2, [96,144) 2^8 = mh h0 + ml h1, [144,192) 1 = ml h0
            const uint32_t d = tmem + 192u * rail, b0 = (bBase + rail * kKSteps * kBStep) >> 4;
            umma_i8 (d, kDescA | aHi, kDescB | b0, id_ss48, 0u);
            umma_i8 (d + 48, kDescA | aLo, kDescB | b0, id_us144, 0u);
            umma_i8 (d + 48, kDescA | aHi, kDescB | (b0 + ((6 * 256) >> 4)), id_ss96, 1u);
#pragma unroll kMmaUnroll
            for (int ks = 1; ks < kKSteps; ks++)
            {
              const uint32_t ao = (uint32_t) (ks * 2 * kChunkBytes) >> 4, bo = (uint32_t) (ks * kBStep) >> 4;
              umma_i8 (d, kDescA | (aHi + ao), kDescB | (b0 + bo), id_ss144, 1u);
              umma_i8 (d + 48, kDescA | (aLo + ao), kDescB | (b0 + bo), id_us144, 1u);
            }
            umma_commit ((rail ? t_full_q : t_full) + (kk & 1));
            if (rail) umma_commit (a_empty + ab);
          }
          __syncwarp ();
        }
      }
    }
  }
  else
  {
    // ========================================== epilogue ==========================================
    const int es = warp >> 2, w = warp & 3, a = lane >> 3, j = lane & 7, q = 4 * w + a;
    float *myPk = sPk + es * (kQ * kJ);
    const float decay = P.alc_decay;
    unsigned kk = 0;
    for (uint32_t g = blockIdx.x; g < P.n_groups; g += gridDim.x)
    {
      const uint32_t gi = P.ginfo[g];
      const bool jvalid = (uint32_t) j < (gi >> 8);
      const uint32_t c = P.chan[P.gstart[g] + min ((uint32_t) j, (gi >> 8) - 1u)];
      const float s0 = P.unit[gi & 0xFFu], s8 = s0 * 256.0f, s16 = s0 * 65536.0f, s24 = s0 * 16777216.0f;
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        if ((int) (kk % kSets) != es) continue;
        const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper);
        const int nblk = (int) (nfr / kBlk);
        const bool last_q = q == nblk - 1;
        // ---- accumulators -> float I, Q: rail by rail, each rail's columns handed back to the MMA issuer as soon as they are in registers
        float zi[kBlk], zq[kBlk];
        const uint32_t taddr = tmem + ((uint32_t) (32 * w) << 16);
        mbar_wait (t_full + (kk & 1), (kk >> 1) & 1);
        tc_fence_after ();
#pragma unroll
        for (int i = 0; i < kBlk / 8; i++)
        {
          uint32_t v0[8], v1[8], v2[8], v3[8];
          tmem_ld8 (taddr + 8 * i, v0); tmem_ld8 (taddr + 48 + 8 * i, v1); tmem_ld8 (taddr + 96 + 8 * i, v2); tmem_ld8 (taddr + 144 + 8 * i, v3);
          tmem_ld_wait ();
#pragma unroll
          for (int n = 0; n < 8; n++)
            zi[8 * i + n] = fmaf (__int2float_rn ((int) v0[n]), s24, fmaf (__int2float_rn ((int) v1[n]), s16, fmaf (__int2float_rn ((int) v2[n]), s8, __int2float_rn ((int) v3[n]) * s0)));
        }
        tc_fence_before ();
        __syncwarp ();
        if (lane == 0) mbar_arrive (t_empty);
        mbar_wait (t_full_q + (kk & 1), (kk >> 1) & 1);
        tc_fence_after ();
#pragma unroll
        for (int i = 0; i < kBlk / 8; i++)
        {
          uint32_t v0[8], v1[8], v2[8], v3[8];
          tmem_ld8 (taddr + 192 + 8 * i, v0); tmem_ld8 (taddr + 240 + 8 * i, v1); tmem_ld8 (taddr + 288 + 8 * i, v2); tmem_ld8 (taddr + 336 + 8 * i, v3);
          tmem_ld_wait ();
#pragma unroll
          for (int n = 0; n < 8; n++)
            zq[8 * i + n] = fmaf (__int2float_rn ((int) v0[n]), s24, fmaf (__int2float_rn ((int) v1[n]), s16, fmaf (__int2float_rn ((int) v2[n]), s8, __int2float_rn ((int) v3[n]) * s0)));
        }
        tc_fence_before ();
        __syncwarp ();
        if (lane == 0) mbar_arrive (t_empty_q);
        // ---- block peak of |I + jQ|: arm_cmplx_mag_f32.c:72 sqrt (re re + im im), each product rounded; sqrt is monotonic and
        //      correctly rounded, so max (sqrt) = sqrt (max)
        float m2 = 0.f;
#pragma unroll
        for (int n = 0; n < kBlk; n++) m2 = fmaxf (m2, __fadd_rn (__fmul_rn (zi[n], zi[n]), __fmul_rn (zq[n], zq[n])));
        myPk[q * kJ + j] = __fsqrt_rn (m2);
        // (every supertile but the CTA's first waits for its predecessor's envelope, also across groups where the value is
        //  not used: no phase of the two-slot carry barrier is ever skipped)
        if (kk != 0) mbar_wait (e_bar + ((kk - 1) & 1), ((kk - 1) >> 1) & 1);
        const float envc = (k == 0) ? __ldcg (P.state + (size_t) c * 8 + 4) : sCarryE[((kk - 1) & 1) * kJ + j];
        named_bar (1 + es, 128);
        // ---- ALC envelope: the oracle's sequential walk env_b = max (peak_b, fl (env_{b-1} * decay))
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
            P.flag[c] = P.flag_final;
          }
          mbar_arrive (e_bar + (kk & 1));
        }
        const float gain = fminf (__fdiv_rn (P.alc_target, fmaxf (e, P.alc_floor)), P.alc_gmax);
        if (q < nblk && jvalid)
        {
          const size_t t0 = (size_t) k * kSuper + (size_t) q * kBlk;
          if (P.iq_dbg)
          {
            float4 *adbg = reinterpret_cast<float4 *> (P.iq_dbg + 2 * ((size_t) c * P.frames + t0));
#pragma unroll
            for (int n = 0; n < kBlk; n += 2) adbg[n / 2] = make_float4 (zi[n], zq[n], zi[n + 1], zq[n + 1]);
          }
          if (P.gain_dbg) P.gain_dbg[(size_t) c * (P.frames / kBlk) + t0 / kBlk] = gain;
          const float g15 = gain * 32768.0f;                                       // arm_scale_f32 then arm_float_to_q15: exact fold
          uint4 *dst = reinterpret_cast<uint4 *> (P.out + (size_t) c * P.frames + t0);
#pragma unroll
          for (int n = 0; n < kBlk; n += 8)
            asm volatile ("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst + n / 4),
                          "r"(pack_iq (zi[n] * g15, zq[n] * g15)), "r"(pack_iq (zi[n + 1] * g15, zq[n + 1] * g15)),
                          "r"(pack_iq (zi[n + 2] * g15, zq[n + 2] * g15)), "r"(pack_iq (zi[n + 3] * g15, zq[n + 3] * g15)),
                          "r"(pack_iq (zi[n + 4] * g15, zq[n + 4] * g15)), "r"(pack_iq (zi[n + 5] * g15, zq[n + 5] * g15)),
                          "r"(pack_iq (zi[n + 6] * g15, zq[n + 6] * g15)), "r"(pack_iq (zi[n + 7] * g15, zq[n + 7] * g15)) : "memory");
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

int launch_tx_ssb_tc (const TxTcLaunch &L, int sm_count, void *stream_)
{
  cudaStream_t stream = (cudaStream_t) stream_;
  if (L.frames % 384u != 0 || L.frames == 0 || L.n_groups == 0) return (int) cudaErrorInvalidValue;
  if ((reinterpret_cast<uintptr_t> (L.in) | reinterpret_cast<uintptr_t> (L.ovl_in) | reinterpret_cast<uintptr_t> (L.ovl_out) | reinterpret_cast<uintptr_t> (L.out) |
       reinterpret_cast<uintptr_t> (L.planes)) & 15u)
    return (int) cudaErrorMisalignedAddress;
  KParams P;
  P.in = reinterpret_cast<const uint32_t *> (L.in); P.out = reinterpret_cast<uint32_t *> (L.out);
  P.iq_dbg = L.iq_dbg; P.gain_dbg = L.gain_dbg;
  P.ovl_in = reinterpret_cast<const uint32_t *> (L.ovl_in); P.ovl_out = reinterpret_cast<uint32_t *> (L.ovl_out);
  P.state = L.state; P.flag = L.flag; P.chan = L.chan; P.gstart = L.gstart; P.ginfo = L.ginfo; P.planes = L.planes;
  for (int i = 0; i < SLB_MAX_MASKS; i++) P.unit[i] = L.unit[i];
  P.flag_final = L.flag_final; P.n_groups = L.n_groups; P.frames = L.frames; P.supers = (L.frames + kSuper - 1) / kSuper;
  P.alc_target = L.alc_target; P.alc_decay = L.alc_decay; P.alc_floor = L.alc_floor; P.alc_gmax = L.alc_gmax;
  cudaError_t e = cudaFuncSetAttribute (tx_ssb_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) Smem::bytes);
  if (e != cudaSuccess) return (int) e;
  uint32_t grid = (uint32_t) sm_count;
  if (grid > L.n_groups) grid = L.n_groups;
  if (const char *gs = std::getenv ("SELENITE_B200_TC_GRID")) { const long v = std::atol (gs); if (v > 0 && (uint32_t) v <= grid) grid = (uint32_t) v; }   // profiling / test knob
  tx_ssb_tc_kernel<<<grid, kThreads, Smem::bytes, stream>>> (P);
  return (int) cudaGetLastError ();
}

}  // namespace sl
