// RX-SSB-f32, AM channels (FT-817 mode byte 0x04), on the tensor cores: the complex-detector variant of sl_rx_ssb_tc.cu.
//
// The oracle chain for AM (oracle/chains.inc.c rx_ssb_f32 with `envelope`): overlap-save with the two-sided channel mask ->
// arm_cmplx_mag_f32 of the complex result -> arm_biquad_cascade_df2T_f32 -> AGC -> arm_float_to_q15, written L = R. The
// magnitude sits between the filter and the biquad, so the biquad's block response cannot be folded into the contraction as
// in sl_rx_ssb_tc.cu: the tensor cores deliver both rails of the filter,
//   Re z[n] = sum_d hr[d] I[n-d] - hi[d] Q[n-d],   Im z[n] = sum_d hi[d] I[n-d] + hr[d] Q[n-d],
// from two sets of tap planes (2 x 23 tcgen05.mma kind::i8 per supertile into 2 x 192 accumulator columns, one accumulator
// buffer, the scheme of sl_tx_ssb_tc.cu on the interleaved I/Q byte planes of sl_rx_ssb_tc.cu), and the epilogue takes |z|,
// runs the zero-state recurrence of the cascade itself, then the same state chain, zero-input correction, envelope walk and
// pack as sl_rx_ssb_tc.cu. Roles, pipelines, row mapping (TMEM lane = 8 q + j) and carried state are those kernels'.
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
constexpr int kChunkBytes = kJ * 16;     // one K-chunk (8 frames x {I,Q} bytes) of all 8 channels = one core matrix
constexpr int kChunksHist = kHist / 8;   // 16
constexpr int kChunksNew = kSuper / 8;   // 96
constexpr int kPlaneBytes = (kChunksHist + kChunksNew) * kChunkBytes;   // 14336
constexpr int kKSteps = 11;              // (128 + 48) frames * 2 bytes / 32
constexpr int kBStep = 18 * 256;         // B bytes per K-step and rail: 18 row groups (3 digits x 48) x 2 chunks x 128 B
constexpr int kRawRow = kSuper * 4 + 16;
constexpr int kHistRow = kHist * 4 + 16;
constexpr int kMmaUnroll = 1, kRailUnroll = 1;   // rolled MMA issue loops (instruction fetch, as in the TX / q15 kernels)
constexpr int kSets = 2, kEpiWarps = 4 * kSets, kConvWarps = 2, kRawStages = 2;
constexpr int kMmaWarp = kEpiWarps + kConvWarps, kProdWarp = kMmaWarp + 1;
constexpr int kThreads = 32 * (kProdWarp + 1);
constexpr int kTmemCols = 512;           // I accumulators in columns [0,192), Q in [192,384)

struct Smem
{
  static constexpr size_t a = 0;                                        // [2 buffers][hi plane | lo plane]
  static constexpr size_t b = a + 2 * 2 * kPlaneBytes;                  // tap planes of the current mask: [rail][K-step]
  static constexpr size_t raw = b + kTcAmPlaneBytes;
  static constexpr size_t hist = raw + kRawStages * kJ * kRawRow;
  static constexpr size_t wsum = hist + kRawStages * kJ * kHistRow;     // [sets][4 warps][8][4] floats
  static constexpr size_t pk = wsum + kSets * 4 * kJ * 4 * 4;           // [sets][16][8] floats
  static constexpr size_t carry_s = pk + kSets * kQ * kJ * 4;           // [2][8][4] floats
  static constexpr size_t carry_e = carry_s + 2 * kJ * 4 * 4;           // [2][8] floats
  static constexpr size_t mp = carry_e + 2 * kJ * 4;                    // [4][20] floats: A^(48 a)
  static constexpr size_t zl = mp + 4 * 20 * 4;                         // FM: [sets][4 warps][8] float2, last baseband sample of each warp's four blocks
  static constexpr size_t carry_z = zl + kSets * 4 * kJ * 8;            // FM: [2][8] float2, last baseband sample of a supertile
  static constexpr size_t bars = carry_z + 2 * kJ * 8;
  static constexpr int n_bars = 18;
  static constexpr size_t tmem_ptr = bars + n_bars * 8;
  static constexpr size_t bytes = tmem_ptr + 16;
};

struct KParams
{
  const uint32_t *in; uint32_t *out;            // one u32 = one L/R (in) or I/Q (out) frame
  float *audio_dbg; float *gain_dbg;
  const uint32_t *ovl_in; uint32_t *ovl_out;
  float *state; unsigned *flag;
  const uint32_t *chan; const uint32_t *gstart; const uint32_t *ginfo;
  const uint8_t *planes;
  float unit[SLB_MAX_MASKS];
  unsigned flag_final;
  uint32_t n_groups, frames, supers;
  float agc_target, agc_decay, agc_floor, agc_gmax;
  TcBiquadTables tab;
};

#include "sl_tc_common.cuh"

__device__ __forceinline__ uint32_t pack_lr (float x_times_32768)
{
  // arm_float_to_q15.c:147 : (q15_t) __SSAT((q31_t)(x * 32768.0f), 16): truncation toward zero, then saturation
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

// FM limiter-discriminator, operation by operation as the oracle chain composes it: prev' = conj (prev) (arm_cmplx_conj_f32.c:71),
// w = z * prev' (arm_cmplx_mult_cmplx_f32.c:72: re = a c - b d, im = a d + b c with every product and sum rounded — the
// oracle build does not contract), m = |w| (arm_cmplx_mag_f32.c:72), d = Im w / max (m, floor).
__device__ __forceinline__ float fm_discriminator (float a, float b, float pr, float pi)
{
  const float c = pr, d = -pi;
  const float re = __fsub_rn (__fmul_rn (a, c), __fmul_rn (b, d)), im = __fadd_rn (__fmul_rn (a, d), __fmul_rn (b, c));
  // Im w / max (|w|, floor) = Im w * rsqrt (max (|w|^2, floor^2)): one MUFU.RSQ and a multiply instead of an IEEE square root and an
  // IEEE division (a quarter of this kernel's instructions, which are what bounds it). rsqrt.approx is good to 2^-22: the detector
  // output moves by <= 2e-7 of its value, against the chain's bar of 1e-5 (tests/test_gpu_rx_fm_f32.py, golden fixture included).
  // The oracle's two roundings (an IEEE square root and division) are recorded in DESIGN.md.
  const float s = fmaf (re, re, im * im);
  return im * rsqrtf (fmaxf (s, kFmFloor * kFmFloor));
}

__global__ void __launch_bounds__ (kThreads, 1) rx_am_tc_kernel (const __grid_constant__ KParams P)
{
  extern __shared__ __align__ (1024) unsigned char smem[];
  unsigned char *sA = smem + Smem::a, *sB = smem + Smem::b, *sRaw = smem + Smem::raw, *sHist = smem + Smem::hist;
  float *sW = reinterpret_cast<float *> (smem + Smem::wsum), *sPk = reinterpret_cast<float *> (smem + Smem::pk);
  float *sCarryS = reinterpret_cast<float *> (smem + Smem::carry_s), *sCarryE = reinterpret_cast<float *> (smem + Smem::carry_e);
  float *sMp = reinterpret_cast<float *> (smem + Smem::mp);
  uint64_t *bars = reinterpret_cast<uint64_t *> (smem + Smem::bars);
  uint64_t *raw_full = bars, *raw_empty = bars + 2, *a_full = bars + 4, *a_empty = bars + 6, *t_empty = bars + 8;
  uint64_t *e_bar = bars + 9, *b_full = bars + 11, *drain = bars + 12, *t_full = bars + 13, *s_bar = bars + 15;   // t_full: two slots (one accumulator buffer)
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *> (smem + Smem::tmem_ptr);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0)
  {
    for (int i = 0; i < 2; i++)
    {
      mbar_init (raw_full + i, 1); mbar_init (raw_empty + i, kConvWarps); mbar_init (a_full + i, kConvWarps); mbar_init (a_empty + i, 1);
      mbar_init (e_bar + i, kJ); mbar_init (t_full + i, 1); mbar_init (s_bar + i, kJ);
    }
    mbar_init (t_empty, 4); mbar_init (b_full, 1); mbar_init (drain, 1);
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

  if (warp == kProdWarp)
  {
    // ======================================= bulk-copy producer (as sl_rx_ssb_tc.cu) =======================================
    // lane j < 8 owns row j of the group: it reads its channel index once per group and issues the row's copies, so the eight
    // copies of a supertile go out together instead of behind eight dependent index loads of one lane
    {
      unsigned kk = 0;
      for (uint32_t g = blockIdx.x; g < P.n_groups; g += gridDim.x)
      {
        const uint32_t gs = P.gstart[g], nv = P.ginfo[g] >> 8;
        const uint32_t c = P.chan[gs + min ((uint32_t) (lane & 7), nv - 1u)];
        const uint32_t *src = P.in + (size_t) c * P.frames;
        for (uint32_t k = 0; k < supers; k++, kk++)
        {
          const int rb = kk & 1;
          const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper);
          if (lane == 0)
          {
            mbar_wait_guarded (raw_empty + rb, ((kk >> 1) & 1) ^ 1);
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
    // ========================================== converters (as sl_rx_ssb_tc.cu) ==========================================
    const int cw = warp - kEpiWarps, j = lane & 7, c4 = lane >> 3;
    unsigned kk = 0;
    for (uint32_t g = blockIdx.x; g < P.n_groups; g += gridDim.x)
    {
      const uint32_t nvalid = P.ginfo[g] >> 8, gs = P.gstart[g];
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        const int rb = kk & 1, ab = kk & 1;
        const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper);
        unsigned char *Ahi = sA + ab * 2 * kPlaneBytes;
        mbar_wait (raw_full + rb, (kk >> 1) & 1);
        mbar_wait (a_empty + ab, ((kk >> 1) & 1) ^ 1);
        if (cw == 0 && k == 0)
        {
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
        if (cw == kConvWarps - 1 && k != 0)
        {
          const unsigned char *prev = sA + (ab ^ 1) * 2 * kPlaneBytes + kChunksNew * kChunkBytes;
#pragma unroll
          for (int i = 0; i < 2 * kChunksHist * kJ / 32; i++)
          {
            const int e = lane + 32 * i, plane = e >> 7, o = (e & 127) * 16;
            *reinterpret_cast<uint4 *> (Ahi + plane * kPlaneBytes + o) = *reinterpret_cast<const uint4 *> (prev + plane * kPlaneBytes + o);
          }
        }
        {
          const int per = (int) (nfr / 32) / kConvWarps;                          // 12 (6 for the half supertile at the end of a stream)
          const unsigned char *src = sRaw + (rb * kJ + j) * kRawRow + (c4 + 4 * cw * per) * 32;
          unsigned char *dst = Ahi + (kChunksHist + c4 + 4 * cw * per) * kChunkBytes + j * 16;
          for (int t0 = 0; t0 < per; t0 += 6)
          {
            uint4 v[12];
#pragma unroll
            for (int t = 0; t < 6; t++) { v[2 * t] = *reinterpret_cast<const uint4 *> (src + (t0 + t) * 128); v[2 * t + 1] = *reinterpret_cast<const uint4 *> (src + (t0 + t) * 128 + 16); }
#pragma unroll
            for (int t = 0; t < 6; t++)
            {
              const uint4 v0 = v[2 * t], v1 = v[2 * t + 1];
              *reinterpret_cast<uint4 *> (dst + (t0 + t) * 4 * kChunkBytes) =
                  make_uint4 (__byte_perm (v0.x, v0.y, 0x7531), __byte_perm (v0.z, v0.w, 0x7531), __byte_perm (v1.x, v1.y, 0x7531), __byte_perm (v1.z, v1.w, 0x7531));
              *reinterpret_cast<uint4 *> (dst + kPlaneBytes + (t0 + t) * 4 * kChunkBytes) =
                  make_uint4 (__byte_perm (v0.x, v0.y, 0x6420), __byte_perm (v0.z, v0.w, 0x6420), __byte_perm (v1.x, v1.y, 0x6420), __byte_perm (v1.z, v1.w, 0x6420));
            }
          }
        }
        if (cw == 0 && k + 1 == supers)
        {
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
    // descriptors: LBO = 128 (A and B), SBO = 768 (A: a block is 6 chunks further on, aliased row groups) / 256 (B), version 1
    constexpr uint64_t kDescA = ((uint64_t) (kChunkBytes >> 4) << 16) | ((uint64_t) ((6 * kChunkBytes) >> 4) << 32) | (1ull << 46);
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
          mbar_expect_tx (b_full, (unsigned) kTcAmPlaneBytes);
          bulk_g2s (sB, P.planes + (size_t) slot * kTcAmPlaneBytes, (unsigned) kTcAmPlaneBytes, b_full);
        }
        __syncwarp ();
        mbar_wait (b_full, b_loads & 1); b_loads++;
        cur_slot = slot;
      }
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        const int ab = kk & 1;
        mbar_wait_guarded (a_full + ab, (kk >> 1) & 1);
        mbar_wait_guarded (t_empty, (kk & 1) ^ 1);                                     // the epilogue has read the accumulators of supertile kk - 1
        tc_fence_after ();
        const uint32_t aHi = (aBase + ab * 2 * kPlaneBytes) >> 4, aLo = aHi + (kPlaneBytes >> 4);
        if (elect_one ())
        {
#pragma unroll kRailUnroll
          for (int rail = 0; rail < 2; rail++)
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
          }
          umma_commit (t_full + (kk & 1));
          umma_commit (a_empty + ab);
        }
        __syncwarp ();
      }
    }
  }
  else
  {
    // ========================================== epilogue ==========================================
    const int es = warp >> 2, w = warp & 3, a = lane >> 3, j = lane & 7, q = 4 * w + a;
    float *myW = sW + es * (4 * kJ * 4), *myPk = sPk + es * (kQ * kJ);
    float2 *myZ = reinterpret_cast<float2 *> (smem + Smem::zl) + es * (4 * kJ), *sCarryZ = reinterpret_cast<float2 *> (smem + Smem::carry_z);
    const float *cf = P.tab.coef;
    const float decay = P.agc_decay;
    unsigned kk = 0;
    for (uint32_t g = blockIdx.x; g < P.n_groups; g += gridDim.x)
    {
      const uint32_t gi = P.ginfo[g];
      const bool jvalid = (uint32_t) j < (gi >> 8);
      const uint32_t c = P.chan[P.gstart[g] + min ((uint32_t) j, (gi >> 8) - 1u)];
      const float s0 = P.unit[gi & 0xFFu], s8 = s0 * 256.0f, s16 = s0 * 65536.0f, s24 = s0 * 16777216.0f;
      const bool fm = (gi & 0xFFu) == (uint32_t) kFmMaskSlot;                 // the group's detector: envelope (AM) or limiter-discriminator (FM)
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        if ((int) (kk % kSets) != es) continue;
        const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper);
        const int nblk = (int) (nfr / kBlk);
        const bool last_q = q == nblk - 1;
        mbar_wait (t_full + (kk & 1), (kk >> 1) & 1);
        tc_fence_after ();
        // ---- accumulators -> float Re z, Im z -> detector.
        //   AM: envelope |z| (arm_cmplx_mag_f32.c:72: sqrt (re re + im im), each product rounded).
        //   FM: w[n] = z[n] conj (z[n-1]) (arm_cmplx_conj_f32.c:71, arm_cmplx_mult_cmplx_f32.c:72: (ac - bd, ad + bc), products rounded),
        //       d[n] = Im w[n] / max (|w[n]|, floor) (arm_cmplx_mag_f32 + one division): the sine of the carrier's phase step, amplitude
        //       divided out. The oracle chain has no arctangent either (CMSIS-DSP V1.5.3 has none; oracle/chains.inc.c).
        //       z[-1] of the block is the neighbouring thread's last sample: fetched below, d[0] is completed there.
        float y[kBlk];
        float pr = 0.f, pi = 0.f, z0r = 0.f, z0i = 0.f;                            // FM: previous sample inside the block; the block's first sample
        const uint32_t taddr = tmem + ((uint32_t) (32 * w) << 16);
#pragma unroll
        for (int i = 0; i < kBlk / 8; i++)
        {
          uint32_t v0[8], v1[8], v2[8], v3[8];
          float zr[8];
          tmem_ld8 (taddr + 8 * i, v0); tmem_ld8 (taddr + 48 + 8 * i, v1); tmem_ld8 (taddr + 96 + 8 * i, v2); tmem_ld8 (taddr + 144 + 8 * i, v3);
          tmem_ld_wait ();
#pragma unroll
          for (int n = 0; n < 8; n++)
            zr[n] = fmaf (__int2float_rn ((int) v0[n]), s24, fmaf (__int2float_rn ((int) v1[n]), s16, fmaf (__int2float_rn ((int) v2[n]), s8, __int2float_rn ((int) v3[n]) * s0)));
          tmem_ld8 (taddr + 192 + 8 * i, v0); tmem_ld8 (taddr + 240 + 8 * i, v1); tmem_ld8 (taddr + 288 + 8 * i, v2); tmem_ld8 (taddr + 336 + 8 * i, v3);
          tmem_ld_wait ();
#pragma unroll
          for (int n = 0; n < 8; n++)
          {
            const float zi = fmaf (__int2float_rn ((int) v0[n]), s24, fmaf (__int2float_rn ((int) v1[n]), s16, fmaf (__int2float_rn ((int) v2[n]), s8, __int2float_rn ((int) v3[n]) * s0)));
            if (!fm) y[8 * i + n] = __fsqrt_rn (__fadd_rn (__fmul_rn (zr[n], zr[n]), __fmul_rn (zi, zi)));
            else
            {
              if (i == 0 && n == 0) { z0r = zr[0]; z0i = zi; y[0] = 0.f; }
              else y[8 * i + n] = fm_discriminator (zr[n], zi, pr, pi);
              pr = zr[n]; pi = zi;
            }
          }
        }
        tc_fence_before ();
        __syncwarp ();
        if (lane == 0) mbar_arrive (t_empty);
        bool carry_waited = false;
        if (fm)
        {
          // ---- FM: the sample before the block. Blocks 1..3 of the warp: the thread 8 lanes down; the warp's first block: the
          // previous warp's last thread through shared memory; the supertile's first block: the previous supertile's last sample
          // (two-slot carry, handed over with the biquad state) or, at the start of a call, the carried state of the channel.
          float qr = __shfl_up_sync (0xffffffffu, pr, 8), qi = __shfl_up_sync (0xffffffffu, pi, 8);
          if (a == 3) myZ[w * kJ + j] = make_float2 (pr, pi);
          if (kk != 0) mbar_wait (s_bar + ((kk - 1) & 1), ((kk - 1) >> 1) & 1);
          carry_waited = true;
          named_bar (5 + es, 128);
          if (a == 0)
          {
            float2 v;
            if (w > 0) v = myZ[(w - 1) * kJ + j];
            else if (k == 0) v = make_float2 (__ldcg (P.state + (size_t) c * 8 + 5), __ldcg (P.state + (size_t) c * 8 + 6));
            else v = sCarryZ[((kk - 1) & 1) * kJ + j];
            qr = v.x; qi = v.y;
          }
          y[0] = fm_discriminator (z0r, z0i, qr, qi);
        }
        // ---- zero-state response of the cascade over the block, per sample as arm_biquad_cascade_df2T_f32.c:551-562:
        //      y = b0 x + d1;  d1 = (b1 x + a1 y) + d2;  d2 = b2 x + a2 y
        float z[4] = { 0.f, 0.f, 0.f, 0.f };
#pragma unroll
        for (int n = 0; n < kBlk; n++)
        {
          const float x = y[n];
          const float y0 = fmaf (cf[0], x, z[0]);
          z[0] = fmaf (cf[3], y0, fmaf (cf[1], x, z[1]));
          z[1] = fmaf (cf[4], y0, cf[2] * x);
          const float y1 = fmaf (cf[5], y0, z[2]);
          z[2] = fmaf (cf[8], y1, fmaf (cf[6], y0, z[3]));
          z[3] = fmaf (cf[9], y1, cf[7] * y0);
          y[n] = y1;
        }
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
          matvec4 (P.tab.Mp[1], Pst, z, We);
          *reinterpret_cast<float4 *> (myW + (w * kJ + j) * 4) = make_float4 (We[0], We[1], We[2], We[3]);
        }
        // ---- carried state: from the previous call (first supertile) or the previous supertile (no carry-barrier phase is skipped)
        float S[4], envc;
        if (kk != 0 && !carry_waited) mbar_wait (s_bar + ((kk - 1) & 1), ((kk - 1) >> 1) & 1);
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
        named_bar (1 + 2 * es, 128);
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
          float en[4];
          matvec4 (P.tab.Mp[1], st, z, en);
          *reinterpret_cast<float4 *> (sCarryS + ((kk & 1) * kJ + j) * 4) = make_float4 (en[0], en[1], en[2], en[3]);
          if (fm) sCarryZ[(kk & 1) * kJ + j] = make_float2 (pr, pi);             // FM: this block's last baseband sample, for the next supertile
          if (k + 1 == supers && jvalid)
          {
            float *stw = P.state + (size_t) c * 8;
            __stcg (stw + 0, en[0]); __stcg (stw + 1, en[1]); __stcg (stw + 2, en[2]); __stcg (stw + 3, en[3]);
            if (fm) { __stcg (stw + 5, pr); __stcg (stw + 6, pi); }
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
        named_bar (2 + 2 * es, 128);
        // ---- AGC envelope: the oracle's sequential walk env_b = max (peak_b, fl (env_{b-1} * decay))
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
          const float g15 = gain * 32768.0f;                                       // exact: power of two
          uint4 *dst = reinterpret_cast<uint4 *> (P.out + (size_t) c * P.frames + t0);
#pragma unroll
          for (int n = 0; n < kBlk; n += 8)
            asm volatile ("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst + n / 4),
                          "r"(pack_lr (y[n] * g15)), "r"(pack_lr (y[n + 1] * g15)), "r"(pack_lr (y[n + 2] * g15)), "r"(pack_lr (y[n + 3] * g15)),
                          "r"(pack_lr (y[n + 4] * g15)), "r"(pack_lr (y[n + 5] * g15)), "r"(pack_lr (y[n + 6] * g15)), "r"(pack_lr (y[n + 7] * g15)) : "memory");
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

int launch_rx_am_tc (const RxAmTcLaunch &L, int sm_count, void *stream_)
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
  for (int i = 0; i < SLB_MAX_MASKS; i++) P.unit[i] = L.unit[i];
  P.flag_final = L.flag_final; P.n_groups = L.n_groups; P.frames = L.frames; P.supers = (L.frames + kSuper - 1) / kSuper;
  P.agc_target = L.agc_target; P.agc_decay = L.agc_decay; P.agc_floor = L.agc_floor; P.agc_gmax = L.agc_gmax;
  P.tab = *L.tables;
  cudaError_t e = cudaFuncSetAttribute (rx_am_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) Smem::bytes);
  if (e != cudaSuccess) return (int) e;
  uint32_t grid = (uint32_t) sm_count;
  if (grid > L.n_groups) grid = L.n_groups;
  if (const char *gs = std::getenv ("SELENITE_B200_TC_GRID")) { const long v = std::atol (gs); if (v > 0 && (uint32_t) v <= grid) grid = (uint32_t) v; }   // profiling / test knob
  rx_am_tc_kernel<<<grid, kThreads, Smem::bytes, stream>>> (P);
  return (int) cudaGetLastError ();
}

}  // namespace sl
