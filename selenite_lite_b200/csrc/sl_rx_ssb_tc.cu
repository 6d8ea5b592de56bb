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
#include <cstdio>
#include <cstdlib>
#include <cstring>
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
#ifndef SL_TC_SETS
#define SL_TC_SETS 2
#endif
#ifndef SL_TC_HALVES
#define SL_TC_HALVES 1                    /* warps per TMEM lane quadrant and epilogue set. 2 = a block's 48 samples are split between two warps (columns [0,24) / [24,48)):
                                             16 epilogue warps of 80 registers instead of 8 of 168. Measured equal (416 vs 423 Gsamples/s at 1024 channels, 461 vs 460 at
                                             8192): the kernel is bound by the L1 / shared-memory data pipe (tensor-core operand reads + LSU wavefronts), not by the
                                             latency of an epilogue set, so more epilogue warps buy nothing; kept as an A/B option */
#endif
#ifndef SL_TC_PAIR
#define SL_TC_PAIR 0                      /* 1: CTA pairs, tcgen05.mma.cta_group::2 (M = 256, each CTA fetches half of the map operand); 0: single CTAs */
#endif
#ifndef SL_TC_RAWSTAGES
#define SL_TC_RAWSTAGES 3
#endif
#ifndef SL_TC_REGSPLIT
#define SL_TC_REGSPLIT 0
#endif
#ifndef SL_TC_BULKOUT
#define SL_TC_BULKOUT 0
#endif
#ifndef SL_TC_MMA_UNROLL
#define SL_TC_MMA_UNROLL 1
#endif
#ifndef SL_TC_STHINT
#define SL_TC_STHINT ".L1::no_allocate"   /* measured: plain 366, .cg 371, .cs 376, .L1::no_allocate 408 Gsamples/s */
#endif
constexpr bool kPair = SL_TC_PAIR != 0;
static_assert (!SL_TC_PAIR, "the CTA-pair variant (tcgen05.mma.cta_group::2, measured slower: 315 vs 403 Gsamples/s at 1024 channels, 370 vs 445 at 8192, "
                            "gpurun_out/s4_*) predates the 32-bit map: its split of the map rows between the two CTAs assumes one N for both data bytes");
constexpr int kMmaUnroll = SL_TC_MMA_UNROLL;
constexpr int kSets = SL_TC_SETS;                 // epilogue warp sets (warpgroups), taking supertiles in turn
constexpr int kRawStages = SL_TC_RAWSTAGES;            // raw stages: a bulk copy takes ~4400 clocks to land (measured), a supertile ~3000
constexpr int kHalves = SL_TC_HALVES;
constexpr int kHalf = kBlk / kHalves;              // samples of a block per epilogue thread
constexpr int kEpiWarps = 4 * kSets * kHalves;
static_assert (kHalves == 1 || (kHalves == 2 && !SL_TC_PAIR && !SL_TC_BULKOUT && !SL_TC_REGSPLIT), "the split epilogue has no CTA-pair / bulk-store / register-split variant");
#ifndef SL_TC_CONVWARPS
#define SL_TC_CONVWARPS 2
#endif
constexpr int kConvWarps = SL_TC_CONVWARPS;        // 2, 3 or 4: the converters' shared-memory accesses queue behind the tensor core's operand reads (latency-bound role)
constexpr int kGroups = kChunksNew / 4;            // groups of 4 chunks (32 frames) of a supertile: 24; warp cw converts the groups t = cw (mod kConvWarps)
static_assert ((kGroups / 2) % kConvWarps == 0, "a half supertile splits evenly too");
constexpr int kMmaWarp = kEpiWarps + kConvWarps, kProdWarp = kMmaWarp + 1;
constexpr int kThreads = 32 * (kProdWarp + 1);   // 16 warps = 4 warpgroups: 3 epilogue sets + {2 converters, MMA issuer, producer}
static_assert (!SL_TC_REGSPLIT || kThreads == 512, "register split below assumes 4 warpgroups");
constexpr int kOutRow = 2 * kBlk * 4 + 16;  // output stage of one epilogue warp (SL_TC_BULKOUT): two blocks of a channel (384 B) + pad, ...
constexpr int kOutStage = kJ * kOutRow;    // ... of all eight channels
constexpr int kTmemCols = 512;           // two accumulator buffers of 256 columns

struct Smem
{
  static constexpr size_t a = 0;                                        // [2 buffers][hi plane | lo plane]
  static constexpr size_t b = a + 2 * 2 * kPlaneBytes;                  // tap planes of the current mask
  static constexpr size_t b_bytes = kPair ? kTcPlaneBytes / 2 : kTcPlaneBytes;   // pair: this CTA's half of the rows of every K-step
  static constexpr size_t raw = b + b_bytes;                            // [stages][8 rows]
  static constexpr size_t hist = raw + kRawStages * kJ * kRawRow;       // [stages][8 rows] carried tail of the previous call
  static constexpr size_t out = hist + kRawStages * kJ * kHistRow;      // [8 rows] packed int16 output of one supertile, stored by bulk copies
  static constexpr size_t wsum = out + (SL_TC_BULKOUT == 2 ? kJ * kRawRow : SL_TC_BULKOUT ? kEpiWarps * kOutStage : 0);                    // [sets][4 warps][8][4] floats
  static constexpr size_t pk = wsum + kSets * 4 * kJ * 4 * 4;           // [sets][halves][16][8] floats
  static constexpr size_t carry_s = pk + kSets * kHalves * kQ * kJ * 4; // [2][8][4] floats
  static constexpr size_t carry_e = carry_s + 2 * kJ * 4 * 4;           // [2][8] floats
  static constexpr size_t mp = carry_e + 2 * kJ * 4;                    // [4][20] floats: A^(48 a), rows padded to 20 (bank spread)
  static constexpr size_t bars = mp + 4 * 20 * 4;
  static constexpr int n_bars = 28;
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
  const uint32_t *pairs;                       // [n_items][2] groups of a CTA pair (same mask slot); 0xFFFFFFFF = none (the CTA idles along on the partner's data)
  const uint8_t *planes;
  float s0[SLB_MAX_MASKS], sz[SLB_MAX_MASKS];
  long long *trace;                            // profiling aid (SELENITE_B200_TC_TRACE): [supertile][16] clock64 stamps of CTA 0
  unsigned flag_final;
  uint32_t n_groups, n_items, frames, supers;   // n_items: work items of the launch = groups (single CTAs) or pairs of groups
  float agc_target, agc_decay, agc_floor, agc_gmax;
  TcBiquadTables tab;
};

#include "sl_tc_common.cuh"

__device__ __forceinline__ uint32_t pack_lr (float x_times_32768)
{
  // arm_float_to_q15.c:147 : (q15_t) __SSAT((q31_t)(x * 32768.0f), 16): truncation toward zero, then saturation.
#ifdef SL_TC_ABLATE_CVT                                                                // (profiling aid: what the conversions cost)
  return __float_as_uint (x_times_32768);
#elif !defined(SL_TC_NOF2I)
  short v;
  asm ("cvt.rzi.sat.s16.f32 %0, %1;" : "=h"(v) : "f"(x_times_32768));
  return __byte_perm ((uint32_t) (uint16_t) v, 0u, 0x1010);   // stereo endpoint, L = R (usbd_audio.c:399-404)
#else
  // A/B alternative without the conversion pipe (-DSL_TC_NOF2I): clamp, add |v| to 1.5 * 2^23 rounding TOWARD ZERO — the
  // sum's low mantissa bits are floor(|v|) — and restore the sign in two's complement. Exact, but 7 instructions instead of 2:
  // measured 266 vs 291 Gsamples/s, the epilogue is bound by instruction count, not by the F2I rate.
  const float c = fmaxf (fminf (x_times_32768, 32767.0f), -32768.0f);
  const int m = __float_as_int (__fadd_rz (fabsf (c), 12582912.0f));
  const int s = __float_as_int (c) >> 31;
  return __byte_perm ((uint32_t) ((m ^ s) - s), 0u, 0x1010);   // stereo endpoint, L = R (usbd_audio.c:399-404)
#endif
}

// y = M x (4x4 row-major, uniform M) + add
__device__ __forceinline__ void matvec4 (const float *M, const float *x, const float *add, float *y)
{
#pragma unroll
  for (int r = 0; r < 4; r++) y[r] = add[r] + (M[4 * r] * x[0] + M[4 * r + 1] * x[1] + M[4 * r + 2] * x[2] + M[4 * r + 3] * x[3]);
}

// split epilogue: the zero-input response of the block's start state added to one half's samples (4 FMA per sample, the only
// biquad arithmetic left on the CUDA cores) and the half's peak (arm_abs_f32 + arm_max_f32). The half is a template parameter so
// that the response table stays an immediate constant-bank operand.
template <int H> __device__ __forceinline__ float corr_half (const KParams &P, float (&y)[kHalf], const float (&st)[4])
{
  float peak = 0.f;
#pragma unroll
  for (int n = 0; n < kHalf; n++)
  {
    const float *C = P.tab.Cresp[H * kHalf + n];
    y[n] = fmaf (C[0], st[0], fmaf (C[1], st[1], fmaf (C[2], st[2], fmaf (C[3], st[3], y[n]))));
    peak = fmaxf (peak, fabsf (y[n]));
  }
  return peak;
}

// pipeline trace (tools/tc_trace.py): build with -DSL_TC_TRACE; the stamps cost 7 % even when no buffer is attached
#ifndef SL_TC_TRACE_CW
#define SL_TC_TRACE_CW 0                  /* which converter warp writes the converter stamps */
#endif
#ifndef SL_TC_TRACE
#define TC_STAMP(slot) do { } while (0)
#else
#define TC_STAMP(slot) do { if (P.trace && blockIdx.x == 0 && lane == 0) P.trace[(size_t) kk * 16 + (slot)] = clock64 (); } while (0)
#endif

// work item -> the channel group this CTA serves. Single CTAs: item = group. CTA pairs: item = two groups of one mask slot, one per
// CTA; a pair with one group only lets its second CTA run along on the partner's channels without storing anything (the MMAs of a
// pair are issued for both CTAs at once, so both must present operands and drain accumulators for every supertile).
struct Item { uint32_t g; bool idle; };
__device__ __forceinline__ Item item_group (const KParams &P, uint32_t it, uint32_t rank)
{
  if (!kPair) return Item{ it, false };
  uint32_t g = P.pairs[2 * it + rank];
  const bool idle = g == 0xFFFFFFFFu;
  if (idle) g = P.pairs[2 * it + (rank ^ 1u)];
  return Item{ g, idle };
}

__global__ void __launch_bounds__ (kThreads, 1) rx_ssb_tc_kernel (const __grid_constant__ KParams P)
{
  extern __shared__ __align__ (1024) unsigned char smem[];
  unsigned char *sA = smem + Smem::a, *sB = smem + Smem::b, *sRaw = smem + Smem::raw, *sHist = smem + Smem::hist;
  float *sW = reinterpret_cast<float *> (smem + Smem::wsum), *sPk = reinterpret_cast<float *> (smem + Smem::pk);
  float *sCarryS = reinterpret_cast<float *> (smem + Smem::carry_s), *sCarryE = reinterpret_cast<float *> (smem + Smem::carry_e);
  float *sMp = reinterpret_cast<float *> (smem + Smem::mp);
#if SL_TC_BULKOUT
  unsigned char *sOut = smem + Smem::out;
#endif
  uint64_t *bars = reinterpret_cast<uint64_t *> (smem + Smem::bars);
  uint64_t *raw_full = bars, *raw_empty = bars + 3, *a_full = bars + 6, *a_empty = bars + 8, *t_empty = bars + 10;
  uint64_t *s_bar = bars + 12, *e_bar = bars + 14, *b_full = bars + 16, *drain = bars + 17, *t_full = bars + 18, *out_free = bars + 22, *b_ready = bars + 26;
  // t_full has FOUR slots although there are two accumulator buffers: an epilogue set may start waiting for supertile
  // kk + 2 while kk is still in flight, and on a two-slot barrier that wait would alias the phase before kk's and pass at once
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *> (smem + Smem::tmem_ptr);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // pair mode: rank 0 of the cluster is the leader (issues the MMAs of both CTAs); a_full, t_empty and b_ready of the LEADER collect
  // arrivals from both CTAs, t_full / a_empty / drain of each CTA are reached by the leader's multicast commits
  const uint32_t rank = kPair ? cluster_ctarank () : 0u;
  const uint32_t item0 = kPair ? cluster_id_x () : blockIdx.x, istride = kPair ? cluster_n_x () : gridDim.x;
  if (tid == 0)
  {
    for (int i = 0; i < kRawStages; i++) { mbar_init (raw_full + i, 1); mbar_init (raw_empty + i, kConvWarps); }
    for (int i = 0; i < 2; i++)
    {
      mbar_init (a_full + i, (kPair ? 2 : 1) * kConvWarps); mbar_init (a_empty + i, 1);
      mbar_init (t_full + i, 1); mbar_init (t_full + 2 + i, 1); mbar_init (t_empty + i, (kPair ? 2 : 1) * 4 * kHalves); mbar_init (s_bar + i, kJ); mbar_init (e_bar + i, kJ);
    }
    mbar_init (b_full, 1); mbar_init (drain, 1); mbar_init (b_ready, 1);
    for (int i = 0; i < 4; i++) mbar_init (out_free + i, 1);                        // (slot 0 in use: SL_TC_BULKOUT == 2)
    asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 64) sMp[(tid >> 4) * 20 + (tid & 15)] = P.tab.Mp[tid >> 4][tid & 15];
  if (warp == kMmaWarp)
  {
    if (kPair)
    {
      // the same warp of both CTAs allocates the same columns in both tensor memories
      asm volatile ("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32 (tmem_ptr)), "n"(kTmemCols) : "memory");
      asm volatile ("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    else
    {
      asm volatile ("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32 (tmem_ptr)), "n"(kTmemCols) : "memory");
      asm volatile ("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before ();
  __syncthreads ();
  if (kPair) cluster_sync_all ();                  // the peer's barriers are initialised before anything arrives on them
  tc_fence_after ();
  const uint32_t tmem = *tmem_ptr;
  const uint32_t a_full_ldr = mapa_u32 (smem_u32 (a_full), 0u), t_empty_ldr = mapa_u32 (smem_u32 (t_empty), 0u), b_ready_ldr = mapa_u32 (smem_u32 (b_ready), 0u);
  const uint32_t supers = P.supers;
  // Columns [0,52) of both accumulator buffers start at zero: the xh MMAs accumulate into them (see the MMA issuer); afterwards
  // the epilogue set that drains a buffer zeroes them again.
  if (warp < 8) tmem_zero<kDig> (tmem + (uint32_t) (warp >> 2) * 256u + ((uint32_t) (32 * (warp & 3)) << 16));
  tc_fence_before ();
  __syncthreads ();
  tc_fence_after ();
  // register split between the warpgroups (the launch gives every thread 128): the epilogue holds a 48-sample block plus
  // 64 accumulator words per thread, the copy / convert / issue roles need little
  // (the whole warpgroup executes ONE setmaxnreg: the three small roles share warpgroup 3 and release together, as a
  // .sync.aligned instruction requires; the epilogue warpgroups acquire at the head of their branch)
#if SL_TC_REGSPLIT
  if (warp >= kEpiWarps) asm volatile ("setmaxnreg.dec.sync.aligned.u32 56;");
#endif

  if (warp == kProdWarp)
  {
    // ======================================= bulk-copy producer =======================================
    // Lane j < 8 owns row j of the group: it reads its channel index ONCE per work item and issues that row's bulk copy for
    // every supertile. (Until round 2 one lane walked the eight rows and read the index from global memory for every row of every
    // supertile — eight dependent L2 round trips of ~400 clocks under load: the producer, not the epilogue or the MMAs, set the
    // kernel's pace of ~3500 clocks per supertile, which is why no epilogue or MMA variant ever moved it.)
    {
      unsigned kk = 0;
#ifdef SL_TC_L2HINT
      uint64_t pol;
      asm volatile ("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
#endif
      for (uint32_t it = item0; it < P.n_items; it += istride)
      {
        const uint32_t g = item_group (P, it, rank).g;
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
            TC_STAMP (0);
            mbar_expect_tx (raw_full + rb, kJ * nfr * 4u + (k == 0 ? kJ * kHist * 4u : 0u));
          }
          __syncwarp ();
          if (lane < kJ)
          {
#ifdef SL_TC_L2HINT
            bulk_g2s_stream (sRaw + (rb * kJ + lane) * kRawRow, src + (size_t) k * kSuper, nfr * 4u, raw_full + rb, pol);
#else
            bulk_g2s (sRaw + (rb * kJ + lane) * kRawRow, src + (size_t) k * kSuper, nfr * 4u, raw_full + rb);
#endif
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
    for (uint32_t it = item0; it < P.n_items; it += istride)
    {
      const Item item = item_group (P, it, rank);
      const uint32_t g = item.g, nvalid = item.idle ? 0u : P.ginfo[g] >> 8, gs = P.gstart[g];
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        const int rb = kk % kRawStages, ab = kk & 1;
        const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper);
        unsigned char *Ahi = sA + ab * 2 * kPlaneBytes;
        mbar_wait_long (raw_full + rb, (kk / kRawStages) & 1);
        if (cw == SL_TC_TRACE_CW) TC_STAMP (1);
        mbar_wait_long (a_empty + ab, ((kk >> 1) & 1) ^ 1);                         // the MMAs of supertile kk - 2 have read this buffer
        if (cw == SL_TC_TRACE_CW) TC_STAMP (2);
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
        if (cw == SL_TC_TRACE_CW) TC_STAMP (3);
        if (lane == 0) { if (kPair) mbar_arrive_cluster (a_full_ldr + ab * 8u); else mbar_arrive (a_full + ab); mbar_arrive (raw_empty + rb); }
      }
    }
  }
  else if (warp == kMmaWarp)
  {
    // ========================================== MMA issuer ==========================================
    // The whole warp walks the loop converged and ONE elected lane issues: with `if (lane == 0)` around the loop the
    // compiler cannot keep descriptors in uniform registers and wraps every tcgen05.mma in a vote / broadcast loop —
    // measured 128 clocks of issue per MMA against 116 of execution (N = 144).
    constexpr uint32_t id_ss = kPair ? umma_idesc_pair (kNhi, 1, 1) : umma_idesc (kNhi, 1, 1), id_us = kPair ? umma_idesc_pair (kN, 0, 1) : umma_idesc (kN, 0, 1);
    const uint32_t aBase = smem_u32 (sA), bBase = smem_u32 (sB);
    // constant upper halves of the descriptors: LBO = 128 (A and B), SBO = 768 (A, aliased row groups) / 256 (B), version 1
    constexpr uint64_t kDescA = ((uint64_t) (kChunkBytes >> 4) << 16) | ((uint64_t) ((6 * kChunkBytes) >> 4) << 32) | (1ull << 46);
    constexpr uint64_t kDescB = ((uint64_t) (128 >> 4) << 16) | ((uint64_t) (256 >> 4) << 32) | (1ull << 46);
    // pair mode: every CTA holds HALF of the map's rows of each K-step (rows [80 rank, 80 rank + 80) of the 160, the split
    // tcgen05.mma.cta_group::2 expects: tools/microbench/umma_cta2.cu), at the same shared-memory offsets in both CTAs
    constexpr uint32_t kBStepS = kPair ? kBStep / 2 : kBStep;            // K-step stride of the planes in shared memory
    unsigned kk = 0, b_loads = 0, drains = 0;
    int cur_slot = -1;
    for (uint32_t it = item0; it < P.n_items; it += istride)
    {
      const uint32_t g = item_group (P, it, rank).g;
      const int slot = (int) (P.ginfo[g] & 0xFFu);                             // (both groups of a pair have the same slot)
      if (slot != cur_slot)
      {
        // (re)load the tap planes of this mask; earlier MMAs may still be reading the old ones (in pair mode: in BOTH CTAs — the
        // leader's commit reaches the drain barrier of both)
        if (kk != 0)
        {
          if (rank == 0 && elect_one ()) { if (kPair) umma_commit_pair (drain); else umma_commit (drain); }
          __syncwarp ();
          mbar_wait (drain, drains & 1); drains++;
        }
        if (elect_one ())
        {
          mbar_expect_tx (b_full, (unsigned) Smem::b_bytes);
          if (kPair)
          {
#pragma unroll 1
            for (int ks = 0; ks < kKSteps; ks++)
              bulk_g2s (sB + ks * kBStepS, P.planes + (size_t) slot * kTcPlaneBytes + (size_t) ks * kBStep + (size_t) rank * kBStepS, kBStepS, b_full);
          }
          else bulk_g2s (sB, P.planes + (size_t) slot * kTcPlaneBytes, (unsigned) kTcPlaneBytes, b_full);
        }
        __syncwarp ();
        mbar_wait (b_full, b_loads & 1);
        if (kPair)
        {
          // the leader may issue only when the follower's half has landed too
          if (rank != 0) { if (lane == 0) mbar_arrive_cluster (b_ready_ldr); }
          else mbar_wait_cluster (b_ready, b_loads & 1);
        }
        b_loads++;
        cur_slot = slot;
      }
      if (rank != 0) { kk += supers; continue; }                               // the follower's MMAs are issued by the leader
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        const int ab = kk & 1, tb = kk & 1;
        if (kPair) mbar_wait_cluster (a_full + ab, (kk >> 1) & 1); else mbar_wait_guarded (a_full + ab, (kk >> 1) & 1);
        TC_STAMP (4);
        // the epilogue (of both CTAs) has drained this accumulator buffer and zeroed its columns [0,52)
        if (kPair) mbar_wait_cluster (t_empty + tb, ((kk >> 1) & 1) ^ 1); else mbar_wait_guarded (t_empty + tb, ((kk >> 1) & 1) ^ 1);
        TC_STAMP (5);
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
#ifdef SL_TC_ABLATE_MMA                                                             // (profiling aid: what the MMAs cost)
            if (ks > 0) break;
#endif
            const uint32_t ao = (uint32_t) (ks * 2 * kChunkBytes) >> 4, bo = (uint32_t) (ks * kBStepS) >> 4;
            if (kPair)
            {
              umma_i8_pair (d + kDig, kDescA | (aLo + ao), kDescB | (b0 + bo), id_us, ks ? 1u : 0u);
              umma_i8_pair (d, kDescA | (aHi + ao), kDescB | (b0 + bo), id_ss, 1u);
            }
            else
            {
              umma_i8 (d + kDig, kDescA | (aLo + ao), kDescB | (b0 + bo), id_us, ks ? 1u : 0u);
              umma_i8 (d, kDescA | (aHi + ao), kDescB | (b0 + bo), id_ss, 1u);
            }
          }
          // accumulators complete -> epilogue; planes read -> converter may overwrite them (pair mode: in both CTAs)
          if (kPair) { umma_commit_pair (t_full + (kk & 3)); umma_commit_pair (a_empty + ab); }
          else { umma_commit (t_full + (kk & 3)); umma_commit (a_empty + ab); }
        }
        __syncwarp ();
        TC_STAMP (6);
      }
    }
  }
  else
  {
    // ========================================== epilogue ==========================================
#if SL_TC_HALVES == 2
    // TMEM lane = 32 w + lane = 8 q + j: the two threads (q, j) of a set — one in each of the two warps that may read lane quadrant
    // w — own firmware block q of channel j of the supertile, half h its samples [24 h, 24 h + 24). Both run the (short) state chain
    // of the block; half 0 hands state and envelope on to the next supertile.
    const int es = warp >> 3, h = (warp >> 2) & 1, w = warp & 3, a = lane >> 3, j = lane & 7, q = 4 * w + a;
    const bool tracer = (w == 0 && h == 0);
    float *myW = sW + es * (4 * kJ * 4), *myPk = sPk + es * (kHalves * kQ * kJ);
    const float decay = P.agc_decay;
    unsigned kk = 0;
    for (uint32_t it = item0; it < P.n_items; it += istride)
    {
      const uint32_t g = it, gi = P.ginfo[g];
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
        mbar_wait_long (t_full + (kk & 3), (kk >> 2) & 1);
        tc_fence_after ();
        if (tracer) TC_STAMP (7);
        // ---- accumulators -> float: y = (D24 2^24 + D16 2^16 + D8 2^8 + D0) * unit (arm_q15_to_float's 1/32768 folded in)
        float y[kHalf];
        const uint32_t taddr = tmem + (uint32_t) tb * 256u + ((uint32_t) (32 * w) << 16);
        const uint32_t tcol = taddr + (uint32_t) (h * kHalf);
#pragma unroll
        for (int i = 0; i < kHalf / 8; i++)
        {
          uint32_t v0[8], v1[8], v2[8], v3[8];
          tmem_ld8 (tcol + 8 * i, v0); tmem_ld8 (tcol + kDig + 8 * i, v1); tmem_ld8 (tcol + 2 * kDig + 8 * i, v2); tmem_ld8 (tcol + 3 * kDig + 8 * i, v3);
          tmem_ld_wait ();
#pragma unroll
          for (int n = 0; n < 8; n++)
            y[8 * i + n] = fmaf (__int2float_rn ((int) v0[n]), s24, fmaf (__int2float_rn ((int) v1[n]), s16, fmaf (__int2float_rn ((int) v2[n]), s8, __int2float_rn ((int) v3[n]) * s0)));
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
        // both warps of the quadrant have read (the state columns are read by both): columns [0,52) are zeroed for the next
        // supertile's xh MMAs, each warp its own audio columns, half 1 the state columns too
        tc_fence_before ();
        named_bar (7 + 4 * es + w, 64);
        tc_fence_after ();
        if (h == 0) tmem_zero<kHalf> (taddr); else tmem_zero<kHalf + 4> (taddr + kHalf);
        tc_fence_before ();
        __syncwarp ();
        if (lane == 0) mbar_arrive (t_empty + tb);                                 // the accumulator buffer now lives in registers
        if (tracer) TC_STAMP (8);
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
        if (a == 3 && h == 0)
        {
          float We[4];
          matvec4 (P.tab.Mp[1], Pst, z, We);                                      // the warp's four blocks from a zero start
          *reinterpret_cast<float4 *> (myW + (w * kJ + j) * 4) = make_float4 (We[0], We[1], We[2], We[3]);
        }
        // ---- carried state of the channel: from the previous call (first supertile) or the previous supertile
        // (every supertile but the CTA's first waits for its predecessor's hand-over, also across items where the value is
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
        if (tracer) TC_STAMP (10);
        named_bar (1 + 3 * es, 128 * kHalves);
        if (tracer) TC_STAMP (11);
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
        if (last_q && h == 0)
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
        // ---- add the zero-input response of the true start state; the half's peak
        const float peak = (h == 0) ? corr_half<0> (P, y, st) : corr_half<1> (P, y, st);
        myPk[(h * kQ + q) * kJ + j] = peak;
        if (kk != 0) mbar_wait (e_bar + ((kk - 1) & 1), ((kk - 1) >> 1) & 1);
        envc = (k == 0) ? __ldcg (P.state + (size_t) c * 8 + 4) : sCarryE[((kk - 1) & 1) * kJ + j];
        if (tracer) TC_STAMP (12);
        named_bar (2 + 3 * es, 128 * kHalves);
        if (tracer) TC_STAMP (13);
        // ---- AGC envelope: the oracle's sequential walk env_b = max(peak_b, fl(env_{b-1} * decay)) over the blocks before and
        // including this one; a block's peak (arm_max_f32 over its 48 samples) is the larger of its halves' peaks
        // (a [half][channel][block] layout read as 16-byte words was measured slower: 396 vs 416 Gsamples/s)
        float e = envc;
#pragma unroll
        for (int qq = 0; qq < kQ; qq++)
        {
          const float p = fmaxf (myPk[qq * kJ + j], myPk[(kQ + qq) * kJ + j]);
          if (qq <= q) e = fmaxf (p, e * decay);
        }
        if (last_q && h == 0)
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
        if (tracer) TC_STAMP (9);
        if (q < nblk && jvalid)
        {
          const size_t t0 = (size_t) k * kSuper + (size_t) q * kBlk + (size_t) (h * kHalf);
          if (P.audio_dbg)
          {
            float4 *adbg = reinterpret_cast<float4 *> (P.audio_dbg + (size_t) c * P.frames + t0);
#pragma unroll
            for (int n = 0; n < kHalf; n += 4) adbg[n / 4] = make_float4 (y[n], y[n + 1], y[n + 2], y[n + 3]);
          }
          if (P.gain_dbg && h == 0) P.gain_dbg[(size_t) c * (P.frames / kBlk) + t0 / kBlk] = gain;
          // ---- gain (arm_scale_f32), pack (arm_float_to_q15) and store: the half block is 96 contiguous bytes. 256-bit stores
          // (sm_100: STG.E.256) that do not allocate in L1 — the shared-memory / L1 data pipe is what the tensor core fetches its
          // operands through
          const float g15 = gain * 32768.0f;                                       // exact: power of two
          uint4 *dst = reinterpret_cast<uint4 *> (P.out + (size_t) c * P.frames + t0);
#ifdef SL_TC_ABLATE_ST                                                              // (profiling aid: what the output stores cost)
          if (g15 == 123.456f)
#endif
#pragma unroll
          for (int n = 0; n < kHalf; n += 8)
            asm volatile ("st.global" SL_TC_STHINT ".v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst + n / 4),
                          "r"(pack_lr (y[n] * g15)), "r"(pack_lr (y[n + 1] * g15)), "r"(pack_lr (y[n + 2] * g15)), "r"(pack_lr (y[n + 3] * g15)),
                          "r"(pack_lr (y[n + 4] * g15)), "r"(pack_lr (y[n + 5] * g15)), "r"(pack_lr (y[n + 6] * g15)), "r"(pack_lr (y[n + 7] * g15)) : "memory");
        }
        if (tracer) TC_STAMP (14);
      }
    }
#else
#if SL_TC_REGSPLIT
    asm volatile ("setmaxnreg.inc.sync.aligned.u32 152;");
#endif
    // TMEM lane = 32 w + lane = 8 q + j: thread (q, j) owns firmware block q of channel j of the supertile.
    const int es = warp >> 2, w = warp & 3, a = lane >> 3, j = lane & 7, q = 4 * w + a;
    float *myW = sW + es * (4 * kJ * 4), *myPk = sPk + es * (kQ * kJ);
    const float decay = P.agc_decay;
    unsigned kk = 0;
    for (uint32_t it = item0; it < P.n_items; it += istride)
    {
      const Item item = item_group (P, it, rank);
      const uint32_t g = item.g, gi = P.ginfo[g];
      const bool jvalid = !item.idle && (uint32_t) j < (gi >> 8);
      const uint32_t c = P.chan[P.gstart[g] + min ((uint32_t) j, (gi >> 8) - 1u)];
      const float s0 = P.s0[gi & 0xFFu], s8 = s0 * 256.0f, s16 = s0 * 65536.0f, s24 = s0 * 16777216.0f, z0s = P.sz[gi & 0xFFu];
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        if ((int) (kk % kSets) != es) continue;
        const int tb = kk & 1;
        const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper);
        const int nblk = (int) (nfr / kBlk);
        const bool last_q = q == nblk - 1;
        mbar_wait_long (t_full + (kk & 3), (kk >> 2) & 1);
        tc_fence_after ();
        if (w == 0) TC_STAMP (7);
        // ---- accumulators -> float: y = (D24 2^24 + D16 2^16 + D8 2^8 + D0) * unit (arm_q15_to_float's 1/32768 folded in)
        float y[kBlk];
        const uint32_t taddr = tmem + (uint32_t) tb * 256u + ((uint32_t) (32 * w) << 16);
#ifndef SL_TC_LDW
#define SL_TC_LDW 16
#endif
        constexpr int kW = SL_TC_LDW;                                              // accumulator columns per tcgen05.ld
#pragma unroll
        for (int i = 0; i < kBlk / kW; i++)
        {
          uint32_t v0[kW], v1[kW], v2[kW], v3[kW];
          if (kW == 16) { tmem_ld16 (taddr + kW * i, v0); tmem_ld16 (taddr + kDig + kW * i, v1); tmem_ld16 (taddr + 2 * kDig + kW * i, v2); tmem_ld16 (taddr + 3 * kDig + kW * i, v3); }
          else { tmem_ld8 (taddr + kW * i, v0); tmem_ld8 (taddr + kDig + kW * i, v1); tmem_ld8 (taddr + 2 * kDig + kW * i, v2); tmem_ld8 (taddr + 3 * kDig + kW * i, v3); }
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
        if (lane == 0) { if (kPair) mbar_arrive_cluster (t_empty_ldr + tb * 8u); else mbar_arrive (t_empty + tb); }   // the accumulator buffer now lives in registers
        if (w == 0) TC_STAMP (8);
#ifdef SL_TC_ABLATE_EPI                                                             // (profiling aid: the kernel without the epilogue's arithmetic and stores)
        if (y[0] != 123.456f || z[0] != 1.0f) continue;
#endif

        // (y[] already IS the zero-state response of the biquad cascade over the block — the operand planes hold the FIR
        //  composed with it — and columns 48..51 of each digit group hold the cascade's end state from a zero start)
        if (w == 0) TC_STAMP (9);
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
        // (every supertile but the CTA's first waits for its predecessor's hand-over, also across items where the value is
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
        if (w == 0) TC_STAMP (10);
        named_bar (1 + 3 * es, 128);
        if (w == 0) TC_STAMP (11);
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
#ifndef SL_TC_ENVSCAN                                                              // (default: the sequential walk; -DSL_TC_ENVSCAN: A/B alternative below)
        myPk[q * kJ + j] = peak;
        if (kk != 0) mbar_wait (e_bar + ((kk - 1) & 1), ((kk - 1) >> 1) & 1);
        envc = (k == 0) ? __ldcg (P.state + (size_t) c * 8 + 4) : sCarryE[((kk - 1) & 1) * kJ + j];
        if (w == 0) TC_STAMP (12);
        named_bar (2 + 3 * es, 128);
        if (w == 0) TC_STAMP (13);
        // ---- AGC envelope: the oracle's sequential walk env_b = max(peak_b, fl(env_{b-1} * decay)) over the blocks before and including this one
        float e = envc;
#pragma unroll
        for (int qq = 0; qq < kQ; qq++)
        {
          const float p = myPk[qq * kJ + j];
          if (qq <= q) e = fmaxf (p, e * decay);
        }
#else
        // ---- AGC envelope: the oracle's sequential walk env_b = max(peak_b, fl(env_{b-1} * decay)) over the blocks before and
        // including this one. x -> fl(x * decay) is monotonic, so fl(max(a, b) * decay) = max(fl(a * decay), fl(b * decay)) and the
        // walk equals a max-scan whose step of distance d applies the rounded multiply d times — bit for bit (the FFT kernel's
        // env_scan, sl_rx_ssb_f32.cu). Inside the warp: its four blocks of channel j sit in lanes j, j + 8, j + 16, j + 24.
        float e = peak;
        {
          const float t1 = __shfl_up_sync (0xffffffffu, e, 8) * decay;
          if (a >= 1) e = fmaxf (e, t1);
          const float t2 = (__shfl_up_sync (0xffffffffu, e, 16) * decay) * decay;
          if (a >= 2) e = fmaxf (e, t2);
        }
        if (a == 3) myPk[w * kJ + j] = e;                                          // the warp's four blocks from a zero envelope
        if (kk != 0) mbar_wait (e_bar + ((kk - 1) & 1), ((kk - 1) >> 1) & 1);
        envc = (k == 0) ? __ldcg (P.state + (size_t) c * 8 + 4) : sCarryE[((kk - 1) & 1) * kJ + j];
        if (w == 0) TC_STAMP (12);
        named_bar (2 + 3 * es, 128);
        if (w == 0) TC_STAMP (13);
        {
          // envelope at the end of the block before the warp's first one, then decayed to this block
          float cin = envc;
#pragma unroll
          for (int ww = 0; ww < 3; ww++)
            if (ww < w) cin = fmaxf (myPk[ww * kJ + j], (((cin * decay) * decay) * decay) * decay);
          float t = cin * decay;
          if (a >= 1) t *= decay;
          if (a >= 2) t *= decay;
          if (a >= 3) t *= decay;
          e = fmaxf (e, t);
        }
#endif
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
#if SL_TC_BULKOUT == 2
        // ---- gain (arm_scale_f32), pack (arm_float_to_q15), store through ONE shared-memory stage of a whole supertile ([8 channels][768
        // frames], rows padded like the raw stage: a 16-byte store of the 8 lanes of a quarter warp hits 8 different bank groups) that the
        // two epilogue sets use in turn: supertile kk takes it when kk - 1's bulk copies have read it (out_free, one phase per
        // supertile), the set's 128 threads lay their blocks in, and lanes 0..7 of the set's first warp send ONE 3072-byte bulk copy
        // per channel — 8 copies per supertile instead of 768 line-sized store wavefronts.
        {
          const float g15 = gain * 32768.0f;                                       // exact: power of two
          if (kk != 0) mbar_wait (out_free, (kk - 1) & 1);
          {
            uint4 *dst = reinterpret_cast<uint4 *> (sOut + j * kRawRow + q * (kBlk * 4));
#pragma unroll
            for (int n = 0; n < kBlk; n += 4)
              dst[n / 4] = make_uint4 (pack_lr (y[n] * g15), pack_lr (y[n + 1] * g15), pack_lr (y[n + 2] * g15), pack_lr (y[n + 3] * g15));
          }
          asm volatile ("fence.proxy.async.shared::cta;" ::: "memory");
          named_bar (9 + es, 128);
          if (w == 0)
          {
            if (lane < kJ)
            {
              if (jvalid) bulk_s2g (P.out + (size_t) c * P.frames + (size_t) k * kSuper, sOut + j * kRawRow, nfr * 4u);
              asm volatile ("cp.async.bulk.commit_group;" ::: "memory");
              asm volatile ("cp.async.bulk.wait_group.read 0;" ::: "memory");
            }
            __syncwarp ();
            if (lane == 0) mbar_arrive (out_free);
          }
        }
#elif SL_TC_BULKOUT
        // ---- gain (arm_scale_f32), pack (arm_float_to_q15), store through a shared-memory stage. A warp holds 4 consecutive blocks of
        // 8 channels = 768 contiguous bytes per channel, but as direct stores every instruction touches 32 different lines (32 L1
        // wavefronts). Here the warp lays two blocks of all eight channels at a time into its private stage (rows of 384 + 16 bytes:
        // the eight lanes of a quarter warp hit eight different 16-byte bank groups, so a 16-byte store of 16 lanes is its two ideal
        // wavefronts) and lanes 0..7 send one 384-byte bulk copy each. No other warp is involved.
        {
          const float g15 = gain * 32768.0f;                                       // exact: power of two
          unsigned char *stage = sOut + warp * kOutStage;
#pragma unroll
          for (int r = 0; r < 2; r++)
          {
            if (lane < 8) asm volatile ("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the stage's previous copies have been read
            __syncwarp ();
            if ((a >> 1) == r)
            {
              uint4 *dst = reinterpret_cast<uint4 *> (stage + j * kOutRow + (a & 1) * (kBlk * 4));
#pragma unroll
              for (int n = 0; n < kBlk; n += 4)
                dst[n / 4] = make_uint4 (pack_lr (y[n] * g15), pack_lr (y[n + 1] * g15), pack_lr (y[n + 2] * g15), pack_lr (y[n + 3] * g15));
            }
            asm volatile ("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp ();
            if (lane < 8)
            {
              // blocks of this round that exist in a short supertile at the end of a stream: 4 w + 2 r .. min (4 w + 2 r + 1, nblk - 1)
              const int q0 = 4 * w + 2 * r, nb = min (2, nblk - q0);
              if (nb > 0 && jvalid)
                bulk_s2g (P.out + (size_t) c * P.frames + (size_t) k * kSuper + (size_t) q0 * kBlk, stage + j * kOutRow, (unsigned) nb * kBlk * 4u);
              asm volatile ("cp.async.bulk.commit_group;" ::: "memory");
            }
          }
        }
#else
        // ---- gain (arm_scale_f32), pack (arm_float_to_q15) and store: the block is 192 contiguous bytes
        if (q < nblk && jvalid)
        {
          const float g15 = gain * 32768.0f;                                       // exact: power of two
#ifdef SL_TC_ABLATE_STADDR                                                          // (profiling aid: the same stores, but to one L2-resident block per thread)
          uint4 *dst = reinterpret_cast<uint4 *> (P.out + ((size_t) blockIdx.x * kThreads + tid) * kBlk);
#else
          uint4 *dst = reinterpret_cast<uint4 *> (P.out + (size_t) c * P.frames + (size_t) k * kSuper + (size_t) q * kBlk);
#endif
#ifdef SL_TC_ABLATE_ST                                                              // (profiling aid: what the output stores cost)
          if (g15 == 123.456f)
#endif
#ifdef SL_TC_ST128
#pragma unroll
          for (int n = 0; n < kBlk; n += 4)
            asm volatile ("st.global" SL_TC_STHINT ".v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(dst + n / 4),
                          "r"(pack_lr (y[n] * g15)), "r"(pack_lr (y[n + 1] * g15)), "r"(pack_lr (y[n + 2] * g15)), "r"(pack_lr (y[n + 3] * g15)) : "memory");
#else
#pragma unroll
          for (int n = 0; n < kBlk; n += 8)
          {
            // 256-bit stores (sm_100: STG.E.256): the 32 lanes of a store hit 32 different lines whatever its width, so the
            // L1 wavefronts per block halve; and the lines must not allocate in L1 — the shared-memory / L1 data pipe is what the
            // tensor core fetches its operands through, and the MMAs are the critical path
            asm volatile ("st.global" SL_TC_STHINT ".v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst + n / 4),
                          "r"(pack_lr (y[n] * g15)), "r"(pack_lr (y[n + 1] * g15)), "r"(pack_lr (y[n + 2] * g15)), "r"(pack_lr (y[n + 3] * g15)),
                          "r"(pack_lr (y[n + 4] * g15)), "r"(pack_lr (y[n + 5] * g15)), "r"(pack_lr (y[n + 6] * g15)), "r"(pack_lr (y[n + 7] * g15)) : "memory");
          }
#endif
        }
#endif
        if (w == 0) TC_STAMP (14);
      }
    }
#if SL_TC_BULKOUT
    if (lane < 8) asm volatile ("cp.async.bulk.wait_group 0;" ::: "memory");    // this warp's output copies complete before the CTA retires
    __syncwarp ();
#endif
#endif
  }

  tc_fence_before ();
  __syncthreads ();
  if (kPair) cluster_sync_all ();                  // neither CTA retires (shared memory, barriers, TMEM) while the peer may still reach into it
  if (warp == kMmaWarp)
  {
    tc_fence_after ();
    if (kPair) asm volatile ("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kTmemCols) : "memory");
    else asm volatile ("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kTmemCols) : "memory");
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
  if (kPair && (L.pairs == nullptr || L.n_pairs == 0)) return (int) cudaErrorInvalidValue;
  KParams P;
  P.in = reinterpret_cast<const uint32_t *> (L.in); P.out = reinterpret_cast<uint32_t *> (L.out);
  P.audio_dbg = L.audio_dbg; P.gain_dbg = L.gain_dbg;
  P.ovl_in = reinterpret_cast<const uint32_t *> (L.ovl_in); P.ovl_out = reinterpret_cast<uint32_t *> (L.ovl_out);
  P.state = L.state; P.flag = L.flag; P.chan = L.chan; P.gstart = L.gstart; P.ginfo = L.ginfo; P.pairs = L.pairs; P.planes = L.planes;
  for (int i = 0; i < SLB_MAX_MASKS; i++) { P.s0[i] = L.s0[i]; P.sz[i] = L.sz[i]; }
  P.flag_final = L.flag_final; P.n_groups = L.n_groups; P.n_items = kPair ? L.n_pairs : L.n_groups; P.frames = L.frames; P.supers = (L.frames + kSuper - 1) / kSuper;
  P.agc_target = L.agc_target; P.agc_decay = L.agc_decay; P.agc_floor = L.agc_floor; P.agc_gmax = L.agc_gmax;
  P.tab = *L.tables;
  static_assert (sizeof (KParams) <= 4000, "kernel parameter block");
  cudaError_t e = cudaFuncSetAttribute (rx_ssb_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) Smem::bytes);
  if (e != cudaSuccess) return (int) e;
  // one CTA per SM; pair mode: one cluster of two CTAs per work item (a TPC), at most sm_count / 2 clusters
  uint32_t ctas_per_item = kPair ? 2u : 1u;
  uint32_t grid_items = (uint32_t) sm_count / ctas_per_item;
  if (grid_items > P.n_items) grid_items = P.n_items;
  if (const char *gs = std::getenv ("SELENITE_B200_TC_GRID")) { const long v = std::atol (gs); if (v > 0 && (uint32_t) v <= grid_items) grid_items = (uint32_t) v; }   // profiling aid
  P.trace = nullptr;
  cudaLaunchConfig_t lc{};
  lc.gridDim = dim3 (grid_items * ctas_per_item); lc.blockDim = dim3 (kThreads); lc.dynamicSmemBytes = Smem::bytes; lc.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = ctas_per_item; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  lc.attrs = at; lc.numAttrs = 1;
#ifdef SL_TC_TRACE
  if (const char *tf = std::getenv ("SELENITE_B200_TC_TRACE"))
  {
    // profiling aid: clock64 stamps of every pipeline role of CTA 0, one row per supertile, dumped as text after the launch
    const size_t n = (size_t) P.supers * ((P.n_items + grid_items - 1) / grid_items) * 16;
    long long *d_tr = nullptr;
    if (cudaMalloc (&d_tr, n * 8) == cudaSuccess)
    {
      cudaMemset (d_tr, 0, n * 8);
      P.trace = d_tr;
      cudaLaunchKernelEx (&lc, rx_ssb_tc_kernel, P);
      cudaDeviceSynchronize ();
      long long *h = (long long *) std::malloc (n * 8);
      cudaMemcpy (h, d_tr, n * 8, cudaMemcpyDeviceToHost);
      if (FILE *f = std::fopen (tf, "w"))
      {
        for (size_t r = 0; r < n / 16; r++) { for (int c = 0; c < 16; c++) std::fprintf (f, "%lld ", h[r * 16 + c] ? h[r * 16 + c] - h[0] : -1ll); std::fprintf (f, "\n"); }
        std::fclose (f);
      }
      std::free (h); cudaFree (d_tr);
      return (int) cudaGetLastError ();
    }
  }
#endif
  e = cudaLaunchKernelEx (&lc, rx_ssb_tc_kernel, P);
  return (int) (e != cudaSuccess ? e : cudaGetLastError ());
}

}  // namespace sl
