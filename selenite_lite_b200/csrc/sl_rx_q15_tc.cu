// RX-SSB-q15 on the 5th-generation tensor cores (tcgen05 + TMEM): the all-integer chain of sl_rx_ssb_q15.cu, bit for bit.
//
//   int16 I/Q --> fir_q15 (I, hI), fir_q15 (Q, hQ) --add/sub (saturating)--> per-48-frame AGC (finite window) --> int16 L=R
//   oracle stage per box as in sl_rx_ssb_q15.cu (arm_fir_q15.c:591, arm_add_q15.c:54 / arm_sub_q15.c:54, arm_abs_q15.c:57,
//   arm_max_q15.c:58, arm_scale_q15.c:56 + our gain law).
//
// The two 64-tap FIRs are a dense contraction of the 64 + 48 frame raw window with Toeplitz matrices of taps, EXACT on the
// integer tensor cores: x = 256 xh + xl (signed high byte, unsigned low byte), h = 256 hh + hl (balanced signed digits),
//   acc = 65536 S2 + 256 S1 + S0,   S2 = sum xh hh,  S1 = sum xh hl + xl hh,  S0 = sum xl hl   (int32 TMEM accumulators)
//   (acc >> 15) = 2 S2 + ((256 S1 + S0) >> 15)                                  (arm_fir_q15.c:642, then __SSAT 16)
// Skeleton of sl_rx_ssb_tc.cu (same byte planes of the interleaved I/Q frames, aliased row groups, roles, pipelines); per
// supertile 7 K-steps x {xh, xl} = 14 tcgen05.mma of N = 192 (rows: rail I hh | rail I hl | rail Q hh | rail Q hl, a rail's
// rows are zero at the other rail's byte positions) into 2 x 192 accumulator columns, one accumulator buffer. The epilogue is
// all integer: thread (block q, channel j) rebuilds the 48 FIR outputs of both rails, mixes, takes the block peak; block
// peaks of the last four supertiles live in shared memory, which is all the finite AGC window (<= 17 blocks) needs.
//
// TX-SSB-q15 (kTx, DESIGN.md §3.7) is the same kernel: the input frames are the mic (L = R), both rails' taps sit at the L byte
// positions of the planes (R gets zero weight, so R is ignored), and the epilogue keeps (I, Q) = (fi, fq) or (fq, fi) by sideband
// instead of mixing, takes the block peak over |I| and |Q|, scales both rails with one gain word and stores I/Q frames.
//
// RX-Q15 (DESIGN.md §3.8) adds two detectors. AM: the same contraction with a real low-pass on both rails, and arm_cmplx_mag_q15
// instead of the mixer. FM: planes of N = 208 that also give each rail's FIR output at frame -1 (the sample before the block,
// whose 64-tap window is frames 0..63 of the 112-frame window), so every block holds z[n-1] for its first sample; the epilogue
// runs arm_cmplx_mag_q15 and the integer limiter-discriminator per sample. A launch of these kinds (and of the SSB kind in a
// context that mixes kinds) works on a list of channels: rxq15_launch groups a channel range by kind.
//
// TX-Q15 (DESIGN.md §3.9) adds two modulators on the TX planes (both rails filter the mic with the mode's low-pass; the epilogue reads
// rail I only): AM adds the scaled audio to the carrier, FM integrates y fm_inc into a per-channel uint32 phase and evaluates the table
// NCO of the f32 chains. The SSB modulator (kTx) takes a channel list too, for the SSB-style channels of a context that mixes kinds.
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include "sl_internal.h"

namespace sl {

namespace {

constexpr int kJ = kTcChannels, kQ = 16, kBlk = 48, kSuper = kQ * kBlk;
constexpr int kTaps = SLB_Q15_TAPS, kWin = SLB_Q15_WIN;
constexpr int kHist = kTaps;             // 64 frames of history (63 needed; 64 keeps the window on a chunk boundary)
constexpr int kChunkBytes = kJ * 16;     // one K-chunk (8 frames x {I,Q} bytes) of all 8 channels
constexpr int kChunksHist = kHist / 8;   // 8
constexpr int kChunksNew = kSuper / 8;   // 96
constexpr int kPlaneBytes = (kChunksHist + kChunksNew) * kChunkBytes;   // 13312
constexpr int kKSteps = 7;               // (64 + 48) frames * 2 bytes / 32
constexpr int kRawRow = kSuper * 4 + 16, kHistRow = kHist * 4 + 16;
// The two epilogue sets alternate supertiles. Splitting every supertile between them, 24 of a block's 48 samples each, is
// bit-identical but slower: 392 vs 467 Gsamples/s (one barrier of all eight warps per supertile puts the sets in lockstep).
constexpr int kSets = 2, kEpiWarps = 4 * kSets, kConvWarps = 2, kRawStages = 4;
constexpr int kMmaUnroll = 1;            // rolled: 489 vs 470 Gsamples/s (the unrolled issue loop costs instruction fetch: gcc requests at 78 % of peak)
constexpr int kMmaWarp = kEpiWarps + kConvWarps, kProdWarp = kMmaWarp + 1, kThreads = 32 * (kProdWarp + 1);
constexpr unsigned kPSlots = 4;
constexpr int kTmemCols = 512;           // xh products in columns [0,N), xl products in [N,2N) (N = 192; FM 208)

// detector kinds (template parameter of the kernel): the two SSB chains on contiguous channels, and the kinds of RX-Q15, which work
// on a channel list (kKindRxList: the SSB detector of kKindRx); TX-Q15's kinds work on a list too (kKindTxList: the modulator of kKindTx)
enum Kind : int { kKindRx = 0, kKindTx = 1, kKindAm = 2, kKindFm = 3, kKindRxList = 4, kKindTxList = 5, kKindTxAm = 6, kKindTxFm = 7 };
template <int K> constexpr int kRowsN = K == kKindFm ? 208 : 192;                  // B rows = MMA N
template <int K> constexpr int kBStepK = kRowsN<K> / 8 * 256;
template <int K> constexpr size_t kPlaneBK = (size_t) kKSteps * kBStepK<K>;   // 43008; FM 46592 (= kTcQ15FmPlaneBytes)
static_assert (kPlaneBK<kKindRx> == kTcQ15PlaneBytes && kPlaneBK<kKindFm> == kTcQ15FmPlaneBytes, "plane sizes");

template <size_t kBBytes, size_t kExtra = 0> struct SmemT
{
  static constexpr size_t a = 0;
  static constexpr size_t b = a + 2 * 2 * kPlaneBytes;
  static constexpr size_t raw = b + kBBytes;
  static constexpr size_t hist = raw + kRawStages * kJ * kRawRow;
  static constexpr size_t pk = hist + kRawStages * kJ * kHistRow;                // [4 tiles][16][8] int: block peaks of the last supertiles
  static constexpr size_t pkc = pk + 4 * kQ * kJ * 4;                            // [sets][16][8] int: peaks before the stream start, by 16 - age
  static constexpr size_t bars = pkc + kSets * kQ * kJ * 4;
  static constexpr int n_bars = 24;
  static constexpr size_t tmem_ptr = bars + n_bars * 8;
  static constexpr size_t extra = tmem_ptr + 16;                                  // kind-specific (TX FM: kTxFmExtra)
  static constexpr size_t bytes = extra + kExtra;
};
// TX FM: arm_sin_f32's table (513 floats), the per-channel phase advance of the last four supertiles ([4][8] uint32, slots as the
// peak tiles) and the scan's per-warp totals ([sets][4 warps][8] uint32)
constexpr size_t kSinBytes = 2064, kTotBytes = 4 * kJ * 4, kTxFmExtra = kSinBytes + kTotBytes + kSets * 4 * kJ * 4;
template <int K> using SmemK = SmemT<kPlaneBK<K>, K == kKindTxFm ? kTxFmExtra : 0>;
using Smem = SmemT<kTcQ15PlaneBytes>;
static_assert (SmemT<kTcQ15FmPlaneBytes>::bytes <= 227 * 1024 && SmemK<kKindTxFm>::bytes <= 227 * 1024, "one CTA per SM");

struct KParams
{
  const uint32_t *in; uint32_t *out;
  const uint32_t *tail_in; uint32_t *tail_out;  // [C][64] raw frames
  const int16_t *peaks_in; int16_t *peaks_out;  // [C][kWin] by age
  const uint8_t *planes; const uint8_t *lsb;
  int16_t *audio_dbg; uint32_t *gain_dbg;
  int16_t rel[kWin];
  uint32_t channels, frames, blocks, supers, gsz, n_groups, window;
  int32_t target, floor_; uint32_t gmax;
  const uint32_t *list; int32_t fm_floor;      // channel list (kinds kKindAm, kKindFm, kKindRxList); FM: the discriminator's floor
  uint32_t *phase; const float *sin513;        // TX FM: [C] phase words (read at the stream start, written at its end); the NCO table
  int32_t am_carrier, fm_inc; float fm_level15; // TX AM: the carrier (q15); TX FM: 2^-32 turn per LSB of y, NCO level x 32768
};

#include "sl_tc_common.cuh"
#include "sl_nco.cuh"

// (cvt.sat.s16.s32 is one instruction but runs on the conversion pipe: 403 vs 467 Gsamples/s. Raw stages with the MMA issue loop rolled: 2 -> 475, 3 -> 486, 4 -> 489 Gsamples/s; with it unrolled 468 .. 470 whatever the stages)
#include "sl_q15.cuh"
// the limiter-discriminator (ours, DESIGN.md §3.8): sat16 (trunc ((x 2^13) / max (m_prev m, floor))), x = a_prev b - b_prev a. |quotient|
// < 2^15 unless it saturates, so a float reciprocal estimate is within one of it and one integer correction makes it exact
__device__ __forceinline__ int fm_disc (int pa, int pb, int pm, int a, int b, int m, int floor_)
{
  const long long x = (long long) pa * b - (long long) pb * a;
  const long long den = max (pm * m, floor_);                                    // pm m <= 23170^2 < 2^31
  const long long N = (x < 0 ? -x : x) << 13;
  int q;
  if (N >= (den << 15)) q = 32768;
  else
  {
    q = (int) ((float) N * __frcp_rn ((float) den));
    const long long r = N - (long long) q * den;
    if (r < 0) q--;
    else if (r >= den) q++;
  }
  return x < 0 ? -q : min (q, 32767);
}

template <int kKind>
__global__ void __launch_bounds__ (kThreads, 1) rx_q15_tc_kernel (const __grid_constant__ KParams P)
{
  constexpr bool kTx = kKind == kKindTx || kKind == kKindTxList, kList = kKind >= kKindAm;
  constexpr bool kMono = kKind == kKindTxAm || kKind == kKindTxFm;               // TX AM / FM: one rail, a = the mic's low-pass
  constexpr int kN = kRowsN<kKind>;                                              // xl products from column kN on
  using Smem = SmemK<kKind>;
  extern __shared__ __align__ (1024) unsigned char smem[];
  unsigned char *sA = smem + Smem::a, *sB = smem + Smem::b, *sRaw = smem + Smem::raw, *sHist = smem + Smem::hist;
  int *sPk = reinterpret_cast<int *> (smem + Smem::pk), *sPkC = reinterpret_cast<int *> (smem + Smem::pkc);
  uint64_t *bars = reinterpret_cast<uint64_t *> (smem + Smem::bars);
  static_assert (kRawStages >= 2 && kRawStages <= 4, "barrier layout");
  uint64_t *raw_full = bars, *raw_empty = bars + 4, *a_full = bars + 8, *a_empty = bars + 10, *t_empty = bars + 12;
  uint64_t *b_full = bars + 15, *t_full = bars + 16, *p_bar = bars + 18;
  // p_bar has FOUR slots: a set arrives for supertile kk BEFORE it waits for its predecessor's peaks, so the other set can arrive for
  // kk + 1 while a warp of this one has not yet looked at kk - 1 (it does whenever the global load at the start of a group takes longer
  // than the MMAs of kk + 1: seen as a hang at 8192 channels). On two slots kk + 1 completes the phase after kk - 1's on the same
  // barrier and the late wait never returns; on four the next arrival on kk - 1's slot is kk + 3, which needs this set's read-out
  // of kk + 2.
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *> (smem + Smem::tmem_ptr);
  float *sSin = reinterpret_cast<float *> (smem + Smem::extra);
  uint32_t *sTot = reinterpret_cast<uint32_t *> (smem + Smem::extra + kSinBytes), *sScan = sTot + 4 * kJ;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if constexpr (kKind == kKindTxFm)
    for (int i = tid; i < 513; i += kThreads) sSin[i] = P.sin513[i];
  if (tid == 0)
  {
    for (int i = 0; i < kRawStages; i++) { mbar_init (raw_full + i, 1); mbar_init (raw_empty + i, kConvWarps); }
    for (int i = 0; i < 2; i++)
    {
      mbar_init (a_full + i, kConvWarps); mbar_init (a_empty + i, 1);
      mbar_init (t_full + i, 1);
    }
    for (int i = 0; i < kPSlots; i++) mbar_init (p_bar + i, 4);
    mbar_init (t_empty, 4); mbar_init (b_full, 1);
    asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
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
  // channels of group g: [g * gsz, g * gsz + nv); rows beyond nv repeat the last channel and are never stored
  auto group_nv = [&] (uint32_t g) { return min (P.gsz, P.channels - g * P.gsz); };
  // channel of row jj of group g: contiguous, or the list entry (list kinds; P.channels = the list's length)
  auto chan = [&] (uint32_t g, uint32_t jj) -> uint32_t { if constexpr (kList) return P.list[g * P.gsz + jj]; else return g * P.gsz + jj; };

  if (warp == kProdWarp)
  {
    if (lane == 0)
    {
      // the tap planes are the same for every channel: loaded once
      mbar_expect_tx (b_full, (unsigned) kPlaneBK<kKind>);
      bulk_g2s (sB, P.planes, (unsigned) kPlaneBK<kKind>, b_full);
      unsigned kk = 0;
      for (uint32_t g = blockIdx.x; g < P.n_groups; g += gridDim.x)
        for (uint32_t k = 0; k < supers; k++, kk++)
        {
          const int rb = kk % kRawStages;
          const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper), nv = group_nv (g);
          mbar_wait_guarded (raw_empty + rb, ((kk / kRawStages) & 1) ^ 1);
          mbar_expect_tx (raw_full + rb, kJ * nfr * 4u + (k == 0 ? kJ * kHist * 4u : 0u));
#pragma unroll 1
          for (int j = 0; j < kJ; j++)
          {
            const uint32_t c = chan (g, min ((uint32_t) j, nv - 1u));
            bulk_g2s (sRaw + (rb * kJ + j) * kRawRow, P.in + (size_t) c * P.frames + (size_t) k * kSuper, nfr * 4u, raw_full + rb);
            if (k == 0) bulk_g2s (sHist + (rb * kJ + j) * kHistRow, P.tail_in + (size_t) c * kHist, kHist * 4u, raw_full + rb);
          }
        }
      // Watchdog (sl_tc_common.cuh): in this kernel only the producer counts its failed polls (the counter in the MMA issuer's waits cost
      // 5 %: 466 vs 492 Gsamples/s, and so did one more commit of the MMA issuer to a completion barrier) — a deadlock reaches it
      // through the raw stages. After its last copy it goes on waiting for the stages as if it had more to load, which covers the
      // pipeline up to the MMAs of the CTA's third-last supertile (a stage is freed once its planes are written, and that needs the
      // MMAs two supertiles back). Only a barrier the producer follows phase by phase will do here: a late parity wait on a t_full
      // slot cannot tell phase n from phase n + 2 (compute-sanitizer's timing showed exactly that).
      for (unsigned i = kk; i < kk + kRawStages; i++) mbar_wait_guarded (raw_empty + i % kRawStages, ((i / kRawStages) & 1) ^ 1);
    }
    __syncwarp ();
  }
  else if (warp >= kEpiWarps && warp < kEpiWarps + kConvWarps)
  {
    // ========================================== converters: int16 I/Q frames -> byte planes (as sl_rx_ssb_tc.cu) ==========
    const int cw = warp - kEpiWarps, j = lane & 7, c4 = lane >> 3;
    unsigned kk = 0;
    for (uint32_t g = blockIdx.x; g < P.n_groups; g += gridDim.x)
    {
      const uint32_t nv = group_nv (g);
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
#pragma unroll
          for (int t = 0; t < 2; t++)
          {
            const int cc = c4 + 4 * t;
            const uint4 *src = reinterpret_cast<const uint4 *> (sHist + (rb * kJ + j) * kHistRow + cc * 32);
            const uint4 v0 = src[0], v1 = src[1];
            *reinterpret_cast<uint4 *> (Ahi + cc * kChunkBytes + j * 16) =
                make_uint4 (__byte_perm (v0.x, v0.y, 0x7531), __byte_perm (v0.z, v0.w, 0x7531), __byte_perm (v1.x, v1.y, 0x7531), __byte_perm (v1.z, v1.w, 0x7531));
            *reinterpret_cast<uint4 *> (Ahi + kPlaneBytes + cc * kChunkBytes + j * 16) =
                make_uint4 (__byte_perm (v0.x, v0.y, 0x6420), __byte_perm (v0.z, v0.w, 0x6420), __byte_perm (v1.x, v1.y, 0x6420), __byte_perm (v1.z, v1.w, 0x6420));
          }
        }
        if (cw == kConvWarps - 1 && k != 0)
        {
          // history = the last 8 chunks of the previous supertile's planes (always a full supertile)
          const unsigned char *prev = sA + (ab ^ 1) * 2 * kPlaneBytes + kChunksNew * kChunkBytes;
#pragma unroll
          for (int i = 0; i < 2 * kChunksHist * kJ / 32; i++)
          {
            const int e = lane + 32 * i, plane = e >> 6, o = (e & 63) * 16;
            *reinterpret_cast<uint4 *> (Ahi + plane * kPlaneBytes + o) = *reinterpret_cast<const uint4 *> (prev + plane * kPlaneBytes + o);
          }
        }
        {
          // new chunks: warp 0 takes the first half, warp 1 the second (the chunks it copies as history next time are its
          // own); a stream may end on any block (nfr = 48 b)
          const int nchunks = (int) nfr / 8, half = (nchunks / 2) & ~3;
          const int lo = cw == 0 ? 0 : half, hi = cw == 0 ? half : nchunks;
          const unsigned char *src0 = sRaw + (rb * kJ + j) * kRawRow;
          unsigned char *dst0 = Ahi + kChunksHist * kChunkBytes + j * 16;
#pragma unroll 3
          for (int cc = lo + c4; cc < hi; cc += 4)
          {
            const uint4 *src = reinterpret_cast<const uint4 *> (src0 + cc * 32);
            const uint4 v0 = src[0], v1 = src[1];
            *reinterpret_cast<uint4 *> (dst0 + cc * kChunkBytes) =
                make_uint4 (__byte_perm (v0.x, v0.y, 0x7531), __byte_perm (v0.z, v0.w, 0x7531), __byte_perm (v1.x, v1.y, 0x7531), __byte_perm (v1.z, v1.w, 0x7531));
            *reinterpret_cast<uint4 *> (dst0 + kPlaneBytes + cc * kChunkBytes) =
                make_uint4 (__byte_perm (v0.x, v0.y, 0x6420), __byte_perm (v0.z, v0.w, 0x6420), __byte_perm (v1.x, v1.y, 0x6420), __byte_perm (v1.z, v1.w, 0x6420));
          }
        }
        if (cw == 0 && k + 1 == supers)
        {
          // carry the raw tail of the stream for the next call: the last 64 frames of every valid channel. A stream shorter
          // than 64 frames (one block of 48) takes the rest from the tail it started with.
          for (int i = lane; i < kJ * (kHist / 4); i += 32)
          {
            const int jj = i >> 4, o = i & 15;                                   // 16 uint4 = 64 frames per channel
            if ((uint32_t) jj < nv)
            {
              const uint32_t c = chan (g, jj);
              const int f0 = (int) nfr - kHist + 4 * o;                            // first of the four frames, relative to the stage
              uint4 v;
              if (f0 >= 0) v = *reinterpret_cast<const uint4 *> (sRaw + (rb * kJ + jj) * kRawRow + f0 * 4);
              else if (k == 0) v = *reinterpret_cast<const uint4 *> (sHist + (rb * kJ + jj) * kHistRow + (kHist + f0) * 4);
              else v = *reinterpret_cast<const uint4 *> (P.in + (size_t) c * P.frames + (size_t) k * kSuper + f0);   // (nfr = 48 after full supertiles)
              reinterpret_cast<uint4 *> (P.tail_out + (size_t) c * kHist)[o] = v;
            }
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
    constexpr uint32_t id_ss = umma_idesc (kN, 1, 1), id_us = umma_idesc (kN, 0, 1);
    const uint32_t aBase = smem_u32 (sA), b0 = smem_u32 (sB) >> 4;
    constexpr uint64_t kDescA = ((uint64_t) (kChunkBytes >> 4) << 16) | ((uint64_t) ((6 * kChunkBytes) >> 4) << 32) | (1ull << 46);
    constexpr uint64_t kDescB = ((uint64_t) (128 >> 4) << 16) | ((uint64_t) (256 >> 4) << 32) | (1ull << 46);
    mbar_wait (b_full, 0);
    unsigned kk = 0;
    for (uint32_t g = blockIdx.x; g < P.n_groups; g += gridDim.x)
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        const int ab = kk & 1;
        mbar_wait (a_full + ab, (kk >> 1) & 1);
        mbar_wait (t_empty, (kk & 1) ^ 1);
        tc_fence_after ();
        const uint32_t aHi = (aBase + ab * 2 * kPlaneBytes) >> 4, aLo = aHi + (kPlaneBytes >> 4);
        if (elect_one ())
        {
#pragma unroll kMmaUnroll
          for (int ks = 0; ks < kKSteps; ks++)
          {
            const uint32_t ao = (uint32_t) (ks * 2 * kChunkBytes) >> 4, bo = (uint32_t) (ks * kBStepK<kKind>) >> 4;
            umma_i8 (tmem, kDescA | (aHi + ao), kDescB | (b0 + bo), id_ss, ks != 0);          // xh * [hhI|hlI|hhQ|hlQ] -> [0,N)
            umma_i8 (tmem + kN, kDescA | (aLo + ao), kDescB | (b0 + bo), id_us, ks != 0);     // xl * [...]             -> [N,2N)
          }
          umma_commit (t_full + (kk & 1));
          umma_commit (a_empty + ab);
        }
        __syncwarp ();
      }
  }
  else
  {
    // ========================================== epilogue (all integer) ==========================================
    const int es = warp >> 2, w = warp & 3, a = lane >> 3, j = lane & 7, q = 4 * w + a;
    int *myC = sPkC + es * (kQ * kJ);
    const int window = (int) P.window;
    unsigned kk = 0;
    for (uint32_t g = blockIdx.x; g < P.n_groups; g += gridDim.x)
    {
      const uint32_t nv = group_nv (g);
      const bool jvalid = (uint32_t) j < nv;
      const uint32_t c = chan (g, min ((uint32_t) j, nv - 1u));
      const bool sub = P.lsb[c] != 0;
      uint32_t fm_end = 0;                        // TX FM: the phase after this set's last supertile of the group
      for (uint32_t k = 0; k < supers; k++, kk++)
      {
        if ((int) (kk % kSets) != es) continue;
        const uint32_t nfr = min ((uint32_t) kSuper, P.frames - k * kSuper);
        const int nblk = (int) (nfr / kBlk);
        mbar_wait (t_full + (kk & 1), (kk >> 1) & 1);
        tc_fence_after ();
        // ---- accumulators -> the two FIR outputs (arm_fir_q15.c:642 + __SSAT), mix (arm_add_q15 / arm_sub_q15), |.| (arm_abs_q15);
        //      TX: the rail order, |.| of both rails
        int aud[kBlk];
        int pk = 0;
        const uint32_t taddr = tmem + ((uint32_t) (32 * w) << 16);
        // FM: z[-1] = the FIR outputs at frame -1 (rows 192 .. 195: rail I hh, hl, rail Q hh, hl) and its magnitude
        int pa = 0, pb = 0, pm = 0;
        if constexpr (kKind == kKindFm)
        {
          uint32_t h4[4], l4[4];
          tmem_ld4 (taddr + 192, h4); tmem_ld4 (taddr + kN + 192, l4);
          tmem_ld_wait ();
          pa = sat16 (2 * (int) h4[0] + ((256 * ((int) h4[1] + (int) l4[0]) + (int) l4[1]) >> 15));
          pb = sat16 (2 * (int) h4[2] + ((256 * ((int) h4[3] + (int) l4[2]) + (int) l4[3]) >> 15));
          pm = cmag_q15 (pa, pb);
        }
#pragma unroll
        for (int i = 0; i < kBlk / 8; i++)
        {
          uint32_t s2[8], s1a[8], s1b[8], s0[8];
          int fi[8];
          tmem_ld8 (taddr + 8 * i, s2); tmem_ld8 (taddr + 48 + 8 * i, s1a); tmem_ld8 (taddr + kN + 8 * i, s1b); tmem_ld8 (taddr + kN + 48 + 8 * i, s0);
          tmem_ld_wait ();
#pragma unroll
          for (int n = 0; n < 8; n++) fi[n] = sat16 (2 * (int) s2[n] + ((256 * ((int) s1a[n] + (int) s1b[n]) + (int) s0[n]) >> 15));
          if constexpr (kMono)
          {
            // TX AM / FM: a = rail I (rail Q holds the same FIR), |.| for the block peak (arm_abs_q15 + arm_max_q15)
#pragma unroll
            for (int n = 0; n < 8; n++) { aud[8 * i + n] = fi[n]; pk = max (pk, min (abs (fi[n]), 32767)); }
            continue;
          }
          tmem_ld8 (taddr + 96 + 8 * i, s2); tmem_ld8 (taddr + 144 + 8 * i, s1a); tmem_ld8 (taddr + kN + 96 + 8 * i, s1b); tmem_ld8 (taddr + kN + 144 + 8 * i, s0);
          tmem_ld_wait ();
#pragma unroll
          for (int n = 0; n < 8; n++)
          {
            const int fq = sat16 (2 * (int) s2[n] + ((256 * ((int) s1a[n] + (int) s1b[n]) + (int) s0[n]) >> 15));
            if constexpr (kKind == kKindAm)
            {
              // arm_cmplx_mag_q15 (2.14, >= 0: arm_abs_q15 leaves it as it is)
              const int v = cmag_q15 (fi[n], fq);
              aud[8 * i + n] = v;
              pk = max (pk, v);
            }
            else if constexpr (kKind == kKindFm)
            {
              const int m = cmag_q15 (fi[n], fq);
              const int v = fm_disc (pa, pb, pm, fi[n], fq, m, P.fm_floor);
              pa = fi[n]; pb = fq; pm = m;
              aud[8 * i + n] = v;
              pk = max (pk, min (abs (v), 32767));
            }
            else if constexpr (kTx)
            {
              // the rail order is the sideband: LSB / CW-R (I, Q) = (fi, fq), the others (fq, fi); the pair stays packed (I | Q << 16)
              const int vi = sub ? fi[n] : fq, vq = sub ? fq : fi[n];
              aud[8 * i + n] = (int) __byte_perm ((uint32_t) vi, (uint32_t) vq, 0x5410);
              pk = max (pk, max (min (abs (vi), 32767), min (abs (vq), 32767)));
            }
            else
            {
              const int v = sat16 (sub ? fi[n] - fq : fi[n] + fq);
              aud[8 * i + n] = v;
              pk = max (pk, min (abs (v), 32767));
            }
          }
        }
        tc_fence_before ();
        __syncwarp ();
        if (lane == 0) mbar_arrive (t_empty);
        // ---- block peaks: this supertile's into tile kk & 3; at a stream start the peaks before it (carried by age) into
        //      this set's carry tile, laid out like a previous supertile (block 16 - age)
        sPk[((kk & 3) * kQ + q) * kJ + j] = pk;
        // (loading it at the group's start instead costs one more live register in the epilogue: 430 vs 492 Gsamples/s)
        if (k == 0) myC[q * kJ + j] = (16 - q <= kWin - 1) ? (int) P.peaks_in[(size_t) c * kWin + (16 - q) - 1] : 0;
        __syncwarp ();
        // (TX FM arrives after its phase advance is published, below)
        if constexpr (kKind != kKindTxFm) { if (lane == 0) mbar_arrive (p_bar + (kk % kPSlots)); }
        // (every supertile but the CTA's first waits for its predecessor's peaks, also across groups where they are not used)
        if (kk != 0) mbar_wait (p_bar + ((kk - 1) % kPSlots), ((kk - 1) / kPSlots) & 1);
        named_bar (1 + es, 128);
        const int *own = sPk + (kk & 3) * kQ * kJ, *prev = (k == 0) ? myC : sPk + ((kk - 1) & 3) * kQ * kJ;
        // ---- envelope over the peak window (ours): max over ages 1 .. window-1 of (peak * rel[age]) >> 15
        int e = 0;
        for (int age = 1; age < window; age++)
        {
          const int bq = q - age;
          const int p = (bq >= 0) ? own[bq * kJ + j] : prev[(16 + bq) * kJ + j];
          e = max (e, (p * (int) P.rel[age]) >> 15);
        }
        // ---- gain (ours): q = min ((target << 15) / max (env, floor), gmax); scaleFract = q >> s with the smallest s that makes
        // it fit a q15; arm_scale_q15.c: __SSAT ((in * scaleFract) >> (15 - s), 16)
        const unsigned gq = min ((unsigned) (P.target << 15) / (unsigned) max (max (e, pk), P.floor_), P.gmax);
        const int sh = max (0, 17 - __clz (gq)), m = (int) (gq >> sh);
        uint32_t ph = 0;                                                          // TX FM: the phase before this thread's block
        if constexpr (kMono)
        {
          if (q < nblk && jvalid && P.audio_dbg)
          {
            // pre-ALC (a, 0) frames, int16 [C][T][2]
            uint4 *ad = reinterpret_cast<uint4 *> (P.audio_dbg + 2 * ((size_t) c * P.frames + ((size_t) k * kQ + q) * kBlk));
#pragma unroll
            for (int n = 0; n < kBlk; n += 4)
              ad[n / 4] = make_uint4 ((uint32_t) (uint16_t) aud[n], (uint32_t) (uint16_t) aud[n + 1], (uint32_t) (uint16_t) aud[n + 2], (uint32_t) (uint16_t) aud[n + 3]);
          }
          // y = arm_scale_q15 (a, q >> s, s)
#pragma unroll
          for (int n = 0; n < kBlk; n++) aud[n] = sat16 ((aud[n] * m) >> (15 - sh));
        }
        if constexpr (kKind == kKindTxFm)
        {
          // ---- the phase (ours, DESIGN.md §3.9): inc[n] = y[n] fm_inc (|.| < 2^31), phi[n] = phi[n-1] + inc[n] mod 2^32. A block's advance,
          //      an inclusive scan over the channel's 16 blocks (lanes j + 8 a of the set's four warps hold blocks 4 w + a), and the phase at
          //      the supertile's start: the state word at the group's first two supertiles, else this set's own end two supertiles back;
          //      plus the other set's advance over the supertile in between (published before its p_bar arrival, which this set has waited
          //      for). Blocks past the end of the stream advance nothing. The advance needs this supertile's gains, i.e. kk - 1's peaks, so
          //      this kind arrives for kk only after its wait for kk - 1: the p_bar sequence becomes a strict chain, and no slot can complete
          //      its next phase before every waiter has seen the current one (DESIGN.md §5A).
          uint32_t adv = 0;
          if (q < nblk)
#pragma unroll
            for (int n = 0; n < kBlk; n++) adv += (uint32_t) (aud[n] * P.fm_inc);
          uint32_t x = adv, t = __shfl_up_sync (0xffffffffu, x, 8);
          if (a >= 1) x += t;
          t = __shfl_up_sync (0xffffffffu, x, 16);
          if (a >= 2) x += t;
          if (a == 3) sScan[(es * 4 + w) * kJ + j] = x;
          named_bar (1 + es, 128);
          uint32_t tot = 0, before = x - adv;
#pragma unroll
          for (int w2 = 0; w2 < 4; w2++) { const uint32_t v = sScan[(es * 4 + w2) * kJ + j]; tot += v; if (w2 < w) before += v; }
          const uint32_t start = (k < 2 ? P.phase[c] : fm_end) + (k == 0 ? 0u : sTot[((kk - 1) & 3) * kJ + j]);
          fm_end = start + tot; ph = start + before;
          if (q == 0) sTot[(kk & 3) * kJ + j] = tot;
          __syncwarp ();
          if (lane == 0) mbar_arrive (p_bar + (kk % kPSlots));
        }
        if (q < nblk && jvalid)
        {
          const size_t blk = (size_t) k * kQ + q, t0 = blk * kBlk;
          if (P.gain_dbg) P.gain_dbg[(size_t) c * P.blocks + blk] = gq;
          if constexpr (kMono)
          {
            uint4 *dst = reinterpret_cast<uint4 *> (P.out + (size_t) c * P.frames + t0);
#pragma unroll
            for (int n = 0; n < kBlk; n += 8)
            {
              uint32_t o[8];
#pragma unroll
              for (int u = 0; u < 8; u++)
              {
                if constexpr (kKind == kKindTxAm)
                  // I = arm_add_q15 (arm_scale_q15 (y, am_carrier, 0), am_carrier), Q = 0
                  o[u] = (uint32_t) (uint16_t) sat16 (sat16 ((aud[n + u] * P.am_carrier) >> 15) + P.am_carrier);
                else
                {
                  ph += (uint32_t) (aud[n + u] * P.fm_inc);
                  o[u] = fm_nco (ph, sSin, P.fm_level15);
                }
              }
              asm volatile ("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst + n / 4),
                            "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
            }
          }
          else if constexpr (kTx)
          {
            if (P.audio_dbg)
            {
              // pre-ALC (I, Q) frames, int16 [C][T][2]
              uint4 *ad = reinterpret_cast<uint4 *> (P.audio_dbg + 2 * ((size_t) c * P.frames + t0));
#pragma unroll
              for (int n = 0; n < kBlk; n += 4) ad[n / 4] = make_uint4 ((uint32_t) aud[n], (uint32_t) aud[n + 1], (uint32_t) aud[n + 2], (uint32_t) aud[n + 3]);
            }
            uint4 *dst = reinterpret_cast<uint4 *> (P.out + (size_t) c * P.frames + t0);
            // arm_scale_q15 on each rail with the same gain word: I from the low half, Q (arithmetic shift) from the high half. Its __SSAT
            // is left out because it cannot fire here: the envelope is never below the block's peak over both rails and q rounds down,
            // so |y| <= target for |v| <= 32767, and v = -32768 (peak 32767) meets q <= 32768 and gives y >= -32768 (DESIGN.md §3.7).
            // Bit-identical to the saturating form; 316 vs 254 Gsamples/s at 1024 channels (the per-sample store arithmetic bounds TX).
#define SL_Q15_TXOUT(n) __byte_perm ((uint32_t) ((((int) (int16_t) aud[n]) * m) >> (15 - sh)), (uint32_t) (((aud[n] >> 16) * m) >> (15 - sh)), 0x5410)
#pragma unroll
            for (int n = 0; n < kBlk; n += 8)
              asm volatile ("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst + n / 4),
                            "r"(SL_Q15_TXOUT (n)), "r"(SL_Q15_TXOUT (n + 1)), "r"(SL_Q15_TXOUT (n + 2)), "r"(SL_Q15_TXOUT (n + 3)),
                            "r"(SL_Q15_TXOUT (n + 4)), "r"(SL_Q15_TXOUT (n + 5)), "r"(SL_Q15_TXOUT (n + 6)), "r"(SL_Q15_TXOUT (n + 7)) : "memory");
#undef SL_Q15_TXOUT
          }
          else
          {
            if (P.audio_dbg)
            {
              uint4 *ad = reinterpret_cast<uint4 *> (P.audio_dbg + (size_t) c * P.frames + t0);
#pragma unroll
              for (int n = 0; n < kBlk; n += 8)
                ad[n / 8] = make_uint4 ((uint32_t) (uint16_t) aud[n] | ((uint32_t) (uint16_t) aud[n + 1] << 16), (uint32_t) (uint16_t) aud[n + 2] | ((uint32_t) (uint16_t) aud[n + 3] << 16),
                                        (uint32_t) (uint16_t) aud[n + 4] | ((uint32_t) (uint16_t) aud[n + 5] << 16), (uint32_t) (uint16_t) aud[n + 6] | ((uint32_t) (uint16_t) aud[n + 7] << 16));
            }
            uint4 *dst = reinterpret_cast<uint4 *> (P.out + (size_t) c * P.frames + t0);
#define SL_Q15_OUT(n) __byte_perm ((uint32_t) sat16 ((aud[n] * m) >> (15 - sh)), 0u, 0x1010)
#pragma unroll
            for (int n = 0; n < kBlk; n += 8)
              asm volatile ("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst + n / 4),
                            "r"(SL_Q15_OUT (n)), "r"(SL_Q15_OUT (n + 1)), "r"(SL_Q15_OUT (n + 2)), "r"(SL_Q15_OUT (n + 3)),
                            "r"(SL_Q15_OUT (n + 4)), "r"(SL_Q15_OUT (n + 5)), "r"(SL_Q15_OUT (n + 6)), "r"(SL_Q15_OUT (n + 7)) : "memory");
#undef SL_Q15_OUT
          }
        }
        if (k + 1 == supers && jvalid)
        {
          // ---- the end of the call: the peak window by age (age a = the block a before the end); this thread takes ages q + 1
          //      and q + 17. Blocks of this call come from the last tiles, older ones from the window the call started with.
          const int blocks = (int) P.blocks;
#pragma unroll
          for (int h = 0; h < 2; h++)
          {
            const int age = q + 1 + 16 * h;
            if (age <= kWin - 1)
            {
              const int bi = blocks - age;
              int v;
              if (bi >= 0)
              {
                const unsigned tk = kk - (k - (unsigned) (bi / 16));                // running index of the supertile that holds block bi
                v = sPk[((tk & 3) * kQ + (bi & 15)) * kJ + j];
              }
              else v = (age - blocks <= kWin - 1) ? (int) P.peaks_in[(size_t) c * kWin + (age - blocks) - 1] : 0;
              P.peaks_out[(size_t) c * kWin + age - 1] = (int16_t) v;
            }
          }
        }
        // The window above may reach back to tile kk - 2 (a short last supertile), which this set's NEXT supertile kk + 2 overwrites
        // — a warp that is through here could be there before a slower one has read it (inside a group only tiles kk and kk - 1
        // are read, and kk + 2 cannot touch those). Found under compute-sanitizer's timing; one barrier per group closes it.
        if (k + 1 == supers) named_bar (1 + es, 128);
        // TX FM: the phase after the group goes back to the state word only here, after the barrier above. Its readers are the group's
        // first two supertiles: this set's warps read it before they reached that barrier, and the other set's warps read it before
        // their p_bar arrival for that supertile, which the strict p_bar chain puts before this set's last wait (DESIGN.md §5A).
        if constexpr (kKind == kKindTxFm)
          if (k + 1 == supers && jvalid && q == 0) P.phase[c] = fm_end;
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

// taps -> B operand: rows [rail I: hh (48) | hl (48) | rail Q: hh | hl], K byte m = 32 ks + kk = frame m / 2 of the 112-frame
// window (64 before the block), rail m & 1; output n of the block meets tap d = 64 + n - frame. false when a tap does not
// split into two signed bytes (|tap| >= 32640). tx: both rails filter the mic, so both place their taps at the L bytes (m = 2 frame)
// and the R bytes get zero weight. fm (RX-Q15's FM planes, N = 208): the same 192 rows, then the outputs at frame n = -1 in rows
// 192 + 2 rail + digit and 12 zero rows; so every section a thread reads starts on an 8-column boundary, as in the 192-row planes.
static int q15_row (int rail, int digit, int n) { return n >= 0 ? rail * 96 + digit * 48 + n : 192 + 2 * rail + digit; }
static size_t q15_plane_at (int rows, int m, int row)
{
  const int ks = m / 32, kk = m % 32;
  return (size_t) ks * (rows / 8 * 256) + (row / 8) * 256 + (kk / 16) * 128 + (row % 8) * 16 + (kk % 16);
}
static bool build_planes (const int16_t *taps_i, const int16_t *taps_q, uint8_t *planes, bool tx, bool fm)
{
  const int rows = fm ? 208 : 192;
  std::memset (planes, 0, (size_t) kKSteps * rows / 8 * 256);
  for (int rail = 0; rail < 2; rail++)
    for (int n = fm ? -1 : 0; n < 48; n++)
      for (int f = 0; f < 112; f++)
      {
        const int d = 64 + n - f;
        if (d < 0 || d >= kTaps) continue;
        const int h = rail ? taps_q[d] : taps_i[d];
        const int hl = ((h + 128) & 255) - 128, hh = (h - hl) >> 8;
        if (hh < -128 || hh > 127) return false;
        const int m = 2 * f + (tx ? 0 : rail);
        const int dg[2] = { hh, hl };
        for (int g = 0; g < 2; g++) planes[q15_plane_at (rows, m, q15_row (rail, g, n))] = (uint8_t) (int8_t) dg[g];
      }
  return true;
}
bool q15_tc_build_planes (const int16_t *taps_i, const int16_t *taps_q, uint8_t *planes, bool tx) { return build_planes (taps_i, taps_q, planes, tx, false); }
bool q15_tc_build_fm_planes (const int16_t *taps, uint8_t *planes) { return build_planes (taps, taps, planes, false, true); }

// host-side evaluation of the planes on one raw window (design check, tests/test_tc_math.py): the integer contraction the
// kernel runs and its reconstruction of arm_fir_q15's result, outputs n = n0 .. 47 of rail I, then of rail Q
static void apply_planes (const uint8_t *planes, int rows, int n0, const int16_t *window, int32_t *out)
{
  const int per = 48 - n0;
  for (int rail = 0; rail < 2; rail++)
    for (int n = n0; n < 48; n++)
    {
      long long s2 = 0, s1 = 0, s0 = 0;
      const int r_hh = q15_row (rail, 0, n), r_hl = q15_row (rail, 1, n);
      for (int m = 0; m < 224; m++)
      {
        const int x = window[m], xl = x & 255, xh = (x - xl) >> 8;
        const int hh = (int8_t) planes[q15_plane_at (rows, m, r_hh)], hl = (int8_t) planes[q15_plane_at (rows, m, r_hl)];
        s2 += xh * hh; s1 += xh * hl + xl * hh; s0 += xl * hl;
      }
      const long long v = 2 * s2 + ((256 * s1 + s0) >> 15);
      out[rail * per + n - n0] = (int32_t) (v > 32767 ? 32767 : (v < -32768 ? -32768 : v));
    }
}
// out[0..47] = rail I, out[48..95] = rail Q. The same for TX planes: the contraction runs over all 224 bytes of the window as the
// kernel's does, and the R bytes meet zero weight there
void q15_tc_apply_planes (const uint8_t *planes, const int16_t *window /* [112][2] */, int32_t *out96) { apply_planes (planes, 192, 0, window, out96); }
// FM planes: out[0..48] = rail I at n = -1 .. 47, out[49..97] = rail Q
void q15_tc_apply_fm_planes (const uint8_t *planes, const int16_t *window /* [112][2] */, int32_t *out98) { apply_planes (planes, 208, -1, window, out98); }

int launch_rx_q15_tc (const RxQ15TcLaunch &L, int sm_count, void *stream)
{
  KParams P{};
  P.in = reinterpret_cast<const uint32_t *> (L.in); P.out = reinterpret_cast<uint32_t *> (L.out);
  P.tail_in = L.tail_in; P.tail_out = L.tail_out; P.peaks_in = L.peaks_in; P.peaks_out = L.peaks_out;
  P.planes = L.planes; P.lsb = L.lsb; P.audio_dbg = L.audio_dbg; P.gain_dbg = L.gain_dbg;
  std::memcpy (P.rel, L.rel, sizeof P.rel);
  P.channels = L.channels; P.frames = L.frames; P.blocks = L.frames / kBlk; P.supers = (L.frames + kSuper - 1) / kSuper;
  P.gsz = (uint32_t) std::min<uint64_t> (kJ, std::max<uint64_t> (1, ((uint64_t) L.channels + (uint64_t) sm_count - 1) / (uint64_t) sm_count));
  P.n_groups = (L.channels + P.gsz - 1) / P.gsz;
  P.window = L.window; P.target = L.target; P.floor_ = L.floor_; P.gmax = L.gmax;
  P.list = L.list; P.fm_floor = L.fm_floor;
  P.phase = L.phase; P.sin513 = L.sin513; P.am_carrier = L.am_carrier; P.fm_inc = L.fm_inc; P.fm_level15 = L.fm_level * 32768.0f;
  void (*kernel) (KParams) = nullptr; size_t smem_bytes = Smem::bytes;
  switch (L.kind)
  {
    case kQ15Ssb: kernel = L.list ? rx_q15_tc_kernel<kKindRxList> : rx_q15_tc_kernel<kKindRx>; break;
    case kQ15Tx: kernel = L.list ? rx_q15_tc_kernel<kKindTxList> : rx_q15_tc_kernel<kKindTx>; break;
    case kQ15TxAm: kernel = rx_q15_tc_kernel<kKindTxAm>; break;
    case kQ15TxFm: kernel = rx_q15_tc_kernel<kKindTxFm>; smem_bytes = SmemK<kKindTxFm>::bytes; break;
    case kQ15Am: kernel = rx_q15_tc_kernel<kKindAm>; break;
    case kQ15Fm: kernel = rx_q15_tc_kernel<kKindFm>; smem_bytes = SmemT<kTcQ15FmPlaneBytes>::bytes; break;
    default: return (int) cudaErrorInvalidValue;
  }
  if (L.kind >= kQ15Am && !L.list) return (int) cudaErrorInvalidValue;
  cudaError_t e = cudaFuncSetAttribute (kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem_bytes);
  if (e != cudaSuccess) return (int) e;
  uint32_t grid = (uint32_t) sm_count;
  if (grid > P.n_groups) grid = P.n_groups;
  if (const char *gs = std::getenv ("SELENITE_B200_TC_GRID")) { const long v = std::atol (gs); if (v > 0 && (uint32_t) v <= grid) grid = (uint32_t) v; }
  kernel<<<grid, kThreads, smem_bytes, (cudaStream_t) stream>>> (P);
  return (int) cudaGetLastError ();
}

}  // namespace sl
