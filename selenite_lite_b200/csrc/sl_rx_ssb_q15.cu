// RX-SSB-q15: the all-integer receive chain (phasing-method SSB demodulator), one fused kernel, bit-exact against the
// reference's q15 routines; every sample crosses HBM once (4 B in, 4 B out).
//
//   int16 I/Q --de-interleave--> fir_q15(I, hI), fir_q15(Q, hQ) --add/sub (saturating)--> per-48-frame AGC --> int16 L=R
//   oracle stage per box (reference = /root/reference/Drivers/CMSIS/DSP/Source/...):
//     FIR     FilteringFunctions/arm_fir_q15.c:591 (64 taps; q63 accumulator, >> 15, __SSAT 16)
//     mix     BasicMathFunctions/arm_add_q15.c:54 / arm_sub_q15.c:54 (saturating)
//     AGC     BasicMathFunctions/arm_abs_q15.c:57, StatisticsFunctions/arm_max_q15.c:58, arm_scale_q15.c:56 (+ our gain law)
//   The COMPOSITION and the gain law are ours (SURVEY.md §0 / Appendix B); the arithmetic of each box is the reference's.
//
// Why tensor cores here and nowhere else: a 64-tap FIR is 128 integer MACs per complex sample for the two rails, which on
// the CUDA cores (IMAD, half rate) caps the chain near 18 % of the HBM roof. The FIR of a block of 16 outputs is a dense
// contraction with a 16 x 80 Toeplitz matrix of taps (81 % non-zero), and it is EXACT on the integer tensor-core path:
// samples and taps are split into a signed high byte and an unsigned low byte, x h = 65536 xh hh + 256 (xh hl + xl hh) +
// xl hl, each partial sum of <= 64 byte products fits an int32 accumulator with 9 bits to spare, and
//   (acc >> 15) = 2 S2 + ((256 S1 + S0) >> 15)      (S2 = sum xh hh, S1 = sum xh hl + xl hh, S0 = sum xl hl)
// reproduces arm_fir_q15's 64-bit accumulator bit for bit. mma.sync.m16n8k32 (SASS IMMA.16832) measured at 0.48 per clock
// per SM (tools/microbench/imma_rate.cu) keeps this stage below the HBM time of the samples it consumes.
//
// Structure. A warp owns 8 channels (the MMA's N dimension) and walks a segment of their streams in time; A fragments =
// the Toeplitz taps, constant in registers; B fragments = byte planes of 4 consecutive frames of the lane's channel,
// kept as a sliding window in registers (one 16-byte shared-memory load + 8 PRMT per 16 frames); raw frames are staged
// by bulk asynchronous copies (TMA engine) into a per-warp double buffer, one chunk of 96 frames ahead.
// The AGC law has FINITE memory (a window of block peaks with a release table), so segments of one channel are
// independent given the input: a segment that does not start at the stream start first re-derives the peaks of the
// window-1 blocks before it (FIR only, nothing stored). No cross-CTA hand-over exists in this kernel.
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "sl_internal.h"

namespace sl {

namespace {

constexpr int kTaps = SLB_Q15_TAPS;              // 64
constexpr int kWin = SLB_Q15_WIN;                // peak ring length (>= agc_window)
constexpr int kBlk = 48;                         // AGC block = firmware block at 48 kHz = 3 MMA blocks of 16 frames
constexpr int kChunkBlocks = 2;                  // AGC blocks per staged chunk
constexpr int kChunk = kChunkBlocks * kBlk;      // 96 frames
constexpr int kRowWords = kTaps + kChunk + 16;   // words per channel row of a raw stage: 64 history + 96 new + 16 pad;
                                                 // 704 B = 64 mod 128, so the 16-byte loads of lanes (ch, tig), (ch+1, tig)
                                                 // fall into different bank halves
constexpr int kWarps = 4;
constexpr int kThreads = 32 * kWarps;
constexpr int kStageWords = 8 * kRowWords;
constexpr size_t kWarpSmem = 2 * kStageWords * 4 + 8 * kWin * 2 + 16;   // two raw stages + peak ring + two mbarriers
constexpr size_t kSmemBytes = kWarps * kWarpSmem;

struct KParams
{
  const uint32_t *in; uint32_t *out;            // [C][frames] u32 = (I, Q) in, (L, R) out
  const uint32_t *tail_in; uint32_t *tail_out;  // [C][64] last raw frames of the previous call (ping-pong)
  const int16_t *peaks_in; int16_t *peaks_out;  // [C][kWin] block peaks by age at the call boundary (ping-pong)
  const uint32_t *afrag;                        // [rail][plane][10][32] Toeplitz tap fragments
  const uint8_t *lsb;                           // [C] 0: I' + Q', 1: I' - Q'
  int16_t *audio_dbg; uint32_t *gain_dbg;       // optional [C][frames], [C][frames / 48]
  int16_t rel[kWin];
  uint32_t channels, frames, blocks, groups, seg_blocks, segs, window;
  int32_t target, floor_; uint32_t gmax;
};

// output stores that do not allocate in L1 (every lane of a fragment store hits its own line)
__device__ __forceinline__ void st_na_u32 (uint32_t *p, uint32_t v)
{
  asm volatile ("st.global.L1::no_allocate.b32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t smem_u32 (const void *p) { return (uint32_t) __cvta_generic_to_shared (p); }
__device__ __forceinline__ void mbar_init (uint64_t *bar, unsigned count)
{
  asm volatile ("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32 (bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx (uint64_t *bar, unsigned bytes)
{
  asm volatile ("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32 (bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait (uint64_t *bar, unsigned parity)
{
  asm volatile (
      "{\n .reg .pred p;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}\n"
      ::"r"(smem_u32 (bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s (void *dst, const void *src, unsigned bytes, uint64_t *bar)
{
  asm volatile ("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                ::"r"(smem_u32 (dst)), "l"(src), "r"(bytes), "r"(smem_u32 (bar)) : "memory");
}

// D (16 x 8, s32) += A (16 x 32, taps) * B (32 x 8, samples); TA / TB = s8 or u8. SASS IMMA.16832
#define SL_IMMA32(TA, TB, d, a, b)                                                                                          \
  asm volatile ("mma.sync.aligned.m16n8k32.row.col.s32." TA "." TB ".s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};" \
                : "+r"((d)[0]), "+r"((d)[1]), "+r"((d)[2]), "+r"((d)[3])                                                    \
                : "r"((a)[0]), "r"((a)[1]), "r"((a)[2]), "r"((a)[3]), "r"((b)[0]), "r"((b)[1]))
#define SL_IMMA16(TA, TB, d, a, b)                                                                                          \
  asm volatile ("mma.sync.aligned.m16n8k16.row.col.s32." TA "." TB ".s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"      \
                : "+r"((d)[0]), "+r"((d)[1]), "+r"((d)[2]), "+r"((d)[3])                                                    \
                : "r"((a)[0]), "r"((a)[1]), "r"((b)[0]))

__device__ __forceinline__ int sat16 (int v) { return max (-32768, min (32767, v)); }

// four consecutive frames (u32 = I lo, I hi, Q lo, Q hi bytes) -> the four byte planes, frame 0 in the low byte
__device__ __forceinline__ void planes_of (const uint4 w, uint32_t &ilo, uint32_t &ihi, uint32_t &qlo, uint32_t &qhi)
{
  const uint32_t t0 = __byte_perm (w.x, w.y, 0x5140), t1 = __byte_perm (w.z, w.w, 0x5140);   // (a.b0, b.b0, a.b1, b.b1)
  const uint32_t t2 = __byte_perm (w.x, w.y, 0x7362), t3 = __byte_perm (w.z, w.w, 0x7362);   // (a.b2, b.b2, a.b3, b.b3)
  ilo = __byte_perm (t0, t1, 0x5410); ihi = __byte_perm (t0, t1, 0x7632);
  qlo = __byte_perm (t2, t3, 0x5410); qhi = __byte_perm (t2, t3, 0x7632);
}

__global__ void __launch_bounds__ (kThreads, 4) rx_ssb_q15_kernel (const __grid_constant__ KParams P)
{
  extern __shared__ __align__ (128) unsigned char smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, tig = lane & 3;       // MMA coordinates: g = B column (input channel) and D row; tig = D column pair
  unsigned char *ws = smem + (size_t) warp * kWarpSmem;
  uint32_t *sRaw = reinterpret_cast<uint32_t *> (ws);
  int16_t *sPeak = reinterpret_cast<int16_t *> (ws + 2 * kStageWords * 4);      // [8][kWin], indexed by absolute block & 31
  uint64_t *sBar = reinterpret_cast<uint64_t *> (ws + 2 * kStageWords * 4 + 8 * kWin * 2);
  if (lane == 0) { mbar_init (sBar, 1); mbar_init (sBar + 1, 1); asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  __syncwarp ();

  // Toeplitz tap fragments: [rail I|Q][plane hi|lo][k-step 0 (4 regs), k-step 1 (4 regs), k-step 2 (k = 16: 2 regs)]
  uint32_t aI_h[10], aI_l[10], aQ_h[10], aQ_l[10];
#pragma unroll
  for (int i = 0; i < 10; i++)
  {
    aI_h[i] = P.afrag[(0 * 10 + i) * 32 + lane]; aI_l[i] = P.afrag[(1 * 10 + i) * 32 + lane];
    aQ_h[i] = P.afrag[(2 * 10 + i) * 32 + lane]; aQ_l[i] = P.afrag[(3 * 10 + i) * 32 + lane];
  }
  const int window = (int) P.window;
  unsigned use[2] = { 0u, 0u };                   // how often each raw stage has been filled (mbarrier phase)

  const unsigned total_items = P.groups * P.segs;
  for (unsigned item = blockIdx.x * kWarps + warp; item < total_items; item += gridDim.x * kWarps)
  {
    const uint32_t grp = item % P.groups, seg = item / P.groups;
    const uint32_t ch_in = grp * 8 + g;                                          // channel whose frames this lane unpacks
    const uint32_t ch_o0 = grp * 8 + 2 * tig, ch_o1 = ch_o0 + 1;                 // channels whose outputs this lane holds
    const bool ok0 = ch_o0 < P.channels, ok1 = ch_o1 < P.channels;
    const uint32_t b_emit = seg * P.seg_blocks;                                  // first block this item writes
    const uint32_t b_end = min (P.blocks, b_emit + P.seg_blocks);
    // blocks re-derived (not stored) so that the peak window of block b_emit is complete; whole chunks only. The segment that ends
    // the call reaches back kWin - 1 blocks whatever the window: it carries every age to the next call, whose window may be longer
    const uint32_t reach = (b_end == P.blocks) ? (uint32_t) (kWin - 1) : (uint32_t) (window - 1);
    uint32_t b_first = (b_emit >= reach) ? b_emit - reach : 0u;
    b_first -= b_first % kChunkBlocks;
    const bool sub0 = ok0 && P.lsb[ch_o0], sub1 = ok1 && P.lsb[ch_o1];

    // peaks of blocks before the call come from the carried state (age-indexed) when the window reaches back that far
    if (b_first == 0)
      for (int i = lane; i < 8 * (kWin - 1); i += 32)
      {
        const int c = i / (kWin - 1), age = i % (kWin - 1) + 1;                  // block index -age
        const uint32_t ch = grp * 8 + c;
        sPeak[c * kWin + ((0 - age) & (kWin - 1))] = (ch < P.channels) ? P.peaks_in[(size_t) ch * kWin + age - 1] : (int16_t) 0;
      }

    // ---- staging: chunk q covers blocks [b_first + 2 q, +2); row = 64 frames of history + 96 new frames
    const uint32_t n_chunks = (b_end - b_first + kChunkBlocks - 1) / kChunkBlocks;
    auto issue = [&] (uint32_t q, int stage) {
      const uint32_t t = (b_first + q * kChunkBlocks) * kBlk;                    // first new frame of the chunk
      const uint32_t new_frames = min ((uint32_t) kChunk, P.frames - t);
      uint32_t *dst = sRaw + stage * kStageWords + g * kRowWords;                // lanes with tig == 0 copy channel g
      const uint32_t nch = min (8u, P.channels - grp * 8);
      if (lane == 0) mbar_expect_tx (sBar + stage, nch * (kTaps + new_frames) * 4u);
      __syncwarp ();
      if (tig == 0 && ch_in < P.channels)
      {
        const uint32_t *src = P.in + (size_t) ch_in * P.frames;
        if (t == 0)
        {
          bulk_g2s (dst, P.tail_in + (size_t) ch_in * kTaps, kTaps * 4u, sBar + stage);
          bulk_g2s (dst + kTaps, src, new_frames * 4u, sBar + stage);
        }
        else
          bulk_g2s (dst, src + t - kTaps, (kTaps + new_frames) * 4u, sBar + stage);
      }
    };
    issue (0, 0);
    if (n_chunks > 1) issue (1, 1);

    uint32_t wIl[5], wIh[5], wQl[5], wQh[5];       // sliding window of byte planes: group j = frames 16 j + 4 tig .. + 3 of the 80
    int aud0[6], aud1[6];                          // audio of one AGC block for channels ch_o0 / ch_o1: rows g, g + 8 of 3 MMA blocks

    for (uint32_t q = 0; q < n_chunks; q++)
    {
      const int stage = q & 1;
      mbar_wait (sBar + stage, use[stage] & 1); use[stage]++;
      const uint32_t *row = sRaw + stage * kStageWords + g * kRowWords + 4 * tig;
      if (q == 0)
      {
        // window groups 0..3 = the 64 frames of history before the first block
#pragma unroll
        for (int j = 0; j < 4; j++) planes_of (*reinterpret_cast<const uint4 *> (row + 16 * j), wIl[j], wIh[j], wQl[j], wQh[j]);
      }
      const uint32_t blocks_here = min ((uint32_t) kChunkBlocks, b_end - (b_first + q * kChunkBlocks));
      for (uint32_t bb = 0; bb < blocks_here; bb++)
      {
        const uint32_t b = b_first + q * kChunkBlocks + bb;                      // absolute block index in this call
        int pk0 = 0, pk1 = 0;
#pragma unroll
        for (int mb = 0; mb < 3; mb++)
        {
          // ---- new group of the window: the block's own 16 frames
          planes_of (*reinterpret_cast<const uint4 *> (row + kTaps + (bb * 3 + mb) * 16), wIl[4], wIh[4], wQl[4], wQh[4]);
          // ---- the two FIRs of 16 frames x 8 channels: out[m] = sum_t h[t] x[n0 + m - t], k <-> frame n0 - 64 + k
          int s2i[4] = { 0, 0, 0, 0 }, s1i[4] = { 0, 0, 0, 0 }, s0i[4] = { 0, 0, 0, 0 };
          int s2q[4] = { 0, 0, 0, 0 }, s1q[4] = { 0, 0, 0, 0 }, s0q[4] = { 0, 0, 0, 0 };
#pragma unroll
          for (int ks = 0; ks < 2; ks++)
          {
            const uint32_t bIh[2] = { wIh[2 * ks], wIh[2 * ks + 1] }, bIl[2] = { wIl[2 * ks], wIl[2 * ks + 1] };
            const uint32_t bQh[2] = { wQh[2 * ks], wQh[2 * ks + 1] }, bQl[2] = { wQl[2 * ks], wQl[2 * ks + 1] };
            SL_IMMA32 ("s8", "s8", s2i, aI_h + 4 * ks, bIh); SL_IMMA32 ("s8", "u8", s1i, aI_h + 4 * ks, bIl);
            SL_IMMA32 ("u8", "s8", s1i, aI_l + 4 * ks, bIh); SL_IMMA32 ("u8", "u8", s0i, aI_l + 4 * ks, bIl);
            SL_IMMA32 ("s8", "s8", s2q, aQ_h + 4 * ks, bQh); SL_IMMA32 ("s8", "u8", s1q, aQ_h + 4 * ks, bQl);
            SL_IMMA32 ("u8", "s8", s1q, aQ_l + 4 * ks, bQh); SL_IMMA32 ("u8", "u8", s0q, aQ_l + 4 * ks, bQl);
          }
          {
            const uint32_t bIh[1] = { wIh[4] }, bIl[1] = { wIl[4] }, bQh[1] = { wQh[4] }, bQl[1] = { wQl[4] };
            SL_IMMA16 ("s8", "s8", s2i, aI_h + 8, bIh); SL_IMMA16 ("s8", "u8", s1i, aI_h + 8, bIl);
            SL_IMMA16 ("u8", "s8", s1i, aI_l + 8, bIh); SL_IMMA16 ("u8", "u8", s0i, aI_l + 8, bIl);
            SL_IMMA16 ("s8", "s8", s2q, aQ_h + 8, bQh); SL_IMMA16 ("s8", "u8", s1q, aQ_h + 8, bQl);
            SL_IMMA16 ("u8", "s8", s1q, aQ_l + 8, bQh); SL_IMMA16 ("u8", "u8", s0q, aQ_l + 8, bQl);
          }
          // ---- slide the window by 16 frames
#pragma unroll
          for (int j = 0; j < 4; j++) { wIl[j] = wIl[j + 1]; wIh[j] = wIh[j + 1]; wQl[j] = wQl[j + 1]; wQh[j] = wQh[j + 1]; }
          // ---- arm_fir_q15.c: (q15_t) __SSAT (acc >> 15, 16); arm_add_q15 / arm_sub_q15: __SSAT (a +- b, 16); arm_abs_q15
          // D element e: row g + 8 (e >> 1), column 2 tig + (e & 1)
#pragma unroll
          for (int e = 0; e < 4; e++)
          {
            const int fi = sat16 (2 * s2i[e] + ((256 * s1i[e] + s0i[e]) >> 15));
            const int fq = sat16 (2 * s2q[e] + ((256 * s1q[e] + s0q[e]) >> 15));
            const bool sub = (e & 1) ? sub1 : sub0;
            const int a = sat16 (sub ? fi - fq : fi + fq);
            const int ab = min (abs (a), 32767);
            if (e & 1) { aud1[2 * mb + (e >> 1)] = a; pk1 = max (pk1, ab); }
            else { aud0[2 * mb + (e >> 1)] = a; pk0 = max (pk0, ab); }
          }
        }
        // ---- block peak per channel (arm_max_q15 over the 48 frames): reduce over the 8 lanes that share tig
#pragma unroll
        for (int d = 4; d < 32; d <<= 1)
        {
          pk0 = max (pk0, __shfl_xor_sync (0xffffffffu, pk0, d));
          pk1 = max (pk1, __shfl_xor_sync (0xffffffffu, pk1, d));
        }
        // ---- envelope over the peak window: lane g takes ages g + 1, g + 9, ... of its two channels
        int e0 = 0, e1 = 0;
        for (int age = g + 1; age < window; age += 8)
        {
          const int slot = ((int) b - age) & (kWin - 1), r = P.rel[age];
          e0 = max (e0, ((int) sPeak[(2 * tig) * kWin + slot] * r) >> 15);
          e1 = max (e1, ((int) sPeak[(2 * tig + 1) * kWin + slot] * r) >> 15);
        }
#pragma unroll
        for (int d = 4; d < 32; d <<= 1)
        {
          e0 = max (e0, __shfl_xor_sync (0xffffffffu, e0, d));
          e1 = max (e1, __shfl_xor_sync (0xffffffffu, e1, d));
        }
        __syncwarp ();                                                            // every lane has read the ring
        if (g == 0) { sPeak[(2 * tig) * kWin + (b & (kWin - 1))] = (int16_t) pk0; sPeak[(2 * tig + 1) * kWin + (b & (kWin - 1))] = (int16_t) pk1; }
        __syncwarp ();
        if (b >= b_emit)
        {
          // ---- gain (ours): q = min ((target << 15) / max (env, floor), gmax); scaleFract = q >> s with the smallest s
          // that makes it fit a q15; arm_scale_q15.c: __SSAT ((in * scaleFract) >> (15 - s), 16)
          const unsigned q0 = min ((unsigned) (P.target << 15) / (unsigned) max (max (e0, pk0), P.floor_), P.gmax);
          const unsigned q1 = min ((unsigned) (P.target << 15) / (unsigned) max (max (e1, pk1), P.floor_), P.gmax);
          const int sh0 = max (0, 17 - __clz (q0)), sh1 = max (0, 17 - __clz (q1));
          const int m0 = (int) (q0 >> sh0), m1 = (int) (q1 >> sh1);
          const size_t t0 = (size_t) b * kBlk;
          if (P.gain_dbg && g == 0)
          {
            if (ok0) P.gain_dbg[(size_t) ch_o0 * P.blocks + b] = q0;
            if (ok1) P.gain_dbg[(size_t) ch_o1 * P.blocks + b] = q1;
          }
#pragma unroll
          for (int i = 0; i < 6; i++)
          {
            const size_t t = t0 + (i >> 1) * 16 + (i & 1) * 8 + g;               // MMA block i >> 1, row g + 8 (i & 1)
            const int y0 = sat16 ((aud0[i] * m0) >> (15 - sh0)), y1 = sat16 ((aud1[i] * m1) >> (15 - sh1));
            if (ok0) st_na_u32 (P.out + (size_t) ch_o0 * P.frames + t, __byte_perm ((uint32_t) y0, 0u, 0x1010));   // L = R
            if (ok1) st_na_u32 (P.out + (size_t) ch_o1 * P.frames + t, __byte_perm ((uint32_t) y1, 0u, 0x1010));
            if (P.audio_dbg)
            {
              if (ok0) P.audio_dbg[(size_t) ch_o0 * P.frames + t] = (int16_t) aud0[i];
              if (ok1) P.audio_dbg[(size_t) ch_o1 * P.frames + t] = (int16_t) aud1[i];
            }
          }
        }
      }
      // ---- the end of the call: carry the raw tail and the peak window
      const bool last_chunk = (b_first + (q + 1) * kChunkBlocks >= P.blocks);
      if (last_chunk)
      {
        const uint32_t new_frames = P.frames - (b_first + q * kChunkBlocks) * kBlk;   // frames of this chunk (48 or 96)
        if (ch_in < P.channels)
          for (int i = tig; i < kTaps; i += 4) P.tail_out[(size_t) ch_in * kTaps + i] = (row - 4 * tig)[new_frames + i];
        for (int i = lane; i < 8 * (kWin - 1); i += 32)
        {
          const int c = i / (kWin - 1), age = i % (kWin - 1) + 1;
          const uint32_t ch = grp * 8 + c;
          if (ch < P.channels) P.peaks_out[(size_t) ch * kWin + age - 1] = sPeak[c * kWin + (((int) P.blocks - age) & (kWin - 1))];
        }
      }
      __syncwarp ();                                                              // the stage has been consumed by every lane
      if (q + 2 < n_chunks) { asm volatile ("fence.proxy.async.shared::cta;" ::: "memory"); issue (q + 2, stage); }
    }
    __syncwarp ();
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------------------------
// host side: state object owned by the context
// ------------------------------------------------------------------------------------------------------------------
struct RxQ15State
{
  uint32_t channels = 0;
  bool tx = false;                      // TX-SSB-q15: the tcgen05 kernel's kTx form, with TX planes (no mma.sync form, no biquad)
  bool all_mode = false;                // RX-Q15 (TX-Q15 with tx): the tcgen05 kernel only (no biquad), one launch per kind present in a range
  slb_rx_q15_params prm{};
  slb_rx_q15_mode_params mprm{};        // RX-Q15: AM / FM taps and the discriminator's floor
  slb_tx_q15_mode_params tmprm{};       // TX-Q15: AM / FM taps and the modulators' constants
  uint8_t *d_am_planes = nullptr, *d_fm_planes = nullptr;   // RX-Q15: the AM and FM planes; TX-Q15: TX planes of the AM and FM taps
  uint32_t *d_phase = nullptr; float *d_sin513 = nullptr;   // TX-Q15: the FM phase word per channel (in place), arm_sin_f32's table
  uint32_t *d_tail[2] = { nullptr, nullptr }; int16_t *d_peaks[2] = { nullptr, nullptr }; int parity = 0;
  uint32_t *d_afrag = nullptr; uint8_t *d_lsb = nullptr;
  uint8_t *d_tc_planes = nullptr; bool tc_ok = false;   // tcgen05 form of the same FIRs (sl_rx_q15_tc.cu)
  int16_t *dbg_audio = nullptr; uint32_t *dbg_gain = nullptr;
  // optional integer biquad between mixer and AGC (prm.bq_stages > 0): state [C][4 x stages], and the staging of the three-kernel path
  int16_t *d_bq = nullptr; int16_t *d_aud = nullptr; int16_t *d_blkpk = nullptr; int16_t *d_pk_dummy = nullptr; int16_t *d_rel = nullptr; size_t aud_cap = 0, blk_cap = 0;
};

// AGC + scale of the three-kernel path (the chain with the optional biquad): block peaks of the filtered audio (arm_abs_q15 + arm_max_q15),
// the finite-window envelope and gain word exactly as in the fused kernels, arm_scale_q15, L = R. One CTA per channel.
__global__ void __launch_bounds__ (128) q15_agc_kernel (const int16_t *__restrict__ aud, uint32_t *__restrict__ out, const int16_t *__restrict__ peaks_in,
                                                        int16_t *__restrict__ peaks_out, int16_t *__restrict__ blkpk, uint32_t frames, uint32_t window,
                                                        int target, int floor_, uint32_t gmax, const int16_t *__restrict__ rel, uint32_t *__restrict__ gain_dbg)
{
  const uint32_t c = blockIdx.x, blocks = frames / kBlk;
  const int16_t *a = aud + (size_t) c * frames;
  int16_t *pk = blkpk + (size_t) c * blocks;
  const int16_t *pin = peaks_in + (size_t) c * kWin;
  __shared__ int16_t s_rel[kWin];
  if (threadIdx.x < kWin) s_rel[threadIdx.x] = rel[threadIdx.x];
  for (uint32_t b = threadIdx.x; b < blocks; b += blockDim.x)
  {
    int m = 0;
    for (int n = 0; n < kBlk; n++) m = max (m, min (abs ((int) a[(size_t) b * kBlk + n]), 32767));
    pk[b] = (int16_t) m;
  }
  __syncthreads ();
  for (uint32_t b = threadIdx.x; b < blocks; b += blockDim.x)
  {
    int e = pk[b];
    for (uint32_t age = 1; age < window; age++)
    {
      const int p = (b >= age) ? (int) pk[b - age] : (int) pin[age - b - 1];
      e = max (e, (p * (int) s_rel[age]) >> 15);
    }
    const unsigned gq = min ((unsigned) (target << 15) / (unsigned) max (e, floor_), gmax);
    const int sh = max (0, 17 - __clz (gq)), m = (int) (gq >> sh);
    if (gain_dbg) gain_dbg[(size_t) c * blocks + b] = gq;
    uint32_t *o = out + (size_t) c * frames + (size_t) b * kBlk;
    for (int n = 0; n < kBlk; n++)
    {
      const int v = max (-32768, min (32767, ((int) a[(size_t) b * kBlk + n] * m) >> (15 - sh)));
      o[n] = __byte_perm ((uint32_t) v, 0u, 0x1010);
    }
  }
  // the peak window by age for the next call
  for (uint32_t age = 1 + threadIdx.x; age < (uint32_t) kWin; age += blockDim.x)
  {
    int v;
    if (blocks >= age) v = pk[blocks - age];
    else v = (age - blocks <= (uint32_t) kWin - 1) ? (int) pin[age - blocks - 1] : 0;
    peaks_out[(size_t) c * kWin + age - 1] = (int16_t) v;
  }
  if (threadIdx.x == 0) peaks_out[(size_t) c * kWin + kWin - 1] = 0;
}

// A[m][k] = h[m + 64 - k] (0 outside 0..ntaps-1), k-steps 0, 1 (32 wide) and 2 (16 wide), split into the signed high
// byte and the unsigned low byte, in the per-lane register layout of mma.sync m16n8k32 / m16n8k16 (row-major A):
// reg 0: row g, cols 4 tig ..; reg 1: row g + 8, same cols; reg 2: row g, cols 16 + 4 tig ..; reg 3: row g + 8, cols 16 + ..
static void pack_afrag (const int16_t *taps, uint32_t ntaps, uint32_t *hi /* [10][32] */, uint32_t *lo)
{
  auto A = [&] (int m, int k) -> int { const int t = m + 64 - k; return (t >= 0 && t < (int) ntaps) ? (int) taps[t] : 0; };
  for (int lane = 0; lane < 32; lane++)
  {
    const int g = lane >> 2, tig = lane & 3;
    for (int r = 0; r < 10; r++)
    {
      const int ks = r < 4 ? 0 : (r < 8 ? 1 : 2), rr = r - 4 * ks;
      const int row = g + 8 * (rr & 1), col0 = 32 * ks + 16 * (rr >> 1) + 4 * tig;
      uint32_t h = 0, l = 0;
      for (int i = 0; i < 4; i++)
      {
        const int v = A (row, col0 + i);
        const int vh = v >> 8, vl = v & 255;                                     // v = 256 vh + vl, vh signed, vl unsigned
        h |= (uint32_t) (vh & 255) << (8 * i); l |= (uint32_t) vl << (8 * i);
      }
      hi[r * 32 + lane] = h; lo[r * 32 + lane] = l;
    }
  }
}

int rxq15_create (slb_ctx *ctx, uint32_t channels, uint32_t fs, bool tx, bool all_mode, RxQ15State **out)
{
  if (fs != 48000u) return ctx_fail (ctx, SLB_ERR_UNSUPPORTED, "the q15 kernels are built for 48 kHz (48-frame firmware blocks)");
  RxQ15State *st = new RxQ15State ();
  st->channels = channels; st->tx = tx; st->all_mode = all_mode;
  bool ok = true;
  for (int p = 0; p < 2; p++)
  {
    ok = ok && cudaMalloc (&st->d_tail[p], (size_t) channels * kTaps * 4) == cudaSuccess;
    ok = ok && cudaMalloc (&st->d_peaks[p], (size_t) channels * kWin * 2) == cudaSuccess;
  }
  ok = ok && cudaMalloc (&st->d_afrag, 4 * 10 * 32 * 4) == cudaSuccess;
  ok = ok && cudaMalloc (&st->d_lsb, channels) == cudaSuccess;
  ok = ok && cudaMalloc (&st->d_tc_planes, kTcQ15PlaneBytes) == cudaSuccess;
  ok = ok && cudaMalloc (&st->d_bq, (size_t) channels * 16 * 2) == cudaSuccess && cudaMalloc (&st->d_pk_dummy, (size_t) channels * kWin * 2) == cudaSuccess && cudaMalloc (&st->d_rel, kWin * 2) == cudaSuccess;
  if (all_mode) ok = ok && cudaMalloc (&st->d_am_planes, kTcQ15PlaneBytes) == cudaSuccess && cudaMalloc (&st->d_fm_planes, tx ? kTcQ15PlaneBytes : kTcQ15FmPlaneBytes) == cudaSuccess;
  if (all_mode && tx)
    ok = ok && cudaMalloc (&st->d_phase, (size_t) channels * 4) == cudaSuccess && cudaMalloc (&st->d_sin513, 513 * sizeof (float)) == cudaSuccess &&
         cudaMemcpy (st->d_sin513, host_sin_table (), 513 * sizeof (float), cudaMemcpyHostToDevice) == cudaSuccess;
  if (!ok) { rxq15_destroy (st); return ctx_fail (ctx, SLB_ERR_CUDA, "RX-SSB-q15 state allocation failed"); }
  slb_rx_q15_params p; design_default_rx_q15 (fs, &p);
  int rc = rxq15_set_params (ctx, st, &p);
  if (rc == SLB_OK && all_mode && !tx)
  {
    slb_rx_q15_mode_params mp; design_default_rx_q15_modes (fs, &mp);
    rc = rxq15_set_mode_params (ctx, st, &mp);
  }
  if (rc == SLB_OK && all_mode && tx)
  {
    slb_tx_q15_mode_params mp; design_default_tx_q15_modes (fs, &mp);
    rc = rxq15_set_tx_mode_params (ctx, st, &mp);
  }
  if (rc == SLB_OK) rc = rxq15_reset (ctx, st);
  if (rc == SLB_OK && cudaMemset (st->d_lsb, 0, channels) != cudaSuccess) rc = ctx_fail (ctx, SLB_ERR_CUDA, "memset failed");
  if (rc != SLB_OK) { rxq15_destroy (st); return rc; }
  *out = st;
  return SLB_OK;
}

void rxq15_destroy (RxQ15State *st)
{
  if (!st) return;
  for (int p = 0; p < 2; p++) { cudaFree (st->d_tail[p]); cudaFree (st->d_peaks[p]); }
  cudaFree (st->d_afrag); cudaFree (st->d_lsb); cudaFree (st->d_tc_planes); cudaFree (st->d_am_planes); cudaFree (st->d_fm_planes);
  cudaFree (st->d_phase); cudaFree (st->d_sin513);
  cudaFree (st->d_bq); cudaFree (st->d_aud); cudaFree (st->d_blkpk); cudaFree (st->d_pk_dummy); cudaFree (st->d_rel);
  delete st;
}

int rxq15_reset (slb_ctx *ctx, RxQ15State *st)
{
  for (int p = 0; p < 2; p++)
    if (cudaMemset (st->d_tail[p], 0, (size_t) st->channels * kTaps * 4) != cudaSuccess || cudaMemset (st->d_peaks[p], 0, (size_t) st->channels * kWin * 2) != cudaSuccess)
      return ctx_fail (ctx, SLB_ERR_CUDA, "RX-SSB-q15 state reset failed");
  if (cudaMemset (st->d_bq, 0, (size_t) st->channels * 16 * 2) != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, "RX-SSB-q15 state reset failed");
  if (st->d_phase && cudaMemset (st->d_phase, 0, (size_t) st->channels * 4) != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, "TX-Q15 state reset failed");
  st->parity = 0;
  return SLB_OK;
}

int rxq15_set_params (slb_ctx *ctx, RxQ15State *st, const slb_rx_q15_params *p)
{
  if (p->ntaps != (uint32_t) kTaps || p->agc_block != (uint32_t) kBlk) return ctx_fail (ctx, SLB_ERR_UNSUPPORTED, "this build has a kernel for ntaps=64, agc_block=48 only");
  if (p->agc_window < 1 || p->agc_window > (uint32_t) kWin || p->agc_floor < 1 || p->agc_target < 1 || p->agc_gmax_q15 < 1 || p->agc_gmax_q15 > (255u << 15))
    return ctx_fail (ctx, SLB_ERR_ARG, "AGC constants out of range");
  if (p->bq_stages > (uint32_t) SLB_MAX_STAGES || p->bq_postshift < 0 || p->bq_postshift > 14) return ctx_fail (ctx, SLB_ERR_ARG, "optional biquad: 0..4 stages, postshift 0..14");
  // the tcgen05 kernel serves the chain when every tap splits into two signed bytes and the AGC window fits the peaks it keeps
  std::vector<uint8_t> planes (kTcQ15PlaneBytes);
  const bool tc_ok = q15_tc_build_planes (p->taps_i, p->taps_q, planes.data (), st->tx) && p->agc_window <= 17;
  // TX-SSB-q15 and RX-Q15 have the tcgen05 kernel only, and no audio filter: refused before anything changes
  if (st->tx && st->all_mode && (p->bq_stages != 0 || !tc_ok))
    return ctx_fail (ctx, SLB_ERR_UNSUPPORTED, "TX-Q15 runs on the tcgen05 kernel only: bq_stages = 0, every tap < 32640, agc_window <= 17");
  if (st->tx && (p->bq_stages != 0 || !tc_ok))
    return ctx_fail (ctx, SLB_ERR_UNSUPPORTED, "TX-SSB-q15 runs on the tcgen05 kernel only: bq_stages = 0, every tap < 32640, agc_window <= 17");
  if (st->all_mode && (p->bq_stages != 0 || !tc_ok))
    return ctx_fail (ctx, SLB_ERR_UNSUPPORTED, "RX-Q15 runs on the tcgen05 kernel only: bq_stages = 0, every tap < 32640, agc_window <= 17");
  if (p->bq_stages != st->prm.bq_stages || std::memcmp (p->bq_coeffs, st->prm.bq_coeffs, sizeof p->bq_coeffs) != 0)
    if (cudaMemset (st->d_bq, 0, (size_t) st->channels * 16 * 2) != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, "RX-SSB-q15 state reset failed");   // a new filter starts from rest
  if (cudaMemcpy (st->d_rel, p->rel, kWin * 2, cudaMemcpyHostToDevice) != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, "release table upload failed");
  std::vector<uint32_t> frag (4 * 10 * 32);
  pack_afrag (p->taps_i, p->ntaps, frag.data (), frag.data () + 320);
  pack_afrag (p->taps_q, p->ntaps, frag.data () + 640, frag.data () + 960);
  if (cudaMemcpy (st->d_afrag, frag.data (), frag.size () * 4, cudaMemcpyHostToDevice) != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, "tap upload failed");
  st->tc_ok = tc_ok;
  if (st->tc_ok && cudaMemcpy (st->d_tc_planes, planes.data (), planes.size (), cudaMemcpyHostToDevice) != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, "tap upload failed");
  st->prm = *p;
  return SLB_OK;
}
const slb_rx_q15_params *rxq15_params (const RxQ15State *st) { return &st->prm; }
int rxq15_set_mode_params (slb_ctx *ctx, RxQ15State *st, const slb_rx_q15_mode_params *p)
{
  if (!st->all_mode || st->tx) return ctx_fail (ctx, SLB_ERR_STATE, "not an RX-Q15 context");
  std::vector<uint8_t> am (kTcQ15PlaneBytes), fm (kTcQ15FmPlaneBytes);
  if (!q15_tc_build_planes (p->am_taps, p->am_taps, am.data (), false) || !q15_tc_build_fm_planes (p->fm_taps, fm.data ()) || p->fm_floor < 1)
    return ctx_fail (ctx, SLB_ERR_UNSUPPORTED, "RX-Q15 runs on the tcgen05 kernel only: every AM / FM tap < 32640, fm_floor >= 1");
  if (cudaMemcpy (st->d_am_planes, am.data (), am.size (), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy (st->d_fm_planes, fm.data (), fm.size (), cudaMemcpyHostToDevice) != cudaSuccess)
    return ctx_fail (ctx, SLB_ERR_CUDA, "tap upload failed");
  st->mprm = *p;
  return SLB_OK;
}
const slb_rx_q15_mode_params *rxq15_mode_params (const RxQ15State *st) { return st->all_mode && !st->tx ? &st->mprm : nullptr; }
int rxq15_set_tx_mode_params (slb_ctx *ctx, RxQ15State *st, const slb_tx_q15_mode_params *p)
{
  if (!st->all_mode || !st->tx) return ctx_fail (ctx, SLB_ERR_STATE, "not a TX-Q15 context");
  std::vector<uint8_t> am (kTcQ15PlaneBytes), fm (kTcQ15PlaneBytes);
  if (!q15_tc_build_planes (p->am_taps, p->am_taps, am.data (), true) || !q15_tc_build_planes (p->fm_taps, p->fm_taps, fm.data (), true) ||
      p->am_carrier < 0 || p->am_depth < 1 || p->fm_target < 1 || p->fm_inc > 65535 || p->fm_inc < -65535)
    return ctx_fail (ctx, SLB_ERR_UNSUPPORTED, "TX-Q15 runs on the tcgen05 kernel only: every AM / FM tap < 32640, am_carrier >= 0, am_depth >= 1, "
                                               "fm_target >= 1, |fm_inc| <= 65535 (y fm_inc stays in int32)");
  if (cudaMemcpy (st->d_am_planes, am.data (), am.size (), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy (st->d_fm_planes, fm.data (), fm.size (), cudaMemcpyHostToDevice) != cudaSuccess)
    return ctx_fail (ctx, SLB_ERR_CUDA, "tap upload failed");
  st->tmprm = *p;
  return SLB_OK;
}
const slb_tx_q15_mode_params *rxq15_tx_mode_params (const RxQ15State *st) { return st->all_mode && st->tx ? &st->tmprm : nullptr; }
void rxq15_set_debug (RxQ15State *st, int16_t *audio, uint32_t *gain) { st->dbg_audio = audio; st->dbg_gain = gain; }

int rxq15_set_sideband (slb_ctx *ctx, RxQ15State *st, uint32_t ch0, uint32_t n, int lsb)
{
  if (cudaMemset (st->d_lsb + ch0, lsb ? 1 : 0, n) != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, "sideband upload failed");
  return SLB_OK;
}

int rxq15_launch (slb_ctx *ctx, RxQ15State *st, const int16_t *d_in, int16_t *d_out, uint32_t ch0, uint32_t nch, uint32_t frames,
                  int sm_count, void *stream, bool with_debug)
{
  if (frames == 0 || frames % kBlk != 0) return ctx_fail (ctx, SLB_ERR_ARG, "frames must be a multiple of the 48-frame firmware block");
  if (reinterpret_cast<uintptr_t> (d_in) & 15u) return ctx_fail (ctx, SLB_ERR_ARG, "input must be 16-byte aligned (bulk copies)");
  const char *path_env = std::getenv ("SELENITE_B200_Q15_PATH");                 // A/B and test knob: "legacy" = the mma.sync kernel below
  const bool legacy_only = path_env && std::strcmp (path_env, "legacy") == 0;
  // With the optional biquad the chain runs as three kernels: (1) the fused kernel for FIRs + mixer, its audio tap as the product and
  // its own AGC output / peak window discarded, (2) arm_biquad_cascade_df1_q15 per channel, (3) AGC + scale on the filtered audio.
  const bool with_bq = st->prm.bq_stages != 0;
  int16_t *aud_tap = with_debug ? st->dbg_audio : nullptr; uint32_t *gain_tap = with_debug ? st->dbg_gain : nullptr;
  int16_t *pk_out = st->d_peaks[st->parity ^ 1] + (size_t) ch0 * kWin;
  if (with_bq)
  {
    const size_t need_a = (size_t) nch * frames, need_b = (size_t) nch * (frames / kBlk);
    if (need_a > st->aud_cap || need_b > st->blk_cap)
    {
      cudaStreamSynchronize ((cudaStream_t) stream);
      cudaFree (st->d_aud); cudaFree (st->d_blkpk); st->d_aud = st->d_blkpk = nullptr; st->aud_cap = st->blk_cap = 0;
      if (cudaMalloc (&st->d_aud, need_a * 2) != cudaSuccess || cudaMalloc (&st->d_blkpk, need_b * 2) != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, "RX-SSB-q15: staging allocation failed");
      st->aud_cap = need_a; st->blk_cap = need_b;
    }
    aud_tap = st->d_aud; gain_tap = nullptr; pk_out = st->d_pk_dummy + (size_t) ch0 * kWin;
  }
  auto finish_bq = [&] () -> int
  {
    if (!with_bq) return SLB_OK;
    cudaStream_t s_ = (cudaStream_t) stream;
    int e = launch_biquad_df1_q15 (st->prm.bq_coeffs, st->prm.bq_stages, st->prm.bq_postshift, st->d_bq + (size_t) ch0 * 4 * st->prm.bq_stages, st->d_aud, st->d_aud, nch, frames, stream);
    if (e != 0) return ctx_fail (ctx, SLB_ERR_CUDA, cudaGetErrorString ((cudaError_t) e));
    q15_agc_kernel<<<nch, 128, 0, s_>>> (st->d_aud, reinterpret_cast<uint32_t *> (d_out), st->d_peaks[st->parity] + (size_t) ch0 * kWin,
                                          st->d_peaks[st->parity ^ 1] + (size_t) ch0 * kWin, st->d_blkpk, frames, st->prm.agc_window, st->prm.agc_target, st->prm.agc_floor,
                                          st->prm.agc_gmax_q15, st->d_rel, with_debug ? st->dbg_gain : nullptr);
    cudaError_t ce = cudaGetLastError ();
    if (ce == cudaSuccess && with_debug && st->dbg_audio) ce = cudaMemcpyAsync (st->dbg_audio, st->d_aud, (size_t) nch * frames * 2, cudaMemcpyDeviceToDevice, s_);
    if (ce != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, cudaGetErrorString (ce));
    ctx_count_launch (ctx, 2);
    return SLB_OK;
  };
  if (st->tx || st->all_mode || (st->tc_ok && !legacy_only))                      // (TX, RX-Q15: the only kernel; set_params guarantees tc_ok)
  {
    RxQ15TcLaunch L{};
    L.in = d_in; L.out = d_out;
    L.tail_in = st->d_tail[st->parity] + (size_t) ch0 * kTaps; L.tail_out = st->d_tail[st->parity ^ 1] + (size_t) ch0 * kTaps;
    L.peaks_in = st->d_peaks[st->parity] + (size_t) ch0 * kWin; L.peaks_out = pk_out;
    L.planes = st->d_tc_planes; L.lsb = st->d_lsb + ch0;
    L.audio_dbg = aud_tap; L.gain_dbg = gain_tap;
    L.rel = st->prm.rel; L.channels = nch; L.frames = frames; L.window = st->prm.agc_window;
    L.target = st->prm.agc_target; L.floor_ = st->prm.agc_floor; L.gmax = st->prm.agc_gmax_q15;
    L.kind = st->tx ? kQ15Tx : kQ15Ssb; L.list = nullptr;
    // RX-Q15 / TX-Q15: the kinds in the range (a range of SSB-style channels only runs exactly as RX-SSB-q15 / TX-SSB-q15, with no list)
    Q15KindLists kl{};
    if (st->all_mode) { const int rc = q15_kind_lists (ctx, ch0, nch, &kl); if (rc) return rc; }
    if (!st->all_mode || kl.n[0] == nch)
    {
      const int e = launch_rx_q15_tc (L, sm_count, stream);
      if (e != 0) return ctx_fail (ctx, SLB_ERR_CUDA, cudaGetErrorString ((cudaError_t) e));
      ctx_count_launch (ctx);
      return finish_bq ();
    }
    // RX-Q15 / TX-Q15 with AM or FM channels in the range: one launch per kind present, each over its list
    static const int kKinds[2][3] = { { kQ15Ssb, kQ15Am, kQ15Fm }, { kQ15Tx, kQ15TxAm, kQ15TxFm } };
    for (int k = 0; k < 3; k++)
    {
      if (kl.n[k] == 0) continue;
      L.kind = kKinds[st->tx][k]; L.list = kl.d[k]; L.channels = kl.n[k];
      L.planes = k == 1 ? st->d_am_planes : (k == 2 ? st->d_fm_planes : st->d_tc_planes);
      L.fm_floor = st->mprm.fm_floor;
      if (st->tx)
      {
        // TX-Q15: the modulator's own ALC target; the phase words are carried in place
        L.target = k == 1 ? st->tmprm.am_depth : (k == 2 ? st->tmprm.fm_target : st->prm.agc_target);
        L.am_carrier = st->tmprm.am_carrier; L.fm_inc = st->tmprm.fm_inc; L.fm_level = st->tmprm.fm_level;
        L.phase = st->d_phase + ch0; L.sin513 = st->d_sin513;
      }
      const int e = launch_rx_q15_tc (L, sm_count, stream);
      if (e != 0) return ctx_fail (ctx, SLB_ERR_CUDA, cudaGetErrorString ((cudaError_t) e));
      ctx_count_launch (ctx);
    }
    return SLB_OK;
  }
  KParams P{};
  P.in = reinterpret_cast<const uint32_t *> (d_in); P.out = reinterpret_cast<uint32_t *> (d_out);
  P.tail_in = st->d_tail[st->parity] + (size_t) ch0 * kTaps; P.tail_out = st->d_tail[st->parity ^ 1] + (size_t) ch0 * kTaps;
  P.peaks_in = st->d_peaks[st->parity] + (size_t) ch0 * kWin; P.peaks_out = pk_out;
  P.afrag = st->d_afrag; P.lsb = st->d_lsb + ch0;
  P.audio_dbg = aud_tap; P.gain_dbg = gain_tap;
  std::memcpy (P.rel, st->prm.rel, sizeof P.rel);
  P.channels = nch; P.frames = frames; P.blocks = frames / kBlk; P.groups = (nch + 7) / 8; P.window = st->prm.agc_window;
  P.target = st->prm.agc_target; P.floor_ = st->prm.agc_floor; P.gmax = st->prm.agc_gmax_q15;

  if (cudaFuncSetAttribute (rx_ssb_q15_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) kSmemBytes) != cudaSuccess)
    return ctx_fail (ctx, SLB_ERR_CUDA, "cudaFuncSetAttribute failed");
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor (&per_sm, rx_ssb_q15_kernel, kThreads, kSmemBytes) != cudaSuccess || per_sm < 1) per_sm = 1;
  // segments: independent given the input (finite AGC window), each pays window-1 blocks of re-derived peaks. Aim at two
  // waves of resident warps, never shorter than 8 windows (<= 12 % overhead)
  const uint32_t resident = (uint32_t) sm_count * per_sm * kWarps;
  uint32_t segs = (2 * resident + P.groups - 1) / P.groups;
  const uint32_t min_seg = 8 * st->prm.agc_window;
  if (segs > P.blocks / min_seg) segs = P.blocks / min_seg;
  if (segs < 1) segs = 1;
  uint32_t seg_blocks = (P.blocks + segs - 1) / segs;
  seg_blocks = (seg_blocks + kChunkBlocks - 1) / kChunkBlocks * kChunkBlocks;    // whole chunks
  P.seg_blocks = seg_blocks; P.segs = (P.blocks + seg_blocks - 1) / seg_blocks;
  const uint64_t items = (uint64_t) P.groups * P.segs;
  uint64_t grid = ((uint64_t) items + kWarps - 1) / kWarps;
  if (grid > (uint64_t) sm_count * per_sm) grid = (uint64_t) sm_count * per_sm;
  rx_ssb_q15_kernel<<<(unsigned) grid, kThreads, kSmemBytes, (cudaStream_t) stream>>> (P);
  cudaError_t e = cudaGetLastError ();
  if (e != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, cudaGetErrorString (e));
  ctx_count_launch (ctx);
  return finish_bq ();
}
void rxq15_advance (RxQ15State *st) { st->parity ^= 1; }
// per-channel cadence: channels [ch0, ch0 + nch) sat this call out — their carried state moves to the buffers the next call reads
int rxq15_carry_idle (RxQ15State *st, uint32_t ch0, uint32_t nch, void *stream)
{
  cudaError_t e = cudaMemcpyAsync (st->d_tail[st->parity ^ 1] + (size_t) ch0 * kTaps, st->d_tail[st->parity] + (size_t) ch0 * kTaps, (size_t) nch * kTaps * sizeof (*st->d_tail[0]),
                                   cudaMemcpyDeviceToDevice, (cudaStream_t) stream);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync (st->d_peaks[st->parity ^ 1] + (size_t) ch0 * kWin, st->d_peaks[st->parity] + (size_t) ch0 * kWin, (size_t) nch * kWin * sizeof (*st->d_peaks[0]),
                         cudaMemcpyDeviceToDevice, (cudaStream_t) stream);
  return (int) e;
}

// TX-Q15: the same sections, then the phase words
size_t rxq15_state_bytes (const RxQ15State *st) { return (size_t) st->channels * (kTaps * 4 + kWin * 2 + 1 + 16 * 2 + (st->d_phase ? 4 : 0)); }
int rxq15_state_save (RxQ15State *st, char *dst)
{
  const size_t C = st->channels;
  if (cudaMemcpy (dst, st->d_tail[st->parity], C * kTaps * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
  if (cudaMemcpy (dst + C * kTaps * 4, st->d_peaks[st->parity], C * kWin * 2, cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
  if (cudaMemcpy (dst + C * (kTaps * 4 + kWin * 2), st->d_lsb, C, cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
  if (cudaMemcpy (dst + C * (kTaps * 4 + kWin * 2 + 1), st->d_bq, C * 16 * 2, cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
  if (st->d_phase && cudaMemcpy (dst + C * (kTaps * 4 + kWin * 2 + 1 + 16 * 2), st->d_phase, C * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
  return 0;
}
int rxq15_state_load (RxQ15State *st, const char *src)
{
  const size_t C = st->channels;
  if (cudaMemcpy (st->d_tail[st->parity], src, C * kTaps * 4, cudaMemcpyHostToDevice) != cudaSuccess) return 1;
  if (cudaMemcpy (st->d_peaks[st->parity], src + C * kTaps * 4, C * kWin * 2, cudaMemcpyHostToDevice) != cudaSuccess) return 1;
  if (cudaMemcpy (st->d_lsb, src + C * (kTaps * 4 + kWin * 2), C, cudaMemcpyHostToDevice) != cudaSuccess) return 1;
  if (cudaMemcpy (st->d_bq, src + C * (kTaps * 4 + kWin * 2 + 1), C * 16 * 2, cudaMemcpyHostToDevice) != cudaSuccess) return 1;
  if (st->d_phase && cudaMemcpy (st->d_phase, src + C * (kTaps * 4 + kWin * 2 + 1 + 16 * 2), C * 4, cudaMemcpyHostToDevice) != cudaSuccess) return 1;
  return 0;
}

}  // namespace sl
