// CHAN-64-q15 (DESIGN.md §3.10): the all-integer channelizer, bit-exact. The sibling of CHAN-64-f32 (sl_chan64.cu) on the integer
// CMSIS-DSP stages: 192 kHz wideband streams -> 64 narrowband channels of 3 kHz -> product or envelope detector -> q15 AGC.
//
//   int16 I/Q wideband --> 64-branch polyphase arm_fir_q15 (8 taps/branch, rails I and Q apart) --> arm_cfft_q15 (64) per hop
//        --> Re or arm_cmplx_mag_q15 --> per-1-ms AGC (3 narrowband samples, finite window) --> int16 L=R [stream][bin][hop]
//   oracle stage per box (reference = CMSIS-DSP V1.5.3 Source/...):
//     branch FIR  FilteringFunctions/arm_fir_q15.c:591 (q63 accumulator, >> 15, __SSAT 16; the sums are exact, so any order)
//     FFT         TransformFunctions/arm_cfft_q15.c:77, the ARM_MATH_DSP branch of a Cortex-M4 build (sl_fft_fixed.cu), output X / 64
//     envelope    ComplexMathFunctions/arm_cmplx_mag_q15.c:120 (AM)      AGC  arm_abs_q15.c, arm_max_q15.c, arm_scale_q15.c + the
//                                                                              finite-window gain law of RX-SSB-q15 (DESIGN.md §3.3)
//
// Structure. Work item = (stream, tile of 48 hops = 3072 wideband frames), dealt tile-major to a persistent, co-resident grid
// (cooperative launch) of 256-thread CTAs, several per SM. Per item, each phase separated by a CTA barrier:
//   * the tile's raw frames and the 7 hops of FIR history before them are copied to shared memory (tile 0: the history is the
//     carried state);
//   * polyphase FIR: thread (branch r, quarter of the tile) runs 12 consecutive hops of both rails with its 8 taps in registers and a
//     sliding window of 8 inputs;
//   * FFT: a half-warp per hop, one radix-4 butterfly per lane and stage in shared memory, then the detector reads the bins in
//     natural order (the bit reversal of arm_bitreversal_16 is the index of that read);
//   * block peaks (arm_abs_q15 + arm_max_q15) of the 64 x 16 blocks of the tile. They depend on the input only, so they are published
//     at once (global memory + a release flag per item). The gain law of block q looks at the peaks of up to 16 blocks before it,
//     i.e. at most the whole previous tile of the stream (agc_window <= 17), and those come from that tile's published peaks: the
//     only wait of an item is on the flag of its predecessor, which never waits on anything later (items are taken in order and
//     publish before they wait), so the co-resident grid always makes progress;
//   * gains and arm_scale_q15, stored L = R.
#include <cuda_runtime.h>
#include <cstdint>
#include <cstring>
#include <vector>
#include "sl_internal.h"

namespace sl {

namespace {
#include "sl_stress.cuh"
#include "sl_q15.cuh"

constexpr int kBins = SLB_CHAN_BINS;             // branches = FFT length = decimation
constexpr int kTaps = SLB_CHAN_TAPS;             // taps per branch (prototype = 512 taps)
constexpr int kHistHops = kTaps - 1;             // hops of input history a tile needs
constexpr int kTileHops = 48;                    // hops per tile = 16 AGC blocks of 3
constexpr int kBlk = 3;                          // AGC block: 1 ms = 192 wideband frames = 3 narrowband samples
constexpr int kTileBlocks = kTileHops / kBlk;
constexpr int kPeakWin = kTileBlocks;            // peaks carried per bin: the most the gain law looks back (agc_window <= 17)
constexpr int kMaxWindow = kPeakWin + 1;
constexpr int kThreads = 256;
constexpr int kFirHops = kTileHops / (kThreads / kBins);    // 12 consecutive hops per FIR thread
constexpr int kSpecStride = 80;                  // words per hop of the FFT buffer: the two half-warps of a warp touch opposite bank halves
constexpr int kAudStride = 50;                   // int16 per bin row of the detector output: 25 words, odd, so the bins of one hop spread over the banks
constexpr int kTwWords = 3 * kBins / 4;          // twiddleCoef_64_q15: 48 (cos, sin) pairs
static_assert (kThreads == 4 * kBins && kTileHops % 4 == 0, "four FIR threads per branch");

constexpr size_t kRawBytes = (size_t) (kTileHops + kHistHops) * kBins * 4;
constexpr size_t kSpecBytes = (size_t) kTileHops * kSpecStride * 4;
constexpr size_t kAudBytes = ((size_t) kBins * kAudStride * 2 + 15) / 16 * 16;
constexpr size_t kHpBytes = (size_t) kBins * 2 * kPeakWin * 2;
constexpr size_t kSmemBytes = kRawBytes + kSpecBytes + kAudBytes + kHpBytes + kTwWords * 4 + 32 * 2;   // ... twiddles, release table

struct KParams
{
  const uint32_t *in; uint32_t *out;            // in [S][frames] u32 I/Q; out [S][64][hops] u32 L=R
  const uint32_t *hist_in; uint32_t *hist_out;  // [S][7*64] raw frames carried between calls (ping-pong)
  const int16_t *peaks_in; int16_t *peaks_out;  // [S][64][16] block peaks by age (peaks[j] = j+1 blocks ago), ping-pong
  unsigned *flag;                               // [S][tiles]: 1 = the tile's block peaks are published (zeroed per launch)
  int16_t *tile_peaks;                          // [S][tiles][64][16]
  const int16_t *coef;                          // [64][8]: e_r[p] = h[64 p + 63 - r]
  const uint32_t *tw;                           // twiddleCoef_64_q15, (cos, sin) packed like a q15 complex word
  int16_t *audio_dbg; uint32_t *gain_dbg;       // optional: [S][64][hops], [S][64][hops/3]
  int16_t rel[kMaxWindow];
  uint32_t streams, hops, tiles, envelope, window;
  int32_t target, floor_; uint32_t gmax;
};

__device__ __forceinline__ unsigned ld_acquire (const unsigned *p)
{
  unsigned v; asm volatile ("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void st_release (unsigned *p, unsigned v)
{
  sl_jitter ();
  asm volatile ("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// arm_abs_q15: (x > 0) ? x : (x == -32768 ? 32767 : -x)
__device__ __forceinline__ int abs_q15 (int x) { return x > 0 ? x : (x == -32768 ? 32767 : -x); }

__global__ void __launch_bounds__ (kThreads) chan64_q15_kernel (const __grid_constant__ KParams P)
{
  extern __shared__ __align__ (128) unsigned char smem[];
  uint32_t *sRaw = reinterpret_cast<uint32_t *> (smem);
  uint32_t *sSpec = reinterpret_cast<uint32_t *> (smem + kRawBytes);
  int16_t *sAud = reinterpret_cast<int16_t *> (smem + kRawBytes + kSpecBytes);
  int16_t *sHp = reinterpret_cast<int16_t *> (smem + kRawBytes + kSpecBytes + kAudBytes);         // [64][32]: 16 peaks before the tile, then the tile's 16
  uint32_t *sTw = reinterpret_cast<uint32_t *> (smem + kRawBytes + kSpecBytes + kAudBytes + kHpBytes);
  int16_t *sRel = reinterpret_cast<int16_t *> (sTw + kTwWords);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned total = P.streams * P.tiles;
  for (int i = tid; i < kTwWords; i += kThreads) sTw[i] = P.tw[i];
  if (tid < kMaxWindow) sRel[tid] = P.rel[tid];
  // this thread's FIR branch and its taps
  const int r = tid & (kBins - 1), fq = tid / kBins;
  int c[kTaps];
#pragma unroll
  for (int p = 0; p < kTaps; p++) c[p] = P.coef[r * kTaps + p];
  __syncthreads ();

  for (unsigned item = blockIdx.x; item < total; item += gridDim.x)
  {
    const uint32_t tile = item / P.streams, s = item % P.streams;
    const uint32_t hops_here = min ((uint32_t) kTileHops, P.hops - tile * kTileHops);
    const int nblk = (int) hops_here / kBlk;

    // ---- raw frames: row j of sRaw holds hop j - 7 of the tile
    {
      const uint4 *src = reinterpret_cast<const uint4 *> (P.in + (size_t) s * P.hops * kBins + (size_t) tile * kTileHops * kBins) - kHistHops * kBins / 4;
      const uint4 *hist = reinterpret_cast<const uint4 *> (P.hist_in + (size_t) s * kHistHops * kBins);
      uint4 *dst = reinterpret_cast<uint4 *> (sRaw);
      const int n4 = (int) (hops_here + kHistHops) * kBins / 4;
      for (int i = tid; i < n4; i += kThreads) dst[i] = (tile == 0 && i < kHistHops * kBins / 4) ? __ldg (hist + i) : __ldg (src + i);
    }
    __syncthreads ();

    // ---- polyphase branch FIRs: v_r[m] = sat16 ((sum_p e_r[p] x_r[m - p]) >> 15), x_r[m - p] in row m + 7 - p
    {
      const int m0 = fq * kFirHops;
      if ((uint32_t) m0 < hops_here)
      {
        uint32_t w[kTaps];                                           // at hop m the sample x_r[m - p] sits in slot (m - p) & 7
#pragma unroll
        for (int j = 0; j < kHistHops; j++) w[(j + 1) & 7] = sRaw[(m0 + j) * kBins + r];
#pragma unroll
        for (int mm = 0; mm < kFirHops; mm++)
        {
          w[mm & 7] = sRaw[(m0 + mm + kHistHops) * kBins + r];
          long long ai = 0, aq = 0;
#pragma unroll
          for (int p = 0; p < kTaps; p++)
          {
            const C16 x = unpack16 (w[(mm - p) & 7]);
            ai += (long long) (c[p] * x.x); aq += (long long) (c[p] * x.y);
          }
          sSpec[(m0 + mm) * kSpecStride + r] = pack16 (C16{ sat16 ((int) (ai >> 15)), sat16 ((int) (aq >> 15)) });
        }
      }
    }
    __syncthreads ();

    // ---- 64-point arm_cfft_q15 per hop (radix-4, three stages, arm_cfft_radix4_q15.c:156-560) and the detector
    {
      const int l = lane & 15;
#pragma unroll 1
      for (int h = 2 * warp + (lane >> 4); h < kTileHops; h += 2 * (kThreads / 32))
      {
        const bool act = (uint32_t) h < hops_here;                  // (both halves of the warp reach every __syncwarp)
        uint32_t *sp = sSpec + h * kSpecStride;
        if (act)
        {
          // first stage: inputs >> 2, saturating sums, twiddles W^l, W^2l, W^3l
          uint32_t *p0 = sp + l, *p1 = p0 + 16, *p2 = p1 + 16, *p3 = p2 + 16;
          C16 a = shr (unpack16 (*p0), 2), b = shr (unpack16 (*p1), 2), cc = shr (unpack16 (*p2), 2), d = shr (unpack16 (*p3), 2);
          const C16 R = qadd (a, cc), S = qsub (a, cc), T = qadd (b, d), T2 = qsub (b, d);
          *p0 = pack16 (hadd (R, T));
          *p1 = pack16 (twid<false> (unpack16 (sTw[2 * l]), qsub (R, T)));
          *p2 = pack16 (twid<false> (unpack16 (sTw[l]), qsax (S, T2)));
          *p3 = pack16 (twid<false> (unpack16 (sTw[3 * l]), qasx (S, T2)));
        }
        __syncwarp ();
        if (act)
        {
          // middle stage: groups of 16, outputs halved, twiddle index 4 j
          const int j = l & 3, ic = 4 * j;
          uint32_t *p0 = sp + (l >> 2) * 16 + j, *p1 = p0 + 4, *p2 = p1 + 4, *p3 = p2 + 4;
          const C16 a = unpack16 (*p0), b = unpack16 (*p1), cc = unpack16 (*p2), d = unpack16 (*p3);
          const C16 R = qadd (a, cc), S = qsub (a, cc), T = qadd (b, d), T2 = qsub (b, d);
          *p0 = pack16 (shr (hadd (R, T), 1));
          *p1 = pack16 (twid<false> (unpack16 (sTw[2 * ic]), hsub (R, T)));
          *p2 = pack16 (twid<false> (unpack16 (sTw[ic]), hsax (S, T2)));
          *p3 = pack16 (twid<false> (unpack16 (sTw[3 * ic]), hasx (S, T2)));
        }
        __syncwarp ();
        if (act)
        {
          // last stage: four neighbours, no twiddles
          uint4 *q = reinterpret_cast<uint4 *> (sp) + l;
          const uint4 v = *q;
          const C16 a = unpack16 (v.x), b = unpack16 (v.y), cc = unpack16 (v.z), d = unpack16 (v.w);
          const C16 R = qadd (a, cc), T = qadd (b, d), S = qsub (a, cc), U = qsub (b, d);
          *q = make_uint4 (pack16 (hadd (R, T)), pack16 (hsub (R, T)), pack16 (hsax (S, U)), pack16 (hasx (S, U)));
        }
        __syncwarp ();
        if (act)
        {
          // bin k sits at the bit-reversed position; product detector (Re) or envelope (arm_cmplx_mag_q15, 2.14)
#pragma unroll
          for (int qd = 0; qd < 4; qd++)
          {
            const int k = l + 16 * qd;
            const C16 z = unpack16 (sp[__brev ((unsigned) k) >> 26]);
            sAud[k * kAudStride + h] = (int16_t) (P.envelope ? cmag_q15 (z.x, z.y) : z.x);
          }
        }
        __syncwarp ();
      }
    }
    __syncthreads ();

    // ---- block peaks of the tile: published at once for the successor tile; optional pre-AGC tap
    const size_t prow = ((size_t) s * P.tiles + tile) * kBins;
#pragma unroll
    for (int i = 0; i < kBins * kTileBlocks / kThreads; i++)
    {
      const int idx = tid + kThreads * i, k = idx / kTileBlocks, q = idx % kTileBlocks;
      if (q < nblk)
      {
        const int16_t *a = sAud + k * kAudStride + kBlk * q;
        const int pk = max (max (abs_q15 (a[0]), abs_q15 (a[1])), abs_q15 (a[2]));
        sHp[k * 2 * kPeakWin + kPeakWin + q] = (int16_t) pk;
        P.tile_peaks[(prow + k) * kTileBlocks + q] = (int16_t) pk;
        if (P.audio_dbg)
        {
          int16_t *ad = P.audio_dbg + ((size_t) s * kBins + k) * P.hops + (size_t) tile * kTileHops + kBlk * q;
          ad[0] = a[0]; ad[1] = a[1]; ad[2] = a[2];
        }
      }
    }
    __threadfence ();
    __syncthreads ();
    if (tid == 0 && tile + 1 < P.tiles) st_release (P.flag + (size_t) s * P.tiles + tile, 1u);

    // ---- the 16 block peaks before the tile: the carried state (tile 0) or the predecessor's published ones
    if (tile == 0)
    {
#pragma unroll
      for (int i = 0; i < kBins * kPeakWin / kThreads; i++)
      {
        const int idx = tid + kThreads * i, k = idx / kPeakWin, j = idx % kPeakWin;
        sHp[k * 2 * kPeakWin + kPeakWin - 1 - j] = P.peaks_in[((size_t) s * kBins + k) * kPeakWin + j];
      }
    }
    else
    {
      if (tid == 0)
      {
        const unsigned *f = P.flag + (size_t) s * P.tiles + tile - 1;
        unsigned spins = 0;
        while (ld_acquire (f) == 0u)
        {
          if (++spins > (1u << 23)) __trap ();                      // (seconds: a predecessor tile never published — an error, not a hung GPU)
          sl_jitter ();
          __nanosleep (40);
        }
      }
      __syncthreads ();
      const int16_t *pp = P.tile_peaks + (prow - kBins) * kTileBlocks;
#pragma unroll
      for (int i = 0; i < kBins * kPeakWin / kThreads; i++)
      {
        const int idx = tid + kThreads * i, k = idx / kPeakWin, j = idx % kPeakWin;
        sHp[k * 2 * kPeakWin + j] = __ldcg (pp + k * kTileBlocks + j);
      }
    }
    __syncthreads ();

    // ---- gain law of RX-SSB-q15 per (bin, block), arm_scale_q15, L = R store
#pragma unroll
    for (int i = 0; i < kBins * kTileBlocks / kThreads; i++)
    {
      const int idx = tid + kThreads * i, k = idx / kTileBlocks, q = idx % kTileBlocks;
      if (q < nblk)
      {
        const int16_t *hp = sHp + k * 2 * kPeakWin + kPeakWin + q;   // hp[-j] = the peak j blocks ago
        int env = hp[0];
        for (int j = 1; j < (int) P.window; j++) env = max (env, ((int) hp[-j] * (int) sRel[j]) >> 15);
        const uint32_t den = (uint32_t) max (env, P.floor_);
        const uint32_t g = min (((uint32_t) P.target << 15) / den, P.gmax);
        const int sh = max (0, 17 - (int) __clz (g));                // the least shift with (g >> sh) <= 32767
        const int kf = (int) (g >> sh);
        const int16_t *a = sAud + k * kAudStride + kBlk * q;
        uint32_t *o = P.out + ((size_t) s * kBins + k) * P.hops + (size_t) tile * kTileHops + kBlk * q;
#pragma unroll
        for (int e = 0; e < kBlk; e++)
        {
          const uint32_t y = (uint16_t) sat16 (((int) a[e] * kf) >> (15 - sh));
          o[e] = y | (y << 16);
        }
        if (P.gain_dbg) P.gain_dbg[((size_t) s * kBins + k) * (P.hops / kBlk) + (size_t) tile * kTileBlocks + q] = g;
      }
    }

    // ---- carried state at the end of the stream: the last 7 hops of raw frames, the last 16 block peaks by age
    if (tile == P.tiles - 1)
    {
      for (int i = tid; i < kHistHops * kBins; i += kThreads) P.hist_out[(size_t) s * kHistHops * kBins + i] = sRaw[hops_here * kBins + i];
#pragma unroll
      for (int i = 0; i < kBins * kPeakWin / kThreads; i++)
      {
        const int idx = tid + kThreads * i, k = idx / kPeakWin, j = idx % kPeakWin;
        P.peaks_out[((size_t) s * kBins + k) * kPeakWin + j] = sHp[k * 2 * kPeakWin + kPeakWin + nblk - 1 - j];
      }
    }
    __syncthreads ();
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
struct ChanQ15State
{
  uint32_t streams = 0;
  slb_chan_q15_params prm{};
  int16_t *d_coef = nullptr; uint32_t *d_tw = nullptr;
  uint32_t *d_hist[2] = { nullptr, nullptr }; int16_t *d_peaks[2] = { nullptr, nullptr }; int parity = 0;
  int16_t *dbg_audio = nullptr; uint32_t *dbg_gain = nullptr;
  bool attr_set = false;
};

static size_t hist_bytes (const ChanQ15State *st) { return (size_t) st->streams * kHistHops * kBins * 4; }
static size_t peak_bytes (const ChanQ15State *st) { return (size_t) st->streams * kBins * kPeakWin * 2; }

static int chanq15_upload (slb_ctx *ctx, ChanQ15State *st)
{
  std::vector<int16_t> coef ((size_t) kBins * kTaps);
  for (int r = 0; r < kBins; r++) for (int p = 0; p < kTaps; p++) coef[(size_t) r * kTaps + p] = st->prm.proto[kBins * p + (kBins - 1 - r)];
  if (cudaMemcpy (st->d_coef, coef.data (), coef.size () * 2, cudaMemcpyHostToDevice) != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, "chan64-q15: coefficient upload failed");
  return SLB_OK;
}

void chanq15_destroy (ChanQ15State *st)
{
  if (!st) return;
  cudaFree (st->d_coef); cudaFree (st->d_tw);
  for (int p = 0; p < 2; p++) { cudaFree (st->d_hist[p]); cudaFree (st->d_peaks[p]); }
  delete st;
}

int chanq15_reset (slb_ctx *ctx, ChanQ15State *st)
{
  for (int p = 0; p < 2; p++)
    if (cudaMemset (st->d_hist[p], 0, hist_bytes (st)) != cudaSuccess || cudaMemset (st->d_peaks[p], 0, peak_bytes (st)) != cudaSuccess)
      return ctx_fail (ctx, SLB_ERR_CUDA, "chan64-q15: state reset failed");
  st->parity = 0;
  return SLB_OK;
}

int chanq15_create (slb_ctx *ctx, uint32_t streams, uint32_t fs, ChanQ15State **out)
{
  ChanQ15State *st = new ChanQ15State ();
  st->streams = streams;
  design_default_chan_q15 (fs, &st->prm);
  bool ok = cudaMalloc (&st->d_coef, (size_t) kBins * kTaps * 2) == cudaSuccess && cudaMalloc (&st->d_tw, kTwWords * 4) == cudaSuccess;
  for (int p = 0; p < 2; p++) ok = ok && cudaMalloc (&st->d_hist[p], hist_bytes (st)) == cudaSuccess && cudaMalloc (&st->d_peaks[p], peak_bytes (st)) == cudaSuccess;
  if (!ok) { chanq15_destroy (st); return ctx_fail (ctx, SLB_ERR_CUDA, "chan64-q15: allocation failed"); }
  int rc = cudaMemcpy (st->d_tw, fft_twiddle_q15 (kBins), kTwWords * 4, cudaMemcpyHostToDevice) == cudaSuccess ? SLB_OK : ctx_fail (ctx, SLB_ERR_CUDA, "chan64-q15: twiddle upload failed");
  if (rc == SLB_OK) rc = chanq15_upload (ctx, st);
  if (rc == SLB_OK) rc = chanq15_reset (ctx, st);
  if (rc != SLB_OK) { chanq15_destroy (st); return rc; }
  *out = st;
  return SLB_OK;
}

int chanq15_set_params (slb_ctx *ctx, ChanQ15State *st, const slb_chan_q15_params *p)
{
  if (p->bins != (uint32_t) kBins || p->taps_per_branch != (uint32_t) kTaps || p->agc_block != (uint32_t) kBlk)
    return ctx_fail (ctx, SLB_ERR_UNSUPPORTED, "this build has a kernel for bins=64, taps_per_branch=8, agc_block=3 only");
  if (p->agc_window > (uint32_t) kMaxWindow)
    return ctx_fail (ctx, SLB_ERR_UNSUPPORTED, "agc_window <= 17: a tile's gains see the peaks of its own 16 blocks and of the tile before");
  if (p->agc_window < 1 || p->agc_floor < 1 || p->agc_target < 1 || p->agc_gmax_q15 < 1 || p->agc_gmax_q15 > (255u << 15) || p->envelope > 1)
    return ctx_fail (ctx, SLB_ERR_ARG, "AGC constants or detector out of range");
  st->prm = *p;
  return chanq15_upload (ctx, st);
}
const slb_chan_q15_params *chanq15_params (const ChanQ15State *st) { return &st->prm; }
void chanq15_set_debug (ChanQ15State *st, int16_t *audio, uint32_t *gain) { st->dbg_audio = audio; st->dbg_gain = gain; }
// checkpoint section: the raw history [S][7*64] u32, then the block peaks [S][64][16] int16
size_t chanq15_state_bytes (const ChanQ15State *st) { return hist_bytes (st) + peak_bytes (st); }
int chanq15_state_save (ChanQ15State *st, char *dst)
{
  if (cudaMemcpy (dst, st->d_hist[st->parity], hist_bytes (st), cudaMemcpyDeviceToHost) != cudaSuccess) return SLB_ERR_CUDA;
  if (cudaMemcpy (dst + hist_bytes (st), st->d_peaks[st->parity], peak_bytes (st), cudaMemcpyDeviceToHost) != cudaSuccess) return SLB_ERR_CUDA;
  return SLB_OK;
}
int chanq15_state_load (ChanQ15State *st, const char *src)
{
  st->parity = 0;
  if (cudaMemcpy (st->d_hist[0], src, hist_bytes (st), cudaMemcpyHostToDevice) != cudaSuccess) return SLB_ERR_CUDA;
  if (cudaMemcpy (st->d_peaks[0], src + hist_bytes (st), peak_bytes (st), cudaMemcpyHostToDevice) != cudaSuccess) return SLB_ERR_CUDA;
  return SLB_OK;
}

// one launch over streams [s0, s0 + ns) of the context (the host bulk path cuts the batch into stream groups)
int chanq15_launch (slb_ctx *ctx, ChanQ15State *st, const int16_t *d_in, int16_t *d_out, uint32_t s0, uint32_t ns, uint32_t frames,
                    int sm_count, void *stream_, bool with_debug)
{
  cudaStream_t stream = (cudaStream_t) stream_;
  if (frames == 0 || frames % (kBins * 12) != 0) return ctx_fail (ctx, SLB_ERR_ARG, "frames must be a multiple of 768 (4 firmware blocks at 192 kHz)");
  KParams P{};
  P.streams = ns; P.hops = frames / kBins; P.tiles = (P.hops + kTileHops - 1) / kTileHops;
  // published flags and block peaks of this launch, per stream group (concurrent launches of one context use disjoint regions)
  const size_t flag_bytes = ((size_t) st->streams * P.tiles * 4 + 255) / 256 * 256, peaks_per_stream = (size_t) P.tiles * kBins * kTileBlocks * 2;
  char *scr = static_cast<char *> (ctx_scratch (ctx, flag_bytes + (size_t) st->streams * peaks_per_stream));
  if (!scr) return SLB_ERR_CUDA;
  P.flag = reinterpret_cast<unsigned *> (scr) + (size_t) s0 * P.tiles;
  P.tile_peaks = reinterpret_cast<int16_t *> (scr + flag_bytes + (size_t) s0 * peaks_per_stream);
  if (cudaMemsetAsync (P.flag, 0, (size_t) ns * P.tiles * 4, stream) != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, "chan64-q15: flag reset failed");
  P.in = reinterpret_cast<const uint32_t *> (d_in); P.out = reinterpret_cast<uint32_t *> (d_out);
  P.hist_in = st->d_hist[st->parity] + (size_t) s0 * kHistHops * kBins; P.hist_out = st->d_hist[st->parity ^ 1] + (size_t) s0 * kHistHops * kBins;
  P.peaks_in = st->d_peaks[st->parity] + (size_t) s0 * kBins * kPeakWin; P.peaks_out = st->d_peaks[st->parity ^ 1] + (size_t) s0 * kBins * kPeakWin;
  P.coef = st->d_coef; P.tw = st->d_tw;
  P.audio_dbg = with_debug ? st->dbg_audio : nullptr; P.gain_dbg = with_debug ? st->dbg_gain : nullptr;
  std::memcpy (P.rel, st->prm.rel, sizeof P.rel);
  P.envelope = st->prm.envelope; P.window = st->prm.agc_window;
  P.target = st->prm.agc_target; P.floor_ = st->prm.agc_floor; P.gmax = st->prm.agc_gmax_q15;

  if (!st->attr_set)
  {
    cudaError_t e = cudaFuncSetAttribute (chan64_q15_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) kSmemBytes);
    if (e != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, cudaGetErrorString (e));
    st->attr_set = true;
  }
  int per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor (&per_sm, chan64_q15_kernel, kThreads, kSmemBytes);
  if (e != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, cudaGetErrorString (e));
  if (per_sm < 1) per_sm = 1;
  const uint64_t items = (uint64_t) ns * P.tiles;
  uint64_t grid = (uint64_t) sm_count * per_sm;          // co-resident: an item may wait for its predecessor's flag
  if (grid > items) grid = items;
  cudaLaunchConfig_t lc{};
  lc.gridDim = dim3 ((unsigned) grid); lc.blockDim = dim3 (kThreads); lc.dynamicSmemBytes = kSmemBytes; lc.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeCooperative; at[0].val.cooperative = 1;
  lc.attrs = at; lc.numAttrs = 1;
  e = cudaLaunchKernelEx (&lc, chan64_q15_kernel, P);
  if (e == cudaSuccess) e = cudaGetLastError ();
  if (e != cudaSuccess) return ctx_fail (ctx, SLB_ERR_CUDA, cudaGetErrorString (e));
  ctx_count_launch (ctx, 1);
  return SLB_OK;
}
void chanq15_advance (ChanQ15State *st) { st->parity ^= 1; }

}  // namespace sl
