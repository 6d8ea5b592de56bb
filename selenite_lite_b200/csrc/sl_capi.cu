// Host library + C ABI (include/selenite_b200.h). Mirrors the reference module Core/Src/dsp_if.c: same entry points,
// same argument meaning, ring index arithmetic identical; the sample movement and the inserted chain run on the GPU.
#include <cuda_runtime.h>
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include "sl_internal.h"

using namespace sl;

namespace {
std::string g_create_error;
constexpr int kBulkSlots = 3;          // pipeline depth of the host bulk path
}  // namespace

struct slb_ctx
{
  slb_config cfg{};
  Geometry geo{ 48000 };
  int sm_count = 148;
  std::string err;
  uint64_t launches = 0;
  cudaStream_t stream = nullptr;

  // chain configuration
  slb_rx_f32_params rx{};
  slb_tx_f32_params tx{};
  slb_tx_mod_params tx_mod{};          // SLB_CHAIN_TX_F32: AM / FM modulator constants
  BiquadScanTables tables{};
  std::vector<float> masks_host;       // [SLB_MAX_MASKS][2*fft_len], unscaled, as set
  std::vector<uint8_t> slot_host;      // [C]
  std::vector<uint8_t> mode_host;      // [C]
  bool tx_mode = false;
  Chan64State *chan = nullptr;         // SLB_CHAIN_CHAN64_F32 only
  ChanQ15State *chanq = nullptr;       // SLB_CHAIN_CHAN64_Q15 only
  RxQ15State *q15 = nullptr;           // SLB_CHAIN_RX_SSB_Q15, SLB_CHAIN_TX_SSB_Q15, SLB_CHAIN_RX_Q15 and SLB_CHAIN_TX_Q15 only

  // device: chain constants + carried state
  float *d_masks = nullptr; uint8_t *d_slot = nullptr; float *d_twiddle = nullptr;
  // tensor-core path of the RX-SSB-f32 chain (sl_rx_ssb_tc.cu): tap planes per mask slot, which slots it can serve
  uint8_t *d_planes = nullptr; bool tc_ok[SLB_MAX_MASKS] = {}; float tc_s0[SLB_MAX_MASKS] = {}; float tc_sz[SLB_MAX_MASKS] = {}; TcBiquadTables tc_tables{};
  uint8_t *d_tx_planes = nullptr; float tx_unit[SLB_MAX_MASKS] = {};
  uint8_t *d_am_planes = nullptr; float am_unit[SLB_MAX_MASKS] = {};   // RX contexts: the AM slot's two-rail planes (sl_rx_am_tc.cu)   // TX-SSB-f32 contexts: tc_ok[] then refers to these planes
  // a device uint32_t list of one channel range: grow-only buffer, stamped with the version of the host state it was built from
  struct DevList { uint32_t *d = nullptr; size_t cap = 0; uint64_t version = ~0ull; };
  // channel lists of the tensor-core launches, cached per channel range (the bulk paths cut the batch the same way every
  // call) and rebuilt when a mode or a mask changes (mode_version)
  struct TcLists : DevList { uint32_t groups = 0, groups_ssb = 0; std::vector<uint8_t> on_tc; };
  std::map<uint64_t, TcLists> tc_lists; uint64_t mode_version = 0;
  bool force_fft = false;              // slb_set_rx_path (SLB_RX_PATH_FFT)
  // per-channel tuning (slb_set_tune, DESIGN.md §3.5): NCO increments (2^-32 turn per sample), empty until a non-zero offset is set;
  // the list {row, inc} of a channel range (tuned rows, then the untuned ones with inc = 0) is cached per range like tc_lists and
  // rebuilt when an offset changes (tune_version)
  std::vector<int32_t> tune_inc; uint32_t n_tuned = 0;
  struct TuneList : DevList { uint32_t n = 0, n_all = 0; };
  std::map<uint64_t, TuneList> tune_lists; uint64_t tune_version = 0;
  // RX-Q15: the channels of a range by detector kind (q15_kind_lists), cached per range like tc_lists and rebuilt on mode_version
  struct KindList : DevList { uint32_t n[3] = {}; };
  std::map<uint64_t, KindList> q15_lists;
  int16_t *d_ovl[2] = { nullptr, nullptr }; int ovl_parity = 0;
  float *d_state = nullptr; unsigned *d_flag = nullptr;
  unsigned flag_base = 0;
  float *dbg_audio = nullptr, *dbg_gain = nullptr; uint32_t *dbg_phase = nullptr;

  // device: firmware rings (de-interleaved planes) + per-call block staging
  RingPtrs ring_in, ring_out;
  // per-channel cadence (SLB_DSP_*_Ch): once switched on, the pointers of every channel live on the device
  bool ring_pc = false; uint32_t *d_rptr[2] = { nullptr, nullptr }; uint8_t *d_active = nullptr;
  // ... and with a super-block chain behind the RX ring every channel fills its own super-block (frames accumulated so far)
  std::vector<uint32_t> acc_fill_pc; uint32_t *d_acc_off = nullptr;
  int16_t *d_ring[2][2] = { { nullptr, nullptr }, { nullptr, nullptr } };   // [which][i|q]
  int16_t *d_blk = nullptr; size_t blk_frames = 0;                           // [C][blk_frames][2]
  // chain at the 1 ms cadence: accumulate `hop` frames, process, feed the ring from the previous super-block
  int16_t *d_acc = nullptr; int16_t *d_proc[2] = { nullptr, nullptr }; uint32_t acc_fill = 0; int proc_cur = 0;

  // CW side-tone (dsp_if.c:218): one second of the tone as q15, key state and phase counter per channel
  uint32_t tone_hz = 0; float tone_level = 0.f; int16_t *d_tone = nullptr; float *d_sin513 = nullptr; uint8_t *d_key = nullptr; uint32_t *d_tone_cnt = nullptr;
  bool any_key = false;

  // scratch for the stage library (coefficients, FIR history double buffer)
  void *d_scratch = nullptr; size_t scratch_bytes = 0;
  cudaStream_t scratch_stream = nullptr; bool scratch_used = false; cudaEvent_t scratch_ev = nullptr;   // last stream that staged data in d_scratch

  // host bulk path
  int16_t *d_bulk_in[kBulkSlots] = {}; int16_t *d_bulk_out[kBulkSlots] = {}; size_t bulk_bytes = 0;
  cudaStream_t bulk_stream[kBulkSlots] = {};
  cudaEvent_t slice_ev[kBulkSlots][3] = {};   // time-sliced SSB host path: H2D landed / kernel done / D2H done, per staging slot
};

#define CK(ctx, call)                                                                              \
  do {                                                                                             \
    cudaError_t e_ = (cudaError_t) (call);                                                         \
    if (e_ != cudaSuccess) {                                                                       \
      char b_[512]; std::snprintf (b_, sizeof b_, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString (e_)); \
      (ctx)->err = b_; return SLB_ERR_CUDA;                                                        \
    }                                                                                              \
  } while (0)

// the two f32 transmit chains share everything but the modes they accept (check_mode): kernels, state, ring handling
static inline bool is_f32_tx_chain (uint32_t chain) { return chain == SLB_CHAIN_TX_SSB_F32 || chain == SLB_CHAIN_TX_F32; }
static inline bool is_ssb_chain (uint32_t chain) { return chain == SLB_CHAIN_RX_SSB_F32 || is_f32_tx_chain (chain); }
// the direction a context was created for: slb_tx_process_* serve these chains, slb_rx_process_* the others
static inline bool is_tx_direction (uint32_t chain) { return is_f32_tx_chain (chain) || chain == SLB_CHAIN_TX_SSB_Q15 || chain == SLB_CHAIN_TX_Q15; }
static inline bool is_q15_chain (uint32_t chain)
{
  return chain == SLB_CHAIN_RX_SSB_Q15 || chain == SLB_CHAIN_TX_SSB_Q15 || chain == SLB_CHAIN_RX_Q15 || chain == SLB_CHAIN_TX_Q15;
}

// the two channelizers: wideband streams in, bulk calls only (no firmware ring, no single-channel path)
static inline bool is_chan (const slb_ctx *ctx) { return ctx->chan || ctx->chanq; }

static int fail (slb_ctx *ctx, int code, const char *msg) { if (ctx) ctx->err = msg; else g_create_error = msg; return code; }

// A kernel of an earlier call may still be reading a cached channel list (any stream): lists change rarely, so the device is idle
// before a list is replaced, and again after the copy (a pageable copy may still be in flight when cudaMemcpy returns; the kernels
// that read the list run on non-blocking streams).
static int upload_list (slb_ctx *ctx, slb_ctx::DevList &l, const std::vector<uint32_t> &pack)
{
  CK (ctx, cudaDeviceSynchronize ());
  if (pack.size () > l.cap) { CK (ctx, cudaFree (l.d)); l.d = nullptr; CK (ctx, cudaMalloc (&l.d, pack.size () * 4)); l.cap = pack.size (); }
  CK (ctx, cudaMemcpy (l.d, pack.data (), pack.size () * 4, cudaMemcpyHostToDevice));
  CK (ctx, cudaDeviceSynchronize ());
  return SLB_OK;
}
// frees a list cache once it holds more than `keep` channel ranges
template <class Lists> static int drop_lists (slb_ctx *ctx, Lists &lists, size_t keep)
{
  if (lists.size () <= keep) return SLB_OK;
  CK (ctx, cudaDeviceSynchronize ());
  for (auto &kv : lists) cudaFree (kv.second.d);
  lists.clear ();
  return SLB_OK;
}

// What every chain launch carries from one call to the next, from channel ch0 on (the launch structs share these field names):
// the raw-input tail (ping-pong by ovl_parity), the per-channel state record and hand-over flag
template <class Launch> static void set_carry (Launch &L, const slb_ctx *ctx, uint32_t ch0)
{
  const size_t ovl = ctx->rx.fft_len - ctx->rx.hop;
  L.ovl_in = ctx->d_ovl[ctx->ovl_parity] + ch0 * ovl * 2; L.ovl_out = ctx->d_ovl[ctx->ovl_parity ^ 1] + ch0 * ovl * 2;
  L.state = ctx->d_state + (size_t) ch0 * 8; L.flag = ctx->d_flag + ch0;
}
template <class Launch> static void set_rx_agc (Launch &L, const slb_rx_f32_params &p)
{
  L.agc_target = p.agc_target; L.agc_decay = p.agc_decay; L.agc_floor = p.agc_floor; L.agc_gmax = p.agc_gmax;
}

namespace sl {
int ctx_device (const slb_ctx *ctx) { return ctx->cfg.device; }
size_t ctx_channels (const slb_ctx *ctx) { return ctx->cfg.channels; }
int ctx_fail (slb_ctx *ctx, int code, const char *msg) { return fail (ctx, code, msg); }
// RX-Q15 (sl_internal.h): the channels of [ch0, ch0 + nch) by kind. A range of SSB-style channels only needs no list and gets none.
int q15_kind_lists (slb_ctx *ctx, uint32_t ch0, uint32_t nch, Q15KindLists *out)
{
  auto kind = [&] (uint32_t c) { const uint8_t m = ctx->mode_host[ch0 + c]; return m == SLB_MODE_AM ? 1 : (m == SLB_MODE_FM ? 2 : 0); };
  *out = Q15KindLists{};
  for (uint32_t c = 0; c < nch; c++) out->n[kind (c)]++;
  if (out->n[0] == nch) return SLB_OK;
  slb_ctx::KindList &l = ctx->q15_lists[((uint64_t) ch0 << 32) | nch];
  if (l.version != ctx->mode_version)
  {
    std::vector<uint32_t> pack;
    pack.reserve (nch);
    for (int k = 0; k < 3; k++)
      for (uint32_t c = 0; c < nch; c++)
        if (kind (c) == k) pack.push_back (c);
    const int rc = upload_list (ctx, l, pack); if (rc) return rc;
    for (int k = 0; k < 3; k++) l.n[k] = out->n[k];
    l.version = ctx->mode_version;
  }
  out->d[0] = l.d; out->d[1] = l.d + l.n[0]; out->d[2] = l.d + l.n[0] + l.n[1];
  return SLB_OK;
}
void ctx_count_launch (slb_ctx *ctx, unsigned n) { ctx->launches += n; }
void *ctx_scratch (slb_ctx *ctx, size_t bytes)
{
  if (bytes <= ctx->scratch_bytes) return ctx->d_scratch;
  cudaDeviceSynchronize ();
  cudaFree (ctx->d_scratch); ctx->d_scratch = nullptr; ctx->scratch_bytes = 0;
  const size_t want = bytes < (1u << 20) ? (1u << 20) : bytes * 2;
  if (cudaMalloc (&ctx->d_scratch, want) != cudaSuccess) { ctx->err = "scratch allocation failed"; return nullptr; }
  ctx->scratch_bytes = want;
  return ctx->d_scratch;
}
// The same for callers that stage per-call data at the start of the buffer (coefficients, tables, temporaries) and consume it on
// `stream`: a call on another stream than the previous one first waits for everything queued there, so two stage calls of one
// context on different streams cannot overwrite each other's staged data (calls on one stream are ordered anyway).
void *ctx_scratch_on (slb_ctx *ctx, size_t bytes, void *stream_)
{
  cudaStream_t stream = (cudaStream_t) stream_;
  if (ctx->scratch_used && ctx->scratch_stream != stream)
  {
    if (!ctx->scratch_ev && cudaEventCreateWithFlags (&ctx->scratch_ev, cudaEventDisableTiming) != cudaSuccess) { ctx->err = "event creation failed"; return nullptr; }
    if (cudaEventRecord (ctx->scratch_ev, ctx->scratch_stream) != cudaSuccess || cudaStreamWaitEvent (stream, ctx->scratch_ev, 0) != cudaSuccess)
    { ctx->err = "scratch hand-over between streams failed"; return nullptr; }
  }
  ctx->scratch_stream = stream; ctx->scratch_used = true;
  return ctx_scratch (ctx, bytes);
}
}  // namespace sl

static int upload_chain_constants (slb_ctx *ctx)
{
  ctx->mode_version++;
  const uint32_t N = ctx->rx.fft_len;
  std::vector<float> scaled (ctx->masks_host.size ());
  // arm_cfft_f32.c:604-614 scales by 1/L after the inverse transform and arm_q15_to_float.c:87 by 1/32768 before the
  // forward one; both are powers of two, so folding them into the mask changes no bit of the result
  const float inv = 1.0f / ((float) N * 32768.0f);
  for (int m = 0; m < SLB_MAX_MASKS; m++)
    rx_ssb_f32_pack_mask (ctx->masks_host.data () + (size_t) m * 2 * N, inv, scaled.data () + (size_t) m * 2 * N);
  CK (ctx, cudaMemcpyAsync (ctx->d_masks, scaled.data (), scaled.size () * sizeof (float), cudaMemcpyHostToDevice, ctx->stream));
  CK (ctx, cudaMemcpyAsync (ctx->d_slot, ctx->slot_host.data (), ctx->slot_host.size (), cudaMemcpyHostToDevice, ctx->stream));
  // the same masks as 24-bit FIR taps in tensor-core layout, one plane set for the context's direction; a mask whose impulse
  // response does not fit 129 taps (a caller-supplied one may not) and the AM slot (two outputs per sample) stay on the FFT kernel.
  // The host buffers live until the stream synchronise at the end.
  const float *mask = ctx->masks_host.data ();
  std::vector<uint8_t> planes, amp;
  if (is_f32_tx_chain (ctx->cfg.chain))
  {
    planes.assign ((size_t) SLB_MAX_MASKS * kTcTxPlaneBytes, 0);
    for (int m = 0; m < SLB_MAX_MASKS; m++)
      ctx->tc_ok[m] = N == 512 && m < kAmMaskSlot && tc_build_tx_planes (mask + (size_t) m * 2 * N, planes.data () + (size_t) m * kTcTxPlaneBytes, &ctx->tx_unit[m]);
    CK (ctx, cudaMemcpyAsync (ctx->d_tx_planes, planes.data (), planes.size (), cudaMemcpyHostToDevice, ctx->stream));
  }
  else
  {
    amp.assign (2 * kTcAmPlaneBytes, 0);
    uint8_t *am = amp.data (), *fm = amp.data () + kTcAmPlaneBytes;
    // the AM slot: both rails of the filter on the tensor cores, envelope and biquad in the epilogue (sl_rx_am_tc.cu).
    // Measured slower than the FFT kernel (135.7 vs 144.8 Gsamples/s at 1024 channels: 46 MMAs per supertile, one accumulator
    // buffer, and the biquad recurrence back on the CUDA cores), so AM channels take it only on request: SELENITE_B200_AM_PATH=tc
    const char *am_env = std::getenv ("SELENITE_B200_AM_PATH");
    ctx->tc_ok[kAmMaskSlot] = am_env && std::strcmp (am_env, "tc") == 0 && N == 512 && tc_build_am_planes (mask + (size_t) kAmMaskSlot * 2 * N, am, &ctx->am_unit[kAmMaskSlot]);
    CK (ctx, cudaMemcpyAsync (ctx->d_am_planes + (size_t) kAmMaskSlot * kTcAmPlaneBytes, am, kTcAmPlaneBytes, cudaMemcpyHostToDevice, ctx->stream));
    // the FM slot: the same two-rail planes; the limiter-discriminator exists on the complex-detector tensor-core kernel only
    // (sl_rx_am_tc.cu), so an FM mask must be a 129-tap FIR (slb_set_mask refuses others)
    ctx->tc_ok[kFmMaskSlot] = N == 512 && tc_build_am_planes (mask + (size_t) kFmMaskSlot * 2 * N, fm, &ctx->am_unit[kFmMaskSlot]);
    CK (ctx, cudaMemcpyAsync (ctx->d_am_planes + (size_t) kFmMaskSlot * kTcAmPlaneBytes, fm, kTcAmPlaneBytes, cudaMemcpyHostToDevice, ctx->stream));
    planes.assign ((size_t) SLB_MAX_MASKS * kTcPlaneBytes, 0);
    for (int m = 0; m < kAmMaskSlot; m++)
      ctx->tc_ok[m] = N == 512 && tc_build_planes (mask + (size_t) m * 2 * N, ctx->rx.biquad, planes.data () + (size_t) m * kTcPlaneBytes, &ctx->tc_s0[m], &ctx->tc_sz[m]);
    CK (ctx, cudaMemcpyAsync (ctx->d_planes, planes.data (), planes.size (), cudaMemcpyHostToDevice, ctx->stream));
  }
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  design_biquad_scan_tables (ctx->rx.biquad, &ctx->tables);
  design_biquad_tc_tables (ctx->rx.biquad, &ctx->tc_tables);
  return SLB_OK;
}

// Zero the samples of both rings and everything the chain carries from one call to the next: filter history, biquad and AGC / ALC
// state, hand-over flags, the pending super-blocks. The ring pointers and the per-channel fill levels (acc_fill_pc) are left alone.
static int clear_chain_state (slb_ctx *ctx)
{
  const uint32_t C = ctx->cfg.channels, R = ctx->geo.ring_frames, ovl = ctx->rx.fft_len - ctx->rx.hop, hop = ctx->rx.hop;
  for (int w = 0; w < 2; w++) for (int k = 0; k < 2; k++) CK (ctx, cudaMemsetAsync (ctx->d_ring[w][k], 0, (size_t) C * R * 2, ctx->stream));
  for (int p = 0; p < 2; p++) CK (ctx, cudaMemsetAsync (ctx->d_ovl[p], 0, (size_t) C * ovl * 4, ctx->stream));
  CK (ctx, cudaMemsetAsync (ctx->d_state, 0, (size_t) C * 8 * sizeof (float), ctx->stream));
  CK (ctx, cudaMemsetAsync (ctx->d_flag, 0, (size_t) C * sizeof (unsigned), ctx->stream));
  CK (ctx, cudaMemsetAsync (ctx->d_acc, 0, (size_t) C * hop * 4, ctx->stream));
  for (int p = 0; p < 2; p++) CK (ctx, cudaMemsetAsync (ctx->d_proc[p], 0, (size_t) C * hop * 4, ctx->stream));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  ctx->flag_base = 0; ctx->ovl_parity = 0; ctx->acc_fill = 0; ctx->proc_cur = 0;
  return SLB_OK;
}

static int reset_state (slb_ctx *ctx)
{
  { const int rc = clear_chain_state (ctx); if (rc) return rc; }
  const uint32_t C = ctx->cfg.channels, R = ctx->geo.ring_frames;
  ctx->ring_in.reset (R); ctx->ring_out.reset (R);
  ctx->ring_pc = false;
  if (ctx->d_key) { CK (ctx, cudaMemset (ctx->d_key, 0, C)); CK (ctx, cudaMemset (ctx->d_tone_cnt, 0, (size_t) C * 4)); ctx->any_key = false; }
  if (ctx->chan) return chan64_reset (ctx, ctx->chan);
  if (ctx->chanq) return chanq15_reset (ctx, ctx->chanq);
  if (ctx->q15) return rxq15_reset (ctx, ctx->q15);
  return SLB_OK;
}

extern "C" {

const char *slb_version (void) { return "selenite-b200 0.1 (sm_100a)"; }
const char *slb_last_error (const slb_ctx *ctx) { return ctx ? ctx->err.c_str () : g_create_error.c_str (); }
uint64_t slb_kernel_launches (const slb_ctx *ctx) { return ctx ? ctx->launches : 0; }

int slb_default_rx_f32_params (uint32_t fs, slb_rx_f32_params *out) { return design_default_rx_f32 (fs, out); }
int slb_default_tx_f32_params (uint32_t fs, slb_tx_f32_params *out) { return design_default_tx_f32 (fs, out); }
int slb_default_tx_mod_params (uint32_t fs, slb_tx_mod_params *out) { return design_default_tx_mod (fs, out); }
int slb_default_mask (uint32_t fs, uint32_t fft_len, uint8_t mode, float *mask_out) { return design_default_mask (fs, fft_len, mode, mask_out); }

int slb_create (const slb_config *cfg, slb_ctx **out)
{
  if (!cfg || !out) return fail (nullptr, SLB_ERR_ARG, "null argument");
  *out = nullptr;
  if (cfg->channels == 0) return fail (nullptr, SLB_ERR_ARG, "channels must be > 0");
  if (cfg->fs != 48000u && cfg->fs != 96000u && cfg->fs != 192000u) return fail (nullptr, SLB_ERR_ARG, "fs must be 48000, 96000 or 192000");
  if (cfg->chain != SLB_CHAIN_PASS && !is_ssb_chain (cfg->chain) && cfg->chain != SLB_CHAIN_CHAN64_F32 && cfg->chain != SLB_CHAIN_CHAN64_Q15 && !is_q15_chain (cfg->chain))
    return fail (nullptr, SLB_ERR_ARG, "unknown chain");
  if (cfg->chain == SLB_CHAIN_CHAN64_Q15 && cfg->fs != 192000u) return fail (nullptr, SLB_ERR_ARG, "the integer channelizer takes 192 kHz wideband streams only");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount (&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail (nullptr, SLB_ERR_CUDA, "no CUDA device: selenite-b200 has no CPU fallback (cudaGetDeviceCount failed or returned 0)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail (nullptr, SLB_ERR_ARG, "device ordinal out of range");
  if ((e = cudaSetDevice (cfg->device)) != cudaSuccess) return fail (nullptr, SLB_ERR_CUDA, cudaGetErrorString (e));

  slb_ctx *ctx = new slb_ctx ();
  ctx->cfg = *cfg; ctx->geo = Geometry (cfg->fs);
  cudaDeviceGetAttribute (&ctx->sm_count, cudaDevAttrMultiProcessorCount, cfg->device);
  // the float chains keep 48-frame AGC / ALC blocks at every rate (the kernels' block; the release time is kept by scaling the
  // decay with fs in design_default_*): 1 ms at 48 kHz, half a firmware block at 96 kHz, a quarter at 192 kHz
  design_default_rx_f32 (cfg->fs, &ctx->rx);
  design_default_tx_f32 (cfg->fs, &ctx->tx);
  design_default_tx_mod (cfg->fs, &ctx->tx_mod);
  const uint32_t C = cfg->channels, N = ctx->rx.fft_len, hop = ctx->rx.hop, ovl = N - hop, R = ctx->geo.ring_frames;

  ctx->masks_host.assign ((size_t) SLB_MAX_MASKS * 2 * N, 0.0f);
  const uint8_t modes[8] = { SLB_MODE_LSB, SLB_MODE_USB, SLB_MODE_CW, SLB_MODE_CWR, SLB_MODE_DIG, SLB_MODE_PKT, SLB_MODE_AM, SLB_MODE_FM };
  for (uint8_t m : modes) design_default_mask (cfg->fs, N, m, ctx->masks_host.data () + (size_t) mode_to_mask_slot (m) * 2 * N);
  ctx->mode_host.assign (C, SLB_MODE_USB);
  ctx->slot_host.assign (C, (uint8_t) mode_to_mask_slot (SLB_MODE_USB));

#define CKC(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { g_create_error = std::string (#call) + " -> " + cudaGetErrorString (e_); slb_destroy (ctx); return SLB_ERR_CUDA; } } while (0)
  CKC (cudaStreamCreateWithFlags (&ctx->stream, cudaStreamNonBlocking));
  CKC (cudaMalloc (&ctx->d_masks, (size_t) SLB_MAX_MASKS * 2 * N * sizeof (float)));
  CKC (cudaMalloc (&ctx->d_planes, (size_t) SLB_MAX_MASKS * kTcPlaneBytes));
  CKC (cudaMalloc (&ctx->d_tx_planes, (size_t) SLB_MAX_MASKS * kTcTxPlaneBytes));
  CKC (cudaMalloc (&ctx->d_am_planes, (size_t) SLB_MAX_MASKS * kTcAmPlaneBytes));
  CKC (cudaMalloc (&ctx->d_slot, C));
  CKC (cudaMalloc (&ctx->d_twiddle, kTwiddleFloats * sizeof (float)));
  CKC (cudaMalloc (&ctx->d_sin513, 513 * sizeof (float)));   // arm_sin_f32's table: the side-tone and the FM NCO
  CKC (cudaMemcpy (ctx->d_sin513, host_sin_table (), 513 * sizeof (float), cudaMemcpyHostToDevice));
  for (int p = 0; p < 2; p++) CKC (cudaMalloc (&ctx->d_ovl[p], (size_t) C * ovl * 4));
  CKC (cudaMalloc (&ctx->d_state, (size_t) C * 8 * sizeof (float)));
  CKC (cudaMalloc (&ctx->d_flag, (size_t) C * sizeof (unsigned)));
  for (int w = 0; w < 2; w++) for (int k = 0; k < 2; k++) CKC (cudaMalloc (&ctx->d_ring[w][k], (size_t) C * R * 2));
  ctx->blk_frames = R;
  CKC (cudaMalloc (&ctx->d_blk, (size_t) C * ctx->blk_frames * 4));
  CKC (cudaMalloc (&ctx->d_acc, (size_t) C * hop * 4));
  for (int p = 0; p < 2; p++) CKC (cudaMalloc (&ctx->d_proc[p], (size_t) C * hop * 4));
  {
    std::vector<float> tw (kTwiddleFloats);
    rx_ssb_f32_pack_twiddles (tw.data ());
    CKC (cudaMemcpy (ctx->d_twiddle, tw.data (), tw.size () * sizeof (float), cudaMemcpyHostToDevice));
  }
#undef CKC
  int rc = upload_chain_constants (ctx);
  if (rc == SLB_OK) rc = reset_state (ctx);
  if (rc == SLB_OK && cfg->chain == SLB_CHAIN_CHAN64_F32) rc = chan64_create (ctx, C, cfg->fs, &ctx->chan);
  if (rc == SLB_OK && cfg->chain == SLB_CHAIN_CHAN64_Q15) rc = chanq15_create (ctx, C, cfg->fs, &ctx->chanq);
  if (rc == SLB_OK && is_q15_chain (cfg->chain)) rc = rxq15_create (ctx, C, cfg->fs, is_tx_direction (cfg->chain), cfg->chain == SLB_CHAIN_RX_Q15 || cfg->chain == SLB_CHAIN_TX_Q15, &ctx->q15);
  if (rc != SLB_OK) { g_create_error = ctx->err; slb_destroy (ctx); return rc; }
  *out = ctx;
  return SLB_OK;
}

void slb_destroy (slb_ctx *ctx)
{
  if (!ctx) return;
  cudaSetDevice (ctx->cfg.device);
  cudaDeviceSynchronize ();
  chan64_destroy (ctx->chan);
  chanq15_destroy (ctx->chanq);
  rxq15_destroy (ctx->q15);
  cudaFree (ctx->d_masks); cudaFree (ctx->d_slot); cudaFree (ctx->d_twiddle); cudaFree (ctx->d_planes); cudaFree (ctx->d_tx_planes); cudaFree (ctx->d_am_planes);
  drop_lists (ctx, ctx->tc_lists, 0); drop_lists (ctx, ctx->tune_lists, 0); drop_lists (ctx, ctx->q15_lists, 0);
  for (int p = 0; p < 2; p++) { cudaFree (ctx->d_ovl[p]); cudaFree (ctx->d_proc[p]); }
  cudaFree (ctx->d_state); cudaFree (ctx->d_flag);
  cudaFree (ctx->d_acc_off);
  cudaFree (ctx->d_tone); cudaFree (ctx->d_sin513); cudaFree (ctx->d_key); cudaFree (ctx->d_tone_cnt);
  for (int w = 0; w < 2; w++) for (int k = 0; k < 2; k++) cudaFree (ctx->d_ring[w][k]);
  cudaFree (ctx->d_blk); cudaFree (ctx->d_acc); cudaFree (ctx->d_scratch); if (ctx->scratch_ev) cudaEventDestroy (ctx->scratch_ev);
  cudaFree (ctx->d_rptr[0]); cudaFree (ctx->d_rptr[1]); cudaFree (ctx->d_active);
  for (int s = 0; s < kBulkSlots; s++)
  {
    cudaFree (ctx->d_bulk_in[s]); cudaFree (ctx->d_bulk_out[s]);
    if (ctx->bulk_stream[s]) cudaStreamDestroy (ctx->bulk_stream[s]);
    for (int e = 0; e < 3; e++) if (ctx->slice_ev[s][e]) cudaEventDestroy (ctx->slice_ev[s][e]);
  }
  if (ctx->stream) cudaStreamDestroy (ctx->stream);
  delete ctx;
}

int slb_sync (slb_ctx *ctx)
{
  if (!ctx) return SLB_ERR_ARG;
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  return SLB_OK;
}

int slb_set_rx_f32_params (slb_ctx *ctx, const slb_rx_f32_params *p)
{
  if (!ctx || !p) return SLB_ERR_ARG;
  if (p->fft_len != 512 || p->hop != 384 || p->n_stages != 2 || p->agc_block != (uint32_t) kAgcBlock)
    return fail (ctx, SLB_ERR_UNSUPPORTED, "this build has kernels for fft_len=512, hop=384, n_stages=2, agc_block=48 only");
  if (!(p->agc_decay > 0.f && p->agc_decay <= 1.f) || !(p->agc_floor > 0.f) || !(p->agc_gmax > 0.f) || !(p->agc_target > 0.f))
    return fail (ctx, SLB_ERR_ARG, "AGC constants out of range");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  ctx->rx = *p;
  return upload_chain_constants (ctx);
}
int slb_get_rx_f32_params (const slb_ctx *ctx, slb_rx_f32_params *p) { if (!ctx || !p) return SLB_ERR_ARG; *p = ctx->rx; return SLB_OK; }

int slb_set_tx_f32_params (slb_ctx *ctx, const slb_tx_f32_params *p)
{
  if (!ctx || !p) return SLB_ERR_ARG;
  if (p->fft_len != 512 || p->hop != 384 || p->alc_block != (uint32_t) kAgcBlock)
    return fail (ctx, SLB_ERR_UNSUPPORTED, "this build has kernels for fft_len=512, hop=384, alc_block=48 only");
  if (!(p->alc_decay > 0.f && p->alc_decay <= 1.f) || !(p->alc_floor > 0.f) || !(p->alc_gmax > 0.f) || !(p->alc_target > 0.f))
    return fail (ctx, SLB_ERR_ARG, "ALC constants out of range");
  ctx->tx = *p;
  return SLB_OK;
}
int slb_get_tx_f32_params (const slb_ctx *ctx, slb_tx_f32_params *p) { if (!ctx || !p) return SLB_ERR_ARG; *p = ctx->tx; return SLB_OK; }

int slb_set_tx_mod_params (slb_ctx *ctx, const slb_tx_mod_params *p)
{
  if (!ctx || !p) return SLB_ERR_ARG;
  if (ctx->cfg.chain != SLB_CHAIN_TX_F32) return fail (ctx, SLB_ERR_STATE, "AM / FM modulator constants belong to SLB_CHAIN_TX_F32 contexts");
  // carrier and level below full scale, depth at most 100 % (no overmodulation), deviation at most fs / 4 (|increment| <= a quarter turn:
  // the q31 increment cannot saturate)
  if (!(p->am_carrier > 0.f && p->am_carrier < 1.f) || !(p->am_depth > 0.f && p->am_depth <= 1.f) || !(p->fm_level > 0.f && p->fm_level < 1.f)
      || !(p->fm_deviation_hz > 0.f && p->fm_deviation_hz <= 0.25f * (float) ctx->cfg.fs))
    return fail (ctx, SLB_ERR_ARG, "modulator constants out of range (0 < carrier, level < 1; 0 < depth <= 1; 0 < deviation <= fs / 4)");
  ctx->tx_mod = *p;
  return SLB_OK;
}
int slb_get_tx_mod_params (const slb_ctx *ctx, slb_tx_mod_params *p) { if (!ctx || !p) return SLB_ERR_ARG; *p = ctx->tx_mod; return SLB_OK; }

int slb_set_mask (slb_ctx *ctx, uint8_t mode, const float *mask)
{
  if (!ctx || !mask) return SLB_ERR_ARG;
  const int slot = mode_to_mask_slot (mode);
  if (slot < 0) return fail (ctx, SLB_ERR_UNSUPPORTED, "not an FT-817 mode byte");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  float *dst = ctx->masks_host.data () + (size_t) slot * 2 * ctx->rx.fft_len;
  const std::vector<float> before (dst, dst + (size_t) 2 * ctx->rx.fft_len);
  std::memcpy (dst, mask, (size_t) 2 * ctx->rx.fft_len * sizeof (float));
  int rc = upload_chain_constants (ctx);
  if (rc == SLB_OK && slot == kFmMaskSlot && ctx->cfg.chain == SLB_CHAIN_RX_SSB_F32 && !ctx->tc_ok[kFmMaskSlot])
  {
    // the discriminator runs on the complex-detector tensor-core kernel only: the FM mask must be the DFT of a 129-tap filter
    std::memcpy (dst, before.data (), before.size () * sizeof (float));
    rc = upload_chain_constants (ctx);
    return rc ? rc : fail (ctx, SLB_ERR_UNSUPPORTED, "an FM mask must be the DFT of a filter of at most 129 taps (the discriminator runs on the tensor-core kernel)");
  }
  return rc;
}
int slb_set_rx_path (slb_ctx *ctx, int path)
{
  if (!ctx || (path != SLB_RX_PATH_AUTO && path != SLB_RX_PATH_FFT)) return SLB_ERR_ARG;
  ctx->force_fft = path == SLB_RX_PATH_FFT;
  ctx->mode_version++;                 // the channel lists of run_rx_kernel depend on it
  return SLB_OK;
}
int slb_get_mask (const slb_ctx *ctx, uint8_t mode, float *mask)
{
  if (!ctx || !mask) return SLB_ERR_ARG;
  const int slot = mode_to_mask_slot (mode);
  if (slot < 0) return SLB_ERR_UNSUPPORTED;
  std::memcpy (mask, ctx->masks_host.data () + (size_t) slot * 2 * ctx->rx.fft_len, (size_t) 2 * ctx->rx.fft_len * sizeof (float));
  return SLB_OK;
}

int slb_default_rx_q15_params (uint32_t fs, slb_rx_q15_params *out) { return design_default_rx_q15 (fs, out); }
int slb_set_rx_q15_params (slb_ctx *ctx, const slb_rx_q15_params *p)
{
  if (!ctx || !p) return SLB_ERR_ARG;
  if (!ctx->q15) return fail (ctx, SLB_ERR_STATE, "not an RX-SSB-q15 or TX-SSB-q15 context");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  return rxq15_set_params (ctx, ctx->q15, p);
}
int slb_get_rx_q15_params (const slb_ctx *ctx, slb_rx_q15_params *p)
{
  if (!ctx || !p || !ctx->q15) return SLB_ERR_ARG;
  *p = *rxq15_params (ctx->q15);
  return SLB_OK;
}
int slb_default_rx_q15_mode_params (uint32_t fs, slb_rx_q15_mode_params *out) { return design_default_rx_q15_modes (fs, out); }
int slb_set_rx_q15_mode_params (slb_ctx *ctx, const slb_rx_q15_mode_params *p)
{
  if (!ctx || !p) return SLB_ERR_ARG;
  if (!ctx->q15 || ctx->cfg.chain != SLB_CHAIN_RX_Q15) return fail (ctx, SLB_ERR_STATE, "not an RX-Q15 context");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  return rxq15_set_mode_params (ctx, ctx->q15, p);
}
int slb_get_rx_q15_mode_params (const slb_ctx *ctx, slb_rx_q15_mode_params *p)
{
  if (!ctx || !p) return SLB_ERR_ARG;
  if (!ctx->q15 || !rxq15_mode_params (ctx->q15)) return SLB_ERR_STATE;
  *p = *rxq15_mode_params (ctx->q15);
  return SLB_OK;
}
int slb_default_tx_q15_mode_params (uint32_t fs, slb_tx_q15_mode_params *out) { return design_default_tx_q15_modes (fs, out); }
int slb_set_tx_q15_mode_params (slb_ctx *ctx, const slb_tx_q15_mode_params *p)
{
  if (!ctx || !p) return SLB_ERR_ARG;
  if (!ctx->q15 || ctx->cfg.chain != SLB_CHAIN_TX_Q15) return fail (ctx, SLB_ERR_STATE, "not a TX-Q15 context");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  return rxq15_set_tx_mode_params (ctx, ctx->q15, p);
}
int slb_get_tx_q15_mode_params (const slb_ctx *ctx, slb_tx_q15_mode_params *p)
{
  if (!ctx || !p) return SLB_ERR_ARG;
  if (!ctx->q15 || !rxq15_tx_mode_params (ctx->q15)) return SLB_ERR_STATE;
  *p = *rxq15_tx_mode_params (ctx->q15);
  return SLB_OK;
}
int slb_rx_q15_set_debug_taps (slb_ctx *ctx, int16_t *d_audio, uint32_t *d_gain)
{
  if (ctx && ctx->chanq) { chanq15_set_debug (ctx->chanq, d_audio, d_gain); return SLB_OK; }
  if (!ctx || !ctx->q15) return SLB_ERR_ARG;
  rxq15_set_debug (ctx->q15, d_audio, d_gain);
  return SLB_OK;
}

// LSB and CW-R take the lower sideband (subtract the quadrature rail); AM / FM are not SSB-style demodulators
static int mode_to_lsb (uint8_t mode)
{
  switch (mode)
  {
    case SLB_MODE_LSB: case SLB_MODE_CWR: return 1;
    case SLB_MODE_USB: case SLB_MODE_CW: case SLB_MODE_DIG: case SLB_MODE_PKT: return 0;
    default: return -1;
  }
}

int slb_rx_set_debug_taps (slb_ctx *ctx, float *d_audio, float *d_gain)
{
  if (!ctx) return SLB_ERR_ARG;
  ctx->dbg_audio = d_audio; ctx->dbg_gain = d_gain;
  if (ctx->chan) chan64_set_debug (ctx->chan, d_audio, d_gain);
  return SLB_OK;
}
int slb_tx_set_phase_tap (slb_ctx *ctx, uint32_t *d_phase)
{
  if (!ctx) return SLB_ERR_ARG;
  if (ctx->cfg.chain != SLB_CHAIN_TX_F32) return fail (ctx, SLB_ERR_STATE, "the FM phase tap belongs to SLB_CHAIN_TX_F32 contexts");
  ctx->dbg_phase = d_phase;
  return SLB_OK;
}

// ---- per-channel tuning (DESIGN.md §3.5) ----
static int check_tune_chain (slb_ctx *ctx)
{
  if (!is_ssb_chain (ctx->cfg.chain))
    return fail (ctx, SLB_ERR_UNSUPPORTED, "tuning is served by the RX-SSB-f32, TX-SSB-f32 and TX-f32 chains only");
  return SLB_OK;
}
// inc = llround (hz 2^32 / fs) in double; the offset is refused unless |inc| <= 2^31 - 1 (strictly inside +-fs/2)
static bool tune_increment (const slb_ctx *ctx, double hz, int32_t *inc)
{
  const double v = hz * 4294967296.0 / (double) ctx->cfg.fs;
  if (!(std::fabs (v) < 2147483647.5)) return false;   // (also refuses NaN and infinities)
  *inc = (int32_t) std::llround (v);
  return true;
}
static void tune_store (slb_ctx *ctx, uint32_t ch0, const int32_t *inc, uint32_t n)
{
  bool any = false;
  for (uint32_t i = 0; i < n; i++) any = any || inc[i] != 0;
  if (!any && ctx->tune_inc.empty ()) return;                         // never tuned: nothing to keep
  if (ctx->tune_inc.empty ()) ctx->tune_inc.assign (ctx->cfg.channels, 0);
  std::copy (inc, inc + n, ctx->tune_inc.begin () + ch0);
  ctx->n_tuned = (uint32_t) std::count_if (ctx->tune_inc.begin (), ctx->tune_inc.end (), [] (int32_t v) { return v != 0; });
  ctx->tune_version++;   // run_rx_kernel rebuilds its lists, after the device has finished every call that reads the old ones
}
int slb_set_tune (slb_ctx *ctx, const double *offset_hz)
{
  if (!ctx) return SLB_ERR_ARG;
  { const int rc = check_tune_chain (ctx); if (rc) return rc; }
  const uint32_t C = ctx->cfg.channels;
  std::vector<int32_t> inc (C, 0);
  if (offset_hz)
    for (uint32_t c = 0; c < C; c++)
      if (!tune_increment (ctx, offset_hz[c], &inc[c])) return fail (ctx, SLB_ERR_ARG, "tuning offset out of range (|offset| < fs / 2)");
  tune_store (ctx, 0, inc.data (), C);
  return SLB_OK;
}
int slb_set_tune_channel (slb_ctx *ctx, uint32_t ch, double offset_hz)
{
  if (!ctx) return SLB_ERR_ARG;
  { const int rc = check_tune_chain (ctx); if (rc) return rc; }
  if (ch >= ctx->cfg.channels) return fail (ctx, SLB_ERR_ARG, "channel out of range");
  int32_t inc = 0;
  if (!tune_increment (ctx, offset_hz, &inc)) return fail (ctx, SLB_ERR_ARG, "tuning offset out of range (|offset| < fs / 2)");
  tune_store (ctx, ch, &inc, 1);
  return SLB_OK;
}
int slb_get_tune_channel (const slb_ctx *ctx, uint32_t ch, int32_t *inc, double *realized_hz)
{
  if (!ctx || ch >= ctx->cfg.channels) return SLB_ERR_ARG;
  if (!is_ssb_chain (ctx->cfg.chain)) return SLB_ERR_UNSUPPORTED;
  const int32_t v = ctx->tune_inc.empty () ? 0 : ctx->tune_inc[ch];
  if (inc) *inc = v;
  if (realized_hz) *realized_hz = (double) v * (double) ctx->cfg.fs / 4294967296.0;
  return SLB_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Firmware API, batched
// ------------------------------------------------------------------------------------------------------------------
int SLB_DSP_Init (slb_ctx *ctx)                       // dsp_if.c:377-383 (+ i2s_buff_init :74-83: zero the buffers)
{
  if (!ctx) return SLB_ERR_ARG;
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  ctx->tx_mode = false;
  return reset_state (ctx);
}
// DSP_Set_RX / DSP_Set_TX (dsp_if.c:347 / :357, called from ptt_set_rx / ptt_set_tx, rxtx_if.c:306 / :269). The firmware hands the switch to
// the codec, which mutes every path, re-routes ADC and DAC (I/Q <-> microphone, headphones <-> exciter) and unmutes (codec_if.c:230-345).
// The codec itself is out of scope; what its mute means for the sample path is: nothing that was captured or queued under the OLD
// routing may come out under the new one. So a real switch of direction flushes the samples of BOTH rings (as DSP_Out_Buff_Mute does for
// one, dsp_if.c:188-195: samples to zero, pointers untouched — the cadence on both sides goes on), and the chain forgets the signal it was
// following (filter history, biquad state, AGC / ALC envelope, the pending super-block), like a context that has just been created.
static int switch_direction (slb_ctx *ctx, bool tx)
{
  if (ctx->tx_mode == tx) return SLB_OK;                                                   // ptt_set_tx / ptt_set_rx act on a change only
  ctx->tx_mode = tx;
  if (is_chan (ctx)) return SLB_OK;                                                        // the channelizers have no firmware rings
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  { const int rc = clear_chain_state (ctx); if (rc) return rc; }
  if (ctx->q15) return rxq15_reset (ctx, ctx->q15);
  return SLB_OK;
}
int SLB_DSP_Set_RX (slb_ctx *ctx) { if (!ctx) return SLB_ERR_ARG; return switch_direction (ctx, false); }
int SLB_DSP_Set_TX (slb_ctx *ctx) { if (!ctx) return SLB_ERR_ARG; return switch_direction (ctx, true); }
int slb_get_direction (const slb_ctx *ctx) { return ctx ? (ctx->tx_mode ? 1 : 0) : SLB_ERR_ARG; }

// ---- CW side-tone at the hook the firmware marks (dsp_if.c:218) ----
int SLB_DSP_Set_Sidetone (slb_ctx *ctx, uint32_t freq_hz, float level)
{
  if (!ctx) return SLB_ERR_ARG;
  if (is_chan (ctx)) return fail (ctx, SLB_ERR_UNSUPPORTED, "the channelizer chains have no firmware ring (bulk calls only)");
  if (freq_hz >= ctx->cfg.fs / 2 || !(level >= 0.f) || !(level < 1.0f)) return fail (ctx, SLB_ERR_ARG, "side-tone: 0 <= freq < fs / 2, 0 <= level < 1");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  const uint32_t C = ctx->cfg.channels, fs = ctx->cfg.fs;
  if (!ctx->d_tone)
  {
    CK (ctx, cudaMalloc (&ctx->d_tone, (size_t) fs * 2));
    CK (ctx, cudaMalloc (&ctx->d_key, C)); CK (ctx, cudaMalloc (&ctx->d_tone_cnt, (size_t) C * 4));
    CK (ctx, cudaMemset (ctx->d_key, 0, C)); CK (ctx, cudaMemset (ctx->d_tone_cnt, 0, (size_t) C * 4));
  }
  ctx->tone_hz = freq_hz; ctx->tone_level = level;
  CK (ctx, launch_tone_table (ctx->d_tone, fs, level, ctx->d_sin513, ctx->stream));
  CK (ctx, cudaMemsetAsync (ctx->d_tone_cnt, 0, (size_t) C * 4, ctx->stream));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  ctx->launches++;
  return SLB_OK;
}
int SLB_DSP_Key (slb_ctx *ctx, const uint8_t *key_down)
{
  if (!ctx) return SLB_ERR_ARG;
  if (!ctx->d_tone) return fail (ctx, SLB_ERR_STATE, "SLB_DSP_Set_Sidetone first");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  const uint32_t C = ctx->cfg.channels;
  if (key_down) CK (ctx, cudaMemcpy (ctx->d_key, key_down, C, cudaMemcpyHostToDevice)); else CK (ctx, cudaMemset (ctx->d_key, 0, C));
  // any_key stays set for one more read after the last key-up so that the released channels' phase counters are reset
  bool any = false; if (key_down) for (uint32_t c = 0; c < C; c++) any = any || key_down[c] != 0;
  ctx->any_key = ctx->any_key || any;
  if (!any) { CK (ctx, cudaMemset (ctx->d_tone_cnt, 0, (size_t) C * 4)); ctx->any_key = false; }
  return SLB_OK;
}

// which FT-817 mode bytes (rxtx_if.h:33-43) a chain has a demodulator / modulator for
static int check_mode (slb_ctx *ctx, uint8_t mode)
{
  if (mode_to_mask_slot (mode) < 0) return fail (ctx, SLB_ERR_UNSUPPORTED, "not an FT-817 mode byte (LSB, USB, CW, CW-R, AM, FM, DIG, PKT are served; rxtx_if.h:33-43)");
  const bool all_mode = ctx->cfg.chain == SLB_CHAIN_RX_SSB_F32 || ctx->cfg.chain == SLB_CHAIN_PASS || ctx->cfg.chain == SLB_CHAIN_TX_F32 || ctx->cfg.chain == SLB_CHAIN_RX_Q15 ||
                        ctx->cfg.chain == SLB_CHAIN_TX_Q15;
  if (mode == SLB_MODE_AM && !all_mode)
    return fail (ctx, SLB_ERR_UNSUPPORTED, "AM is served by the RX-SSB-f32 and RX-Q15 chains (envelope detector), the channelizer and the TX-f32 and TX-Q15 chains (AM modulator) only; "
                                           "TX-SSB-f32, RX-SSB-q15 and TX-SSB-q15 are SSB-only");
  if (mode == SLB_MODE_FM && !all_mode)
    return fail (ctx, SLB_ERR_UNSUPPORTED, "FM is served by the RX-SSB-f32 and RX-Q15 chains (limiter-discriminator) and the TX-f32 and TX-Q15 chains (FM modulator) only; "
                                           "TX-SSB-f32, RX-SSB-q15 and TX-SSB-q15 are SSB-only");
  if (mode == SLB_MODE_FM && ctx->cfg.chain == SLB_CHAIN_RX_SSB_F32 && !ctx->tc_ok[kFmMaskSlot])
    return fail (ctx, SLB_ERR_UNSUPPORTED, "the FM slot has no tensor-core planes (fft_len must be 512 and the FM mask a 129-tap FIR)");
  return SLB_OK;
}

int SLB_DSP_Set_Mode_Channel (slb_ctx *ctx, uint32_t ch, uint8_t mode)
{
  if (!ctx || ch >= ctx->cfg.channels) return SLB_ERR_ARG;
  const int slot = mode_to_mask_slot (mode);
  { const int rc = check_mode (ctx, mode); if (rc) return rc; }
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  if (ctx->q15)
  {
    CK (ctx, cudaStreamSynchronize (ctx->stream));
    ctx->mode_host[ch] = mode; ctx->mode_version++;                    // (RX-Q15: the kind lists follow the modes)
    return rxq15_set_sideband (ctx, ctx->q15, ch, 1, mode_to_lsb (mode));
  }
  ctx->mode_host[ch] = mode; ctx->slot_host[ch] = (uint8_t) slot; ctx->mode_version++;
  CK (ctx, cudaMemcpyAsync (ctx->d_slot + ch, &ctx->slot_host[ch], 1, cudaMemcpyHostToDevice, ctx->stream));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  return SLB_OK;
}
int SLB_DSP_Set_Mode (slb_ctx *ctx, uint8_t mode)     // dsp_if.c:367-370 is the empty hook this fills
{
  if (!ctx) return SLB_ERR_ARG;
  if (ctx->chan)                                       // channelizer: the mode picks the per-bin detector
  {
    if (mode == SLB_MODE_FM) return fail (ctx, SLB_ERR_UNSUPPORTED, "no FM discriminator in the channelizer chain");
    slb_chan_params p = *chan64_params (ctx->chan);
    p.envelope = (mode == SLB_MODE_AM) ? 1u : 0u;
    CK (ctx, cudaSetDevice (ctx->cfg.device));
    return chan64_set_params (ctx, ctx->chan, &p);
  }
  if (ctx->chanq)
  {
    if (mode == SLB_MODE_FM) return fail (ctx, SLB_ERR_UNSUPPORTED, "no FM discriminator in the channelizer chain");
    slb_chan_q15_params p = *chanq15_params (ctx->chanq);
    p.envelope = (mode == SLB_MODE_AM) ? 1u : 0u;
    CK (ctx, cudaSetDevice (ctx->cfg.device));
    CK (ctx, cudaDeviceSynchronize ());
    return chanq15_set_params (ctx, ctx->chanq, &p);
  }
  const int slot = mode_to_mask_slot (mode);
  { const int rc = check_mode (ctx, mode); if (rc) return rc; }
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  std::fill (ctx->mode_host.begin (), ctx->mode_host.end (), mode);
  if (ctx->q15)
  {
    CK (ctx, cudaStreamSynchronize (ctx->stream));
    ctx->mode_version++;
    return rxq15_set_sideband (ctx, ctx->q15, 0, ctx->cfg.channels, mode_to_lsb (mode));
  }
  std::fill (ctx->slot_host.begin (), ctx->slot_host.end (), (uint8_t) slot); ctx->mode_version++;
  CK (ctx, cudaMemcpyAsync (ctx->d_slot, ctx->slot_host.data (), ctx->slot_host.size (), cudaMemcpyHostToDevice, ctx->stream));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  return SLB_OK;
}

// The FFT kernel over the contiguous channel range [ch0, ch0 + nch)
static int run_rx_fft_kernel (slb_ctx *ctx, const int16_t *d_in, int16_t *d_out, uint32_t ch0, uint32_t nch, uint32_t frames,
                              float *dbg_audio, float *dbg_gain, cudaStream_t stream, uint32_t *dbg_phase = nullptr)
{
  RxF32Launch L{};
  L.in = d_in; L.out = d_out; L.audio_dbg = dbg_audio; L.gain_dbg = dbg_gain;
  set_carry (L, ctx, ch0);
  L.masks = ctx->d_masks; L.mask_slot = ctx->d_slot + ch0; L.twiddle = ctx->d_twiddle;
  L.flag_base = ctx->flag_base; L.channels = nch; L.frames = frames;
  L.tx = is_f32_tx_chain (ctx->cfg.chain);
  L.tx_mod = ctx->cfg.chain == SLB_CHAIN_TX_F32;
  if (L.tx_mod)
  {
    const slb_tx_mod_params &m = ctx->tx_mod;
    L.am_depth = m.am_depth; L.am_carrier = m.am_carrier; L.fm_level = m.fm_level;
    L.fm_target = 2.0f * m.fm_deviation_hz / (float) ctx->cfg.fs;                 // half-turns per sample (oracle: the same float expression)
    L.phase_dbg = dbg_phase; L.sin513 = ctx->d_sin513;
  }
  if (L.tx) { L.agc_target = ctx->tx.alc_target; L.agc_decay = ctx->tx.alc_decay; L.agc_floor = ctx->tx.alc_floor; L.agc_gmax = ctx->tx.alc_gmax; }
  else set_rx_agc (L, ctx->rx);
  L.tables = &ctx->tables;
  CK (ctx, launch_rx_ssb_f32 (L, ctx->sm_count, stream));
  ctx->launches += rx_ssb_f32_launches_per_call ();
  return SLB_OK;
}

// SELENITE_B200_RX_PATH=fft keeps every channel on the FFT kernel (A/B measurements, tests of that kernel)
static bool tc_path_enabled ()
{
  static const bool on = [] { const char *e = std::getenv ("SELENITE_B200_RX_PATH"); return !(e && std::strcmp (e, "fft") == 0); } ();
  return on;
}

// The channels of [ch0, ch0 + nch) as a device list {row, inc}, the n tuned ones first (cached per range), nullptr when none is tuned
static int tune_list (slb_ctx *ctx, uint32_t ch0, uint32_t nch, const slb_ctx::TuneList **out)
{
  *out = nullptr;
  if (ctx->n_tuned == 0) return SLB_OK;
  slb_ctx::TuneList &tl = ctx->tune_lists[((uint64_t) ch0 << 32) | nch];
  if (tl.version != ctx->tune_version)
  {
    std::vector<uint32_t> pack;
    for (int tuned = 1; tuned >= 0; tuned--)
      for (uint32_t i = 0; i < nch; i++)
        if ((ctx->tune_inc[ch0 + i] != 0) == (tuned != 0)) { pack.push_back (i); pack.push_back ((uint32_t) ctx->tune_inc[ch0 + i]); }
    uint32_t n = 0;
    while (n < nch && pack[2 * n + 1] != 0) n++;
    if (n != 0) { const int rc = upload_list (ctx, tl, pack); if (rc) return rc; }
    tl.n = n; tl.n_all = nch; tl.version = ctx->tune_version;
  }
  if (tl.n) *out = &tl;
  return SLB_OK;
}

// One pass of the SSB chain over channels [ch0, ch0 + nch); d_in / d_out / debug taps point at channel ch0.
// RX: every channel whose mask is a 129-tap FIR goes to the tensor-core kernel — in groups of up to 8 channels of one
// mask slot; which kernel serves a channel depends on its mode only, never on how the batch is cut, so shards and
// channel groups reproduce the whole bit for bit. AM channels, caller-supplied masks that are no FIR, and TX stay on
// the FFT kernel (contiguous runs).
// Tuned channels (slb_set_tune) are mixed in front of an RX chain and behind a TX chain, on `stream`. in_owned: d_in is the library's
// own buffer, consumed by this pass only, so RX mixes it in place (tuned rows only); a caller's input (slb_rx_process_device) is
// staged through scratch: the same launch mixes the tuned rows into it and copies the others.
static int run_rx_chain (slb_ctx *ctx, const int16_t *d_in, int16_t *d_out, uint32_t ch0, uint32_t nch, uint32_t frames,
                         float *dbg_audio, float *dbg_gain, cudaStream_t stream, uint32_t *dbg_phase);
static int run_rx_kernel (slb_ctx *ctx, const int16_t *d_in, int16_t *d_out, uint32_t ch0, uint32_t nch, uint32_t frames,
                          float *dbg_audio, float *dbg_gain, cudaStream_t stream, bool in_owned, uint32_t *dbg_phase = nullptr)
{
  const slb_ctx::TuneList *tu = nullptr;
  { const int rc = tune_list (ctx, ch0, nch, &tu); if (rc) return rc; }
  if (!tu) return run_rx_chain (ctx, d_in, d_out, ch0, nch, frames, dbg_audio, dbg_gain, stream, dbg_phase);
  const bool is_tx = is_f32_tx_chain (ctx->cfg.chain);
  float *state = ctx->d_state + (size_t) ch0 * 8;
  if (!is_tx)
  {
    int16_t *mixed = const_cast<int16_t *> (d_in);
    if (!in_owned)
    {
      mixed = static_cast<int16_t *> (ctx_scratch_on (ctx, (size_t) nch * frames * 4, stream));
      if (!mixed) return SLB_ERR_CUDA;
    }
    CK (ctx, launch_tune (d_in, mixed, tu->d, in_owned ? tu->n : tu->n_all, tu->n, state, frames, false, ctx->d_sin513, stream));
    ctx->launches += 2;
    return run_rx_chain (ctx, mixed, d_out, ch0, nch, frames, dbg_audio, dbg_gain, stream, dbg_phase);
  }
  const int rc = run_rx_chain (ctx, d_in, d_out, ch0, nch, frames, dbg_audio, dbg_gain, stream, dbg_phase);
  if (rc) return rc;
  CK (ctx, launch_tune (d_out, d_out, tu->d, tu->n, tu->n, state, frames, true, ctx->d_sin513, stream));
  ctx->launches += 2;
  return SLB_OK;
}
static int run_rx_chain (slb_ctx *ctx, const int16_t *d_in, int16_t *d_out, uint32_t ch0, uint32_t nch, uint32_t frames,
                         float *dbg_audio, float *dbg_gain, cudaStream_t stream, uint32_t *dbg_phase)
{
  const bool is_tx = is_f32_tx_chain (ctx->cfg.chain);
  if (ctx->cfg.chain != SLB_CHAIN_RX_SSB_F32 && !is_tx)
    return run_rx_fft_kernel (ctx, d_in, d_out, ch0, nch, frames, dbg_audio, dbg_gain, stream);
  // slb_set_rx_path (SLB_RX_PATH_FFT) / SELENITE_B200_RX_PATH=fft keep every channel on the FFT kernel — except FM, whose
  // discriminator exists on the complex-detector tensor-core kernel only
  const bool fft_only = !tc_path_enabled () || ctx->force_fft;
  slb_ctx::TcLists &tl = ctx->tc_lists[((uint64_t) ch0 << 32) | nch];
  if (tl.version != ctx->mode_version)
  {
    std::vector<uint32_t> by_slot[SLB_MAX_MASKS];
    tl.on_tc.assign (nch, 0);
    size_t n_tc = 0;
    for (uint32_t i = 0; i < nch; i++)
    {
      const uint8_t slot = ctx->slot_host[ch0 + i];
      if (slot < SLB_MAX_MASKS && ctx->tc_ok[slot] && (!fft_only || slot == kFmMaskSlot)) { by_slot[slot].push_back (i); tl.on_tc[i] = 1; n_tc++; }
    }
    std::vector<uint32_t> chan, gstart, ginfo;
    chan.reserve (n_tc);
    // a group fills the 8 channel rows of one CTA; with fewer than 8 channels per SM the groups are made smaller (rows of
    // a short group repeat its last channel and are not stored), so that every SM has one: 1024 channels -> 147 groups of 7
    const size_t gsz = std::min<size_t> (kTcChannels, std::max<size_t> (1, (n_tc + (size_t) ctx->sm_count - 1) / (size_t) ctx->sm_count));
    for (uint32_t slot = 0; slot < SLB_MAX_MASKS; slot++)
      for (size_t i = 0; i < by_slot[slot].size (); i += gsz)
      {
        const uint32_t n = (uint32_t) std::min<size_t> (gsz, by_slot[slot].size () - i);
        gstart.push_back ((uint32_t) chan.size ()); ginfo.push_back (slot | (n << 8));
        chan.insert (chan.end (), by_slot[slot].begin () + i, by_slot[slot].begin () + i + n);
      }
    const uint32_t G = (uint32_t) gstart.size ();
    tl.groups_ssb = G;
    for (uint32_t gi = 0; gi < G; gi++) if ((ginfo[gi] & 0xFFu) >= (uint32_t) kAmMaskSlot) { tl.groups_ssb = gi; break; }   // slot-major: AM and FM groups (complex detector) are last
    if (G != 0)
    {
      std::vector<uint32_t> pack (2 * (size_t) G + chan.size ());
      std::memcpy (pack.data (), gstart.data (), G * 4); std::memcpy (pack.data () + G, ginfo.data (), G * 4);
      std::memcpy (pack.data () + 2 * (size_t) G, chan.data (), chan.size () * 4);
      const int rc = upload_list (ctx, tl, pack); if (rc) return rc;
    }
    tl.groups = G; tl.version = ctx->mode_version;
  }
  const std::vector<uint8_t> &on_tc = tl.on_tc;
  const unsigned flag_final = ctx->flag_base + rx_ssb_f32_tiles (frames);
  if (tl.groups != 0 && is_tx)
  {
    const uint32_t G = tl.groups;
    TxTcLaunch L{};
    L.in = d_in; L.out = d_out; L.iq_dbg = dbg_audio; L.gain_dbg = dbg_gain;
    set_carry (L, ctx, ch0);
    L.gstart = tl.d; L.ginfo = tl.d + G; L.chan = tl.d + 2 * (size_t) G;
    L.planes = ctx->d_tx_planes; L.unit = ctx->tx_unit;
    L.flag_final = flag_final;
    L.n_groups = G; L.frames = frames;
    L.alc_target = ctx->tx.alc_target; L.alc_decay = ctx->tx.alc_decay; L.alc_floor = ctx->tx.alc_floor; L.alc_gmax = ctx->tx.alc_gmax;
    CK (ctx, launch_tx_ssb_tc (L, ctx->sm_count, stream));
    ctx->launches++;
  }
  else if (tl.groups != 0)
  {
    const uint32_t G = tl.groups, Gs = tl.groups_ssb;
    if (Gs != 0)
    {
      RxTcLaunch L{};
      L.in = d_in; L.out = d_out; L.audio_dbg = dbg_audio; L.gain_dbg = dbg_gain;
      set_carry (L, ctx, ch0);
      L.gstart = tl.d; L.ginfo = tl.d + G; L.chan = tl.d + 2 * (size_t) G;
      L.planes = ctx->d_planes; L.s0 = ctx->tc_s0; L.sz = ctx->tc_sz;
      L.flag_final = flag_final;
      L.n_groups = Gs; L.frames = frames;
      set_rx_agc (L, ctx->rx);
      L.tables = &ctx->tc_tables;
      CK (ctx, launch_rx_ssb_tc (L, ctx->sm_count, stream));
      ctx->launches++;
    }
    if (Gs != G)
    {
      RxAmTcLaunch L{};
      L.in = d_in; L.out = d_out; L.audio_dbg = dbg_audio; L.gain_dbg = dbg_gain;
      set_carry (L, ctx, ch0);
      L.gstart = tl.d + Gs; L.ginfo = tl.d + G + Gs; L.chan = tl.d + 2 * (size_t) G;
      L.planes = ctx->d_am_planes; L.unit = ctx->am_unit;
      L.flag_final = flag_final;
      L.n_groups = G - Gs; L.frames = frames;
      set_rx_agc (L, ctx->rx);
      L.tables = &ctx->tc_tables;
      CK (ctx, launch_rx_am_tc (L, ctx->sm_count, stream));
      ctx->launches++;
    }
  }
  for (uint32_t i = 0; i < nch;)
  {
    if (on_tc[i]) { i++; continue; }
    uint32_t e = i; while (e < nch && !on_tc[e]) e++;
    const int rc = run_rx_fft_kernel (ctx, d_in + (size_t) i * frames * 2, d_out + (size_t) i * frames * 2, ch0 + i, e - i, frames,
                                      dbg_audio ? dbg_audio + (size_t) i * frames * (is_tx ? 2 : 1) : nullptr, dbg_gain ? dbg_gain + (size_t) i * (frames / kAgcBlock) : nullptr, stream,
                                      dbg_phase ? dbg_phase + (size_t) i * frames : nullptr);
    if (rc) return rc;
    i = e;
  }
  return SLB_OK;
}
// after ALL channels have been advanced by `frames`
static void rx_advance (slb_ctx *ctx, uint32_t frames) { ctx->flag_base += rx_ssb_f32_tiles (frames); ctx->ovl_parity ^= 1; }

static int ensure_blk (slb_ctx *ctx, size_t frames)
{
  if (frames <= ctx->blk_frames) return SLB_OK;
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  CK (ctx, cudaFree (ctx->d_blk)); ctx->d_blk = nullptr;
  CK (ctx, cudaMalloc (&ctx->d_blk, (size_t) ctx->cfg.channels * frames * 4));
  ctx->blk_frames = frames;
  return SLB_OK;
}

// switch to per-channel pointers: every channel starts from the shared host-side state
static int ring_pc_enable (slb_ctx *ctx)
{
  if (ctx->ring_pc) return SLB_OK;
  const uint32_t C = ctx->cfg.channels;
  for (int w = 0; w < 2; w++) if (!ctx->d_rptr[w]) CK (ctx, cudaMalloc (&ctx->d_rptr[w], (size_t) C * 4 * sizeof (uint32_t)));
  if (!ctx->d_active) CK (ctx, cudaMalloc (&ctx->d_active, C));
  const RingPtrs *rp[2] = { &ctx->ring_in, &ctx->ring_out };
  std::vector<uint32_t> h ((size_t) C * 4);
  for (int w = 0; w < 2; w++)
  {
    for (uint32_t c = 0; c < C; c++) { h[4 * c] = rp[w]->enable; h[4 * c + 1] = rp[w]->rd; h[4 * c + 2] = rp[w]->wr; h[4 * c + 3] = 0; }
    CK (ctx, cudaMemcpyAsync (ctx->d_rptr[w], h.data (), h.size () * sizeof (uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    CK (ctx, cudaStreamSynchronize (ctx->stream));
  }
  if (is_ssb_chain (ctx->cfg.chain))
  {
    // from here on d_proc[0] alone holds every channel's previously processed super-block (a channel's row is rewritten only after
    // its eight blocks have gone into the ring), and every channel counts its own accumulated frames
    const uint32_t hop = ctx->rx.hop;
    if (ctx->proc_cur == 1) { CK (ctx, cudaMemcpyAsync (ctx->d_proc[0], ctx->d_proc[1], (size_t) C * hop * 4, cudaMemcpyDeviceToDevice, ctx->stream)); ctx->proc_cur = 0; }
    if (!ctx->d_acc_off) CK (ctx, cudaMalloc (&ctx->d_acc_off, (size_t) C * 4));
    ctx->acc_fill_pc.assign (C, 0u);
    CK (ctx, cudaStreamSynchronize (ctx->stream));
  }
  ctx->ring_pc = true;
  return SLB_OK;
}
// maximal runs [first, first + count) of channels for which pred holds
static std::vector<std::pair<uint32_t, uint32_t>> channel_runs (uint32_t C, const std::function<bool (uint32_t)> &pred)
{
  std::vector<std::pair<uint32_t, uint32_t>> r;
  for (uint32_t c = 0; c < C;)
  {
    if (!pred (c)) { c++; continue; }
    uint32_t e = c; while (e < C && pred (e)) e++;
    r.emplace_back (c, e - c); c = e;
  }
  return r;
}
// device copy of the activity mask of this call (nullptr = all channels)
static int ring_pc_mask (slb_ctx *ctx, const uint8_t *active, const uint8_t **d_out)
{
  *d_out = nullptr;
  if (!active) return SLB_OK;
  CK (ctx, cudaMemcpyAsync (ctx->d_active, active, ctx->cfg.channels, cudaMemcpyHostToDevice, ctx->stream));
  *d_out = ctx->d_active;
  return SLB_OK;
}

static int ring_write_common (slb_ctx *ctx, int which, const void *pbuf, uint32_t frames, const uint8_t *active = nullptr, bool per_channel = false)
{
  if (is_chan (ctx)) return fail (ctx, SLB_ERR_UNSUPPORTED, "the channelizer chains have no firmware ring (bulk calls only)");
  const uint32_t C = ctx->cfg.channels, R = ctx->geo.ring_frames;
  if (!pbuf || frames == 0 || frames + 1 > R) return fail (ctx, SLB_ERR_ARG, "block must hold 1..DSP_BUFF_SIZE-1 frames");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  RingPtrs &rp = which ? ctx->ring_out : ctx->ring_in;
  // every chain sits where the codec's I2S half enters (dsp_if.c:286-289): RX chains demodulate the I/Q there, the TX
  // modulator takes the microphone the codec delivers on both ADC channels in TX (codec_if.c:304-306); the TX ring passes
  const bool chain = (which == 0 && is_ssb_chain (ctx->cfg.chain));
  if (per_channel || ctx->ring_pc)
  {
    if (which == 0 && !ctx->ring_pc && is_ssb_chain (ctx->cfg.chain) && ctx->acc_fill != 0)
      return fail (ctx, SLB_ERR_STATE, "switch to per-channel cadence on a super-block boundary");
    int rc = ring_pc_enable (ctx); if (rc) return rc;
    const uint8_t *d_act = nullptr;
    rc = ring_pc_mask (ctx, active, &d_act); if (rc) return rc;
    rc = ensure_blk (ctx, frames); if (rc) return rc;
    CK (ctx, cudaMemcpyAsync (ctx->d_blk, pbuf, (size_t) C * frames * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK (ctx, launch_ring_plan (ctx->d_rptr[which], d_act, C, R, true, which != 0, frames, ctx->stream));
    auto is_on = [&] (uint32_t c) { return !active || active[c] != 0; };
    if (which == 0 && ctx->q15)
    {
      // the integer chains demodulate (or modulate) a block in the call that delivers it (dsp_if.c:286-289): the channels that fired run through the
      // kernel (one launch per run of neighbours), the others carry their state over unchanged
      if (frames % ctx->geo.block_frames != 0) return fail (ctx, SLB_ERR_ARG, "with a q15 chain the block must be a whole number of 48-frame firmware blocks");
      rc = drop_lists (ctx, ctx->q15_lists, 64); if (rc) return rc;        // (RX-Q15: the runs of active channels change from call to call)
      for (auto &r : channel_runs (C, is_on))
      {
        rc = rxq15_launch (ctx, ctx->q15, ctx->d_blk + (size_t) r.first * frames * 2, ctx->d_proc[0] + (size_t) r.first * frames * 2, r.first, r.second, frames, ctx->sm_count, ctx->stream, false);
        if (rc) return rc;
      }
      for (auto &r : channel_runs (C, [&] (uint32_t c) { return !is_on (c); })) CK (ctx, rxq15_carry_idle (ctx->q15, r.first, r.second, ctx->stream));
      rxq15_advance (ctx->q15);
      CK (ctx, launch_ring_write_pc (ctx->d_proc[0], frames, ctx->d_ring[0][0], ctx->d_ring[0][1], C, R, ctx->d_rptr[0], frames, ctx->stream));
      ctx->launches += 2;
    }
    else if (which == 0 && is_ssb_chain (ctx->cfg.chain))
    {
      // dsp_if.c:252-300 per channel with the demodulator in front: the block joins the channel's own super-block, the ring takes the
      // block at the same position of the channel's previously processed super-block (384 frames of latency, as under the shared
      // cadence), and the channels whose super-block is now complete run through the fused chain
      const uint32_t hop = ctx->rx.hop;
      if (hop % frames != 0) return fail (ctx, SLB_ERR_ARG, "with a chain the block size must divide the hop (384)");
      for (uint32_t c = 0; c < C; c++) if (is_on (c) && ctx->acc_fill_pc[c] % frames != 0) return fail (ctx, SLB_ERR_ARG, "with a chain the block size must divide the hop (384)");
      CK (ctx, cudaMemcpyAsync (ctx->d_acc_off, ctx->acc_fill_pc.data (), (size_t) C * 4, cudaMemcpyHostToDevice, ctx->stream));
      CK (ctx, launch_acc_store_pc (ctx->d_acc, hop, ctx->d_blk, C, frames, ctx->d_acc_off, ctx->d_rptr[0], ctx->stream));
      CK (ctx, launch_ring_write_pc (ctx->d_proc[0], hop, ctx->d_ring[0][0], ctx->d_ring[0][1], C, R, ctx->d_rptr[0], frames, ctx->stream, ctx->d_acc_off));
      ctx->launches += 3;
      CK (ctx, cudaStreamSynchronize (ctx->stream));                       // (acc_fill_pc is host memory the copy above reads)
      for (uint32_t c = 0; c < C; c++) if (is_on (c)) ctx->acc_fill_pc[c] += frames;
      auto ready = [&] (uint32_t c) { return ctx->acc_fill_pc[c] == hop; };
      const auto runs = channel_runs (C, ready);
      if (!runs.empty ())
      {
        // (lists are cached per channel range, and the runs of ready channels change from call to call)
        rc = drop_lists (ctx, ctx->tc_lists, 64); if (rc) return rc;
        rc = drop_lists (ctx, ctx->tune_lists, 64); if (rc) return rc;
        const uint32_t ovl = ctx->rx.fft_len - hop;
        for (auto &r : runs)
        {
          rc = run_rx_kernel (ctx, ctx->d_acc + (size_t) r.first * hop * 2, ctx->d_proc[0] + (size_t) r.first * hop * 2, r.first, r.second, hop, nullptr, nullptr, ctx->stream, true);
          if (rc) return rc;
        }
        // the other channels sit this launch out: their raw tail and hand-over counter move on unchanged
        for (auto &r : channel_runs (C, [&] (uint32_t c) { return !ready (c); }))
        {
          CK (ctx, cudaMemcpyAsync (ctx->d_ovl[ctx->ovl_parity ^ 1] + (size_t) r.first * ovl * 2, ctx->d_ovl[ctx->ovl_parity] + (size_t) r.first * ovl * 2, (size_t) r.second * ovl * 4,
                                    cudaMemcpyDeviceToDevice, ctx->stream));
          CK (ctx, launch_fill_u32 (ctx->d_flag + r.first, r.second, ctx->flag_base + rx_ssb_f32_tiles (hop), ctx->stream));
        }
        rx_advance (ctx, hop);
        for (uint32_t c = 0; c < C; c++) if (ready (c)) ctx->acc_fill_pc[c] = 0;
      }
    }
    else
    {
      CK (ctx, launch_ring_write_pc (ctx->d_blk, frames, ctx->d_ring[which][0], ctx->d_ring[which][1], C, R, ctx->d_rptr[which], frames, ctx->stream));
      ctx->launches += 2;
    }
    CK (ctx, cudaStreamSynchronize (ctx->stream));
    return SLB_OK;
  }
  if (which == 0 && ctx->q15)
  {
    // the integer chains work at the firmware's own block size: the block is demodulated (or modulated) and enters the ring in the same
    // call, where the firmware would have called it (dsp_if.c:286-289), with no added latency
    if (frames % ctx->geo.block_frames != 0) return fail (ctx, SLB_ERR_ARG, "with a q15 chain the block must be a whole number of 48-frame firmware blocks");
    int rc = ensure_blk (ctx, frames); if (rc) return rc;
    CK (ctx, cudaMemcpyAsync (ctx->d_blk, pbuf, (size_t) C * frames * 4, cudaMemcpyHostToDevice, ctx->stream));
    rc = rxq15_launch (ctx, ctx->q15, ctx->d_blk, ctx->d_proc[0], 0, C, frames, ctx->sm_count, ctx->stream, false);
    if (rc) return rc;
    rxq15_advance (ctx->q15);
    const uint32_t wr0 = rp.plan_write (false, frames);
    CK (ctx, launch_ring_write (ctx->d_proc[0], frames, ctx->d_ring[0][0], ctx->d_ring[0][1], C, R, wr0, frames, ctx->stream));
    ctx->launches++;
  }
  else if (!chain)
  {
    int rc = ensure_blk (ctx, frames); if (rc) return rc;
    CK (ctx, cudaMemcpyAsync (ctx->d_blk, pbuf, (size_t) C * frames * 4, cudaMemcpyHostToDevice, ctx->stream));
    const uint32_t wr0 = rp.plan_write (which != 0, frames);
    CK (ctx, launch_ring_write (ctx->d_blk, frames, ctx->d_ring[which][0], ctx->d_ring[which][1], C, R, wr0, frames, ctx->stream));
    ctx->launches++;
  }
  else
  {
    const uint32_t hop = ctx->rx.hop;
    if (hop % frames != 0 || ctx->acc_fill % frames != 0) return fail (ctx, SLB_ERR_ARG, "with a chain the block size must divide the hop (384)");
    // 1. this block joins the super-block being accumulated
    CK (ctx, cudaMemcpy2DAsync (ctx->d_acc + (size_t) ctx->acc_fill * 2, (size_t) hop * 4, pbuf, (size_t) frames * 4, (size_t) frames * 4, C,
                                cudaMemcpyHostToDevice, ctx->stream));
    // 2. the ring is fed, at the same cadence, from the previously processed super-block (chain latency = hop frames)
    const uint32_t wr0 = rp.plan_write (false, frames);
    CK (ctx, launch_ring_write (ctx->d_proc[ctx->proc_cur] + (size_t) ctx->acc_fill * 2, hop, ctx->d_ring[0][0], ctx->d_ring[0][1], C, R, wr0,
                                frames, ctx->stream));
    ctx->launches++;
    ctx->acc_fill += frames;
    // 3. a full super-block runs through the fused chain
    if (ctx->acc_fill == hop)
    {
      int rc = run_rx_kernel (ctx, ctx->d_acc, ctx->d_proc[ctx->proc_cur ^ 1], 0, C, hop, nullptr, nullptr, ctx->stream, true);
      if (rc) return rc;
      rx_advance (ctx, hop);
      ctx->proc_cur ^= 1; ctx->acc_fill = 0;
    }
  }
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  return SLB_OK;
}

static int ring_read_common (slb_ctx *ctx, int which, void *pbuf, uint32_t frames, const uint8_t *active = nullptr, bool per_channel = false)
{
  if (is_chan (ctx)) return fail (ctx, SLB_ERR_UNSUPPORTED, "the channelizer chains have no firmware ring (bulk calls only)");
  const uint32_t C = ctx->cfg.channels, R = ctx->geo.ring_frames;
  if (!pbuf || frames == 0) return fail (ctx, SLB_ERR_ARG, "empty read");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  int rc = ensure_blk (ctx, frames); if (rc) return rc;
  const uint32_t *d_first = nullptr;     // per-channel cadence: the pointer records, which mark the channels skipped this call
  if (per_channel || ctx->ring_pc)
  {
    if (which == 0 && !ctx->ring_pc && ctx->cfg.chain != SLB_CHAIN_PASS && ctx->acc_fill != 0)
      return fail (ctx, SLB_ERR_STATE, "switch to per-channel cadence on a super-block boundary");
    rc = ring_pc_enable (ctx); if (rc) return rc;
    const uint8_t *d_act = nullptr;
    rc = ring_pc_mask (ctx, active, &d_act); if (rc) return rc;
    CK (ctx, launch_ring_plan (ctx->d_rptr[which], d_act, C, R, false, which != 0, frames, ctx->stream));
    CK (ctx, launch_ring_read_pc (ctx->d_blk, ctx->d_ring[which][0], ctx->d_ring[which][1], C, R, ctx->d_rptr[which], frames, ctx->stream));
    ctx->launches += 2;
    d_first = ctx->d_rptr[which];
  }
  else
  {
    RingPtrs &rp = which ? ctx->ring_out : ctx->ring_in;
    const uint32_t rd0 = rp.plan_read (which != 0, frames);
    CK (ctx, launch_ring_read (ctx->d_blk, ctx->d_ring[which][0], ctx->d_ring[which][1], C, R, rd0, frames, ctx->stream));
    ctx->launches++;
  }
  if (which == 1 && ctx->any_key && ctx->tone_hz)                                                        // "mix CW tone to speaker signal here" (dsp_if.c:218)
  { CK (ctx, launch_sidetone_mix (ctx->d_blk, C, frames, ctx->d_key, ctx->d_tone_cnt, d_first, ctx->d_tone, ctx->tone_hz, ctx->cfg.fs, ctx->stream)); ctx->launches++; }
  CK (ctx, cudaMemcpyAsync (pbuf, ctx->d_blk, (size_t) C * frames * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  return SLB_OK;
}

// the block size of a buffer call, in half-words (I2S side) or in bytes (USB side): whole frames of two 16-bit words either way
static int check_halfwords (slb_ctx *ctx, uint32_t size)
{
  if (!ctx) return SLB_ERR_ARG;
  return (size < 2 || (size & 1)) ? fail (ctx, SLB_ERR_ARG, "size must be an even number of half-words >= 2") : SLB_OK;
}
static int check_bytes (slb_ctx *ctx, uint32_t size)
{
  if (!ctx) return SLB_ERR_ARG;
  return (size < 4 || (size & 3)) ? fail (ctx, SLB_ERR_ARG, "size must be a multiple of 4 bytes") : SLB_OK;
}
int SLB_DSP_In_Buff_Write (slb_ctx *ctx, const uint16_t *pbuf, uint16_t size)
{ const int rc = check_halfwords (ctx, size); return rc ? rc : ring_write_common (ctx, 0, pbuf, size / 2u); }
int SLB_DSP_In_Buff_Read (slb_ctx *ctx, uint8_t *pbuf, uint32_t size)
{ const int rc = check_bytes (ctx, size); return rc ? rc : ring_read_common (ctx, 0, pbuf, size / 4u); }
int SLB_DSP_Out_Buff_Write (slb_ctx *ctx, const uint8_t *pbuf, uint32_t size)
{ const int rc = check_bytes (ctx, size); return rc ? rc : ring_write_common (ctx, 1, pbuf, size / 4u); }
int SLB_DSP_Out_Buff_Read (slb_ctx *ctx, uint16_t *pbuf, uint16_t size)
{ const int rc = check_halfwords (ctx, size); return rc ? rc : ring_read_common (ctx, 1, pbuf, size / 2u); }

int SLB_DSP_In_Buff_Write_Ch (slb_ctx *ctx, const uint16_t *pbuf, uint16_t size, const uint8_t *active)
{ const int rc = check_halfwords (ctx, size); return rc ? rc : ring_write_common (ctx, 0, pbuf, size / 2u, active, true); }
int SLB_DSP_In_Buff_Read_Ch (slb_ctx *ctx, uint8_t *pbuf, uint32_t size, const uint8_t *active)
{ const int rc = check_bytes (ctx, size); return rc ? rc : ring_read_common (ctx, 0, pbuf, size / 4u, active, true); }
int SLB_DSP_Out_Buff_Write_Ch (slb_ctx *ctx, const uint8_t *pbuf, uint32_t size, const uint8_t *active)
{ const int rc = check_bytes (ctx, size); return rc ? rc : ring_write_common (ctx, 1, pbuf, size / 4u, active, true); }
int SLB_DSP_Out_Buff_Read_Ch (slb_ctx *ctx, uint16_t *pbuf, uint16_t size, const uint8_t *active)
{ const int rc = check_halfwords (ctx, size); return rc ? rc : ring_read_common (ctx, 1, pbuf, size / 2u, active, true); }
int slb_ring_get_ptrs_channel (slb_ctx *ctx, int which, uint32_t channel, uint32_t out[3])
{
  if (!ctx || !out || which < 0 || which > 1 || channel >= ctx->cfg.channels) return SLB_ERR_ARG;
  if (!ctx->ring_pc) return slb_ring_get_ptrs (ctx, which, out);
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  CK (ctx, cudaMemcpy (out, ctx->d_rptr[which] + 4 * (size_t) channel, 3 * sizeof (uint32_t), cudaMemcpyDeviceToHost));
  return SLB_OK;
}

int SLB_AUDIO_AudioCmd (slb_ctx *ctx, uint8_t *pbuf, uint32_t size, uint8_t cmd)     // usbd_audio_if.c:179-202
{
  if (!ctx) return SLB_ERR_ARG;
  switch (cmd)
  {
    case 1: return SLB_OK;                                                             // AUDIO_CMD_START
    case 2: return SLB_DSP_Out_Buff_Write (ctx, pbuf, size);                           // AUDIO_CMD_PLAY
    case 3: return SLB_DSP_Out_Buff_Mute (ctx);                                        // AUDIO_CMD_STOP
    case 4: return SLB_DSP_In_Buff_Read (ctx, pbuf, size);                             // AUDIO_CMD_RECORD
    default: return SLB_OK;                                                            // the firmware ignores unknown opcodes
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Host stream feeder
// ------------------------------------------------------------------------------------------------------------------
// Both feeders (stream and live) replay the one shared cadence of a context that has firmware rings; a chain behind the RX ring
// takes whole super-blocks
static int check_feeder (slb_ctx *ctx, bool with_rx, uint32_t ticks)
{
  if (is_chan (ctx)) return fail (ctx, SLB_ERR_UNSUPPORTED, "the channelizer chains have no firmware ring (bulk calls only)");
  if (ctx->ring_pc) return fail (ctx, SLB_ERR_STATE, "the feeder replays one shared cadence; per-channel cadence is on");
  if (with_rx && is_ssb_chain (ctx->cfg.chain) && (ticks % (ctx->rx.hop / ctx->geo.block_frames) != 0 || ctx->acc_fill != 0))
    return fail (ctx, SLB_ERR_ARG, "with an FFT chain the feeder moves whole 384-frame super-blocks (ticks % 8 == 0)");
  return SLB_OK;
}
// {write index, read index} of every tick, the firmware's arithmetic in call order: the TX ring is read, then written, per tick;
// the RX ring is written, then read
static void plan_ticks (RingPtrs &rp, bool is_out, uint32_t *plan, uint32_t ticks, uint32_t B)
{
  for (uint32_t t = 0; t < ticks; t++)
    if (is_out) { plan[2 * t + 1] = rp.plan_read (true, B); plan[2 * t] = rp.plan_write (true, B); }
    else { plan[2 * t] = rp.plan_write (false, B); plan[2 * t + 1] = rp.plan_read (false, B); }
}
// TX ring: the USB stream in, the DAC stream out, with the side-tone of all `ticks` reads at once (keys constant over the run)
static int replay_tx (slb_ctx *ctx, const int16_t *d_usb_out, int16_t *d_dac, const uint32_t *d_plan, uint32_t ticks, cudaStream_t st)
{
  const uint32_t C = ctx->cfg.channels, R = ctx->geo.ring_frames, B = ctx->geo.block_frames, frames = ticks * B;
  CK (ctx, launch_ring_replay (false, nullptr, 0, 0, d_usb_out, frames, d_dac, ctx->d_ring[1][0], ctx->d_ring[1][1], C, R, d_plan, ticks, B, st));
  ctx->launches++;
  if (ctx->any_key && ctx->tone_hz)
  { CK (ctx, launch_sidetone_mix (d_dac, C, frames, ctx->d_key, ctx->d_tone_cnt, nullptr, ctx->d_tone, ctx->tone_hz, ctx->cfg.fs, st)); ctx->launches++; }
  return SLB_OK;
}
// RX ring: the ADC stream through the chain (d_prc: its output, d_adc may be overwritten), the USB stream out
static int replay_rx (slb_ctx *ctx, int16_t *d_adc, int16_t *d_prc, int16_t *d_usb_in, const uint32_t *d_plan, uint32_t ticks, cudaStream_t st)
{
  const uint32_t C = ctx->cfg.channels, R = ctx->geo.ring_frames, B = ctx->geo.block_frames, hop = ctx->rx.hop, frames = ticks * B;
  const bool f32 = is_ssb_chain (ctx->cfg.chain);        // RX demodulator or TX modulator: both sit where the I2S half enters
  const int16_t *src_a = nullptr, *src_b = d_adc; uint32_t stride_a = 0, ticks_a = 0;
  if (ctx->q15)
  {
    int rc = rxq15_launch (ctx, ctx->q15, d_adc, d_prc, 0, C, frames, ctx->sm_count, st, false);
    if (rc) return rc;
    rxq15_advance (ctx->q15);
    src_b = d_prc;
  }
  else if (f32)
  {
    // the ring is fed from the PREVIOUS processed super-block (the chain's 384 frames of latency, as behind the per-call
    // API): the first 8 ticks come from the carried super-block, the last super-block of this run becomes the carry
    int rc = run_rx_kernel (ctx, d_adc, d_prc, 0, C, frames, nullptr, nullptr, st, true);
    if (rc) return rc;
    rx_advance (ctx, frames);
    src_a = ctx->d_proc[ctx->proc_cur]; stride_a = hop; ticks_a = hop / B; src_b = d_prc;
  }
  CK (ctx, launch_ring_replay (true, src_a, stride_a, ticks_a, src_b, frames, d_usb_in, ctx->d_ring[0][0], ctx->d_ring[0][1], C, R, d_plan, ticks, B, st));
  ctx->launches++;
  if (f32)
  {
    CK (ctx, cudaMemcpy2DAsync (ctx->d_proc[ctx->proc_cur ^ 1], (size_t) hop * 4, reinterpret_cast<const char *> (d_prc) + (size_t) (frames - hop) * 4, (size_t) frames * 4,
                                (size_t) hop * 4, C, cudaMemcpyDeviceToDevice, st));
    ctx->proc_cur ^= 1;
  }
  return SLB_OK;
}

int slb_feeder_run (slb_ctx *ctx, const slb_feeder_io *io, uint32_t ticks)
{
  if (!ctx || !io || ticks == 0) return SLB_ERR_ARG;
  if ((io->adc == nullptr) != (io->usb_in == nullptr) || (io->usb_out == nullptr) != (io->dac == nullptr)) return fail (ctx, SLB_ERR_ARG, "give both buffers of a direction or neither");
  { const int rc = check_feeder (ctx, io->adc != nullptr, ticks); if (rc) return rc; }
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  const size_t frames = (size_t) ticks * ctx->geo.block_frames, bytes = (size_t) ctx->cfg.channels * frames * 4;
  // scratch: raw stream, processed stream, ring output, plan
  char *scr = static_cast<char *> (ctx_scratch_on (ctx, 3 * bytes + (size_t) ticks * 8 + 256, ctx->stream));
  if (!scr) return SLB_ERR_CUDA;
  int16_t *d_raw = reinterpret_cast<int16_t *> (scr), *d_prc = reinterpret_cast<int16_t *> (scr + bytes), *d_out = reinterpret_cast<int16_t *> (scr + 2 * bytes);
  uint32_t *d_plan = reinterpret_cast<uint32_t *> (scr + 3 * bytes);
  std::vector<uint32_t> plan ((size_t) ticks * 2);
  cudaStream_t st = ctx->stream;
  if (io->usb_out)
  {
    plan_ticks (ctx->ring_out, true, plan.data (), ticks, ctx->geo.block_frames);
    CK (ctx, cudaMemcpyAsync (d_plan, plan.data (), plan.size () * 4, cudaMemcpyHostToDevice, st));
    CK (ctx, cudaMemcpyAsync (d_raw, io->usb_out, bytes, cudaMemcpyHostToDevice, st));
    { const int rc = replay_tx (ctx, d_raw, d_out, d_plan, ticks, st); if (rc) return rc; }
    CK (ctx, cudaMemcpyAsync (io->dac, d_out, bytes, cudaMemcpyDeviceToHost, st));
    CK (ctx, cudaStreamSynchronize (st));
  }
  if (io->adc)
  {
    plan_ticks (ctx->ring_in, false, plan.data (), ticks, ctx->geo.block_frames);
    CK (ctx, cudaMemcpyAsync (d_plan, plan.data (), plan.size () * 4, cudaMemcpyHostToDevice, st));
    CK (ctx, cudaMemcpyAsync (d_raw, io->adc, bytes, cudaMemcpyHostToDevice, st));
    { const int rc = replay_rx (ctx, d_raw, d_prc, d_out, d_plan, ticks, st); if (rc) return rc; }
    CK (ctx, cudaMemcpyAsync (io->usb_in, d_out, bytes, cudaMemcpyDeviceToHost, st));
    CK (ctx, cudaStreamSynchronize (st));
  }
  return SLB_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Live feeder: chunks of ticks through a three-stream pipeline (H2D | chain + ring replay | D2H) with pinned staging
// ------------------------------------------------------------------------------------------------------------------
struct slb_live
{
  slb_ctx *ctx = nullptr;
  uint32_t ticks = 0, depth = 0; bool rx = false, tx = false;
  size_t frames = 0, bytes = 0;
  struct Slot
  {
    int16_t *h_adc = nullptr, *h_usb_out = nullptr, *h_usb_in = nullptr, *h_dac = nullptr;   // pinned
    uint32_t *h_plan = nullptr;                                                               // pinned, [2 rings][ticks][2]
    int16_t *d_adc = nullptr, *d_usb_out = nullptr, *d_prc = nullptr, *d_usb_in = nullptr, *d_dac = nullptr; uint32_t *d_plan = nullptr;
    cudaEvent_t in_done = nullptr, work_done = nullptr, out_done = nullptr;
    std::chrono::steady_clock::time_point pushed;
  };
  std::vector<Slot> slots;
  cudaStream_t s_in = nullptr, s_work = nullptr, s_out = nullptr;
  uint64_t n_pushed = 0, n_popped = 0;
};

int slb_live_open (slb_ctx *ctx, uint32_t ticks_per_chunk, uint32_t depth, int with_rx, int with_tx, slb_live **out)
{
  if (!ctx || !out || ticks_per_chunk == 0 || depth < 2 || depth > 8 || (!with_rx && !with_tx)) return SLB_ERR_ARG;
  *out = nullptr;
  { const int rc = check_feeder (ctx, with_rx != 0, ticks_per_chunk); if (rc) return rc; }
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  slb_live *lv = new slb_live ();
  lv->ctx = ctx; lv->ticks = ticks_per_chunk; lv->depth = depth; lv->rx = with_rx != 0; lv->tx = with_tx != 0;
  lv->frames = (size_t) ticks_per_chunk * ctx->geo.block_frames; lv->bytes = (size_t) ctx->cfg.channels * lv->frames * 4;
  lv->slots.resize (depth);
  bool ok = cudaStreamCreateWithFlags (&lv->s_in, cudaStreamNonBlocking) == cudaSuccess && cudaStreamCreateWithFlags (&lv->s_work, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags (&lv->s_out, cudaStreamNonBlocking) == cudaSuccess;
  const size_t plan_bytes = (size_t) ticks_per_chunk * 2 * 2 * sizeof (uint32_t);
  for (auto &sl : lv->slots)
  {
    if (!ok) break;
    if (lv->rx) ok = ok && cudaHostAlloc (&sl.h_adc, lv->bytes, cudaHostAllocDefault) == cudaSuccess && cudaHostAlloc (&sl.h_usb_in, lv->bytes, cudaHostAllocDefault) == cudaSuccess &&
                     cudaMalloc (&sl.d_adc, lv->bytes) == cudaSuccess && cudaMalloc (&sl.d_prc, lv->bytes) == cudaSuccess && cudaMalloc (&sl.d_usb_in, lv->bytes) == cudaSuccess;
    if (lv->tx) ok = ok && cudaHostAlloc (&sl.h_usb_out, lv->bytes, cudaHostAllocDefault) == cudaSuccess && cudaHostAlloc (&sl.h_dac, lv->bytes, cudaHostAllocDefault) == cudaSuccess &&
                     cudaMalloc (&sl.d_usb_out, lv->bytes) == cudaSuccess && cudaMalloc (&sl.d_dac, lv->bytes) == cudaSuccess;
    ok = ok && cudaHostAlloc (&sl.h_plan, plan_bytes, cudaHostAllocDefault) == cudaSuccess && cudaMalloc (&sl.d_plan, plan_bytes) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags (&sl.in_done, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags (&sl.work_done, cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags (&sl.out_done, cudaEventDisableTiming) == cudaSuccess;
  }
  if (!ok) { slb_live_close (lv); return fail (ctx, SLB_ERR_CUDA, "live feeder: allocation failed"); }
  CK (ctx, cudaStreamSynchronize (ctx->stream));                  // whatever the per-call API left running is ordered before the first chunk
  *out = lv;
  return SLB_OK;
}

void slb_live_close (slb_live *lv)
{
  if (!lv) return;
  cudaSetDevice (lv->ctx->cfg.device);
  if (lv->s_in) cudaStreamSynchronize (lv->s_in);
  if (lv->s_work) cudaStreamSynchronize (lv->s_work);
  if (lv->s_out) cudaStreamSynchronize (lv->s_out);
  for (auto &sl : lv->slots)
  {
    cudaFreeHost (sl.h_adc); cudaFreeHost (sl.h_usb_out); cudaFreeHost (sl.h_usb_in); cudaFreeHost (sl.h_dac); cudaFreeHost (sl.h_plan);
    cudaFree (sl.d_adc); cudaFree (sl.d_usb_out); cudaFree (sl.d_prc); cudaFree (sl.d_usb_in); cudaFree (sl.d_dac); cudaFree (sl.d_plan);
    if (sl.in_done) cudaEventDestroy (sl.in_done);
    if (sl.work_done) cudaEventDestroy (sl.work_done);
    if (sl.out_done) cudaEventDestroy (sl.out_done);
  }
  if (lv->s_in) cudaStreamDestroy (lv->s_in);
  if (lv->s_work) cudaStreamDestroy (lv->s_work);
  if (lv->s_out) cudaStreamDestroy (lv->s_out);
  delete lv;
}

int slb_live_in_flight (const slb_live *lv) { return lv ? (int) (lv->n_pushed - lv->n_popped) : SLB_ERR_ARG; }

int slb_live_push (slb_live *lv, const int16_t *adc, const int16_t *usb_out)
{
  if (!lv || (lv->rx && !adc) || (lv->tx && !usb_out)) return SLB_ERR_ARG;
  slb_ctx *ctx = lv->ctx;
  if (lv->n_pushed - lv->n_popped >= lv->depth) return fail (ctx, SLB_ERR_STATE, "live feeder: every slot is in flight (pop first)");
  if (ctx->ring_pc) return fail (ctx, SLB_ERR_STATE, "the feeder replays one shared cadence; per-channel cadence is on");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  slb_live::Slot &sl = lv->slots[lv->n_pushed % lv->depth];
  const uint32_t ticks = lv->ticks;
  sl.pushed = std::chrono::steady_clock::now ();
  // 1. staging (pinned) and the pointer plan of every tick of the chunk — the firmware's arithmetic, on the host, in call order
  uint32_t *plan_tx = sl.h_plan, *plan_rx = sl.h_plan + (size_t) ticks * 2;
  if (lv->tx)
  {
    std::memcpy (sl.h_usb_out, usb_out, lv->bytes);
    plan_ticks (ctx->ring_out, true, plan_tx, ticks, ctx->geo.block_frames);
  }
  if (lv->rx)
  {
    std::memcpy (sl.h_adc, adc, lv->bytes);
    plan_ticks (ctx->ring_in, false, plan_rx, ticks, ctx->geo.block_frames);
  }
  // 2. copy in (stream s_in)
  CK (ctx, cudaMemcpyAsync (sl.d_plan, sl.h_plan, (size_t) ticks * 4 * sizeof (uint32_t), cudaMemcpyHostToDevice, lv->s_in));
  if (lv->tx) CK (ctx, cudaMemcpyAsync (sl.d_usb_out, sl.h_usb_out, lv->bytes, cudaMemcpyHostToDevice, lv->s_in));
  if (lv->rx) CK (ctx, cudaMemcpyAsync (sl.d_adc, sl.h_adc, lv->bytes, cudaMemcpyHostToDevice, lv->s_in));
  CK (ctx, cudaEventRecord (sl.in_done, lv->s_in));
  // 3. the chunk's kernels (stream s_work: chunks in order — chain state and rings carry from one to the next)
  CK (ctx, cudaStreamWaitEvent (lv->s_work, sl.in_done, 0));
  cudaStream_t st = lv->s_work;
  if (lv->tx) { const int rc = replay_tx (ctx, sl.d_usb_out, sl.d_dac, sl.d_plan, ticks, st); if (rc) return rc; }
  if (lv->rx) { const int rc = replay_rx (ctx, sl.d_adc, sl.d_prc, sl.d_usb_in, sl.d_plan + (size_t) ticks * 2, ticks, st); if (rc) return rc; }
  CK (ctx, cudaEventRecord (sl.work_done, st));
  // 4. copy out (stream s_out)
  CK (ctx, cudaStreamWaitEvent (lv->s_out, sl.work_done, 0));
  if (lv->tx) CK (ctx, cudaMemcpyAsync (sl.h_dac, sl.d_dac, lv->bytes, cudaMemcpyDeviceToHost, lv->s_out));
  if (lv->rx) CK (ctx, cudaMemcpyAsync (sl.h_usb_in, sl.d_usb_in, lv->bytes, cudaMemcpyDeviceToHost, lv->s_out));
  CK (ctx, cudaEventRecord (sl.out_done, lv->s_out));
  lv->n_pushed++;
  return SLB_OK;
}

int slb_live_pop (slb_live *lv, int16_t *usb_in, int16_t *dac, float *latency_us)
{
  if (!lv || (lv->rx && !usb_in) || (lv->tx && !dac)) return SLB_ERR_ARG;
  slb_ctx *ctx = lv->ctx;
  if (lv->n_pushed == lv->n_popped) return fail (ctx, SLB_ERR_STATE, "live feeder: nothing in flight");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  slb_live::Slot &sl = lv->slots[lv->n_popped % lv->depth];
  CK (ctx, cudaEventSynchronize (sl.out_done));
  if (latency_us) *latency_us = std::chrono::duration<float, std::micro> (std::chrono::steady_clock::now () - sl.pushed).count ();
  if (lv->rx) std::memcpy (usb_in, sl.h_usb_in, lv->bytes);
  if (lv->tx) std::memcpy (dac, sl.h_dac, lv->bytes);
  lv->n_popped++;
  return SLB_OK;
}

int SLB_DSP_Out_Buff_Mute (slb_ctx *ctx)                                           // dsp_if.c:188-195: zero the samples, keep the pointers
{
  if (!ctx) return SLB_ERR_ARG;
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  const size_t bytes = (size_t) ctx->cfg.channels * ctx->geo.ring_frames * 2;
  CK (ctx, cudaMemsetAsync (ctx->d_ring[1][0], 0, bytes, ctx->stream));
  CK (ctx, cudaMemsetAsync (ctx->d_ring[1][1], 0, bytes, ctx->stream));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  return SLB_OK;
}

int slb_ring_get_ptrs (const slb_ctx *ctx, int which, uint32_t out[3])
{
  if (!ctx || !out || which < 0 || which > 1) return SLB_ERR_ARG;
  const RingPtrs &rp = which ? ctx->ring_out : ctx->ring_in;
  out[0] = rp.enable; out[1] = rp.rd; out[2] = rp.wr;
  return SLB_OK;
}
int slb_ring_get_iq (slb_ctx *ctx, int which, int16_t *i, int16_t *q)
{
  if (!ctx || !i || !q || which < 0 || which > 1) return SLB_ERR_ARG;
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  const size_t bytes = (size_t) ctx->cfg.channels * ctx->geo.ring_frames * 2;
  CK (ctx, cudaMemcpy (i, ctx->d_ring[which][0], bytes, cudaMemcpyDeviceToHost));
  CK (ctx, cudaMemcpy (q, ctx->d_ring[which][1], bytes, cudaMemcpyDeviceToHost));
  return SLB_OK;
}

// one planning step of a ring whose pointers {enable, rd, wr} the caller keeps
static uint32_t ring_plan (bool write, uint32_t ring_frames, int is_out, uint32_t state[3], uint32_t frames)
{
  RingPtrs rp; rp.size = ring_frames; rp.enable = state[0]; rp.rd = state[1]; rp.wr = state[2];
  const uint32_t first = write ? rp.plan_write (is_out != 0, frames) : rp.plan_read (is_out != 0, frames);
  state[0] = rp.enable; state[1] = rp.rd; state[2] = rp.wr;
  return first;
}
uint32_t slb_ring_plan_write (uint32_t ring_frames, int is_out, uint32_t state[3], uint32_t frames) { return ring_plan (true, ring_frames, is_out, state, frames); }
uint32_t slb_ring_plan_read (uint32_t ring_frames, int is_out, uint32_t state[3], uint32_t frames) { return ring_plan (false, ring_frames, is_out, state, frames); }
int slb_biquad_scan_tables (const float coef10[10], float *Mpow96, float *Cresp96)
{
  if (!coef10 || !Mpow96 || !Cresp96) return SLB_ERR_ARG;
  BiquadScanTables t; design_biquad_scan_tables (coef10, &t);
  std::memcpy (Mpow96, t.Mpow, sizeof t.Mpow); std::memcpy (Cresp96, t.Cresp, sizeof t.Cresp);
  return SLB_OK;
}

int slb_rx_spectrum_device (slb_ctx *ctx, const int16_t *d_iq, float *d_power, uint32_t N, void *stream)
{
  if (!ctx || !d_iq || !d_power) return SLB_ERR_ARG;
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  float *tmp = static_cast<float *> (sl::ctx_scratch_on (ctx, (size_t) ctx->cfg.channels * 2 * N * sizeof (float), stream));
  if (!tmp) return SLB_ERR_CUDA;
  int rc = slb_st_q15_to_float (ctx, d_iq, tmp, 2 * N, stream);                 // arm_q15_to_float.c:65
  if (!rc) rc = slb_st_cfft_f32 (ctx, tmp, N, 1, 0, stream);                      // arm_cfft_f32.c:562, forward
  if (!rc) rc = slb_st_cmplx_mag_squared_f32 (ctx, tmp, d_power, N, stream);      // arm_cmplx_mag_squared_f32.c:70
  return rc;
}
int slb_design_tc_taps (const float *mask_re_im, double taps_re[129], double taps_im[129])
{
  if (!mask_re_im || !taps_re || !taps_im) return SLB_ERR_ARG;
  return tc_design_taps (mask_re_im, taps_re, taps_im) ? SLB_OK : SLB_ERR_UNSUPPORTED;
}
int slb_design_tc_block (const float *mask_re_im, const float coef10[10], const int16_t *window, double out52[52])
{
  if (!mask_re_im || !coef10 || !window || !out52) return SLB_ERR_ARG;
  std::vector<uint8_t> planes (kTcPlaneBytes);
  float ua = 0.f, uz = 0.f;
  if (!tc_build_planes (mask_re_im, coef10, planes.data (), &ua, &uz)) return SLB_ERR_UNSUPPORTED;
  tc_apply_planes (planes.data (), ua, uz, window, out52);
  return SLB_OK;
}
int slb_design_tc_tx_block (const float *mask_re_im, const int16_t *window, double out_iq[96])
{
  if (!mask_re_im || !window || !out_iq) return SLB_ERR_ARG;
  std::vector<uint8_t> planes (kTcTxPlaneBytes);
  float u = 0.f;
  if (!tc_build_tx_planes (mask_re_im, planes.data (), &u)) return SLB_ERR_UNSUPPORTED;
  tc_apply_tx_planes (planes.data (), u, window, out_iq);
  return SLB_OK;
}
int slb_design_q15_tc_block (const int16_t taps_i[64], const int16_t taps_q[64], const int16_t *window, int32_t out96[96])
{
  if (!taps_i || !taps_q || !window || !out96) return SLB_ERR_ARG;
  std::vector<uint8_t> planes (kTcQ15PlaneBytes);
  if (!q15_tc_build_planes (taps_i, taps_q, planes.data (), false)) return SLB_ERR_UNSUPPORTED;
  q15_tc_apply_planes (planes.data (), window, out96);
  return SLB_OK;
}
int slb_design_q15_tc_fm_block (const int16_t taps[64], const int16_t *window, int32_t out98[98])
{
  if (!taps || !window || !out98) return SLB_ERR_ARG;
  std::vector<uint8_t> planes (kTcQ15FmPlaneBytes);
  if (!q15_tc_build_fm_planes (taps, planes.data ())) return SLB_ERR_UNSUPPORTED;
  q15_tc_apply_fm_planes (planes.data (), window, out98);
  return SLB_OK;
}
int slb_design_q15_tc_tx_block (const int16_t taps_i[64], const int16_t taps_q[64], const int16_t *window, int32_t out96[96])
{
  if (!taps_i || !taps_q || !window || !out96) return SLB_ERR_ARG;
  std::vector<uint8_t> planes (kTcQ15PlaneBytes);
  if (!q15_tc_build_planes (taps_i, taps_q, planes.data (), true)) return SLB_ERR_UNSUPPORTED;
  q15_tc_apply_planes (planes.data (), window, out96);
  return SLB_OK;
}
int slb_design_mask (uint32_t fs, uint8_t mode, float *mask_re_im)
{
  if (!mask_re_im) return SLB_ERR_ARG;
  return design_default_mask (fs, 512, mode, mask_re_im) == 0 ? SLB_OK : SLB_ERR_UNSUPPORTED;
}
int slb_biquad_tc_tables (const float coef10[10], float *Mp64, float *M192, float *Cresp192)
{
  if (!coef10 || !Mp64 || !M192 || !Cresp192) return SLB_ERR_ARG;
  TcBiquadTables t; design_biquad_tc_tables (coef10, &t);
  std::memcpy (Mp64, t.Mp, sizeof t.Mp); std::memcpy (M192, t.M192, sizeof t.M192); std::memcpy (Cresp192, t.Cresp, sizeof t.Cresp);
  return SLB_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Bulk path
// ------------------------------------------------------------------------------------------------------------------
static int process_device (slb_ctx *ctx, const int16_t *d_in, int16_t *d_out, uint32_t frames, void *stream, bool want_tx)
{
  if (!ctx || !d_in || !d_out || frames == 0) return SLB_ERR_ARG;
  if (is_chan (ctx)) return fail (ctx, SLB_ERR_STATE, "channelizer context: use slb_chan_process_*");
  if (want_tx != is_tx_direction (ctx->cfg.chain)) return fail (ctx, SLB_ERR_STATE, "context was created for the other direction (cfg.chain)");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  if (ctx->cfg.chain == SLB_CHAIN_PASS)
  {
    CK (ctx, launch_copy_iq (d_in, d_out, (size_t) ctx->cfg.channels * frames, stream));
    ctx->launches++;
    return SLB_OK;
  }
  if (ctx->q15)
  {
    int rc = rxq15_launch (ctx, ctx->q15, d_in, d_out, 0, ctx->cfg.channels, frames, ctx->sm_count, stream, true);
    if (rc) return rc;
    rxq15_advance (ctx->q15);
    return SLB_OK;
  }
  if (frames % ctx->rx.hop != 0) return fail (ctx, SLB_ERR_ARG, "frames must be a multiple of the hop (384)");
  int rc = run_rx_kernel (ctx, d_in, d_out, 0, ctx->cfg.channels, frames, ctx->dbg_audio, ctx->dbg_gain, (cudaStream_t) stream, false, ctx->dbg_phase);
  if (rc) return rc;
  rx_advance (ctx, frames);
  return SLB_OK;
}

int slb_rx_process_device (slb_ctx *ctx, const int16_t *d_in, int16_t *d_out, uint32_t frames, void *stream) { return process_device (ctx, d_in, d_out, frames, stream, false); }
int slb_tx_process_device (slb_ctx *ctx, const int16_t *d_in, int16_t *d_out, uint32_t frames, void *stream) { return process_device (ctx, d_in, d_out, frames, stream, true); }

// Staging of the host bulk paths: kBulkSlots slots of two device buffers of at least `bytes` each, and one stream per slot
static int ensure_bulk (slb_ctx *ctx, size_t bytes)
{
  if (bytes <= ctx->bulk_bytes && ctx->bulk_stream[0]) return SLB_OK;
  for (int s = 0; s < kBulkSlots; s++)
  {
    if (ctx->bulk_stream[s]) CK (ctx, cudaStreamSynchronize (ctx->bulk_stream[s]));
    if (bytes > ctx->bulk_bytes)
    {
      CK (ctx, cudaFree (ctx->d_bulk_in[s])); CK (ctx, cudaFree (ctx->d_bulk_out[s]));
      ctx->d_bulk_in[s] = ctx->d_bulk_out[s] = nullptr;
      CK (ctx, cudaMalloc (&ctx->d_bulk_in[s], bytes)); CK (ctx, cudaMalloc (&ctx->d_bulk_out[s], bytes));
    }
    if (!ctx->bulk_stream[s]) CK (ctx, cudaStreamCreateWithFlags (&ctx->bulk_stream[s], cudaStreamNonBlocking));
  }
  ctx->bulk_bytes = std::max (ctx->bulk_bytes, bytes);
  return SLB_OK;
}

// Chains whose channels (or channelizer streams) are independent, through host buffers: the batch is cut into groups of at most
// 48 MiB, and H2D / kernel / D2H of consecutive groups overlap, round-robin over the slot streams. launch (d_in, d_out, c0, n, stream)
// runs the chain on the n channels from c0 staged in d_in.
using GroupLaunch = std::function<int (const int16_t *, int16_t *, uint32_t, uint32_t, cudaStream_t)>;
static int process_host_groups (slb_ctx *ctx, const int16_t *h_in, int16_t *h_out, uint32_t frames, const GroupLaunch &launch)
{
  const uint32_t C = ctx->cfg.channels;
  const size_t ch_bytes = (size_t) frames * 4;          // per channel, in and out alike
  uint32_t group = (uint32_t) ((size_t) (48u << 20) / ch_bytes);
  if (group < 1) group = 1;
  if (group > C) group = C;
  { const int rc = ensure_bulk (ctx, (size_t) group * ch_bytes); if (rc) return rc; }
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  int slot = 0;
  for (uint32_t c0 = 0; c0 < C; c0 += group, slot = (slot + 1) % kBulkSlots)
  {
    const uint32_t n = (C - c0 < group) ? C - c0 : group;
    cudaStream_t st = ctx->bulk_stream[slot];
    const size_t off = (size_t) c0 * ch_bytes, bytes = (size_t) n * ch_bytes;
    CK (ctx, cudaMemcpyAsync (ctx->d_bulk_in[slot], reinterpret_cast<const char *> (h_in) + off, bytes, cudaMemcpyHostToDevice, st));
    { const int rc = launch (ctx->d_bulk_in[slot], ctx->d_bulk_out[slot], c0, n, st); if (rc) return rc; }
    CK (ctx, cudaMemcpyAsync (reinterpret_cast<char *> (h_out) + off, ctx->d_bulk_out[slot], bytes, cudaMemcpyDeviceToHost, st));
  }
  for (int s = 0; s < kBulkSlots; s++) CK (ctx, cudaStreamSynchronize (ctx->bulk_stream[s]));
  return SLB_OK;
}

// SSB chains (f32 and q15) through host buffers: the batch is cut in TIME. Every slice carries all channels (strided 2-D copies
// straight from / to the caller's [channels][frames] arrays), so each launch is as wide as the batch — the tensor-core
// kernel wants one channel group per SM — and the slices are small (~64 MB), so the copy that cannot overlap anything (the
// first H2D, the last D2H) is a few per cent of the call. Slices of one stream depend on each other through the carried
// state: the kernels run in order on one stream, copies on two others, three staging slots in flight.
static int process_host_sliced (slb_ctx *ctx, const int16_t *h_in, int16_t *h_out, uint32_t frames)
{
  const uint32_t C = ctx->cfg.channels;
  // The batch is cut into tiles = (block of channels) x (slice of time) that go through a three-stream pipeline: H2D of tile i + 1,
  // kernel of tile i and D2H of tile i - 1 overlap. Time cuts are multiples of 1536 frames = the FFT kernel's tile and two
  // supertiles of the tensor-core kernel: both kernels give the cut stream bit for bit the result of the uncut one (the carried
  // state lives per channel on the device). Tile size: the pipeline's fill and drain (one tile's H2D before, one tile's D2H after)
  // are what separates this path from the plain duplex copy of the same bytes; measured at 1024 channels x 10 s
  // (tools/bench_e2e_slices.py, profiles/r02_e2e_slices.json): 4 / 8 MiB 0.975 of that ceiling, 32 MiB 0.957, 64 MiB 0.921,
  // 256 MiB 0.888. Wide batches (config 5: 32 768 channels per GPU, where the shortest time slice of ALL channels is 201 MB) are
  // cut into blocks of 1024 channels as well; the kernels take a channel range like under per-channel cadence.
  size_t tile_bytes = (size_t) 8 << 20;
  if (const char *e = std::getenv ("SELENITE_B200_SLICE_BYTES")) { const long long v = std::atoll (e); if (v > 0) tile_bytes = (size_t) v; }   // test / tuning knob
  uint32_t block = C;
  if (C > 1024u && (size_t) C * 1536u * 4u > tile_bytes) block = 1024u;
  if (const char *e = std::getenv ("SELENITE_B200_SLICE_CHANNELS")) { const long v = std::atol (e); if (v > 0 && (uint32_t) v < C) block = (uint32_t) v; }   // test knob
  uint32_t slice = (uint32_t) std::min<size_t> (tile_bytes / ((size_t) block * 4), 0xFFFFFFFFu) / 1536u * 1536u;
  if (slice < 1536u) slice = 1536u;
  if (slice > frames) slice = frames;
  { const int rc = ensure_bulk (ctx, (size_t) block * slice * 4); if (rc) return rc; }
  for (int s = 0; s < kBulkSlots; s++)
    for (int e = 0; e < 3; e++)
      if (!ctx->slice_ev[s][e]) CK (ctx, cudaEventCreateWithFlags (&ctx->slice_ev[s][e], cudaEventDisableTiming));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  cudaStream_t s_in = ctx->bulk_stream[0], s_k = ctx->bulk_stream[1], s_out = ctx->bulk_stream[2];
  const size_t pitch = (size_t) frames * 4;
  uint32_t n_tiles = 0;
  for (uint32_t t0 = 0; t0 < frames; t0 += slice)
  {
    const uint32_t n = (frames - t0 < slice) ? frames - t0 : slice;
    const size_t row = (size_t) n * 4;
    for (uint32_t c0 = 0; c0 < C; c0 += block, n_tiles++)
    {
      const int slot = (int) (n_tiles % kBulkSlots);
      const uint32_t nc = (C - c0 < block) ? C - c0 : block;
      const size_t host_off = ((size_t) c0 * frames + t0) * 4;
      if (n_tiles >= (uint32_t) kBulkSlots) CK (ctx, cudaStreamWaitEvent (s_in, ctx->slice_ev[slot][2], 0));   // the slot's previous result has left
      CK (ctx, cudaMemcpy2DAsync (ctx->d_bulk_in[slot], row, reinterpret_cast<const char *> (h_in) + host_off, pitch, row, nc, cudaMemcpyHostToDevice, s_in));
      CK (ctx, cudaEventRecord (ctx->slice_ev[slot][0], s_in));
      CK (ctx, cudaStreamWaitEvent (s_k, ctx->slice_ev[slot][0], 0));
      if (ctx->q15)
      {
        const int rc = rxq15_launch (ctx, ctx->q15, ctx->d_bulk_in[slot], ctx->d_bulk_out[slot], c0, nc, n, ctx->sm_count, s_k, false); if (rc) return rc;
      }
      else
      {
        const int rc = run_rx_kernel (ctx, ctx->d_bulk_in[slot], ctx->d_bulk_out[slot], c0, nc, n, nullptr, nullptr, s_k, true); if (rc) return rc;
      }
      CK (ctx, cudaEventRecord (ctx->slice_ev[slot][1], s_k));
      CK (ctx, cudaStreamWaitEvent (s_out, ctx->slice_ev[slot][1], 0));
      CK (ctx, cudaMemcpy2DAsync (reinterpret_cast<char *> (h_out) + host_off, pitch, ctx->d_bulk_out[slot], row, row, nc, cudaMemcpyDeviceToHost, s_out));
      CK (ctx, cudaEventRecord (ctx->slice_ev[slot][2], s_out));
    }
    // every channel has taken this time slice: host bookkeeping of the carried state (the launches are stream-ordered)
    if (ctx->q15) rxq15_advance (ctx->q15); else rx_advance (ctx, n);
  }
  for (int s = 0; s < kBulkSlots; s++) CK (ctx, cudaStreamSynchronize (ctx->bulk_stream[s]));
  return SLB_OK;
}

static int process_host (slb_ctx *ctx, const int16_t *h_in, int16_t *h_out, uint32_t frames, bool want_tx)
{
  if (!ctx || !h_in || !h_out || frames == 0) return SLB_ERR_ARG;
  if (is_chan (ctx)) return fail (ctx, SLB_ERR_STATE, "channelizer context: use slb_chan_process_*");
  if (want_tx != is_tx_direction (ctx->cfg.chain)) return fail (ctx, SLB_ERR_STATE, "context was created for the other direction (cfg.chain)");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  const bool chain = is_ssb_chain (ctx->cfg.chain);
  if (chain && frames % ctx->rx.hop != 0) return fail (ctx, SLB_ERR_ARG, "frames must be a multiple of the hop (384)");
  if (ctx->q15 && frames % ctx->geo.block_frames != 0) return fail (ctx, SLB_ERR_ARG, "frames must be a multiple of the 48-frame firmware block");
  if (chain || ctx->q15) return process_host_sliced (ctx, h_in, h_out, frames);   // (the integer chain is exact, so any cut at a block boundary reproduces the uncut stream)
  // PASS (the firmware as shipped)
  return process_host_groups (ctx, h_in, h_out, frames, [&] (const int16_t *d_in, int16_t *d_out, uint32_t, uint32_t n, cudaStream_t st) -> int {
    CK (ctx, launch_copy_iq (d_in, d_out, (size_t) n * frames, st));
    ctx->launches++;
    return SLB_OK;
  });
}
int slb_rx_process_host (slb_ctx *ctx, const int16_t *h_in, int16_t *h_out, uint32_t frames) { return process_host (ctx, h_in, h_out, frames, false); }
int slb_tx_process_host (slb_ctx *ctx, const int16_t *h_in, int16_t *h_out, uint32_t frames) { return process_host (ctx, h_in, h_out, frames, true); }

// ------------------------------------------------------------------------------------------------------------------
// Channelizer bulk path (SLB_CHAIN_CHAN64_F32, SLB_CHAIN_CHAN64_Q15)
// ------------------------------------------------------------------------------------------------------------------
int slb_default_chan_params (uint32_t fs, slb_chan_params *out) { return design_default_chan (fs, out); }
int slb_set_chan_params (slb_ctx *ctx, const slb_chan_params *p)
{
  if (!ctx || !p) return SLB_ERR_ARG;
  if (!ctx->chan) return fail (ctx, SLB_ERR_STATE, "not a channelizer context");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  CK (ctx, cudaDeviceSynchronize ());
  return chan64_set_params (ctx, ctx->chan, p);
}
int slb_get_chan_params (const slb_ctx *ctx, slb_chan_params *p)
{
  if (!ctx || !p || !ctx->chan) return SLB_ERR_ARG;
  *p = *chan64_params (ctx->chan);
  return SLB_OK;
}
int slb_default_chan_q15_params (uint32_t fs, slb_chan_q15_params *out) { return design_default_chan_q15 (fs, out); }
int slb_set_chan_q15_params (slb_ctx *ctx, const slb_chan_q15_params *p)
{
  if (!ctx || !p) return SLB_ERR_ARG;
  if (!ctx->chanq) return fail (ctx, SLB_ERR_STATE, "not a CHAN-64-q15 context");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  CK (ctx, cudaDeviceSynchronize ());
  return chanq15_set_params (ctx, ctx->chanq, p);
}
int slb_get_chan_q15_params (const slb_ctx *ctx, slb_chan_q15_params *p)
{
  if (!ctx || !p) return SLB_ERR_ARG;
  if (!ctx->chanq) return SLB_ERR_STATE;
  *p = *chanq15_params (ctx->chanq);
  return SLB_OK;
}
int slb_chan_process_device (slb_ctx *ctx, const int16_t *d_in, int16_t *d_out, uint32_t frames, void *stream)
{
  if (!ctx || !d_in || !d_out || frames == 0) return SLB_ERR_ARG;
  if (!is_chan (ctx)) return fail (ctx, SLB_ERR_STATE, "not a channelizer context (cfg.chain)");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  if (ctx->chanq)
  {
    const int rc = chanq15_launch (ctx, ctx->chanq, d_in, d_out, 0, ctx->cfg.channels, frames, ctx->sm_count, stream, true);
    if (rc) return rc;
    chanq15_advance (ctx->chanq);
    return SLB_OK;
  }
  int rc = chan64_launch (ctx, ctx->chan, d_in, d_out, 0, ctx->cfg.channels, frames, ctx->sm_count, stream, true);
  if (rc) return rc;
  chan64_advance (ctx->chan);
  return SLB_OK;
}
int slb_chan_process_host (slb_ctx *ctx, const int16_t *h_in, int16_t *h_out, uint32_t frames)
{
  if (!ctx || !h_in || !h_out || frames == 0) return SLB_ERR_ARG;
  if (!is_chan (ctx)) return fail (ctx, SLB_ERR_STATE, "not a channelizer context (cfg.chain)");
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  // (a stream takes as many bytes out as in: 64 bins x frames/64 x 4 B)
  const int rc = process_host_groups (ctx, h_in, h_out, frames, [&] (const int16_t *d_in, int16_t *d_out, uint32_t s0, uint32_t n, cudaStream_t st) {
    return ctx->chanq ? chanq15_launch (ctx, ctx->chanq, d_in, d_out, s0, n, frames, ctx->sm_count, st, false)
                      : chan64_launch (ctx, ctx->chan, d_in, d_out, s0, n, frames, ctx->sm_count, st, false);
  });
  if (rc) return rc;
  if (ctx->chanq) chanq15_advance (ctx->chanq); else chan64_advance (ctx->chan);
  return SLB_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Checkpoint: everything a later call depends on
// ------------------------------------------------------------------------------------------------------------------
namespace {
struct StateHeader
{
  uint32_t magic, channels, fs, chain, fft_len, hop;
  uint32_t flag_base, ovl_parity, acc_fill, proc_cur, tx_mode;
  uint32_t ring[2][4];
  uint32_t ring_pc;                          // 1: the per-channel pointer tables at the end of the blob are live
};
constexpr uint32_t kMagic = 0x534C4233u;   // 'SLB3'
}
// The device sections of the blob, in blob order (after the header and the mode bytes): the raw-input tail, the state records, the
// four ring planes, the super-block being accumulated and the one processed last. The ping-pong buffers are saved from the current
// side; a load resets ovl_parity and proc_cur to 0 first and so restores into side 0.
struct StateSection { void *d; size_t bytes; };
static std::vector<StateSection> state_sections (const slb_ctx *ctx)
{
  const size_t C = ctx->cfg.channels, ovl = ctx->rx.fft_len - ctx->rx.hop, hop = ctx->rx.hop, R = ctx->geo.ring_frames;
  std::vector<StateSection> s = { { ctx->d_ovl[ctx->ovl_parity], C * ovl * 4 }, { ctx->d_state, C * 8 * 4 } };
  for (int w = 0; w < 2; w++) for (int k = 0; k < 2; k++) s.push_back ({ ctx->d_ring[w][k], C * R * 2 });
  s.push_back ({ ctx->d_acc, C * hop * 4 });
  s.push_back ({ ctx->d_proc[ctx->proc_cur], C * hop * 4 });
  return s;
}
static size_t state_bytes (const slb_ctx *ctx)
{
  const size_t C = ctx->cfg.channels;
  size_t n = sizeof (StateHeader) + C /*modes*/;
  for (const StateSection &s : state_sections (ctx)) n += s.bytes;
  return n + (ctx->chan ? chan64_state_bytes (ctx->chan) : 0) + (ctx->chanq ? chanq15_state_bytes (ctx->chanq) : 0) + (ctx->q15 ? rxq15_state_bytes (ctx->q15) : 0) + 2 * C * 4 * sizeof (uint32_t) /* per-channel ring pointers */;
}
int slb_state_size (const slb_ctx *ctx, size_t *bytes) { if (!ctx || !bytes) return SLB_ERR_ARG; *bytes = state_bytes (ctx); return SLB_OK; }

int slb_state_save (slb_ctx *ctx, void *buf, size_t bytes)
{
  if (!ctx || !buf || bytes < state_bytes (ctx)) return SLB_ERR_ARG;
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  const size_t C = ctx->cfg.channels;
  char *p = static_cast<char *> (buf);
  StateHeader h{};
  h.magic = kMagic; h.channels = (uint32_t) C; h.fs = ctx->cfg.fs; h.chain = ctx->cfg.chain; h.fft_len = ctx->rx.fft_len; h.hop = ctx->rx.hop;
  h.flag_base = ctx->flag_base; h.ovl_parity = (uint32_t) ctx->ovl_parity; h.acc_fill = ctx->acc_fill; h.proc_cur = (uint32_t) ctx->proc_cur; h.tx_mode = ctx->tx_mode;
  const RingPtrs *rp[2] = { &ctx->ring_in, &ctx->ring_out };
  for (int w = 0; w < 2; w++) { h.ring[w][0] = rp[w]->size; h.ring[w][1] = rp[w]->enable; h.ring[w][2] = rp[w]->rd; h.ring[w][3] = rp[w]->wr; }
  h.ring_pc = ctx->ring_pc ? 1u : 0u;
  std::memcpy (p, &h, sizeof h); p += sizeof h;
  std::memcpy (p, ctx->mode_host.data (), C); p += C;
  for (const StateSection &s : state_sections (ctx)) { CK (ctx, cudaMemcpy (p, s.d, s.bytes, cudaMemcpyDeviceToHost)); p += s.bytes; }
  if (ctx->chan) { CK (ctx, cudaDeviceSynchronize ()); if (chan64_state_save (ctx->chan, p)) return fail (ctx, SLB_ERR_CUDA, "chan64 state save failed"); p += chan64_state_bytes (ctx->chan); }
  if (ctx->chanq) { CK (ctx, cudaDeviceSynchronize ()); if (chanq15_state_save (ctx->chanq, p)) return fail (ctx, SLB_ERR_CUDA, "chan64-q15 state save failed"); p += chanq15_state_bytes (ctx->chanq); }
  if (ctx->q15) { CK (ctx, cudaDeviceSynchronize ()); if (rxq15_state_save (ctx->q15, p)) return fail (ctx, SLB_ERR_CUDA, "RX-SSB-q15 state save failed"); p += rxq15_state_bytes (ctx->q15); }
  for (int w = 0; w < 2; w++)
  {
    if (ctx->ring_pc) CK (ctx, cudaMemcpy (p, ctx->d_rptr[w], C * 4 * sizeof (uint32_t), cudaMemcpyDeviceToHost));
    else std::memset (p, 0, C * 4 * sizeof (uint32_t));
    // (the 4th word of a pointer record is per-call scratch: in the checkpoint it carries the channel's own super-block fill level)
    if (w == 0 && ctx->ring_pc && ctx->acc_fill_pc.size () == C)
      for (size_t c = 0; c < C; c++) std::memcpy (p + (4 * c + 3) * sizeof (uint32_t), &ctx->acc_fill_pc[c], sizeof (uint32_t));
    p += C * 4 * sizeof (uint32_t);
  }
  return SLB_OK;
}

int slb_state_load (slb_ctx *ctx, const void *buf, size_t bytes)
{
  if (!ctx || !buf || bytes < state_bytes (ctx)) return SLB_ERR_ARG;
  CK (ctx, cudaSetDevice (ctx->cfg.device));
  const size_t C = ctx->cfg.channels;
  const char *p = static_cast<const char *> (buf);
  StateHeader h; std::memcpy (&h, p, sizeof h); p += sizeof h;
  if (h.magic != kMagic || h.channels != C || h.fs != ctx->cfg.fs || h.chain != ctx->cfg.chain || h.fft_len != ctx->rx.fft_len || h.hop != ctx->rx.hop)
    return fail (ctx, SLB_ERR_STATE, "checkpoint does not match this context");
  CK (ctx, cudaStreamSynchronize (ctx->stream));
  for (size_t c = 0; c < C; c++) { ctx->mode_host[c] = (uint8_t) p[c]; int s = mode_to_mask_slot (ctx->mode_host[c]); ctx->slot_host[c] = (uint8_t) (s < 0 ? 1 : s); }
  ctx->mode_version++;
  p += C;
  CK (ctx, cudaMemcpy (ctx->d_slot, ctx->slot_host.data (), C, cudaMemcpyHostToDevice));
  ctx->ovl_parity = 0; ctx->proc_cur = 0;
  for (const StateSection &s : state_sections (ctx)) { CK (ctx, cudaMemcpy (s.d, p, s.bytes, cudaMemcpyHostToDevice)); p += s.bytes; }
  if (ctx->chan) { CK (ctx, cudaDeviceSynchronize ()); if (chan64_state_load (ctx->chan, p)) return fail (ctx, SLB_ERR_CUDA, "chan64 state load failed"); p += chan64_state_bytes (ctx->chan); }
  if (ctx->chanq) { CK (ctx, cudaDeviceSynchronize ()); if (chanq15_state_load (ctx->chanq, p)) return fail (ctx, SLB_ERR_CUDA, "chan64-q15 state load failed"); p += chanq15_state_bytes (ctx->chanq); }
  if (ctx->q15) { CK (ctx, cudaDeviceSynchronize ()); if (rxq15_state_load (ctx->q15, p)) return fail (ctx, SLB_ERR_CUDA, "RX-SSB-q15 state load failed"); p += rxq15_state_bytes (ctx->q15); }
  ctx->ring_pc = false;
  if (h.ring_pc)
  {
    int rc = ring_pc_enable (ctx); if (rc) return rc;
    for (int w = 0; w < 2; w++)
    {
      CK (ctx, cudaMemcpy (ctx->d_rptr[w], p, C * 4 * sizeof (uint32_t), cudaMemcpyHostToDevice));
      if (w == 0 && ctx->acc_fill_pc.size () == C)
        for (size_t c = 0; c < C; c++) std::memcpy (&ctx->acc_fill_pc[c], p + (4 * c + 3) * sizeof (uint32_t), sizeof (uint32_t));
      p += C * 4 * sizeof (uint32_t);
    }
  }
  // per-channel tile counters restart from zero on this context
  CK (ctx, cudaMemset (ctx->d_flag, 0, C * sizeof (unsigned)));
  ctx->flag_base = 0; ctx->acc_fill = h.acc_fill; ctx->tx_mode = h.tx_mode != 0;
  RingPtrs *rp[2] = { &ctx->ring_in, &ctx->ring_out };
  for (int w = 0; w < 2; w++) { rp[w]->size = h.ring[w][0]; rp[w]->enable = h.ring[w][1]; rp[w]->rd = h.ring[w][2]; rp[w]->wr = h.ring[w][3]; }
  return SLB_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Single-channel drop-in with the firmware's names (Core/Inc/dsp_if.h:42-51)
// ------------------------------------------------------------------------------------------------------------------
namespace {
slb_ctx *g_dropin = nullptr;
int g_dropin_status = SLB_OK;
std::mutex g_dropin_mu;
slb_ctx *dropin ()
{
  std::lock_guard<std::mutex> lk (g_dropin_mu);
  if (!g_dropin)
  {
    slb_config cfg{};
    cfg.channels = 1;
    const char *fs = std::getenv ("SELENITE_B200_FS"), *dev = std::getenv ("SELENITE_B200_DEVICE"), *ch = std::getenv ("SELENITE_B200_CHAIN");
    cfg.fs = fs ? (uint32_t) std::atoi (fs) : 48000u;
    cfg.device = dev ? std::atoi (dev) : 0;
    cfg.chain = (ch && std::strcmp (ch, "rx_ssb_f32") == 0) ? SLB_CHAIN_RX_SSB_F32 : (ch && std::strcmp (ch, "tx_ssb_f32") == 0) ? SLB_CHAIN_TX_SSB_F32
              : (ch && std::strcmp (ch, "tx_f32") == 0) ? SLB_CHAIN_TX_F32
              : (ch && std::strcmp (ch, "rx_ssb_q15") == 0) ? SLB_CHAIN_RX_SSB_Q15
              : (ch && std::strcmp (ch, "tx_ssb_q15") == 0) ? SLB_CHAIN_TX_SSB_Q15
              : (ch && std::strcmp (ch, "rx_q15") == 0) ? SLB_CHAIN_RX_Q15
              : (ch && std::strcmp (ch, "tx_q15") == 0) ? SLB_CHAIN_TX_Q15 : SLB_CHAIN_PASS;   // (the channelizer has no single-channel drop-in)
    g_dropin_status = slb_create (&cfg, &g_dropin);
    if (g_dropin_status != SLB_OK) std::fprintf (stderr, "selenite-b200: drop-in context failed: %s\n", slb_last_error (nullptr));
  }
  return g_dropin;
}
}  // namespace

int slb_dropin_status (void) { return g_dropin_status; }
slb_ctx *slb_dropin_ctx (void) { return dropin (); }
#define DROPIN(call) do { slb_ctx *c_ = dropin (); if (c_) g_dropin_status = (call); } while (0)
void DSP_Init (void) { DROPIN (SLB_DSP_Init (c_)); }
void DSP_Set_RX (void) { DROPIN (SLB_DSP_Set_RX (c_)); }
void DSP_Set_TX (void) { DROPIN (SLB_DSP_Set_TX (c_)); }
void DSP_Set_Mode (uint8_t mode) { DROPIN (SLB_DSP_Set_Mode (c_, mode)); }
void DSP_In_Buff_Write (uint16_t *pbuf, uint16_t size) { DROPIN (SLB_DSP_In_Buff_Write (c_, pbuf, size)); }
void DSP_In_Buff_Read (uint8_t *pbuf, uint32_t size) { DROPIN (SLB_DSP_In_Buff_Read (c_, pbuf, size)); }
void DSP_Out_Buff_Write (uint8_t *pbuf, uint32_t size) { DROPIN (SLB_DSP_Out_Buff_Write (c_, pbuf, size)); }
void DSP_Out_Buff_Read (uint16_t *pbuf, uint16_t size) { DROPIN (SLB_DSP_Out_Buff_Read (c_, pbuf, size)); }
void DSP_Out_Buff_Mute (void) { DROPIN (SLB_DSP_Out_Buff_Mute (c_)); }

// the I2S DMA double buffer and its completion callbacks (dsp_if.c:32, :50-67) and the USB class dispatcher
SLB_I2S_Buff_TypeDef i2s_buff;   // storage for the largest geometry; rx at 0, tx at I2S_BUFF_SIZE of the context's rate (dsp_if.h:75-79)
void HAL_I2SEx_TxRxHalfCpltCallback (void *)
{
  slb_ctx *c = dropin (); if (!c) return;
  const uint16_t half = (uint16_t) c->geo.i2s_half_hw;
  uint16_t *rx = i2s_buff.words, *tx = i2s_buff.words + 2u * half;
  DSP_Out_Buff_Read (tx, half);
  DSP_In_Buff_Write (rx, half);
}
void HAL_I2SEx_TxRxCpltCallback (void *)
{
  slb_ctx *c = dropin (); if (!c) return;
  const uint16_t half = (uint16_t) c->geo.i2s_half_hw;
  uint16_t *rx = i2s_buff.words, *tx = i2s_buff.words + 2u * half;
  DSP_Out_Buff_Read (&tx[half], half);
  DSP_In_Buff_Write (&rx[half], half);
}
int8_t AUDIO_AudioCmd_FS (uint8_t *pbuf, uint32_t size, uint8_t cmd) { DROPIN (SLB_AUDIO_AudioCmd (c_, pbuf, size, cmd)); return 0; /* USBD_OK, unconditionally (usbd_audio_if.c:200) */ }

}  // extern "C"
