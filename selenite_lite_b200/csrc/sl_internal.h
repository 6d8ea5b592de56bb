// Internal declarations shared by the host library and the CUDA translation units.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>
#define SLB_BUILDING_LIBRARY 1   /* i2s_buff is declared as raw storage inside the library (include/selenite_b200.h) */
#include "../../include/selenite_b200.h"

namespace sl {

// ---------------------------------------------------------------------------------------------------------
// Geometry of the firmware buffers, Core/Inc/dsp_if.h:69-85 with AUDIO_OUT_PACKET_NUM = 2 (usbd_audio.h:53).
// ---------------------------------------------------------------------------------------------------------
struct Geometry
{
  uint32_t fs;
  uint32_t block_frames;     // DSP_BUFF_PACKET_SIZE      = fs / 1000          (48)
  uint32_t i2s_half_hw;      // I2S_BUFF_HALF_SIZE        = 2 * fs / 1000      (96 half-words)
  uint32_t ring_frames;      // DSP_BUFF_SIZE             = 8 * fs / 1000      (384)
  explicit Geometry (uint32_t fs_) : fs (fs_), block_frames (fs_ / 1000u), i2s_half_hw (2u * fs_ / 1000u), ring_frames (8u * fs_ / 1000u) {}
};

// ---------------------------------------------------------------------------------------------------------
// Host-side index logic of one firmware ring (DSP_Buff_TypeDef, dsp_if.h:87-94). Sample storage is on the GPU;
// all channels of a context share one cadence, hence one set of pointers. plan_*() advance the pointers exactly
// as Core/Src/dsp_if.c does and return where the kernel must put / fetch the frames.
// ---------------------------------------------------------------------------------------------------------
struct RingPtrs
{
  uint32_t size = 0, enable = 0, rd = 0, wr = 0;
  void reset (uint32_t n) { size = n; enable = 0; rd = 0; wr = 0; }
  // returns the ring index the first frame of the block is stored at; `frames`+1 slots get written (last frame twice)
  uint32_t plan_write (bool is_out, uint32_t frames);
  // returns the ring index the first frame is read from
  uint32_t plan_read (bool is_out, uint32_t frames);
};

// ---------------------------------------------------------------------------------------------------------
// Frozen default design (sl_design.cpp)
// ---------------------------------------------------------------------------------------------------------
int design_default_rx_f32 (uint32_t fs, slb_rx_f32_params *out);
int design_default_tx_f32 (uint32_t fs, slb_tx_f32_params *out);
int design_default_tx_mod (uint32_t fs, slb_tx_mod_params *out);
int design_default_mask (uint32_t fs, uint32_t fft_len, uint8_t mode, float *mask_out);
int mode_to_mask_slot (uint8_t mode);   // -1 for a byte that is no FT-817 mode
constexpr int kAmMaskSlot = 6;          // channels on this slot use the envelope detector (arm_cmplx_mag_f32) instead of Re
constexpr int kFmMaskSlot = 7;          // channels on this slot use the limiter-discriminator (complex-detector tensor-core kernel only)
constexpr float kFmFloor = 9.765625e-4f;     // FM soft squelch: |z[n] conj z[n-1]| below this (no carrier, filter start-up) divides by this instead (oracle: SLO_FM_FLOOR)

// Tables the time-parallel biquad needs, derived in double from the 2-stage df2T coefficients (sl_design.cpp).
constexpr int kRun = 24;                // samples per run; a lane of the recurrence warp carries two runs = one AGC block
constexpr int kAgcBlock = 2 * kRun;     // 48 frames = the firmware block at 48 kHz
struct BiquadScanTables
{
  float coef[10];                       // stage 0 {b0,b1,b2,a1,a2}, stage 1 {...}
  float Mpow[6][16];                    // (A^kRun)^(2^k), k = 0..5, row-major 4x4, state order {d1_0,d2_0,d1_1,d2_1}
  float Cresp[kRun][4];                 // zero-input response of the cascade output at sample n of a run per unit state
};
void design_biquad_scan_tables (const float *coef10, BiquadScanTables *t);

// ---------------------------------------------------------------------------------------------------------
// Kernel launchers (sl_ring.cu, sl_rx_ssb_f32.cu). All return cudaError_t as int.
// ---------------------------------------------------------------------------------------------------------
int launch_ring_write (const int16_t *d_blocks, uint32_t block_stride_frames, int16_t *d_ring_i, int16_t *d_ring_q,
                       uint32_t channels, uint32_t ring_frames, uint32_t wr0, uint32_t frames, void *stream);
int launch_ring_read (int16_t *d_blocks, const int16_t *d_ring_i, const int16_t *d_ring_q, uint32_t channels,
                      uint32_t ring_frames, uint32_t rd0, uint32_t frames, void *stream);
int launch_copy_iq (const int16_t *d_in, int16_t *d_out, size_t n_frames_total, void *stream);
// stream feeder: `ticks` firmware ticks of one ring in one launch; d_plan = [ticks][2] {first slot written, first slot read}
int launch_ring_replay (bool write_first, const int16_t *src_a, uint32_t stride_a_frames, uint32_t ticks_a, const int16_t *src_b,
                        uint32_t stride_b_frames, int16_t *dst, int16_t *d_ring_i, int16_t *d_ring_q, uint32_t channels, uint32_t ring_frames,
                        const uint32_t *d_plan, uint32_t ticks, uint32_t block_frames, void *stream);
// per-channel cadence: d_ptr = [C][4] {enable, rd, wr, first slot of this call | 0xFFFFFFFF when skipped}
int launch_ring_plan (uint32_t *d_ptr, const uint8_t *d_active, uint32_t channels, uint32_t ring_frames, bool is_write, bool is_out,
                      uint32_t frames, void *stream);
int launch_ring_write_pc (const int16_t *d_blocks, uint32_t block_stride_frames, int16_t *d_ring_i, int16_t *d_ring_q, uint32_t channels,
                          uint32_t ring_frames, const uint32_t *d_ptr, uint32_t frames, void *stream, const uint32_t *d_src_off = nullptr);
int launch_acc_store_pc (int16_t *d_acc, uint32_t acc_stride_frames, const int16_t *d_blocks, uint32_t channels, uint32_t frames, const uint32_t *d_off,
                         const uint32_t *d_ptr, void *stream);
int launch_fill_u32 (uint32_t *d, uint32_t n, uint32_t v, void *stream);
int launch_ring_read_pc (int16_t *d_blocks, const int16_t *d_ring_i, const int16_t *d_ring_q, uint32_t channels, uint32_t ring_frames,
                         const uint32_t *d_ptr, uint32_t frames, void *stream);

// CW side-tone (the hook "mix CW tone to speaker signal here", dsp_if.c:218). d_tone = one second of the tone as q15
// ([fs] samples: arm_sin_f32 (k * 2 pi / fs) -> arm_scale_f32 (level) -> arm_float_to_q15), built once by launch_tone_table;
// launch_sidetone_mix adds tone[(cnt + n f) mod fs] to both words of frame n of every keyed channel (arm_add_q15, saturating)
// and advances the channel's phase counter; a channel whose key is up has its counter reset (every element starts at phase 0).
// d_first (per-channel cadence, may be null) = the [C][4] pointer words whose 4th entry is 0xFFFFFFFF for a channel skipped this call.
int launch_tone_table (int16_t *d_tone, uint32_t fs, float level, const float *d_sin513, void *stream);
int launch_sidetone_mix (int16_t *d_blocks, uint32_t channels, uint32_t frames, const uint8_t *d_key, uint32_t *d_cnt, const uint32_t *d_first,
                         const int16_t *d_tone, uint32_t freq_hz, uint32_t fs, void *stream);
const float *host_sin_table ();
// fixed-point FFTs (sl_fft_fixed.cu): regenerated twiddle tables (host, cached) and the batched transforms
const int16_t *fft_twiddle_q15 (uint32_t N);
const int32_t *fft_twiddle_q31 (uint32_t N);
int launch_cfft_q15 (int16_t *d_data, uint32_t N, size_t transforms, int ifft, const int16_t *d_tw, void *stream);
int launch_cfft_q31 (int32_t *d_data, uint32_t N, size_t transforms, int ifft, const int32_t *d_tw, void *stream);

struct RxF32Launch
{
  const int16_t *in; int16_t *out;         // [C][T][2]
  float *audio_dbg; float *gain_dbg;       // optional taps
  const int16_t *ovl_in; int16_t *ovl_out; // [C][ovl][2] carried raw-input tail (ping-pong between calls)
  float *state;                            // [C][8] {d1_0,d2_0,d1_1,d2_1,env,-,-,-}
  unsigned *flag;                          // [C] tiles completed, monotonically increasing across calls
  const float *masks;                      // [SLB_MAX_MASKS][2*fft_len] in the kernel's packed layout (rx_ssb_f32_pack_mask)
  const uint8_t *mask_slot;                // [C]
  const float *twiddle;                    // kTwiddleFloats, packed per lane (rx_ssb_f32_pack_twiddles)
  unsigned flag_base;                      // tiles each channel had completed before this launch
  uint32_t channels, frames;
  float agc_target, agc_decay, agc_floor, agc_gmax;
  const BiquadScanTables *tables;          // host pointer, copied into the kernel parameter block
  bool tx;                                 // TX-SSB-f32: mic (L) in, I/Q out through the ALC; audio_dbg is then [C][T][2]
  // TX-f32 (all modes): channels on the AM / FM slots run the modulators of DESIGN.md §3.4 instead of the SSB ALC; the FM phase
  // accumulator is carried in state[c][5] (uint32 bits)
  bool tx_mod;
  float am_depth, am_carrier;              // AM: ALC target, carrier level
  float fm_target, fm_level;               // FM: ALC target 2 deviation / fs (half-turns per sample), output level
  uint32_t *phase_dbg;                     // optional [C][T]: phi[n] of FM channels
  const float *sin513;                     // device, arm_sin_f32's 513-entry table (host_sin_table)
};
int launch_rx_ssb_f32 (const RxF32Launch &L, int sm_count, void *stream);
uint32_t rx_ssb_f32_launches_per_call ();
uint32_t rx_ssb_f32_tiles (uint32_t frames);   // how far a call of `frames` advances the per-channel hand-over flag
void rx_ssb_f32_pack_twiddles (float *out /* kTwiddleFloats */);
void rx_ssb_f32_pack_mask (const float *mask_re_im, float scale, float *out /* 2 * fft_len floats */);
constexpr size_t kTwiddleFloats = 6 * 32 * 4;

// ---- RX-SSB-f32 on the tensor cores (sl_rx_ssb_tc.cu): the overlap-save filter restated as the exact integer FIR it
// is (the mask is the DFT of a 129-tap filter), evaluated by tcgen05.mma kind::i8 on byte planes of samples and taps ----
constexpr int kTcTaps = 129;                       // fft_len - hop + 1
constexpr int kTcChannels = 8;                     // channels of one group = the 8 rows of a shared-memory core matrix
constexpr int kTcDigit = 52;                       // rows of one digit: 48 audio + 4 end-state outputs of a block
constexpr int kTcMapDigits = 4;                    // base-256 digits of a map entry: a 32-bit map. The high data byte meets all four, the low one the top three
constexpr int kTcRowGroups = 26;                   // 4 digits x 52 rows = 208 rows (N = 208 for the xh MMAs; the xl MMAs read the first 160), / 8
constexpr size_t kTcPlaneBytes = 11 * kTcRowGroups * 256;   // operand planes of one mask: [k-step][digit*52+row][32 bytes] in UMMA layout
struct TcBiquadTables
{
  float coef[10];                       // stage 0 {b0,b1,b2,a1,a2}, stage 1 {...}
  float Mp[4][16];                      // A^(48 k), k = 0..3 (k = 0: identity), row-major 4x4, state order {d1_0,d2_0,d1_1,d2_1}
  float M192[16];                       // A^192: one warp of the epilogue = four blocks
  float Cresp[48][4];                   // zero-input response of the cascade output at sample n of a block per unit state
};
void design_biquad_tc_tables (const float *coef10, TcBiquadTables *t);
// taps = IDFT of the (unscaled) mask in double; false when the impulse response does not fit 129 taps (then the FFT kernel
// serves the slot)
bool tc_design_taps (const float *mask_re_im /* [512][2] */, double *hr /* kTcTaps */, double *hi);
// operand planes: FIR taps composed with the zero-state response of the 2-stage biquad (coef10), see sl_design.cpp.
// *unit_a / *unit_z: the float value of one unit of the integer audio / state outputs
bool tc_build_planes (const float *mask_re_im, const float *coef10, uint8_t *planes /* kTcPlaneBytes */, float *unit_a, float *unit_z);
void tc_apply_planes (const uint8_t *planes, float unit_a, float unit_z, const int16_t *window /* [176][2] */, double *out52);
struct RxTcLaunch
{
  const int16_t *in; int16_t *out;         // [C][T][2]
  float *audio_dbg; float *gain_dbg;
  const int16_t *ovl_in; int16_t *ovl_out; // [C][128][2]
  float *state; unsigned *flag;            // as RxF32Launch; flag[c] is left at flag_final so the FFT kernel can take over
  const uint32_t *chan;                    // channels served by this launch, grouped by mask slot
  const uint32_t *gstart;                  // [n_groups] index of the group's first channel in chan[]
  const uint32_t *ginfo;                   // [n_groups] mask slot | channels in the group (1..8) << 8
  const uint32_t *pairs; uint32_t n_pairs; // [n_pairs][2]: the two groups (same mask slot) served by a CTA pair; second = 0xFFFFFFFF when the slot has an odd group
  const uint8_t *planes;                   // [SLB_MAX_MASKS][kTcPlaneBytes]
  const float *s0, *sz;                    // host, [SLB_MAX_MASKS]: units of the audio / state outputs
  unsigned flag_final;
  uint32_t n_groups, frames;
  float agc_target, agc_decay, agc_floor, agc_gmax;
  const TcBiquadTables *tables;
};
int launch_rx_ssb_tc (const RxTcLaunch &L, int sm_count, void *stream);

// ---- TX-SSB-f32 on the tensor cores (sl_tx_ssb_tc.cu): real mic samples x complex taps, two output rails ----
constexpr size_t kTcTxPlaneBytes = 2 * 6 * 18 * 256;   // [rail I|Q][K-step of 32 samples][digit*48+n][32 bytes]
bool tc_build_tx_planes (const float *mask_re_im, uint8_t *planes /* kTcTxPlaneBytes */, float *unit);
void tc_apply_tx_planes (const uint8_t *planes, float unit, const int16_t *window /* [192] mic samples */, double *out_iq /* [48][2] */);
struct TxTcLaunch
{
  const int16_t *in; int16_t *out;         // [C][T][2]: L = R mic frames in, I/Q out
  float *iq_dbg; float *gain_dbg;
  const int16_t *ovl_in; int16_t *ovl_out; // [C][128][2] carried raw tail
  float *state; unsigned *flag;            // envelope at state[c][4]; flag[c] left at flag_final for the FFT kernel
  const uint32_t *chan, *gstart, *ginfo;   // as RxTcLaunch
  const uint8_t *planes;                   // [SLB_MAX_MASKS][kTcTxPlaneBytes]
  const float *unit;                       // host, [SLB_MAX_MASKS]
  unsigned flag_final;
  uint32_t n_groups, frames;
  float alc_target, alc_decay, alc_floor, alc_gmax;
};
int launch_tx_ssb_tc (const TxTcLaunch &L, int sm_count, void *stream);

// ---- CHAN-64-f32 (sl_chan64.cu): state object owned by the context ----
struct Chan64State;
int design_default_chan (uint32_t fs, slb_chan_params *p);
int chan64_create (slb_ctx *ctx, uint32_t streams, uint32_t fs, Chan64State **out);
void chan64_destroy (Chan64State *st);
int chan64_reset (slb_ctx *ctx, Chan64State *st);
int chan64_set_params (slb_ctx *ctx, Chan64State *st, const slb_chan_params *p);
const slb_chan_params *chan64_params (const Chan64State *st);
void chan64_set_debug (Chan64State *st, float *audio, float *gain);
size_t chan64_state_bytes (const Chan64State *st);
int chan64_state_save (Chan64State *st, char *dst);
int chan64_state_load (Chan64State *st, const char *src);
int chan64_launch (slb_ctx *ctx, Chan64State *st, const int16_t *d_in, int16_t *d_out, uint32_t s0, uint32_t ns, uint32_t frames,
                   int sm_count, void *stream, bool with_debug);
void chan64_advance (Chan64State *st);

// ---- RX-SSB-q15 (sl_rx_ssb_q15.cu): state object owned by the context ----
struct RxQ15State;
int design_default_rx_q15 (uint32_t fs, slb_rx_q15_params *p);
int rxq15_create (slb_ctx *ctx, uint32_t channels, uint32_t fs, RxQ15State **out);
void rxq15_destroy (RxQ15State *st);
int rxq15_reset (slb_ctx *ctx, RxQ15State *st);
int rxq15_set_params (slb_ctx *ctx, RxQ15State *st, const slb_rx_q15_params *p);
const slb_rx_q15_params *rxq15_params (const RxQ15State *st);
void rxq15_set_debug (RxQ15State *st, int16_t *audio, uint32_t *gain);
int rxq15_set_sideband (slb_ctx *ctx, RxQ15State *st, uint32_t ch0, uint32_t n, int lsb);
int rxq15_launch (slb_ctx *ctx, RxQ15State *st, const int16_t *d_in, int16_t *d_out, uint32_t ch0, uint32_t nch, uint32_t frames,
                  int sm_count, void *stream, bool with_debug);
void rxq15_advance (RxQ15State *st);
int rxq15_carry_idle (RxQ15State *st, uint32_t ch0, uint32_t nch, void *stream);
int launch_biquad_df1_q15 (const int16_t *coeffs6, uint32_t ns, int32_t postshift, int16_t *d_state, const int16_t *d_src, int16_t *d_dst, uint32_t channels, uint32_t n, void *stream);
size_t rxq15_state_bytes (const RxQ15State *st);
int rxq15_state_save (RxQ15State *st, char *dst);
int rxq15_state_load (RxQ15State *st, const char *src);

// ---- RX-SSB-f32 AM channels on the tensor cores (sl_rx_am_tc.cu): both rails of the complex filter, envelope detector ----
constexpr size_t kTcAmPlaneBytes = 2 * 11 * 18 * 256;   // [rail Re|Im][K-step][digit*48+n][32 bytes]
bool tc_build_am_planes (const float *mask_re_im, uint8_t *planes /* kTcAmPlaneBytes */, float *unit);
struct RxAmTcLaunch
{
  const int16_t *in; int16_t *out; float *audio_dbg; float *gain_dbg;
  const int16_t *ovl_in; int16_t *ovl_out; float *state; unsigned *flag;
  const uint32_t *chan, *gstart, *ginfo;   // as RxTcLaunch
  const uint8_t *planes;                   // [SLB_MAX_MASKS][kTcAmPlaneBytes]
  const float *unit;                       // host, [SLB_MAX_MASKS]
  unsigned flag_final; uint32_t n_groups, frames;
  float agc_target, agc_decay, agc_floor, agc_gmax;
  const TcBiquadTables *tables;
};
int launch_rx_am_tc (const RxAmTcLaunch &L, int sm_count, void *stream);

// ---- RX-SSB-q15 on the tensor cores (sl_rx_q15_tc.cu): same chain, same state, bit-identical results ----
constexpr size_t kTcQ15PlaneBytes = 7 * 24 * 256;
bool q15_tc_build_planes (const int16_t *taps_i, const int16_t *taps_q, uint8_t *planes /* kTcQ15PlaneBytes */);
void q15_tc_apply_planes (const uint8_t *planes, const int16_t *window /* [112][2] */, int32_t *out96);
struct RxQ15TcLaunch
{
  const int16_t *in; int16_t *out;
  const uint32_t *tail_in; uint32_t *tail_out; const int16_t *peaks_in; int16_t *peaks_out;
  const uint8_t *planes, *lsb; int16_t *audio_dbg; uint32_t *gain_dbg;
  const int16_t *rel;                      // host, [SLB_Q15_WIN]
  uint32_t channels, frames, window; int32_t target, floor_; uint32_t gmax;
};
int launch_rx_q15_tc (const RxQ15TcLaunch &L, int sm_count, void *stream);

// ---- context accessors for translation units that do not see the struct (sl_stages.cu, sl_chains.cu) ----
int ctx_device (const slb_ctx *ctx);
size_t ctx_channels (const slb_ctx *ctx);
int ctx_fail (slb_ctx *ctx, int code, const char *msg);
void ctx_count_launch (slb_ctx *ctx, unsigned n = 1);
void *ctx_scratch_on (slb_ctx *ctx, size_t bytes, void *stream);   // the same, ordered after the previous user's stream (per-call staging)
void *ctx_scratch (slb_ctx *ctx, size_t bytes);     // device scratch owned by the context, grown on demand (nullptr + error on failure)

}  // namespace sl
