// Frozen default design of the RX-SSB-f32 chain. NOTHING here comes from the reference: the firmware has no filter
// taps, no AGC constants and no demodulator (SURVEY.md §0; DSP_Set_Mode is empty, Core/Src/dsp_if.c:367-370).
// The designs are closed-form and evaluated in double so that every consumer (product, oracle, tests) gets the same
// numbers from slb_default_*().
#include <cmath>
#include <cstring>
#include <vector>
#include "sl_internal.h"

namespace sl {

static const double kPi = 3.14159265358979323846;

// RBJ-style 2nd-order sections by bilinear transform with pre-warping; returned in the CMSIS layout
// {b0,b1,b2,a1,a2} with the +a1,+a2 feedback sign (arm_biquad_cascade_df1_f32.c:52).
static void biquad_lp (double fc, double q, double fs, float *c)
{
  double w0 = 2.0 * kPi * fc / fs, cw = std::cos (w0), al = std::sin (w0) / (2.0 * q), a0 = 1.0 + al;
  c[0] = (float) ((1.0 - cw) / 2.0 / a0); c[1] = (float) ((1.0 - cw) / a0); c[2] = (float) ((1.0 - cw) / 2.0 / a0);
  c[3] = (float) (2.0 * cw / a0); c[4] = (float) (-(1.0 - al) / a0);
}

int design_default_rx_f32 (uint32_t fs, slb_rx_f32_params *p)
{
  if (!p || (fs != 48000u && fs != 96000u && fs != 192000u)) return SLB_ERR_ARG;
  std::memset (p, 0, sizeof *p);
  p->fft_len = 512; p->hop = 384; p->agc_block = 48; p->n_stages = 2;
  // 4th-order Butterworth audio low-pass at 3 kHz as two sections. (A 200 Hz high-pass section was tried first and
  // dropped: in float32 df2T its poles at r = 0.98 amplify a 1-ulp input perturbation ~30x, which makes ANY two
  // implementations — even the reference against its own restatement — disagree at the 1e-5 level. The mask already
  // removes everything below 300 Hz.)
  biquad_lp (3000.0, 0.54119610014619698, (double) fs, p->biquad);
  biquad_lp (3000.0, 1.30656296487637653, (double) fs, p->biquad + 5);
  p->agc_target = 0.25f;                                                 // -12 dBFS
  p->agc_decay = (float) std::exp (-(48.0 / (double) fs) / 0.300);       // 300 ms release; one step per 48-frame block (1 ms at 48 kHz)
  p->agc_floor = 1.0e-4f;
  p->agc_gmax = 100.0f;                                                  // +40 dB
  return SLB_OK;
}

// TX-SSB-f32: the mode's one-sided mask is band-pass and Hilbert pair in one; what is left to freeze is the ALC.
int design_default_tx_f32 (uint32_t fs, slb_tx_f32_params *p)
{
  if (!p || (fs != 48000u && fs != 96000u && fs != 192000u)) return SLB_ERR_ARG;
  std::memset (p, 0, sizeof *p);
  p->fft_len = 512; p->hop = 384; p->alc_block = 48;
  p->alc_target = 0.5f;                                                  // -6 dBFS peak envelope of I + jQ
  p->alc_decay = (float) std::exp (-(48.0 / (double) fs) / 0.100);       // 100 ms release; one step per 48-frame block (1 ms at 48 kHz)
  p->alc_floor = 1.0e-3f;
  p->alc_gmax = 16.0f;                                                   // +24 dB
  return SLB_OK;
}

// TX AM / FM (SLB_CHAIN_TX_F32): the carrier at -6 dBFS leaves 80 % peak modulation room below full scale (0.5 * 1.8 = 0.9); 2.5 kHz peak
// deviation is narrow-band FM on a 6 kHz audio band (Carson: 2 (2.5 + 3) = 11 kHz); the FM level matches the SSB ALC target.
int design_default_tx_mod (uint32_t fs, slb_tx_mod_params *p)
{
  if (!p || (fs != 48000u && fs != 96000u && fs != 192000u)) return SLB_ERR_ARG;
  p->am_carrier = 0.5f; p->am_depth = 0.8f; p->fm_deviation_hz = 2500.0f; p->fm_level = 0.5f;
  return SLB_OK;
}

int mode_to_mask_slot (uint8_t mode)
{
  switch (mode)
  {
    case SLB_MODE_LSB: return 0; case SLB_MODE_USB: return 1; case SLB_MODE_CW: return 2; case SLB_MODE_CWR: return 3;
    case SLB_MODE_DIG: return 4; case SLB_MODE_PKT: return 5;
    case SLB_MODE_AM: return kAmMaskSlot;                                // two-sided channel filter + envelope detector
    case SLB_MODE_FM: return kFmMaskSlot;                                // two-sided channel filter + limiter-discriminator
    default: return -1;
  }
}

static double bessel_i0 (double x)
{
  double s = 1.0, t = 1.0;
  for (int k = 1; k < 64; k++) { t *= (x / (2.0 * k)) * (x / (2.0 * k)); s += t; if (t < 1e-18 * s) break; }
  return s;
}

// 129-tap (fft_len/4 + 1) Kaiser-windowed-sinc low-pass, heterodyned to the wanted sideband, then its fft_len-point
// DFT. Overlap-save with fft_len - hop = 128 = taps - 1 makes the FFT filter identical to that linear FIR.
int design_default_mask (uint32_t fs, uint32_t N, uint8_t mode, float *out)
{
  if (!out || N < 16 || N > 4096 || (N & (N - 1))) return SLB_ERR_ARG;
  double lo, hi;
  switch (mode)
  {
    case SLB_MODE_USB: lo = 300.0; hi = 2700.0; break;
    case SLB_MODE_LSB: lo = -2700.0; hi = -300.0; break;
    case SLB_MODE_CW:  lo = 450.0; hi = 950.0; break;
    case SLB_MODE_CWR: lo = -950.0; hi = -450.0; break;
    case SLB_MODE_DIG: case SLB_MODE_PKT: lo = 300.0; hi = 3300.0; break;
    case SLB_MODE_AM: lo = -3000.0; hi = 3000.0; break;                  // carrier and both sidebands
    case SLB_MODE_FM: lo = -7500.0; hi = 7500.0; break;                  // narrow-band FM channel: +-5 kHz deviation + 2.5 kHz audio (Carson)
    default: return SLB_ERR_UNSUPPORTED;
  }
  const int taps = (int) N / 4 + 1, mid = (taps - 1) / 2;
  const double fcut = (hi - lo) / 2.0 / (double) fs, fcen = (hi + lo) / 2.0 / (double) fs, beta = 8.0;
  std::vector<double> hr (taps), hi_ (taps);
  double dc = 0.0;
  for (int n = 0; n < taps; n++)
  {
    double m = n - mid, x = 2.0 * fcut * m;
    double sinc = (m == 0) ? 1.0 : std::sin (kPi * x) / (kPi * x);
    double r = (double) m / (double) mid;
    double w = bessel_i0 (beta * std::sqrt (1.0 - r * r)) / bessel_i0 (beta);
    hr[n] = 2.0 * fcut * sinc * w; dc += hr[n];
  }
  for (int n = 0; n < taps; n++)
  {
    double g = hr[n] / dc;                                               // unit pass-band gain for a complex (I/Q) tone
    double ph = 2.0 * kPi * fcen * (n - mid);
    hr[n] = g * std::cos (ph); hi_[n] = g * std::sin (ph);
  }
  for (uint32_t k = 0; k < N; k++)
  {
    double re = 0.0, im = 0.0;
    for (int n = 0; n < taps; n++)
    {
      double ph = -2.0 * kPi * (double) ((uint64_t) k * (uint64_t) n % N) / (double) N, c = std::cos (ph), s = std::sin (ph);
      re += hr[n] * c - hi_[n] * s; im += hr[n] * s + hi_[n] * c;
    }
    out[2 * k] = (float) re; out[2 * k + 1] = (float) im;
  }
  return SLB_OK;
}

// RX-SSB-q15: 64-tap band-pass Hilbert pair (Kaiser-windowed low-pass of half the audio bandwidth, heterodyned to the
// audio centre with 0 / +90 degrees), each rail at half gain so that the wanted sideband sums to unity and the other
// cancels; finite-window AGC. Quantised to q15 by round-to-nearest.
int design_default_rx_q15 (uint32_t fs, slb_rx_q15_params *p)
{
  if (!p || fs != 48000u) return p ? SLB_ERR_UNSUPPORTED : SLB_ERR_ARG;
  std::memset (p, 0, sizeof *p);
  p->ntaps = SLB_Q15_TAPS; p->agc_block = fs / 1000u; p->agc_window = 16;
  const int T = SLB_Q15_TAPS;
  const double lo = 300.0, hi = 2700.0, fcut = (hi - lo) / 2.0 / (double) fs, fcen = (hi + lo) / 2.0 / (double) fs, beta = 6.0, mid = (T - 1) / 2.0;
  double g[SLB_Q15_TAPS], dc = 0.0;
  for (int n = 0; n < T; n++)
  {
    const double m = n - mid, x = 2.0 * fcut * m, r = m / mid;
    g[n] = 2.0 * fcut * (std::sin (kPi * x) / (kPi * x)) * bessel_i0 (beta * std::sqrt (1.0 - r * r)) / bessel_i0 (beta);
    dc += g[n];
  }
  for (int n = 0; n < T; n++)
  {
    const double ph = 2.0 * kPi * fcen * (n - mid), a = g[n] / dc;
    p->taps_i[n] = (int16_t) std::lrint (32768.0 * a * std::cos (ph));
    p->taps_q[n] = (int16_t) std::lrint (-32768.0 * a * std::sin (ph));
  }
  p->rel[0] = 32767;
  for (int j = 1; j < SLB_Q15_WIN; j++) p->rel[j] = (int16_t) std::lrint (32767.0 * std::exp (-(double) j / 6.0));   // ~6 ms time constant
  p->agc_target = 8192;                                                  // -12 dBFS
  p->agc_floor = 16;
  p->agc_gmax_q15 = 64u << 15;                                           // +36 dB
  return SLB_OK;
}

// CHAN-64-q15 (DESIGN.md §3.10): CHAN-64-f32's prototype at DC gain 32, llround to q15. Every branch then sums to about 0.5 (at most
// 0.75 in absolute value), so no branch FIR saturates and an in-bin tone of amplitude A leaves the FFT (which divides by 64) at A / 2;
// at DC gain 1 the branch outputs would lose 6 bits. The AGC is RX-SSB-q15's.
int design_default_chan_q15 (uint32_t fs, slb_chan_q15_params *p)
{
  if (!p) return SLB_ERR_ARG;
  if (fs != 192000u) return SLB_ERR_UNSUPPORTED;
  std::memset (p, 0, sizeof *p);
  p->bins = SLB_CHAN_BINS; p->taps_per_branch = SLB_CHAN_TAPS; p->agc_block = 3; p->envelope = 0;
  double h[SLB_CHAN_BINS * SLB_CHAN_TAPS];
  chan_prototype (h);
  for (int i = 0; i < SLB_CHAN_BINS * SLB_CHAN_TAPS; i++) p->proto[i] = (int16_t) std::llround (32.0 * 32768.0 * h[i]);
  slb_rx_q15_params q;
  design_default_rx_q15 (48000u, &q);
  p->agc_window = q.agc_window; std::memcpy (p->rel, q.rel, sizeof p->rel);
  p->agc_target = q.agc_target; p->agc_floor = q.agc_floor; p->agc_gmax_q15 = q.agc_gmax_q15;
  return SLB_OK;
}

// RX-Q15's AM and FM detectors: 64-tap Kaiser (beta 6) windowed-sinc low-passes with the cut-off (-6 dB) at 3 kHz (AM) and 6 kHz
// (FM), normalised to DC gain 1 in double, then llround to q15 (both rails use the same taps)
int design_default_rx_q15_modes (uint32_t fs, slb_rx_q15_mode_params *p)
{
  if (!p || fs != 48000u) return p ? SLB_ERR_UNSUPPORTED : SLB_ERR_ARG;
  std::memset (p, 0, sizeof *p);
  const int T = SLB_Q15_TAPS;
  const double beta = 6.0, mid = (T - 1) / 2.0;
  auto lowpass = [&] (double fc_hz, int16_t *out)
  {
    const double fc = fc_hz / (double) fs;
    double g[SLB_Q15_TAPS], dc = 0.0;
    for (int n = 0; n < T; n++)
    {
      const double m = n - mid, x = 2.0 * fc * m, r = m / mid;
      g[n] = 2.0 * fc * (std::sin (kPi * x) / (kPi * x)) * bessel_i0 (beta * std::sqrt (1.0 - r * r)) / bessel_i0 (beta);
      dc += g[n];
    }
    for (int n = 0; n < T; n++) out[n] = (int16_t) std::llround (32768.0 * g[n] / dc);
  };
  lowpass (3000.0, p->am_taps);
  lowpass (6000.0, p->fm_taps);
  p->fm_floor = 1 << 18;
  return SLB_OK;
}

// TX-Q15's AM and FM modulators: RX-Q15's AM low-pass (3 kHz) for both; carrier 0.5, AM depth 0.8, FM ALC target 0.25 and an increment
// that puts y = fm_target at 2.5 kHz: llround (2500 2^32 / 48000 / 8192) = 27307; NCO level 0.5
int design_default_tx_q15_modes (uint32_t fs, slb_tx_q15_mode_params *p)
{
  if (!p || fs != 48000u) return p ? SLB_ERR_UNSUPPORTED : SLB_ERR_ARG;
  slb_rx_q15_mode_params rx;
  const int rc = design_default_rx_q15_modes (fs, &rx); if (rc) return rc;
  std::memset (p, 0, sizeof *p);
  std::memcpy (p->am_taps, rx.am_taps, sizeof p->am_taps);
  std::memcpy (p->fm_taps, rx.am_taps, sizeof p->fm_taps);
  p->am_carrier = 16384; p->am_depth = 26214; p->fm_target = 8192;
  p->fm_inc = (int32_t) std::llround (2500.0 * 4294967296.0 / (double) fs / 8192.0);
  p->fm_level = 0.5f;
  return SLB_OK;
}

// -----------------------------------------------------------------------------------------------------------
// Time-parallel evaluation of the 2-stage df2T cascade (arm_biquad_cascade_df2T_f32.c:551-562 per sample):
// with x = 0 the 4-vector s = {d1_0,d2_0,d1_1,d2_1} evolves linearly, s' = A s, and the cascade output is c.s.
// A lane filters its run of kRun samples from a zero state; the true start state s_k of run k then adds
// Cresp[n].s_k to sample n, and run end states chain through M = A^kRun (scan with M, M^2, M^4, ...).
// -----------------------------------------------------------------------------------------------------------
void design_biquad_scan_tables (const float *cf, BiquadScanTables *t)
{
  for (int i = 0; i < 10; i++) t->coef[i] = cf[i];
  const double b0 = cf[5], b1 = cf[6], b2 = cf[7];
  const double a1[2] = { cf[3], cf[8] }, a2[2] = { cf[4], cf[9] };
  double M[4][4];
  for (int col = 0; col < 4; col++)
  {
    double s[4] = { 0, 0, 0, 0 }; s[col] = 1.0;
    for (int n = 0; n < kRun; n++)
    {
      double y0 = s[0];                                  // stage 0, x = 0
      double n0 = a1[0] * y0 + s[1], n1 = a2[0] * y0;
      double y1 = b0 * y0 + s[2];                        // stage 1, x = y0
      double n2 = (b1 * y0 + a1[1] * y1) + s[3], n3 = b2 * y0 + a2[1] * y1;
      t->Cresp[n][col] = (float) y1;
      s[0] = n0; s[1] = n1; s[2] = n2; s[3] = n3;
    }
    for (int r = 0; r < 4; r++) M[r][col] = s[r];
  }
  for (int k = 0; k < 6; k++)
  {
    for (int r = 0; r < 4; r++) for (int c = 0; c < 4; c++) t->Mpow[k][4 * r + c] = (float) M[r][c];
    double P[4][4];
    for (int r = 0; r < 4; r++) for (int c = 0; c < 4; c++) { double a = 0; for (int j = 0; j < 4; j++) a += M[r][j] * M[j][c]; P[r][c] = a; }
    std::memcpy (M, P, sizeof M);
  }
}

// -----------------------------------------------------------------------------------------------------------
// Tables of the tensor-core RX-SSB-f32 kernel (sl_rx_ssb_tc.cu)
// -----------------------------------------------------------------------------------------------------------
// One zero-input step of the 2-stage df2T cascade (arm_biquad_cascade_df2T_f32.c:551-562 with x = 0), in double.
static void cascade_zero_input_step (const float *cf, double *s, double *y_out)
{
  const double b0 = cf[5], b1 = cf[6], b2 = cf[7];
  const double y0 = s[0];
  const double n0 = (double) cf[3] * y0 + s[1], n1 = (double) cf[4] * y0;
  const double y1 = b0 * y0 + s[2];
  const double n2 = (b1 * y0 + (double) cf[8] * y1) + s[3], n3 = b2 * y0 + (double) cf[9] * y1;
  s[0] = n0; s[1] = n1; s[2] = n2; s[3] = n3;
  *y_out = y1;
}
void design_biquad_tc_tables (const float *cf, TcBiquadTables *t)
{
  for (int i = 0; i < 10; i++) t->coef[i] = cf[i];
  double M[4][4];
  for (int col = 0; col < 4; col++)
  {
    double s[4] = { 0, 0, 0, 0 }; s[col] = 1.0;
    for (int n = 0; n < 48; n++) { double y; cascade_zero_input_step (cf, s, &y); t->Cresp[n][col] = (float) y; }
    for (int r = 0; r < 4; r++) M[r][col] = s[r];
  }
  double P[4][4];
  for (int r = 0; r < 4; r++) for (int c = 0; c < 4; c++) P[r][c] = (r == c) ? 1.0 : 0.0;
  for (int k = 0; k <= 4; k++)
  {
    float *dst = (k < 4) ? t->Mp[k] : t->M192;
    for (int r = 0; r < 4; r++) for (int c = 0; c < 4; c++) dst[4 * r + c] = (float) P[r][c];
    double Q[4][4];
    for (int r = 0; r < 4; r++) for (int c = 0; c < 4; c++) { double a = 0; for (int j = 0; j < 4; j++) a += M[r][j] * P[j][c]; Q[r][c] = a; }
    std::memcpy (P, Q, sizeof P);
  }
}

// The mask of a mode is the DFT of a filter of fft_len - hop + 1 = 129 taps, so overlap-save with it IS a 129-tap FIR.
// Recover the taps (inverse DFT in double, 1/N as arm_cfft_f32.c:604-614); false when the impulse response does not fit.
bool tc_design_taps (const float *mask, double *hr /* kTcTaps */, double *hi)
{
  const int N = 512;
  const double two_pi = 6.283185307179586476925286766559;
  std::vector<double> cs (N), sn (N);
  for (int i = 0; i < N; i++) { cs[i] = std::cos (two_pi * i / N); sn[i] = std::sin (two_pi * i / N); }
  double main_e = 0, tail_e = 0;
  for (int d = 0; d < N; d++)
  {
    double ar = 0, ai = 0;
    for (int k = 0; k < N; k++)
    {
      const int ph = (k * d) & (N - 1);
      const double Hr = mask[2 * k], Hi = mask[2 * k + 1];
      ar += Hr * cs[ph] - Hi * sn[ph]; ai += Hr * sn[ph] + Hi * cs[ph];
    }
    ar /= N; ai /= N;
    if (d < kTcTaps) { hr[d] = ar; hi[d] = ai; main_e += ar * ar + ai * ai; } else tail_e += ar * ar + ai * ai;
  }
  return main_e > 0.0 && std::isfinite (main_e) && tail_e <= 1e-13 * main_e;
}

// B operand of the tensor-core kernel. Per firmware block (48 outputs, zero biquad state at the block start) everything up
// to and including the biquad's zero-state response is ONE linear map of the 176-frame raw window:
//   FIR        y[m]  = sum_d hr[d] I[m-d] - hi[d] Q[m-d]                  (m = 0..47 inside the block)
//   audio      a[n]  = sum_{m<=n} g[n-m] y[m]      g = impulse response of the 2-stage df2T cascade (zero state)
//   end state  z_i   = sum_m sigma_i[47-m] y[m]    sigma[t] = cascade state t samples after a unit impulse
// so the taps operand holds W = G T (48 audio rows) and Z = Sigma T (4 state rows) instead of the bare Toeplitz T: the
// tensor cores deliver the block's zero-state audio and end state, the CUDA cores only chain the states and add the
// zero-input response (arm_biquad_cascade_df2T_f32.c:551-562 is linear, so the split is exact). Rows are quantised to 24
// bits (audio and state rows with their own scale), three balanced base-256 digits, rows digit * 52 + r (r < 48 audio,
// 48..51 state; rows 156..159 zero), K-major no-swizzle core matrices; window byte m = 32 ks + kk = frame m / 2, rail m & 1.
bool tc_build_planes (const float *mask, const float *cf, uint8_t *planes, float *unit_a, float *unit_z)
{
  double hr[kTcTaps], hi[kTcTaps];
  if (!tc_design_taps (mask, hr, hi)) return false;
  // cascade impulse response and state trajectory, in double
  double g[48], sig[48][4];
  {
    double st[4] = { 0, 0, 0, 0 };
    for (int t = 0; t < 48; t++)
    {
      const double x = (t == 0) ? 1.0 : 0.0;
      const double y0 = (double) cf[0] * x + st[0];
      const double n0 = ((double) cf[1] * x + (double) cf[3] * y0) + st[1], n1 = (double) cf[2] * x + (double) cf[4] * y0;
      const double y1 = (double) cf[5] * y0 + st[2];
      const double n2 = ((double) cf[6] * y0 + (double) cf[8] * y1) + st[3], n3 = (double) cf[7] * y0 + (double) cf[9] * y1;
      st[0] = n0; st[1] = n1; st[2] = n2; st[3] = n3;
      g[t] = y1;
      for (int i = 0; i < 4; i++) sig[t][i] = st[i];
    }
  }
  // rows x window (176 frames x 2 rails)
  const int R = 52, F = 176;
  std::vector<double> W ((size_t) R * F * 2, 0.0);
  for (int f = 0; f < F; f++)
    for (int m = 0; m < 48; m++)
    {
      const int d = 128 + m - f;
      if (d < 0 || d >= kTcTaps) continue;
      const double tI = hr[d], tQ = -hi[d];
      for (int n = m; n < 48; n++) { W[((size_t) n * F + f) * 2] += g[n - m] * tI; W[((size_t) n * F + f) * 2 + 1] += g[n - m] * tQ; }
      for (int i = 0; i < 4; i++) { W[((size_t) (48 + i) * F + f) * 2] += sig[47 - m][i] * tI; W[((size_t) (48 + i) * F + f) * 2 + 1] += sig[47 - m][i] * tQ; }
    }
  double mx_a = 0, mx_z = 0;
  for (int r = 0; r < R; r++) for (int k = 0; k < F * 2; k++) { double &mx = (r < 48) ? mx_a : mx_z; mx = std::fmax (mx, std::fabs (W[(size_t) r * F * 2 + k])); }
  // 32-bit map, four balanced base-256 digits: 127 (2^24 + 2^16 + 2^8 + 1) is the largest value they hold
  const double lim = 2139062143.0 - 16843009.0;
  // scale: the largest entry takes the full range. The float unit of the integer output is fixed first and the scale derived
  // from it, so that unit * 32768 * scale == 1 holds exactly for the float32 value the kernel multiplies by (the 1/32768 of
  // arm_q15_to_float.c:87 is folded in). The kernel drops the one product class below 2^8 (low data byte x lowest digit), so
  // the unit it is handed belongs to the 2^8 class: 256 map LSBs.
  const float ua = (float) (256.0 * mx_a / (lim * 32768.0)), uz = (float) (256.0 * mx_z / (lim * 32768.0));
  if (!(ua > 1e-30f) || !std::isfinite (ua) || !(uz > 1e-30f) || !std::isfinite (uz)) return false;
  const double sc_a = 256.0 / ((double) ua * 32768.0), sc_z = 256.0 / ((double) uz * 32768.0);
  *unit_a = ua; *unit_z = uz;
  std::memset (planes, 0, kTcPlaneBytes);
  for (int r = 0; r < R; r++)
    for (int m = 0; m < F * 2; m++)
    {
      const long long q = std::llround (W[(size_t) r * F * 2 + m] * (r < 48 ? sc_a : sc_z));
      if (q == 0) continue;
      if (std::llabs (q) > 2139062143ll) return false;          // (lim keeps 0.8 % of headroom under this: the float32 unit moves the scale by up to 6e-8)
      long long h = q;
      int32_t dg[kTcMapDigits];                      // most significant first: accumulator columns 0..51 carry 2^32 (x 2^8 of the high data byte)
      for (int gdig = kTcMapDigits - 1; gdig >= 0; gdig--)
      {
        const long long lo = ((h + 128) & 255) - 128;
        dg[gdig] = (int32_t) lo; h = (h - lo) >> 8;
      }
      if (h != 0) return false;
      const int ks = m / 32, kk = m % 32;
      for (int gdig = 0; gdig < kTcMapDigits; gdig++)
      {
        const int row = gdig * kTcDigit + r;
        planes[(size_t) ks * kTcRowGroups * 256 + (row / 8) * 256 + (kk / 16) * 128 + (row % 8) * 16 + (kk % 16)] = (uint8_t) (int8_t) dg[gdig];
      }
    }
  return true;
}

// host-side evaluation of the planes on one raw window (design check, tests/test_tc_math.py): exactly the integer
// contraction the kernel runs — the high data byte against all four digits, the low one against the top three (the class
// below 2^8 is not computed) — out[0..47] = zero-state audio of the block, out[48..51] = its end state
void tc_apply_planes (const uint8_t *planes, float unit_a, float unit_z, const int16_t *window /* [176][2] */, double *out52)
{
  for (int r = 0; r < 52; r++)
  {
    long long acc = 0;                                // in units of the 2^8 class
    for (int m = 0; m < 352; m++)
    {
      const int ks = m / 32, kk = m % 32;
      long long dg[kTcMapDigits];
      for (int gdig = 0; gdig < kTcMapDigits; gdig++)
      {
        const int row = gdig * kTcDigit + r;
        dg[gdig] = (int8_t) planes[(size_t) ks * kTcRowGroups * 256 + (row / 8) * 256 + (kk / 16) * 128 + (row % 8) * 16 + (kk % 16)];
      }
      const int x = window[m], xl = x & 255, xh = (x - xl) >> 8;
      // x h / 2^8 = xh (h3 2^24 + h2 2^16 + h1 2^8 + h0) + xl (h3 2^16 + h2 2^8 + h1) [+ xl h0 / 2^8, dropped]
      acc += (long long) xh * (((dg[0] * 256 + dg[1]) * 256 + dg[2]) * 256 + dg[3]) + (long long) xl * ((dg[0] * 256 + dg[1]) * 256 + dg[2]);
    }
    out52[r] = (double) acc * (double) (r < 48 ? unit_a : unit_z);
  }
}

// TX: I[n] = sum_d hr[d] m[n-d], Q[n] = sum_d hi[d] m[n-d] on the real mic samples m. Window = 192 samples from 128 before
// the block (6 K-steps of 32; the last 16 reach past the block and meet zero taps); rows digit * 48 + n per rail.
bool tc_build_tx_planes (const float *mask, uint8_t *planes, float *unit)
{
  double hr[kTcTaps], hi[kTcTaps];
  if (!tc_design_taps (mask, hr, hi)) return false;
  double mx = 0;
  for (int d = 0; d < kTcTaps; d++) mx = std::fmax (mx, std::fmax (std::fabs (hr[d]), std::fabs (hi[d])));
  const double lim = 8323071.0;
  const float u = (float) (mx / (lim * 32768.0));
  if (!(u > 1e-30f) || !std::isfinite (u)) return false;
  const double sc = 1.0 / ((double) u * 32768.0);
  *unit = u;
  std::memset (planes, 0, kTcTxPlaneBytes);
  for (int rail = 0; rail < 2; rail++)
    for (int n = 0; n < 48; n++)
      for (int f = 0; f < 192; f++)
      {
        const int d = 128 + n - f;
        if (d < 0 || d >= kTcTaps) continue;
        const long long q = std::llround ((rail ? hi[d] : hr[d]) * sc);
        if (std::llabs (q) > (long long) lim + 1) return false;
        const int32_t h = (int32_t) q;
        const int32_t l0 = ((h + 128) & 255) - 128, r1 = (h - l0) >> 8, l1 = ((r1 + 128) & 255) - 128, l2 = (r1 - l1) >> 8;
        const int32_t dg[3] = { l2, l1, l0 };
        const int ks = f / 32, kk = f % 32;
        for (int g = 0; g < 3; g++)
        {
          const int row = g * 48 + n;
          planes[(size_t) (rail * 6 + ks) * 18 * 256 + (row / 8) * 256 + (kk / 16) * 128 + (row % 8) * 16 + (kk % 16)] = (uint8_t) (int8_t) dg[g];
        }
      }
  return true;
}
void tc_apply_tx_planes (const uint8_t *planes, float unit, const int16_t *window, double *out_iq)
{
  for (int rail = 0; rail < 2; rail++)
    for (int n = 0; n < 48; n++)
    {
      long long acc = 0;
      for (int f = 0; f < 192; f++)
      {
        const int ks = f / 32, kk = f % 32;
        long long h = 0;
        for (int g = 0; g < 3; g++)
        {
          const int row = g * 48 + n;
          h = h * 256 + (int8_t) planes[(size_t) (rail * 6 + ks) * 18 * 256 + (row / 8) * 256 + (kk / 16) * 128 + (row % 8) * 16 + (kk % 16)];
        }
        acc += h * (long long) window[f];
      }
      out_iq[2 * n + rail] = (double) acc * (double) unit;
    }
}

// AM (complex detector): both rails of z = h * x on the interleaved I/Q byte planes, window byte m = 2 frame + rail:
//   Re z[n] = sum_d hr[d] I - hi[d] Q,  Im z[n] = sum_d hi[d] I + hr[d] Q;  rows digit * 48 + n per output rail, 11 K-steps.
bool tc_build_am_planes (const float *mask, uint8_t *planes, float *unit)
{
  double hr[kTcTaps], hi[kTcTaps];
  if (!tc_design_taps (mask, hr, hi)) return false;
  double mx = 0;
  for (int d = 0; d < kTcTaps; d++) mx = std::fmax (mx, std::fmax (std::fabs (hr[d]), std::fabs (hi[d])));
  const double lim = 8323071.0;
  const float u = (float) (mx / (lim * 32768.0));
  if (!(u > 1e-30f) || !std::isfinite (u)) return false;
  const double sc = 1.0 / ((double) u * 32768.0);
  *unit = u;
  std::memset (planes, 0, kTcAmPlaneBytes);
  for (int orail = 0; orail < 2; orail++)
    for (int n = 0; n < 48; n++)
      for (int m = 0; m < 352; m++)
      {
        const int f = m / 2, irail = m & 1, d = 128 + n - f;
        if (d < 0 || d >= kTcTaps) continue;
        const double v = (orail == 0) ? (irail ? -hi[d] : hr[d]) : (irail ? hr[d] : hi[d]);
        const long long q = std::llround (v * sc);
        if (std::llabs (q) > (long long) lim + 1) return false;
        const int32_t h = (int32_t) q;
        const int32_t l0 = ((h + 128) & 255) - 128, r1 = (h - l0) >> 8, l1 = ((r1 + 128) & 255) - 128, l2 = (r1 - l1) >> 8;
        const int32_t dg[3] = { l2, l1, l0 };
        const int ks = m / 32, kk = m % 32;
        for (int g = 0; g < 3; g++)
        {
          const int row = g * 48 + n;
          planes[(size_t) (orail * 11 + ks) * 18 * 256 + (row / 8) * 256 + (kk / 16) * 128 + (row % 8) * 16 + (kk % 16)] = (uint8_t) (int8_t) dg[g];
        }
      }
  return true;
}

// -----------------------------------------------------------------------------------------------------------
// Ring index logic — follows Core/Src/dsp_if.c line by line (cited), with the sample stores left to the kernels.
// -----------------------------------------------------------------------------------------------------------
uint32_t RingPtrs::plan_write (bool is_out, uint32_t frames)
{
  const uint32_t N = size;
  uint32_t gap = 0;
  if (is_out)
  {
    if (!enable)                                   // dsp_if.c:124-134: writer arms the TX ring half a ring ahead
    {
      wr = rd + N / 2; if (wr >= N) wr -= N;
      enable = 1;
    }
    gap = wr; if (rd > wr) gap += N; gap -= rd;    // dsp_if.c:136-143
  }
  else if (enable)                                 // dsp_if.c:254-264: RX gap only once the reader armed the ring
  {
    gap = wr; if (rd > wr) gap += N; gap -= rd;
  }
  gap &= 0xFFFFu;                                  // uint16_t gap
  if (gap > 3u * N / 4u) { if (wr < 1u) wr += N; wr--; }          // dsp_if.c:145-153 / :266-274
  if (gap < N / 4u) { wr++; if (wr >= N) wr -= N; }               // dsp_if.c:155-163 / :276-284
  const uint32_t first = wr;
  // `frames` stores, the duplicate of the last frame, then one step back (dsp_if.c:165-179 / :286-300)
  wr = (wr + frames + 1u) % N;
  if (wr < 1u) wr += N;
  wr--;
  return first;
}

uint32_t RingPtrs::plan_read (bool is_out, uint32_t frames)
{
  const uint32_t N = size;
  if (!is_out && !enable)                          // dsp_if.c:316-326: first read arms; overflow case RESETS TO 0
  {
    rd = wr + N / 2; if (rd >= N) rd = 0;
    enable = 1;
  }
  const uint32_t first = rd;
  rd = (rd + frames) % N;                          // dsp_if.c:206-217 / :328-339
  return first;
}

}  // namespace sl
