/*
 * rx_design.cpp — host control path (see rx_design.h).  Compile with -ffp-contract=off.
 *
 * Every routine states the reference function whose result it reproduces; mixed
 * float/double arithmetic follows the reference expressions term by term because the
 * resulting tables are compared bit-for-bit with the CPU oracle's.
 */
#include "rx_design.h"

#include <math.h>
#include <string.h>

#include "rx_fft.h"
#include "rx_tables_data.h"

namespace t41rx {

namespace {

/* FIR.h:6-16 — single-precision constants used throughout the DSP files */
const float kPiF = 3.1415926535897932384626433832795f;
const float kHalfPiF = 1.5707963267948966192313216916398f;
const float kTwoPiF = 6.283185307179586476925286766559f;

const int kFs = 192000;          /* SampleRate, T41_SDR.ino:129 */
const float kDf1 = 4.0f;
const float kDf = 8.0f;
const float kStopDb = 90.0f;     /* n_att */

float g_host_twiddle[2 * kFft];
bool g_host_twiddle_ready = false;

/* Utility.cpp:213-230 */
float BesselI0Series(float x) {
  const float half = x / 2.0;
  float sum = 1.0;
  float term = 1.0;
  float k = 1.0;
  const float eps = 1e-9;
  do {
    float t = half / k;
    t *= t;
    term *= t;
    sum += term;
    k += 1.0;
  } while (term >= eps * sum);
  return sum;
}

/* Utility.cpp:197-203 */
float SincHalfPi(int m, float fc) {
  const float x = m * kHalfPiF;
  if (m == 0) return 1.0f;
  return sinf(x * fc) / (fc * x);
}

}  // namespace

const float *HostTwiddle512() {
  if (!g_host_twiddle_ready) {
    for (int i = 0; i < kFft; ++i) {
      const double a = 2.0 * 3.14159265358979323846 * (double)i / (double)kFft;
      g_host_twiddle[2 * i] = (float)cos(a);
      g_host_twiddle[2 * i + 1] = (float)sin(a);
    }
    g_host_twiddle[0] = 1.0f;        g_host_twiddle[1] = 0.0f;
    g_host_twiddle[2 * 128] = 0.0f;  g_host_twiddle[2 * 128 + 1] = 1.0f;
    g_host_twiddle[2 * 256] = -1.0f; g_host_twiddle[2 * 256 + 1] = 0.0f;
    g_host_twiddle[2 * 384] = 0.0f;  g_host_twiddle[2 * 384 + 1] = -1.0f;
    g_host_twiddle_ready = true;
  }
  return g_host_twiddle;
}

void HostFft512(float *interleaved) {
  float2 *buf = reinterpret_cast<float2 *>(interleaved);
  const float2 *tw = reinterpret_cast<const float2 *>(HostTwiddle512());
  for (int pass = 0; pass < 3; ++pass)
    for (int b = 0; b < 64; ++b) Radix8Butterfly(buf, tw, pass, b);
  for (unsigned p = 0; p < (unsigned)kFft; ++p) {
    const unsigned r = OctRev3(p);
    if (r > p) {
      const float2 t = buf[p];
      buf[p] = buf[r];
      buf[r] = t;
    }
  }
}

/* CalcFIRCoeffs type 0, FIR.cpp:908-980: n_taps samples of a Kaiser-windowed sinc taken at
 * ii = -n, -n+2, ..., n-2 (centre index n/2: one tap off symmetric, B20). */
void DesignKaiserLowpass(float *taps, int n_taps, float cutoff_hz, float stop_db, float fs_hz) {
  float beta;
  float fc = cutoff_hz / fs_hz;
  if (stop_db < 20.96) beta = 0.0;
  else if (stop_db >= 50.0) beta = 0.1102 * (stop_db - 8.71);
  else beta = 0.5842 * powf((stop_db - 20.96), 0.4) + 0.07886 * (stop_db - 20.96);
  const float i0_beta = BesselI0Series(beta);
  const float fcf = fc * 2.0;
  int out = 0;
  for (int ii = -n_taps; ii < n_taps; ii += 2, ++out) {
    const float x = (float)ii / (float)n_taps;
    const float w = BesselI0Series(beta * sqrtf(1.0f - x * x)) / i0_beta;
    taps[out] = fcf * SincHalfPi(ii, fcf) * w;
  }
}

/* CalcCplxFIRCoeffs, FIR.cpp:1008-1065, 4-term Blackman-Harris window (FIR_filter_window == 1) */
void DesignComplexBandpass(float *taps_re, float *taps_im, int n_taps, float lo_hz, float hi_hz, float fs_hz) {
  const float nFL = lo_hz / fs_hz;
  const float nFH = hi_hz / fs_hz;
  const float nFc = (nFH - nFL) / 2.0;
  const float nFs = kPiF * (nFH + nFL);
  const float centre = 0.5 * (float)(n_taps - 1);
  const float four_pi = 2.0f * kTwoPiF;
  const float six_pi = 3.0f * kTwoPiF;
  for (int i = 0; i < n_taps; ++i) {
    const float x = (float)i - centre;
    const float dist = x > 0 ? x : -x;
    float z;
    if (dist < 0.01) {
      z = 2.0 * nFc;
    } else {
      z = (float)sinf(kTwoPiF * x * nFc) / (kPiF * x) *
          (0.35875 - 0.48829 * cosf((kTwoPiF * i) / (n_taps - 1)) +
           0.14128 * cosf((four_pi * i) / (n_taps - 1)) -
           0.01168 * cosf((six_pi * i) / (n_taps - 1)));
    }
    taps_re[i] = z * cosf(nFs * x);
    taps_im[i] = z * sinf(nFs * x);
  }
}

/* SetIIRCoeffs(3000, 1.3, 24000, lowpass), FIR.cpp:1076-1106; designed once at start-up
 * for the default band and never redone (T41_SDR.ino:560-566, B16). */
void DesignAmLowpass(float *c) {
  float f0 = (float)3000;
  const float q = 1.3;
  const float fs = (float)kFs / kDf;
  if (f0 > fs / 2.0) f0 = fs / 2.0;
  const float w0 = f0 * (kTwoPiF / fs);
  const float sn = sinf(w0);
  const float alpha = sn / (q * 2.0);
  const float cs = cosf(w0);
  const float scale = 1.0 / (1.0 + alpha);
  c[0] = ((1.0 - cs) / 2.0) * scale;
  c[1] = (1.0 - cs) * scale;
  c[2] = c[0];
  c[3] = (2.0 * cs) * scale;
  c[4] = (-1.0 + alpha) * scale;
}

void AgcStickyDefaults(AgcSticky *s) {   /* AGCPrep, DSP_Fn.cpp:444-465 */
  s->hangtime = 0.250;
  s->tau_decay = 0.250;
  s->hang_thresh = 0.250;
}

/* AGCLoadValues, DSP_Fn.cpp:368-435, with AGCPrep's fixed tuning values */
void DesignAgc(AgcSticky *st, int agc_mode, int agc_thresh, AgcConsts *o, int *attack_buffsize) {
  const float tau_attack = 0.001;
  const int n_tau = 4;
  const float max_input = 1.0;
  const float out_targ = 1.0;
  const float var_gain = 1.5;
  const float tau_fast_backaverage = 0.250;
  const float tau_fast_decay = 0.005;
  const float tau_hang_backmult = 0.500;
  const float tau_hang_decay = 0.100;
  const float sample_rate = (float)kFs / kDf;
  switch (agc_mode) {
    case 1: st->hangtime = 2.000; st->tau_decay = 2.000; break;
    case 2: st->hangtime = 1.000; st->tau_decay = 0.5; break;
    case 3: st->hang_thresh = 1.0; st->hangtime = 0.000; st->tau_decay = 0.250; break;
    case 4: st->hang_thresh = 1.0; st->hangtime = 0.0; st->tau_decay = 0.050; break;
    default: break;
  }
  float tmp;
  o->max_gain = powf(10.0, (float)agc_thresh / 20.0);
  *attack_buffsize = (int)ceil(sample_rate * n_tau * tau_attack);
  o->attack_mult = 1.0 - expf(-1.0 / (sample_rate * tau_attack));
  o->decay_mult = 1.0 - expf(-1.0 / (sample_rate * st->tau_decay));
  o->fast_decay_mult = 1.0 - expf(-1.0 / (sample_rate * tau_fast_decay));
  o->fast_backmult = 1.0 - expf(-1.0 / (sample_rate * tau_fast_backaverage));
  o->onemfast_backmult = 1.0 - o->fast_backmult;
  o->out_target = out_targ * (1.0 - expf(-(float)n_tau)) * 0.9999;
  o->min_volts = o->out_target / (var_gain * o->max_gain);
  tmp = log10f(o->out_target / (max_input * var_gain * o->max_gain));
  if (tmp == 0.0) tmp = 1e-16;
  o->slope_constant = (o->out_target * (1.0 - 1.0 / var_gain)) / tmp;
  o->inv_max_input = 1.0 / max_input;
  tmp = powf(10.0, (st->hang_thresh - 1.0) / 0.125);
  o->hang_level = (max_input * tmp + (o->out_target / (var_gain * o->max_gain)) * (1.0 - tmp)) * 0.637;
  o->hang_backmult = 1.0 - expf(-1.0 / (sample_rate * tau_hang_backmult));
  o->onemhang_backmult = 1.0 - o->hang_backmult;
  o->hang_decay_mult = 1.0 - expf(-1.0 / (sample_rate * tau_hang_decay));
  o->hangtime = st->hangtime;
  o->fixed_gain = 20.0;
  o->pop_ratio = 5.0;
  o->hang_enable = 1;
  o->hang_counter_load = (int)(st->hangtime * kFs / kDf);
  o->pad_ = 0;
}

/* CalcFilters -> CalcCplxFIRCoeffs + InitFilterMask + SetDecIntFilters (Filter.cpp:235-418);
 * NFM re-designs the two decimators for nfmFilterBW at every block (Process.cpp:259,
 * Filter.cpp:429-438), which is the same as carrying those taps while the mode is NFM. */
void DesignFilterSet(const t41rx_params &p, FilterSet *fs) {
  memset(fs, 0, sizeof(*fs));
  float re[kMaskTaps], im[kMaskTaps];
  DesignComplexBandpass(re, im, kMaskTaps, (float)p.f_lo_cut, (float)p.f_hi_cut, (float)kFs / kDf);
  for (int i = 0; i < kMaskTaps; ++i) {
    fs->mask[2 * i] = re[i];
    fs->mask[2 * i + 1] = im[i];
  }
  /* InitFilterMask zeroes from float index FFT_length + 1 = 513 on: the imaginary part of
     tap 256 is dropped (B7) */
  for (int i = kFft + 1; i < 2 * kFft; ++i) fs->mask[i] = 0.0;
  HostFft512(fs->mask);

  int widest = p.f_hi_cut;
  if (widest < -p.f_lo_cut) widest = -p.f_lo_cut;
  int lp = widest;
  if (lp > 10000) lp = 10000;
  if (p.mode == T41RX_DEMOD_NFM) {
    DesignKaiserLowpass(fs->dec1, kDec1Taps, (float)p.nfm_filter_bw, kStopDb, (float)kFs);
    DesignKaiserLowpass(fs->dec2, kDec2Taps, (float)p.nfm_filter_bw, kStopDb, (float)(kFs / kDf1));
  } else {
    DesignKaiserLowpass(fs->dec1, kDec1Taps, (float)lp, kStopDb, (float)kFs);
    DesignKaiserLowpass(fs->dec2, kDec2Taps, (float)lp, kStopDb, (float)(kFs / kDf1));
  }
  DesignKaiserLowpass(fs->int1, kInt1Taps, (float)lp, kStopDb, (float)(kFs / kDf1));
  DesignKaiserLowpass(fs->int2, kInt2Taps, (float)lp, kStopDb, (float)kFs);
}

void DesignStreamCfg(const t41rx_params &p, const AgcConsts &agc, int filter_id, StreamCfg *c) {
  const int32_t keep_epoch = c->nco_epoch;
  memset(c, 0, sizeof(*c));
  c->nco_epoch = keep_epoch;
  c->mode = p.mode;
  c->agc_mode = p.agc_mode;
  c->zoom = p.spectrum_zoom;
  c->filter_id = filter_id;
  c->psk31_enable = p.psk31_enable;
  c->mirrored = (p.mode == T41RX_DEMOD_USB || p.mode == T41RX_DEMOD_LSB || p.mode == T41RX_DEMOD_AM ||
                 p.mode == T41RX_DEMOD_SAM) ? 1 : 0;
  c->pixel_add = t41rx_base_offset[p.current_scale] + (int16_t)p.pixel_offset;
  c->wf_base = p.spectrum_noise_floor - p.current_nf;
  c->current_nf = p.current_nf;
  c->eq_on = (p.receive_eq_flag == 1) ? 1 : 0;                       /* Process.cpp:828 */
  c->nr_lms = (p.nr_option == 3) ? 1 : 0;                            /* Process.cpp:852 */
  c->anr_notch = (p.anr_notch_on == 1) ? 1 : 0;                      /* Process.cpp:860 */
  c->cw_filter = (p.cw_receive == 1 && p.cw_filter_index != 5) ? p.cw_filter_index : -1;   /* Process.cpp:878-912 */
  c->nr_kim = (p.nr_option == 1) ? 1 : 0;                            /* Process.cpp:845 */
  c->nr_spectral = (p.nr_option == 2) ? 1 : 0;                       /* Process.cpp:850 */
  c->nb_on = (p.nb_on != 0) ? 1 : 0;                                 /* Process.cpp:873 */
  {
    /* VAD_low / VAD_high (Noise.cpp:141-172 = :429-443,515-529): the bins between the filter cut-offs, bin width
       (SampleRate / DF) / NR_FFT_L = 93.75 Hz; the reference keeps them in uint8_t */
    float lf_freq, uf_freq;
    if (p.f_lo_cut <= 0 && p.f_hi_cut >= 0) {
      lf_freq = 0.0;
      uf_freq = fmax(-(float)p.f_lo_cut, (float)p.f_hi_cut);
    } else if (p.f_lo_cut > 0) {
      lf_freq = (float)p.f_lo_cut;
      uf_freq = (float)p.f_hi_cut;
    } else {
      uf_freq = -(float)p.f_lo_cut;
      lf_freq = -(float)p.f_hi_cut;
    }
    lf_freq /= (((float)kFs / kDf) / 256);
    uf_freq /= (((float)kFs / kDf) / 256);
    uint8_t lo = (uint8_t)(int)lf_freq, hi = (uint8_t)(int)uf_freq;
    if (lo == hi) hi++;
    if (lo < 1) lo = 1;
    else if (lo > 256 / 2 - 2) lo = 256 / 2 - 2;
    if (hi < 1) hi = 1;
    else if (hi > 256 / 2) hi = 256 / 2;
    c->nr_vad_lo = lo;
    c->nr_vad_hi = hi;
  }
  for (int i = 0; i < 14; ++i) {                                     /* Filter.cpp:118-120,136-149 */
    const float level = (float)p.equalizer_rec[i] / 100.0;
    c->eq_scale[i] = (i & 1) ? level : -level;
  }
  int zs = kBlock / (1 << p.spectrum_zoom);
  if (zs > kSpecRes) zs = kSpecRes;
  c->zoom_samples = zs;

  c->rf_gain_value = pow(10, (float)p.rf_gain_all_bands / 20);        /* Process.cpp:117 */
  c->neg_iq_amp = -p.iq_amp_correction;
  c->iq_phase = p.iq_phase_correction;
  float fcut_khz;                                                      /* Process.cpp:482-490 */
  if (p.mode == T41RX_DEMOD_LSB) fcut_khz = -(float)p.f_lo_cut * 0.001;
  else fcut_khz = (float)p.f_hi_cut * 0.001;
  c->vol_scale = 7.0874 * pow(fcut_khz, -1.232);
  {                                                                    /* Process.cpp:929,955-967 */
    const float x = p.audio_volume / 100.0f;
    const float ampl = 5 * x * x * x * x * x;
    c->volume = kDf * ampl;
  }
  c->db_scale = t41rx_db_scale[p.current_scale];
  c->zoom_mult = (float)p.spectrum_zoom;                               /* FFT.cpp:105-108 */
  if (p.spectrum_zoom > 3) c->zoom_mult = (float)(1 << p.spectrum_zoom);
  {                                                                    /* FFT.cpp:38-39 */
    const float fstop = 0.5 * (float)kFs / (1 << p.spectrum_zoom);
    DesignKaiserLowpass(c->zoom_fir, 4, fstop, 60, (float)kFs);
  }
  DesignAmLowpass(c->am_lp);
  c->agc = agc;

  /* FreqShift2 set-up, Freq_Shift.cpp:121-124.  NCO_INC is a float32 and cos()/sin() of a
     float argument resolve to the single-precision overloads under ISO C++ (<cmath>), so
     the rotation matrix holds float-accurate entries widened to double. */
  const float nco_inc = 2.0 * kPiF * (long)p.nco_freq / 192000.0;
  const float cf = cosf(nco_inc);
  const float sf = sinf(nco_inc);
  c->osc_cos = (double)cf;
  c->osc_sin = (double)sf;
  /* closed-form description of the same oscillator: per-sample rotation angle, the radial
     gain rho of the (not exactly orthonormal) matrix, and the amplitude the 1.95 - |V|^2
     control loop settles to: |V|^2 = 1.95 - 1/rho, |Osc| = rho * |V| */
  const long double cl = (long double)c->osc_cos, sl = (long double)c->osc_sin;
  const long double two_pi = 6.283185307179586476925286766559005768L;
  const long double delta = atan2l(sl, cl);
  const long double rho = sqrtl(cl * cl + sl * sl);
  long double blk = fmodl(2048.0L * delta, two_pi);
  if (blk < 0) blk += two_pi;
  const long double r2 = 1.95L - 1.0L / rho;
  c->nco_delta = (double)delta;
  c->nco_block_delta = (double)blk;
  c->nco_rho = (double)rho;
  c->nco_r2_fix = (double)r2;
  c->nco_amp = (double)(rho * sqrtl(r2));
}

int ValidateParams(const t41rx_params &p) {
  switch (p.mode) {
    case T41RX_DEMOD_USB: case T41RX_DEMOD_LSB: case T41RX_DEMOD_AM:
    case T41RX_DEMOD_NFM: case T41RX_DEMOD_PSK31: case T41RX_DEMOD_SAM: break;
    default: return 0;
  }
  if (p.agc_mode < 0 || p.agc_mode > 4) return 0;
  if (p.spectrum_zoom < 0 || p.spectrum_zoom > 4) return 0;
  if (p.current_scale < 0 || p.current_scale > 4) return 0;
  if (p.f_hi_cut <= p.f_lo_cut) return 0;
  if (p.audio_volume < 0 || p.audio_volume > 100) return 0;
  /* the range over which the throughput kernel holds its tolerance (t41rx.h) */
  if (p.rf_gain_all_bands < -T41RX_RF_GAIN_ALL_BANDS_MAX || p.rf_gain_all_bands > T41RX_RF_GAIN_ALL_BANDS_MAX) return 0;
  if (p.nr_option < 0 || p.nr_option > 3) return 0;
  if (p.cw_filter_index < 0 || p.cw_filter_index > 5) return 0;
  return 1;
}

}  // namespace t41rx
