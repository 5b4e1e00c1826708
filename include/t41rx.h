/*
 * t41rx.h — C-ABI of the B200-native T41 receive chain (libt41rx.so).
 *
 * Drop-in boundary for the reference's per-block receive pipeline
 *     void ProcessIQData(void)            software/T41_SDR/Process.h:15, Process.cpp:70-944
 * batched over n_streams independent virtual receivers.  The reference passes
 * every input and output through globals; each of them becomes an explicit
 * argument or a field of t41rx_params here (reference location cited per field).
 * Plain pointers and sizes only; no C++ or torch types cross this boundary.
 *
 * Buffer layouts (row-major):
 *   iq         float  [n_streams][n_blocks][2048][2]   interleaved (I,Q) at 192 kS/s, i.e. what
 *                                                       arm_q15_to_float produced (Process.cpp:107-108;
 *                                                       I = Q_in_R, Q = Q_in_L)
 *   audio      float  [n_streams][n_blocks][2048]      float_buffer_L after the volume scale
 *                                                       (Process.cpp:929), before arm_float_to_q15
 *   spec_rows  int16  [n_streams][n_rows][512]         pixelnew[] (FFT.cpp:157,245)
 *   wf_rows    uint16 [n_streams][n_rows][512]         waterfall[] RGB565 (Display.cpp:459-466);
 *                                                       element 511 is never written by the reference: 0
 *   psk_bits   int8   [n_streams][n_blocks]            -1 = no symbol decision in this block, else 0/1
 *   psk_chars  uint8  [n_streams][n_blocks]            decoded varicode character or 0
 * A block b of a call is "row-producing" (updateDisplayFlag == 1, Display.cpp:261-267) when
 * row_every > 0 and b % row_every == 0; n_rows = ceil(n_blocks / row_every).
 *
 * Every entry point returns 0 on success or a negative T41RX_E* code; the text of the
 * last failure on the calling thread is available from t41rx_last_error().  The library
 * has no CPU fallback: without a CUDA device t41rx_create fails.
 */
#ifndef T41RX_H
#define T41RX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define T41RX_BLOCK_SAMPLES 2048   /* BUFFER_SIZE * N_BLOCKS, T41_SDR.ino:368-369 */
#define T41RX_SPECTRUM_RES 512     /* SPECTRUM_RES, Display.h:12 */

/* demodulation modes: values of SDT.h:57-68 */
#define T41RX_DEMOD_USB 0
#define T41RX_DEMOD_LSB 1
#define T41RX_DEMOD_AM 2
#define T41RX_DEMOD_NFM 3
#define T41RX_DEMOD_PSK31 5
#define T41RX_DEMOD_SAM 8

#define T41RX_OK 0
#define T41RX_EINVAL -1    /* bad argument / parameter out of range */
#define T41RX_ECUDA -2     /* CUDA runtime failure (text in t41rx_last_error) */
#define T41RX_ENOMEM -3
#define T41RX_ENODEV -4    /* no usable CUDA device: there is no CPU path */

/* t41rx_process flags */
#define T41RX_FLAG_EXACT_NCO 1u /* bit-exact kernel, FreqShift2's FP64 oscillator recurrence run step by step:
                                   every output identical to the reference build, slow */
#define T41RX_FLAG_PHASED_KERNEL 2u /* bit-exact kernel with the closed-form FP64 oscillator (all other stages
                                   still rounded operation by operation like the reference) */
#define T41RX_FLAG_SCAN_ROWS 4u /* display spectrum: ZoomFFT's biquad cascade as blocked scans (rows kernel 4 % faster at C4: 23.5 against 22.7 M rows/s); rows
                                   then differ from the reference by at most 1 LSB in < 1 % of the pixels instead of
                                   being identical */
#define T41RX_FLAG_FAST_LMS 8u /* receivers with the LMS noise reduction / automatic notch on also run on the throughput
                                   kernel (by default they stay on the bit-exact one): the notch cancels most of its input,
                                   so FP32 re-ordering shows 20-30 dB stronger in what is left: audio SNR >= 70 dB */
#define T41RX_FLAG_FAST_SAM 16u /* SAM receivers also run on the throughput kernel (by default they stay on the bit-exact
                                   one, ~9x slower): identical to the reference only in the statistical sense while
                                   the PLL pulls in (its acquisition is chaotic: ApproxAtan2's 2 pi quirk), within the
                                   stated tolerance once it is locked */
#define T41RX_FLAG_FUSED_EXACT 32u /* developer / comparison switch: run the bit-exact chain as the single fused kernel
                                   (serial stages on one lane per receiver) instead of its front | serial | back
                                   kernels (serial stages with thread = receiver); same results bit for bit, ~3x slower */
/* flags == 0: the throughput kernel (FP32 with FMA contraction, blocked-scan recurrences): audio within
   the stated tolerance of the reference (SNR >= 90 dB), discrete state identical */

/* rf_gain_all_bands outside +-40 dB is EINVAL (t41rx_set_params*).  The throughput kernel (flags 0) meets its stated
   tolerance across this range, including a step from one end to the other between calls (measured on a B200: >= 101 dB,
   every mode and AGC mode).  Beyond it the margin goes: 94 dB for AM at a 100 dB step, below 90 dB from 120 dB steps
   (AM 88 dB; NFM 68-80 dB at 200 dB), and from about -760 dB the FP32 gain rounds to a denormal or 0,
   where the kernel's gain-normalised DC-block state became 0 / 0 (NaN audio). */
#define T41RX_RF_GAIN_ALL_BANDS_MAX 40

/* Per-receiver parameters = the globals ProcessIQData() samples at block start. */
typedef struct t41rx_params {
  int32_t mode;                 /* bands[currentBand].mode        SDT.h:179-192, Process.cpp:251,615 */
  int32_t f_lo_cut;             /* bands[].FLoCut (Hz)            Filter.cpp:239                      */
  int32_t f_hi_cut;             /* bands[].FHiCut (Hz)            Filter.cpp:239                      */
  int32_t nco_freq;             /* NCOFreq (Hz)                   Freq_Shift.cpp:121                  */
  int32_t agc_mode;             /* AGCMode 0..4                   DSP_Fn.cpp:373,494                  */
  int32_t agc_thresh;           /* bands[].AGC_thresh (dB)        DSP_Fn.cpp:408                      */
  int32_t audio_volume;         /* audioVolume 0..100             Process.cpp:929                     */
  int32_t rf_gain_all_bands;    /* rfGainAllBands (dB), |value| <= T41RX_RF_GAIN_ALL_BANDS_MAX  Process.cpp:117 */
  int32_t rf_gain;              /* bands[].RFgain start value     Process.cpp:133 (then Codec_gain)   */
  int32_t spectrum_zoom;        /* spectrumZoom index 0..4        Process.cpp:185,212                 */
  int32_t current_scale;        /* currentScale 0..4              FFT.cpp:157                         */
  int32_t pixel_offset;         /* bands[].pixel_offset           FFT.cpp:157                         */
  int32_t current_nf;           /* currentNoiseFloor[band]        Display.cpp:250,343                 */
  int32_t spectrum_noise_floor; /* spectrumNoiseFloor             Display.cpp:343                     */
  int32_t nfm_filter_bw;        /* nfmFilterBW (Hz)               Process.cpp:259                     */
  int32_t psk31_enable;         /* DBPSK + varicode tap on the filtered stream (psk31.cpp:235-310)    */
  float iq_amp_correction;      /* IQAmpCorrectionFactor[band]    Process.cpp:166,171                 */
  float iq_phase_correction;    /* IQPhaseCorrectionFactor[band]  Process.cpp:167,172                 */
  int32_t receive_eq_flag;      /* receiveEQFlag (ON = 1)         Process.cpp:827-831                 */
  int32_t equalizer_rec[14];    /* EEPROMData.equalizerRec[] 0..100 (default 100)  Filter.cpp:117-165 */
  int32_t nr_option;            /* nrOptionSelect: 0 off, 1 Kim (Kim1_NR, then x 30), 2 spectral
                                   (SpectralNoiseReduction), 3 LMS (Xanr)   Process.cpp:841-857, Noise.cpp:108-655 */
  int32_t anr_notch_on;         /* ANR_notchOn: automatic notch (Xanr)  Process.cpp:860-865           */
  int32_t cw_receive;           /* T41State == CW_RECEIVE: the CW audio low-pass below is in the chain (the CW decoder
                                   of that state, DoCWReceiveProcessing, is out of scope)  Process.cpp:878 */
  int32_t cw_filter_index;      /* CWFilterIndex 0..4 = 0.8 / 1.0 / 1.3 / 1.8 / 2.0 kHz, 5 = off (default)  Process.cpp:882-912 */
  int32_t nb_on;                /* NB_on: the LPC impulse blanker (NoiseBlanker / AltNoiseBlanking) behind the notch; default 0
                                   Process.cpp:39,873-876, DSP_Fn.cpp:105-362 */
} t41rx_params;

/* Discrete / scalar DSP state for state-transition parity checks. */
typedef struct t41rx_debug {
  int32_t agc_state;            /* DSP_Fn.cpp:483 */
  int32_t agc_decay_type;       /* DSP_Fn.cpp:482 */
  int32_t agc_hang_counter;     /* DSP_Fn.cpp:32  */
  int32_t agc_action;           /* DSP_Fn.cpp:28  */
  int32_t rf_gain;              /* bands[].RFgain after Codec_gain, Process.cpp:1005 */
  int32_t codec_timer;          /* Process.cpp:980 */
  int32_t zoom_sample_ptr;      /* FFT.cpp:13 */
  int32_t first_block;          /* Process.cpp:47 */
  float agc_volts;
  float agc_ring_max;
  float agc_save_volts;
  float agc_fast_backaverage;
  float agc_hang_backaverage;
  float sam_phzerror;           /* Demod.cpp:19 */
  float sam_omega2;             /* Demod.cpp:23 */
  float sam_fil_out;            /* Demod.cpp:21 */
  float dc_state[2];            /* HP_DC_Butter_state2, Process.cpp:42 */
  float am_wold;                /* Process.cpp:73 */
  double osc_vect_q;            /* Freq_Shift.cpp:13 */
  double osc_vect_i;            /* Freq_Shift.cpp:14 */
} t41rx_debug;

/* The control-path tables a receiver currently uses (CalcFilters / AGCLoadValues /
 * ZoomFFTPrep results), for table-level parity checks. */
typedef struct t41rx_tables {
  float dec1[28];               /* FIR_dec1_coeffs  Filter.cpp:412 */
  float dec2[46];               /* FIR_dec2_coeffs  Filter.cpp:413 */
  float int1[48];               /* FIR_int1_coeffs  Filter.cpp:415 */
  float int2[32];               /* FIR_int2_coeffs  Filter.cpp:416 */
  float mask[1024];             /* FIR_filter_mask  Filter.cpp:260-284 */
  float am_lp[5];               /* biquad_lowpass1_coeffs T41_SDR.ino:560-566 */
  float zoom_fir[4];            /* Fir_Zoom_FFT_Decimate_coeffs FFT.cpp:39 */
  float agc[16];                /* max_gain, attack_mult, decay_mult, fast_decay_mult, fast_backmult,
                                   onemfast_backmult, out_target, min_volts, slope_constant, inv_max_input,
                                   hang_level, hang_backmult, onemhang_backmult, hang_decay_mult, hangtime,
                                   fixed_gain (DSP_Fn.cpp:408-434) */
  int32_t attack_buffsize;      /* DSP_Fn.cpp:409 */
  int32_t hang_counter_load;    /* DSP_Fn.cpp:554 */
} t41rx_tables;

typedef struct t41rx_ctx t41rx_ctx;

/* Reference defaults (gwv.cpp:15-25,70-74; bands[] T41_SDR.ino:163-167). */
void t41rx_default_params(t41rx_params *p);
/* FLoCut/FHiCut presets a mode change applies (SetupMode, Filter.cpp:341-385). */
void t41rx_mode_default_cuts(int32_t mode, int32_t *f_lo_cut, int32_t *f_hi_cut);

/* A context owns n_streams receivers on ONE CUDA device (t41rx_create_multi below shards a bank over several
 * devices in one process; one process per GPU with a context each works too).  Every receiver starts in the state
 * InitializeDataArrays() + SoftReset() leave the firmware in (T41_SDR.ino:473-667,753-795). */
int t41rx_create(t41rx_ctx **out, int n_streams, int device);
void t41rx_destroy(t41rx_ctx *ctx);
int t41rx_num_streams(const t41rx_ctx *ctx);

/* Parameter changes take effect at the next block boundary, like CalcFilters() /
 * AGCLoadValues() / ZoomFFTPrep() running between two ProcessIQData() calls
 * (Display.cpp:270-275, MenuProc.cpp:275-284, Display.cpp:1402-1417).
 * set_params applies *p to streams [first, first+count); set_params_each takes count structs. */
int t41rx_set_params(t41rx_ctx *ctx, int first, int count, const t41rx_params *p);
int t41rx_set_params_each(t41rx_ctx *ctx, int first, int count, const t41rx_params *p);
int t41rx_get_params(const t41rx_ctx *ctx, int stream, t41rx_params *p);
int t41rx_get_tables(const t41rx_ctx *ctx, int stream, t41rx_tables *t);
int t41rx_get_debug(t41rx_ctx *ctx, int stream, t41rx_debug *d);
/* Control path only, no GPU needed: the tables a fresh receiver holds after n_seq successive
 * t41rx_set_params calls (sticky AGC tuning included, DSP_Fn.cpp:378-402). */
int t41rx_design_tables(const t41rx_params *seq, int n_seq, t41rx_tables *t);

/* n_blocks ProcessIQData() calls per receiver, HOST buffers (pinned or pageable); copies to and
 * from the device happen inside.  spec_rows / wf_rows may be NULL when row_every == 0;
 * psk_bits / psk_chars may be NULL. */
int t41rx_process(t41rx_ctx *ctx, const float *iq, float *audio, int n_blocks, int row_every,
                  int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars,
                  uint32_t flags);

/* The same call on the firmware's own block format: q15 I/Q in (what the codec queues Q_in_R / Q_in_L hold,
 * interleaved (I,Q): arm_q15_to_float = x / 32768, Process.cpp:107-108) and q15 audio out (what Q_out_L.play
 * gets: arm_float_to_q15 = saturate(trunc(x * 32768)), Process.cpp:936-937).  HOST buffers; the conversions
 * run inside the chain kernels (at their loads and stores), so half as many bytes cross the host link and HBM as
 * with the float entry point.
 *   iq_q15     int16 [n_streams][n_blocks][2048][2]      audio_q15  int16 [n_streams][n_blocks][2048] */
int t41rx_process_q15(t41rx_ctx *ctx, const int16_t *iq_q15, int16_t *audio_q15, int n_blocks, int row_every,
                      int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars,
                      uint32_t flags);

/* Same, with DEVICE pointers (resident in HBM) and an optional cudaStream_t (NULL = the
 * context's own stream).  Asynchronous: returns after enqueueing.
 * Ordering contract: the context records the end of the call on the stream it was given.  t41rx_set_params*,
 * t41rx_get_debug, t41rx_synchronize, t41rx_destroy and the host-buffer entry points wait for that point (and for
 * the context's own streams) before they touch device tables or state, so they are safe after a call on ANY stream.
 * Two t41rx_process_device calls on DIFFERENT streams are not ordered against each other by the library: the
 * receivers' state lives in the context, so the caller must order them (one stream, or an event between them). */
int t41rx_process_device(t41rx_ctx *ctx, const float *iq, float *audio, int n_blocks, int row_every,
                         int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars,
                         uint32_t flags, void *cuda_stream);
/* t41rx_process_device on q15 blocks resident in HBM (layouts of t41rx_process_q15): the firmware's own block format
 * end to end, 12 KiB of HBM traffic per stream-block instead of 24. */
int t41rx_process_device_q15(t41rx_ctx *ctx, const int16_t *iq_q15, int16_t *audio_q15, int n_blocks, int row_every,
                             int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars,
                             uint32_t flags, void *cuda_stream);
int t41rx_synchronize(t41rx_ctx *ctx);

/* ---- a bank over several CUDA devices (SURVEY 8(b), 8(e)) ----
 * n_streams receivers sharded over n_dev devices: device_ids[g] owns the contiguous range [g n / N, (g + 1) n / N) in a
 * single-device context of its own; every call fans out to one host thread per device.  No inter-GPU traffic on the
 * hot path; the optional gather of rows is the only collective.  A device id may be listed more than once (several
 * shards on one GPU).  Failures: negative T41RX_E* code, text in t41rx_multi_last_error() (it names the shard). */
typedef struct t41rx_multi t41rx_multi;
int t41rx_create_multi(t41rx_multi **out, int n_streams, const int *device_ids, int n_dev);
void t41rx_destroy_multi(t41rx_multi *m);
int t41rx_multi_num_devices(const t41rx_multi *m);
int t41rx_multi_num_streams(const t41rx_multi *m);
/* shard g: its device, receiver range and single-device context (for the per-context calls above); any may be NULL */
int t41rx_multi_shard(const t41rx_multi *m, int shard, int *device, int *first, int *count, t41rx_ctx **ctx);
/* receiver indices are those of the whole bank */
int t41rx_multi_set_params(t41rx_multi *m, int first, int count, const t41rx_params *p);
int t41rx_multi_set_params_each(t41rx_multi *m, int first, int count, const t41rx_params *p);
int t41rx_multi_get_debug(t41rx_multi *m, int stream, t41rx_debug *d);
/* t41rx_process / t41rx_process_q15 on HOST buffers of the whole bank: every device works on its slice concurrently */
int t41rx_multi_process(t41rx_multi *m, const float *iq, float *audio, int n_blocks, int row_every, int16_t *spec_rows,
                        uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars, uint32_t flags);
int t41rx_multi_process_q15(t41rx_multi *m, const int16_t *iq_q15, int16_t *audio_q15, int n_blocks, int row_every,
                            int16_t *spec_rows, uint16_t *wf_rows, int8_t *psk_bits, uint8_t *psk_chars, uint32_t flags);
/* device-resident: arrays of n_dev DEVICE pointers, entry g on shard g's device with that shard's receivers
 * ([count][n_blocks][...]); asynchronous on every context's own stream; spec_rows / wf_rows may be NULL */
int t41rx_multi_process_device(t41rx_multi *m, const float *const *iq, float *const *audio, int n_blocks, int row_every,
                               int16_t *const *spec_rows, uint16_t *const *wf_rows, uint32_t flags);
int t41rx_multi_synchronize(t41rx_multi *m);
/* optional collective: the shards' row buffers (rows[g] on shard g's device, bytes_per_receiver bytes per receiver, e.g.
 * n_rows * 512 * 2) gathered into dst on device_ids[0] in receiver order; NCCL send / recv over NVLink / NVSwitch when
 * libnccl can be loaded and the devices are distinct, else peer copies; blocking; *used_nccl (may be NULL) reports it */
int t41rx_multi_gather_rows(t41rx_multi *m, const void *const *rows, size_t bytes_per_receiver, void *dst, int *used_nccl);
const char *t41rx_multi_last_error(void);

/* ---- polyphase channelizer: one wideband capture -> the receivers' iq blocks (DESIGN §3.7) ----
 * The capture x[n] is interleaved complex float at Fs_in = M x 96 kS/s, M = n_channels in {64, 320, 512, 640} (6.144,
 * 30.72, 49.152 or 61.44 MS/s; 30.72 and 61.44 are the LTE-family rates of AD936x / USRP N3xx digitizers, DESIGN
 * §3.10); n counts samples since t41rx_chan_create, x[n < 0] = 0.  Prototype h[0..N), N = 10 M: Kaiser-windowed
 * sinc (beta 8.96), cutoff 96 kHz, designed in FP64, symmetric, unit DC gain, rounded to float: flat to +-60 kHz,
 * <= -90 dB from 132 kHz.  Decimation D = M / 2: every channel comes out at 192 kS/s, channel k centred at
 * (k < M/2 ? k : k - M) x 96 kHz, so any frequency of the capture lies within 48 kHz of some centre.  Sample m of
 * channel k (m counted from the call's start; a call produces n_blocks x 2048 samples per channel):
 *     z_k[m] = conj( sum_{i<N} h[i] x[mD - i] exp(-j 2 pi k (mD - i) / M) )
 * The conjugate mirrors the channel: the chain's front end mirrors USB / LSB / AM / SAM once more (it negates I), so a
 * USB receiver hears the capture's upper sideband.  The channel lags the capture by (N - 1) / 2 capture samples.
 * The zoom x1 display spectrum of a receiver fed this way (it spans +-96 kHz) shows the prototype's roll-off beyond
 * +-60 kHz of the channel centre; a receiver placed by t41rx_chan_tune keeps its widest filter (10 kHz) inside the
 * flat +-60 kHz.  Cutting a run into several calls, or changing the map, gives
 * the same samples bit for bit.  Runs on the FP32 CUDA cores (sm_100a); there is no CPU path.
 * Fine tuning (opt-in, t41rx_chan_set_shift): receiver r mapped to channel k gets its channel rotated,
 *     iq_r[m] = z_k[m] exp(+j 2 pi phi_r(m) / 192000),   phi_r(m) = (P_r + shift_r m_abs) mod 192000  (integers),
 * m_abs counting the outputs since t41rx_chan_create, so the stream is moved up by shift_r Hz.  P_r starts at 0 and
 * t41rx_chan_set_shift sets it so that the phase is continuous at the change: the first output after it has the phase
 * the old shift would have given it.  A receiver whose shift was never set gets z_k bit for bit; cutting a run into
 * calls still gives the same bits, with or without shifts.  The chain's front end rejects the opposite sideband best at
 * NCOFreq 0 (72 dB; 19 dB at 48000, DESIGN §3.7) and decodes PSK31 there: t41rx_chan_place puts a receiver on that
 * operating point, t41rx_chan_tune (no shift) on NCOFreq 48000 +- f_rel. */
typedef struct t41rx_chan t41rx_chan;
/* n_receivers = the n_streams of the context the iq output feeds; every receiver starts unmapped (-1).  ENODEV without
 * a CUDA device, EINVAL for n_channels other than 64 / 320 / 512 / 640. */
int t41rx_chan_create(t41rx_chan **out, int n_channels, int n_receivers, int device);
void t41rx_chan_destroy(t41rx_chan *c);
/* receivers [first, first + count) take channel[i] in [0, n_channels), or -1 = not written (their iq rows keep whatever
 * the caller put there); several receivers may share a channel.  Effective from the next call. */
int t41rx_chan_set_map(t41rx_chan *c, int first, int count, const int32_t *channel);
/* receivers [first, first + count) rotated by shift_hz[i], |shift_hz[i]| < 192000 (EINVAL otherwise); every receiver
 * starts at 0.  Effective from the next call, with continuous phase; waits for the channelizer's calls like set_map. */
int t41rx_chan_set_shift(t41rx_chan *c, int first, int count, const int32_t *shift_hz);
/* DEVICE pointers (8-byte aligned), asynchronous on cuda_stream (NULL = the channelizer's own stream):
 *   capture  float [n_blocks * 2048 * n_channels / 2][2]     the next n_blocks * 2048 * D capture samples
 *   iq       float [n_receivers][n_blocks][2048][2]          t41rx_process_device's iq: block b holds m = 2048 b ...
 * Ordering contract of t41rx_process_device: the end of the call is recorded on the stream it was given, and
 * t41rx_chan_set_map, t41rx_chan_synchronize and t41rx_chan_destroy wait for it.  Two calls on different streams are
 * not ordered against each other by the library (the capture tail lives in the channelizer). */
int t41rx_chan_process_device(t41rx_chan *c, const float *capture, float *iq, int n_blocks, void *cuda_stream);
int t41rx_chan_synchronize(t41rx_chan *c);
/* Host only, no GPU needed: the prototype (10 * n_channels floats, h[0] first; n_channels 64, 128, 320, 512, 640, 800,
 * 1024 or 1280), and where to put a receiver whose carrier or dial point sits offset_hz from the capture's centre: the nearest channel centre (|f_rel| <= 48 kHz) and
 * nco_freq = 48000 + f_rel for USB / LSB / AM / SAM, 48000 - f_rel for NFM / PSK31 (rounded to integer Hz).  EINVAL
 * outside [-Fs_in / 2, Fs_in / 2) or for a mode t41rx_set_params rejects.  Offsets within 48 kHz below +Fs_in / 2 go
 * to channel M / 2, whose centre -Fs_in / 2 is the same frequency.  t41rx_chan_tune / t41rx_chan_place take the
 * complex channel counts 64, 320, 512 and 640. */
int t41rx_chan_taps(int n_channels, float *taps);
int t41rx_chan_tune(int n_channels, int32_t mode, double offset_hz, int32_t *channel, int32_t *nco_freq);
/* Host only, the placement to use with fine tuning: the channel t41rx_chan_tune picks, the shift that brings the
 * carrier or dial point to where the chain runs at *nco_freq, and that NCOFreq (0, the chain's best operating point):
 * shift_hz = 48000 + f_rel for USB / LSB / AM / SAM, f_rel - 48000 for NFM / PSK31 (rounded to integer Hz; the mirrored
 * modes see the stream conjugated).  Same EINVAL rules as t41rx_chan_tune. */
int t41rx_chan_place(int n_channels, int32_t mode, double offset_hz, int32_t *channel, int32_t *shift_hz,
                     int32_t *nco_freq);
/* Real captures (DESIGN §3.8), as a direct-sampling ADC delivers them: s[n] int16 at Fs_in = M x 96 kS/s, M =
 * n_channels in {128, 800, 1024, 1280} (12.288 MS/s: 0 - 6.144 MHz; 76.8 MS/s: 0 - 38.4 MHz, Hermes-Lite 2's ADC
 * clock; 98.304 MS/s: 0 - 49.152 MHz, all of HF; 122.88 MS/s: 0 - 61.44 MHz, the HPSDR family's ADC clock, DESIGN
 * §3.10).  x[n] = s[n] / 32768
 * (as arm_q15_to_float), then the formula above unchanged (prototype N = 10 M, D = M / 2, the conjugate).  Only
 * channels k = 0 ... M / 2 are distinct, channel k centred at +k x 96 kHz; a real tone A cos(2 pi f t) appears in its
 * channel with amplitude A / 2.  Mirror caveat: channel 0 holds its band together with its mirror image about 0 Hz,
 * channel M / 2 the same about Fs_in / 2, so a receiver placed below 48 kHz or above Fs_in / 2 - 48 kHz (channel 0 or
 * M / 2) hears the band and its mirror image at once.
 * t41rx_chan_set_map takes channels in [0, M / 2] on a real channelizer; set_map, set_shift, synchronize, destroy, the
 * iq layout, the phase rule and the ordering contract are those of the complex channelizer.
 * t41rx_chan_create_real: ENODEV without a CUDA device, EINVAL for n_channels other than 128 / 800 / 1024 / 1280.
 * t41rx_chan_process_device_real: capture int16 [n_blocks * 2048 * n_channels / 2], a DEVICE pointer, 16-byte aligned;
 * iq and cuda_stream as t41rx_chan_process_device.  Each kind of channelizer rejects the other kinds' process calls
 * (EINVAL).
 * t41rx_chan_tune_real / t41rx_chan_place_real: host only, freq_hz the absolute frequency in [0, Fs_in / 2] (EINVAL
 * outside it, for NaN, for a mode t41rx_set_params rejects, for n_channels other than 128 / 800 / 1024 / 1280): channel =
 * round(freq_hz / 96000), f_rel = freq_hz - channel x 96000, nco_freq and shift_hz by the rules of t41rx_chan_tune /
 * t41rx_chan_place. */
int t41rx_chan_create_real(t41rx_chan **out, int n_channels, int n_receivers, int device);
int t41rx_chan_process_device_real(t41rx_chan *c, const int16_t *capture, float *iq, int n_blocks, void *cuda_stream);
int t41rx_chan_tune_real(int n_channels, int32_t mode, double freq_hz, int32_t *channel, int32_t *nco_freq);
int t41rx_chan_place_real(int n_channels, int32_t mode, double freq_hz, int32_t *channel, int32_t *shift_hz,
                          int32_t *nco_freq);
/* Complex int16 captures (DESIGN §3.9), as wideband I/Q digitizers stream them (sc16: USRP-class, AD936x / LMS7002,
 * SDRplay): interleaved (I, Q) int16 pairs at Fs_in = M x 96 kS/s, M = n_channels in {64, 320, 512, 640}.  x[n] = (I[n] + j Q[n])
 * / 32768 (as arm_q15_to_float), then the complex channelizer unchanged: channels, fine tuning, t41rx_chan_tune /
 * t41rx_chan_place, set_map (channels [0, M)), set_shift, synchronize, destroy, the iq layout, the n_blocks limit and
 * the ordering contract.  The output is bit for bit that of t41rx_chan_create's channelizer fed with s / 32768 as
 * float (exact), while the capture takes half the bytes and needs no conversion pass.
 * t41rx_chan_create_q15: ENODEV without a CUDA device, EINVAL for n_channels other than 64 / 320 / 512 / 640.
 * t41rx_chan_process_device_q15: capture int16 [n_blocks * 2048 * n_channels / 2][2], a DEVICE pointer, 16-byte
 * aligned; iq and cuda_stream as t41rx_chan_process_device. */
int t41rx_chan_create_q15(t41rx_chan **out, int n_channels, int n_receivers, int device);
int t41rx_chan_process_device_q15(t41rx_chan *c, const int16_t *capture, float *iq, int n_blocks, void *cuda_stream);
/* Diversity (DESIGN §3.11): n_inputs in {2, 3, 4} coherent captures of one kind, sampled on one clock (sample n of every
 * input is the same instant: two to four ADCs of one digitizer), and one complex weight per (receiver, input).
 * Receiver r mapped to channel k gets
 *     iq_r[m] = rot_r(m) sum_a w[r][a] z^(a)_k[m]
 * where z^(a)_k is exactly what the single-input channelizer of that kind delivers for input a (same prototype, D,
 * conjugate; each input keeps its own tail) and rot_r is the fine-tuning rotation with its phase rule.  The weights
 * multiply the channel as delivered, after the conjugate: an input-1 copy c x of a complex interferer x on input 0
 * appears in channel k as conj(c) times input 0's, so it is nulled by w[r][1] = -w[r][0] / conj(c).  Each receiver has
 * its own weights, so each can null a different source or none.
 * kind: T41RX_CHAN_FLOAT, _Q15 or _REAL, with the n_channels that kind's create call takes.  Every receiver starts
 * unmapped, unshifted and with the default weights w[r][0] = 1, w[r][a > 0] = 0, with which it gets the single-input
 * channelizer's output for input 0 bit for bit.  EINVAL for an unknown kind, an n_channels the kind does not take or
 * n_inputs outside 2 ... 4; ENODEV without a CUDA device.
 * t41rx_chan_set_weights: receivers [first, first + count) take w[i][a] = (w[2 (i n_inputs + a)], w[2 (i n_inputs + a)
 * + 1]) (re, im), finite (EINVAL otherwise, and on a single-input channelizer).  Effective from the next call; it waits
 * for the channelizer's calls like set_map.  Weights change in a step at the call boundary: there is no ramp.
 * t41rx_chan_process_device_diversity: captures[a], a < n_inputs, DEVICE pointers with the layout and alignment of the
 * kind's process call (float: 8-byte, int16: 16-byte aligned); iq, the n_blocks limit, cuda_stream and the ordering
 * contract as t41rx_chan_process_device.  set_map, set_shift, synchronize, destroy and tune / place are the kind's.  A
 * diversity channelizer rejects the three single-input process calls, and a single-input one the diversity call
 * (EINVAL, naming the entry point it takes). */
#define T41RX_CHAN_FLOAT 0   /* kinds of t41rx_chan_create, _q15, _real */
#define T41RX_CHAN_Q15   1
#define T41RX_CHAN_REAL  2
int t41rx_chan_create_diversity(t41rx_chan **out, int kind, int n_channels, int n_inputs, int n_receivers, int device);
int t41rx_chan_set_weights(t41rx_chan *c, int first, int count, const float *w);
int t41rx_chan_process_device_diversity(t41rx_chan *c, const void *const *captures, float *iq, int n_blocks,
                                        void *cuda_stream);
/* Image correction (DESIGN §3.12): complex single-input channelizers (t41rx_chan_create, t41rx_chan_create_q15).  An
 * I/Q digitizer's gain, phase and delay mismatch between its I and Q branches puts an image of a signal at +f at -f,
 * so a carrier on channel k leaks into channel kbar = (M - k) mod M.  Each channel has a complex coefficient c_k (0 at
 * creation), and receiver r mapped to channel k gets
 *     y_k[m]  = z_k[m] + c_k conj(z_kbar[m])
 *     iq_r[m] = rot_r(m) y_k[m]
 * z_k being the channel as delivered without correction (after the conjugate); the fine-tuning rotation and its phase
 * rule are applied to y.  Channels 0 and M / 2 are their own mirrors.
 * Model: a frequency-independent imbalance x = mu s + nu conj(s) is removed on every channel by c_k = -conj(nu) / mu.
 * With gain g and phase phi on Q (Q' = g (Q cos phi + I sin phi)): mu = (1 + g e^(j phi)) / 2, nu = (1 - g e^(-j phi))
 * / 2.  An imbalance that varies with frequency (I/Q delay skew) needs a different c_k per channel, and different values
 * on k and kbar.
 * Bits: with every c_k exactly 0 and tracking off a call runs the uncorrected channelizer and gives its bits; a channel
 * whose c_k is 0 gets z_k unmodified (with its rotation rounded as without correction); with fixed coefficients,
 * cutting a run into calls gives the same bits; the q15 channelizer gives the float one's bits on s / 32768.
 * Tracking (opt-in, t41rx_chan_track_image): each call measures every mirror pair k = 0 ... M / 2 on its delivered y,
 * A = sum_m y_k y_kbar (no conjugate), P_k = sum |y_k|^2, P_kbar = sum |y_kbar|^2 over the call's outputs (whether or
 * not a receiver is mapped there), and for k = 1 ... M / 2 - 1 updates the coefficients the next call uses, on the
 * device, without a host synchronisation: if P_k >= T P_kbar, c_kbar -= A / P_k; else if P_kbar >= T P_k, c_k -= A /
 * P_kbar; else the pair is left alone (only the weak side of a pair where the other dominates is corrected).  Channels
 * 0 and M / 2 are never updated.  With tracking, the coefficients, and so the bits, depend on where the call
 * boundaries fall; calls cut the same way give identical bits.  The first tracking call, and any with more blocks
 * than every earlier one, waits for the channelizer's earlier calls while it makes room for its per-tile sums.
 * Every image entry point returns EINVAL on a real or a diversity channelizer (the message says why), and on a null c.
 * t41rx_chan_set_image: channels [first, first + count) take c_k = (coef[2 i], coef[2 i + 1]), finite (EINVAL
 * otherwise, and for a range outside [0, n_channels)).  Effective from the next call; waits for the channelizer's calls
 * like t41rx_chan_set_shift.  Channels outside the range keep their coefficients, including ones tracking has moved.
 * t41rx_chan_get_image: all n_channels coefficients as (re, im) pairs into coef[2 n_channels], including what tracking
 * has made of them (save and restore a calibration per band with it); waits for the channelizer's calls.
 * t41rx_chan_track_image: on != 0 turns tracking on with T = dominance_db (in [T41RX_CHAN_DOMINANCE_MIN_DB,
 * T41RX_CHAN_DOMINANCE_MAX_DB], EINVAL outside it; 20 is a good default), from the next call; on = 0 turns it off
 * (dominance_db is then not read), the coefficients staying where tracking left them.
 * t41rx_chan_image_stats: stats[(M / 2 + 1) x 4], (Re A, Im A, P_k, P_kbar) of pair k = 0 ... M / 2 from the last
 * call that ran with tracking on (EINVAL if none has); waits for the channelizer's calls. */
#define T41RX_CHAN_DOMINANCE_MIN_DB 3.0f
#define T41RX_CHAN_DOMINANCE_MAX_DB 60.0f
int t41rx_chan_set_image(t41rx_chan *c, int first, int count, const float *coef);
int t41rx_chan_get_image(t41rx_chan *c, float *coef);
int t41rx_chan_track_image(t41rx_chan *c, int on, float dominance_db);
int t41rx_chan_image_stats(t41rx_chan *c, double *stats);

/* Audio-spectrum + S-meter by-product of the row-producing blocks (Process.cpp:550-570; NFM: 791-805):
 *   audio_ypixel      int32 [n_streams][n_rows][270]  audioYPixel[k], k < AUDIO_SPEC_BOX_W - 2 (Process.cpp:34,555)
 *   audio_max_sq_ave  float [n_streams][n_rows]       audioMaxSquaredAve after the block (Process.cpp:32,569)
 * Binds where the following t41rx_process / _q15 (HOST pointers) or t41rx_process_device (DEVICE pointers) calls
 * put them, for row_every > 0; either may be NULL; both NULL unbinds (the default: the by-product is not computed).
 * Receivers in the raw PSK31 mode do not update either (Process.cpp:376-387): their rows repeat the last values.
 * While bound the context keeps n_streams * n_rows * 4 KiB of scratch for the masked spectra. */
#define T41RX_AUDIO_SPEC_PIXELS 270
int t41rx_bind_audio_spectrum(t41rx_ctx *ctx, int32_t *audio_ypixel, float *audio_max_sq_ave);
/* What the row-producing blocks write to the PC control app's serial port while controlDataFlag is set
 * (t41Control.cpp:20-48); binding plays the role of the flag:
 *   spec_frames   uint8 [n_streams][n_rows][518]  "FD" + "%03d" of (255 - max) + 512 data bytes + ';' (FFT.cpp:142-194:
 *                                                 data = pixelnew + currentNF shifted so that its maximum is 255);
 *                                                 only ZoomFFTExe sends it: all zeros at spectrum_zoom == 0
 *   audio_frames  uint8 [n_streams][n_rows][270]  min(audioYPixel, 255), no header (Process.cpp:818-825)
 * Same pointer rules as t41rx_bind_audio_spectrum.  spec_frames is built from the spectrum rows: with
 * t41rx_process_device the call's spec_rows must not be NULL. */
#define T41RX_SPEC_FRAME_BYTES 518
int t41rx_bind_control_frames(t41rx_ctx *ctx, uint8_t *spec_frames, uint8_t *audio_frames);
/* The S-meter reading DrawSmeterBar() derives from audioMaxSquaredAve (Display.cpp:959-981, TCVSDR_SMETER build):
 * dBm, given bands[].gainCorrection, bands[].RFgain (t41rx_debug.rf_gain) and rfGainAllBands.  Host arithmetic. */
float t41rx_smeter_dbm(float audio_max_sq_ave, float gain_correction, int32_t rf_gain, int32_t rf_gain_all_bands);
/* Length of the S-meter bar in pixels for that reading (Display.cpp:995-998): map(dbm, S1 = -127, S9 = -73, 0, 9 * 12)
 * in float (Teensy core map()), truncated to int16, limited to 0 .. SMETER_BAR_LENGTH = 180 (Display.h:69). */
int32_t t41rx_smeter_bar(float dbm);

/* Instrumentation for bench.py: kernels launched by this context so far, and the CUDA-event
 * duration (ms) of all kernels of the most recent t41rx_process[_device] call (valid after t41rx_synchronize). */
int64_t t41rx_kernel_launches(const t41rx_ctx *ctx);
/* Bit-exact chain and rows kernel, current device: how many blocks had to re-run their input conditioning serially
 * because a time-parallel chunk's speculative start state differed from the true one in the last bit (the result is
 * exact either way; this only costs time).  -1 on a CUDA error. */
int64_t t41rx_dc_refilter_count(void);
int t41rx_last_kernel_ms(t41rx_ctx *ctx, float *ms);
/* CUDA-event durations (ms) of the most recent launches (oldest first, at most 32) of the dominant kernel,
 * t41rx_stream_rx_kernel; returns how many were written, or a negative error code. */
int t41rx_stream_kernel_times(t41rx_ctx *ctx, float *ms, int max_n);

/* The firmware's WAV test-signal reader (Utility.cpp:773-888: load_wav / readWave; 16-bit mono PCM, format chunk of
 * 16, 18 or 40 bytes), host only.  t41rx_load_wav returns load_wav's own codes: 0, -1 cannot open, -2 format chunk
 * size, -3 not PCM / mono / 16 bit, -4 more than num_samples samples.  t41rx_read_wave returns 1 with size_buf samples
 * x / 32768 in buf, or 0 once the reference's end test (byte position + size_buf >= file size) fires; it then closes
 * the file, like readWave.  Where the reference would convert uninitialised stack (a read running past the end of
 * the file) the samples are 0. */
typedef struct t41rx_wav t41rx_wav;
int t41rx_load_wav(t41rx_wav **out, const char *input_file, uint32_t num_samples);
int t41rx_read_wave(t41rx_wav *w, float *buf, int size_buf);
uint32_t t41rx_wav_sample_rate(const t41rx_wav *w);
void t41rx_wav_close(t41rx_wav *w);

const char *t41rx_last_error(void);
const char *t41rx_version(void);

#ifdef __cplusplus
}
#endif
#endif /* T41RX_H */
