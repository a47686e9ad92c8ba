/* fmgpu.h — C ABI of the B200 channel-batched FM stereo + RDS engine.
 *
 * This is the drop-in boundary for the reference's IQ -> audio + RDS hot path
 * (SURVEY.md §8(b)). Every entry point below replaces one method of the
 * reference's block-processing classes; the C++ classes in
 * fmtuner_sdr_b200/dropin/ (same names and signatures as the reference headers)
 * are thin wrappers over these calls, so the reference's src/main.cpp compiles
 * unchanged against them (INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only; no exceptions cross this boundary.
 * Functions returning int return 0 on success and a negative FMGPU_E* code on
 * failure (fmgpu_last_error gives the text). Functions mirroring a reference
 * method that returns a sample count return that count and 0 for null / empty
 * arguments, as the reference does (stereo_decoder.cpp:94-96,
 * af_post_processor.cpp:50-53, rds_decoder.cpp:76-78, liquid_primitives.cpp:465-467).
 * There is no CPU fallback: every call fails with FMGPU_ENODEV without a CUDA device, and every
 * sample-rate operation of the path — the factor-1 convert and the uint8 re-quantisation of
 * ComplexDecimator::execute included — runs on the device.
 */
#ifndef FMGPU_H_
#define FMGPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FMGPU_OK 0
#define FMGPU_EINVAL (-1)  /* bad argument */
#define FMGPU_ENODEV (-2)  /* no CUDA device / CUDA runtime error */
#define FMGPU_ENOMEM (-3)  /* device allocation failed */
#define FMGPU_ERANGE (-4)  /* a caller-supplied capacity is too small */

typedef struct fmgpu_engine fmgpu_engine;

/* Parameters the reference takes from its constructors and config keys
 * (SURVEY §5: processing.* and tuner.deemphasis; src/main.cpp:640-710). */
typedef struct fmgpu_config {
  int32_t iq_rate;         /* IQ sample rate in: 256000|1024000|2048000 (main.cpp:391-396) or 240000|2400000 */
  int32_t decimation;      /* ComplexDecimator factor: 1, 4, 8 (main.cpp:670-674) or 10 */
  int32_t output_rate;     /* audio rate, 32000 (main.cpp OUTPUT_RATE) */
  int32_t block_samples;   /* processing.dsp_block_samples at the DSP rate, 1024..32768 (default 8192) */
  int32_t max_blocks;      /* logical blocks accepted per fmgpu_process_* call (>= 1) */
  int32_t w0_bandwidth_hz; /* processing.w0_bandwidth_hz (default 194000) */
  int32_t bandwidth_hz;    /* initial FMDemod::setBandwidthHz argument (0 => W0), main.cpp:710 */
  int32_t dsp_agc;         /* FMDemod::DspAgcMode: 0 off, 1 fast, 2 slow */
  int32_t stereo_blend;    /* StereoDecoder::BlendMode: 0 soft, 1 normal, 2 aggressive */
  int32_t deemphasis;      /* tuner.deemphasis: 0 = 50 us, 1 = 75 us, 2 = off (include/config.h:37) */
  int32_t stereo;          /* processing.stereo (0 => mono path, main.cpp:1266-1279) */
  int32_t force_mono;      /* StereoDecoder::setForceMono */
  int32_t decim_taps_per_phase; /* ComplexDecimator::init tapsPerPhase; 0 => main.cpp:672-673 (12/20/28) */
  int32_t decim_atten_db;       /* ComplexDecimator::init stopBandAtten; 0 => 80 dB (main.cpp:674) */
} fmgpu_config;

/* RDSGroup (include/rds_decoder.h:9-15) plus the logical block that emitted it. */
typedef struct fmgpu_rds_group {
  uint16_t a, b, c, d;
  uint8_t errors; /* A<<6|B<<4|C<<2|D ; 0 clean, 1 corrected/had errors, 3 missing (rds_decoder.cpp:29-41) */
  uint8_t pad[3];
  uint32_t block_index;
} fmgpu_rds_group;

/* Per logical block observables the caller reads after each block
 * (main.cpp:1294-1303: isStereo, getPilotLevelTenthsKHz; fm_demod.h:35-36). */
typedef struct fmgpu_block_status {
  int32_t n_audio;      /* 32 kHz frames produced by this block */
  int32_t stereo;       /* StereoDecoder::isStereo() after the block */
  int32_t pilot_tenths; /* StereoDecoder::getPilotLevelTenthsKHz() */
  float clip_ratio;     /* FMDemod::getClippingRatio() */
  int32_t n_groups;     /* RDS groups emitted during this block */
} fmgpu_block_status;

#define FMGPU_RESET_DECIM 1u  /* ComplexDecimator::reset  liquid_primitives.cpp:405-420 */
#define FMGPU_RESET_DEMOD 2u  /* FMDemod::reset           fm_demod.cpp:73-88 */
#define FMGPU_RESET_STEREO 4u /* StereoDecoder::reset     stereo_decoder.cpp:67-86 */
#define FMGPU_RESET_AFPOST 8u /* AFPostProcessor::reset   af_post_processor.cpp:20-29 */
#define FMGPU_RESET_RDS 16u   /* RDSDecoder::reset        rds_decoder.cpp:23-27 */
#define FMGPU_RESET_DSP 15u   /* the dspRuntime reset handler, main.cpp:686-691 */
#define FMGPU_RESET_ALL 31u

/* ---- lifetime ------------------------------------------------------------ */
/* Replaces the constructors at main.cpp:640-674,895. n_channels independent
 * channels share one configuration; per-channel settings can be changed below. */
int fmgpu_engine_create(const fmgpu_config *cfg, int n_channels, int device, fmgpu_engine **out);
void fmgpu_engine_destroy(fmgpu_engine *e);
const char *fmgpu_last_error(const fmgpu_engine *e); /* e may be NULL: last creation error */
int fmgpu_n_channels(const fmgpu_engine *e);
int fmgpu_dsp_rate(const fmgpu_engine *e); /* iq_rate / decimation */

/* ---- per-channel settings; channel = -1 applies to every channel ---------- */
int fmgpu_set_bandwidth_hz(fmgpu_engine *e, int channel, int bw_hz);   /* FMDemod::setBandwidthHz   fm_demod.cpp:99-135 */
int fmgpu_set_bandwidth_mode(fmgpu_engine *e, int channel, int mode);  /* FMDemod::setBandwidthMode fm_demod.cpp:90-97 */
int fmgpu_set_w0_bandwidth_hz(fmgpu_engine *e, int channel, int bw_hz);/* FMDemod::setW0BandwidthHz fm_demod.cpp:137-139 */
int fmgpu_set_agc_mode(fmgpu_engine *e, int channel, int mode);        /* FMDemod::setDspAgcMode    fm_demod.cpp:141-148 */
int fmgpu_set_deemphasis_us(fmgpu_engine *e, int channel, int tau_us); /* FMDemod/AFPostProcessor::setDeemphasis */
int fmgpu_set_deviation_hz(fmgpu_engine *e, double deviation_hz);      /* FMDemod::setDeviation fm_demod.cpp:64-71 (all channels) */
/* Arithmetic of the decimating FIR (ComplexDecimator::executeComplex, liquid_primitives.cpp:461-499),
 * all channels. 0: FP32 FMA chain in the reference's summation order, bit-identical to the CPU
 * oracle. 1: integer contraction on the tensor cores (uint8 samples x taps quantised to 2^-26,
 * exact int32 sums, ONE float rounding): within ~1e-7 of mode 0, about 7x faster. FMGPU_EINVAL when
 * the factor / tap count has no tensor-core form (odd factors, factor 16). The environment variable
 * FMGPU_DECIM_MODE sets the mode an engine starts in. */
int fmgpu_set_decimator_mode(fmgpu_engine *e, int mode);
int fmgpu_get_decimator_mode(const fmgpu_engine *e);
/* The linear first-order recursions of the batched path — the I/Q DC blockers in front of the
 * channel filter (fm_demod.cpp:37-38,164-165) and de-emphasis + DC blocker at 32 kHz
 * (af_post_processor.cpp:66-71) — all channels. 0: serial recursions, one lane per channel,
 * bit-identical to the CPU oracle. 1: the same filters as warp-shuffle parallel scans (one warp per
 * channel row, coalesced accesses; north_star item 5): results agree to float rounding (~1e-7 of
 * full scale), not bit for bit. FMGPU_SCAN_MODE sets the mode an engine starts in. */
int fmgpu_set_scan_mode(fmgpu_engine *e, int mode);
int fmgpu_get_scan_mode(const fmgpu_engine *e);
/* Arithmetic of the stereo decoder's real-tap FIRs — the 19 kHz pilot band-pass and the L/R 15 kHz
 * low-pass (stereo_decoder.cpp:25-63,172-173,233-239) — all channels. 0: FP32 FMA chains in the
 * reference's summation order, bit-identical to the CPU oracle. 1: exact integer contractions on the
 * tensor cores (samples as 24-bit fixed point, taps as 24-bit integers, int32 sums in TMEM, rounded
 * at the end): within ~2e-7 of mode 0. FMGPU_EINVAL when a filter length has no tensor-core form.
 * FMGPU_FIR_MODE sets the mode an engine starts in. */
int fmgpu_set_fir_mode(fmgpu_engine *e, int mode);
int fmgpu_get_fir_mode(const fmgpu_engine *e);
/* Channel filter -> pre-discriminator AGC -> quadrature discriminator (FMDemod::demodulateComplex,
 * fm_demod.cpp:194-199) of the batched path, all channels. 0: three kernels in the reference's
 * arithmetic, bit-identical to the CPU oracle. 1: ONE tensor-core kernel — the channel filter as an
 * exact integer contraction (24-bit fixed-point samples, 24-bit integer taps), the discriminator in
 * its epilogue; the AGC multiplies y[n] by a positive real gain, which arg(y[n] conj(y[n-1])) does
 * not see, so it is left out (its state is not advanced). Used for a call whose channels share one
 * channel filter; otherwise, and for the stage-level entry points, mode 0's kernels run. MPX agrees
 * with mode 0 to ~1e-6. FMGPU_DEMOD_MODE sets the mode an engine starts in. */
int fmgpu_set_demod_mode(fmgpu_engine *e, int mode);
int fmgpu_get_demod_mode(const fmgpu_engine *e);
int fmgpu_set_blend_mode(fmgpu_engine *e, int channel, int mode);      /* StereoDecoder::setBlendMode */
int fmgpu_set_force_mono(fmgpu_engine *e, int channel, int on);        /* StereoDecoder::setForceMono */
int fmgpu_set_force_stereo(fmgpu_engine *e, int channel, int on);      /* StereoDecoder::setForceStereo */
int fmgpu_reset(fmgpu_engine *e, int channel, unsigned what_mask);     /* the reset() methods, see FMGPU_RESET_* */

/* ---- observables ------------------------------------------------------------ */
int fmgpu_is_stereo(fmgpu_engine *e, int channel);       /* StereoDecoder::isStereo */
int fmgpu_pilot_tenths(fmgpu_engine *e, int channel);    /* StereoDecoder::getPilotLevelTenthsKHz */
float fmgpu_clip_ratio(fmgpu_engine *e, int channel);    /* FMDemod::getClippingRatio */
int fmgpu_is_clipping(fmgpu_engine *e, int channel);     /* FMDemod::isClipping */

/* ---- batched whole-pipeline path (the per-block body of main.cpp:1232-1308) ----
 * All channels, n_blocks logical blocks each. Device pointers, asynchronous on
 * `stream` (a cudaStream_t, may be NULL for the default stream).
 *   iq_dev      [C][iq_stride_bytes] uint8 I,Q pairs; each channel holds
 *               n_blocks*block_samples*decimation pairs; base and stride 16-byte aligned
 *   audio_dev   [C][2][audio_cap] float, left row then right row, clamped to +-1
 *   n_audio_dev [C] frames written per channel
 *   groups_dev  [C][group_cap], n_groups_dev [C]
 *   status_dev  [C][n_blocks]
 * Any output pointer may be NULL to skip that output. */
int fmgpu_process_batch(fmgpu_engine *e, const uint8_t *iq_dev, size_t iq_stride_bytes,
                        int n_blocks, float *audio_dev, size_t audio_cap, uint32_t *n_audio_dev,
                        fmgpu_rds_group *groups_dev, size_t group_cap, uint32_t *n_groups_dev,
                        fmgpu_block_status *status_dev, void *stream);

/* Streaming form of fmgpu_process_batch for back-to-back calls (the reference's main loop runs one
 * block after another, main.cpp:992): the pipeline groups start after the work already queued on
 * `stream` (so the IQ must be ready in stream order), but `stream` does NOT wait for them; each
 * group orders itself after its own previous batch, so one call's serial (lane) kernels overlap
 * the next call's FIR kernels. Outputs are complete once fmgpu_join(e, stream) has been queued and
 * `stream` has reached it; give consecutive calls different output buffers if each call's
 * results are needed. */
int fmgpu_process_batch_async(fmgpu_engine *e, const uint8_t *iq_dev, size_t iq_stride_bytes,
                              int n_blocks, float *audio_dev, size_t audio_cap,
                              uint32_t *n_audio_dev, fmgpu_rds_group *groups_dev, size_t group_cap,
                              uint32_t *n_groups_dev, fmgpu_block_status *status_dev, void *stream);
/* Make `stream` wait for every batch queued so far by fmgpu_process_batch_async. */
int fmgpu_join(fmgpu_engine *e, void *stream);

/* Same work with HOST buffers: copies the IQ bytes host->device, runs the batch,
 * copies audio / groups / status back and synchronises. Layouts as above. */
int fmgpu_process_host(fmgpu_engine *e, const uint8_t *iq_host, size_t iq_stride_bytes,
                       int n_blocks, float *audio_host, size_t audio_cap, uint32_t *n_audio_host,
                       fmgpu_rds_group *groups_host, size_t group_cap, uint32_t *n_groups_host,
                       fmgpu_block_status *status_host);
/* Streaming form: fmgpu_submit_host queues the copies and the batch and returns a ticket (0 or 1,
 * negative = error) without waiting; fmgpu_wait_host(ticket) blocks until that submission's
 * outputs are in the host buffers. Two submissions may be in flight, so a caller that submits
 * block k+1 before waiting for block k keeps the PCIe copies and the kernels of consecutive
 * blocks overlapped. The host buffers of a submission must stay valid (and pinned, for the copies
 * to be asynchronous) until its ticket has been waited for. fmgpu_process_host = submit + wait. */
int fmgpu_submit_host(fmgpu_engine *e, const uint8_t *iq_host, size_t iq_stride_bytes,
                      int n_blocks, float *audio_host, size_t audio_cap, uint32_t *n_audio_host,
                      fmgpu_rds_group *groups_host, size_t group_cap, uint32_t *n_groups_host,
                      fmgpu_block_status *status_host);
int fmgpu_wait_host(fmgpu_engine *e, int ticket);

/* ---- RF signal level (SURVEY §8(f) row 2): the per-block meter main.cpp computes from the raw
 * IQ bytes (computeSignalLevel, src/signal_level.cpp:145-203, called at main.cpp:1167).
 * The device pass reduces each logical block of each channel to EXACT integer sums; the host
 * helper finishes them in double precision the way the reference does. */
typedef struct fmgpu_level_sums {
  uint64_t sum_i, sum_q;   /* sum of the I / Q bytes */
  uint64_t sum_ii, sum_qq; /* sum of their squares */
  uint32_t hard_clip;      /* samples with a byte <= 1 or >= 254 (signal_level.cpp:169-171) */
  uint32_t near_clip;      /* samples with a byte <= 8 or >= 247 (signal_level.cpp:172-174) */
  uint32_t n_samples;      /* IQ pairs reduced */
  uint32_t pad;
} fmgpu_level_sums;

typedef struct fmgpu_signal_level { /* SignalLevelResult, include/signal_level.h:7-13 */
  float level120;
  double dbfs, compensated_dbfs, hard_clip_ratio, near_clip_ratio;
} fmgpu_signal_level;

/* sums_dev [C][n_blocks]; iq layout as fmgpu_process_batch. Asynchronous on `stream`. */
int fmgpu_signal_level_batch(fmgpu_engine *e, const uint8_t *iq_dev, size_t iq_stride_bytes,
                             int n_blocks, fmgpu_level_sums *sums_dev, void *stream);
/* Host only: dBFS / 0..120 meter / clip ratios from one block's sums (signal_level.cpp:180-203). */
void fmgpu_signal_level_finish(const fmgpu_level_sums *sums, int applied_gain_db,
                               double gain_comp_factor, double signal_bias_db, double floor_dbfs,
                               double ceil_dbfs, fmgpu_signal_level *out);

/* ---- output formatting (SURVEY §8(f) row 4): what AudioOutput::write / writeWAVData do to the
 * clamped float audio before it reaches a WAV file (src/audio_output.cpp:1445-1464,1386-1391):
 * multiply by the volume scale (0.85 * volume% / 100), clamp to +-1, scale by 32767 and truncate
 * toward zero, left/right interleaved. audio_dev / n_audio_dev as written by
 * fmgpu_process_batch; pcm_dev is [C][2*audio_cap] int16. Asynchronous on `stream`. */
int fmgpu_pack_pcm16(fmgpu_engine *e, const float *audio_dev, size_t audio_cap,
                     const uint32_t *n_audio_dev, float volume_scale, int16_t *pcm_dev,
                     void *stream);

/* ---- XDR / FM-DX view of the RDS stream (SURVEY section 8(f) row 4) -------------------------
 * XDRServer::updateRDS (src/xdr_server.cpp:403-457) with its PI debounce (evaluatePiState,
 * :189-215), one state per channel, for hosts that serve many channels: every group gives up to
 * two text lines, "P<PI>" followed by one '?' per error level of block A once the PI is
 * debounced, and "R<B><C><D><errors>" when block B was received clean. Host-side; no device work. */
typedef struct fmgpu_xdr_rds_state {
  uint16_t pi_buffer[64];
  uint8_t pi_error[8];
  uint8_t pi_fill, pi_pos, pi_last_state, pad;
  uint16_t pi_last_value;
} fmgpu_xdr_rds_state;
/* the state of a constructed server and after every start / retune (xdr_server.cpp:257-266,461-470) */
void fmgpu_xdr_rds_init(fmgpu_xdr_rds_state *s);
/* returns the number of lines written (0..2), each NUL-terminated */
int fmgpu_xdr_rds_lines(fmgpu_xdr_rds_state *s, const fmgpu_rds_group *g, char lines[2][32]);

/* ---- wideband channelizer (BASELINE config 4; SURVEY section 8(f) row 3) --------------------
 * NO reference counterpart: the reference tunes one carrier in the RTL-SDR hardware. One IQ
 * capture at wide_rate (uint8 by default; other sample formats below) holds n_channels carriers, channel k centred first_center_hz +
 * k * spacing_hz away from the capture centre; each is mixed to baseband, low-pass filtered by a
 * Kaiser-windowed sinc of decimation * taps_per_phase taps (cut-off cutoff_hz, atten_db) and
 * decimated to wide_rate / decimation — complex float at the engine's DSP rate, the input of
 * fmgpu_process_batch_cf32 (the FMDemod::processSplitComplex path, fm_demod.cpp:258-274).
 * Definition (what tests/test_gpu_channelizer.py evaluates in float64):
 *   y_k[m] = sum_n h[n] x[m*D - n] exp(-j 2 pi f_k (m*D - n) / wide_rate),
 * x the input pair converted by the object's sample format (FMGPU_IQ_*): cu8 x = (u8 - 127.5)/127.5,
 * cs8 x = s8 / 128, cs16 x = s16 / 32768; m counted from creation, input before the first call = 0.
 * Two evaluations of it: a polyphase bank when the carriers sit on a uniform grid (wide_rate /
 * spacing_hz an integer P <= 1024, n_channels <= P, and first_center_hz / spacing_hz * T an
 * integer for some T <= 8), otherwise the direct form (one complex tap table per carrier, several
 * times slower). FMGPU_CHANNELIZER_DIRECT set in the environment at creation selects the direct form.
 *
 * Many captures: one object may serve n_captures captures that advance together (same wide_rate,
 * decimation, carrier spacing and filter), each with its own centre offset: capture w's carrier k
 * sits first_center_hz[w] + k * spacing_hz from ITS centre. The definition holds per capture, with
 * capture w's input, its own history and its own f_k; m is shared. The polyphase bank is used only
 * when every capture passes the grid test above, so one off-grid offset (e.g. a ppm-corrected
 * centre) selects the slower direct form for all captures. At most 65535 captures.
 * fmgpu_channelizer_create is fmgpu_channelizer_create_multi with one capture.
 *
 * Sample formats: all captures of one object share one format (a mixed fleet uses one object per
 * format). Only the load of a pair differs; the filter, the bank and the outputs' layout do not.
 * bladeRF's SC16_Q11 samples are cs16 with full scale 2048, so their outputs come out 16x smaller,
 * which the scale-invariant discriminator behind the channelizer does not notice.
 *
 * Rational rates (fmgpu_channelizer_create_rate): with U/D the reduced ratio output_rate / wide_rate
 * (gcd(U, D) = 1, U <= 64), the prototype h has L = D * taps_per_phase taps, designed at rate
 * U * wide_rate with cut-off cutoff_hz / (U * wide_rate) and scaled by 2 fc U for unity pass-band
 * gain, and
 *   y_k[m] = sum_{n = 0..L-1, (mD - n) = 0 mod U} h[n] x[(mD - n)/U] exp(-j 2 pi f_k ((mD - n)/U) / wide_rate).
 * Output m reads inputs up to s_m = floor(mD / U) through the phase filter g_q[i] = h[q + iU],
 * q = mD mod U, at most Lin = ceil(L / U) taps. For U = 1 this is the definition above with the same
 * taps. After T pairs per capture since creation, outputs 0 .. ceil(T U / D) - 1 exist, so a call
 * with n_in pairs writes ceil((T + n_in) U / D) - ceil(T U / D) outputs: a count that varies from
 * call to call (fmgpu_channelizer_outputs). create, create_multi and create_format are create_rate's
 * U = 1 objects; fmgpu_channelizer_process_stream serves every object. */
#define FMGPU_IQ_CU8 0  /* uint8 I,Q, offset binary: RTL-SDR */
#define FMGPU_IQ_CS8 1   /* int8 I,Q: HackRF */
#define FMGPU_IQ_CS16 2  /* int16 I,Q, native (little-endian) order: USRP, bladeRF, LimeSDR,
                            SDRplay (SoapySDR CS16) */
typedef struct fmgpu_channelizer fmgpu_channelizer;
int fmgpu_channelizer_create(int device, int wide_rate, int decimation, int n_channels,
                             double first_center_hz, double spacing_hz, int taps_per_phase,
                             double cutoff_hz, float atten_db, fmgpu_channelizer **out);
/* first_center_hz [n_captures] */
int fmgpu_channelizer_create_multi(int device, int n_captures, int wide_rate, int decimation,
                                   int n_channels, const double *first_center_hz, double spacing_hz,
                                   int taps_per_phase, double cutoff_hz, float atten_db,
                                   fmgpu_channelizer **out);
/* fmgpu_channelizer_create_multi for captures of sample_format (FMGPU_IQ_*; FMGPU_EINVAL for any
 * other value); create_multi is this with FMGPU_IQ_CU8. */
int fmgpu_channelizer_create_format(int device, int sample_format, int n_captures, int wide_rate,
                                    int decimation, int n_channels, const double *first_center_hz,
                                    double spacing_hz, int taps_per_phase, double cutoff_hz,
                                    float atten_db, fmgpu_channelizer **out);
/* An object whose output rate is output_rate, a rational fraction U/D of wide_rate (see "Rational
 * rates" above). FMGPU_EINVAL when output_rate < 1, output_rate > wide_rate or U > 64; the other
 * checks are create_format's. With U = 1 it is the create_format object of decimation D, bit for bit. */
int fmgpu_channelizer_create_rate(int device, int sample_format, int n_captures, int wide_rate,
                                  int output_rate, int n_channels, const double *first_center_hz,
                                  double spacing_hz, int taps_per_phase, double cutoff_hz, float atten_db,
                                  fmgpu_channelizer **out);
void fmgpu_channelizer_destroy(fmgpu_channelizer *z);
/* wide_rate * U / D, an exact integer for create_rate objects (wide_rate / decimation, rounded down,
 * for create_format objects) */
int fmgpu_channelizer_output_rate(const fmgpu_channelizer *z);
int fmgpu_channelizer_interpolation(const fmgpu_channelizer *z);   /* U (1 unless create_rate) */
int fmgpu_channelizer_decimation(const fmgpu_channelizer *z);      /* D */
int fmgpu_channelizer_n_captures(const fmgpu_channelizer *z);
/* the FMGPU_IQ_* format the object was created for */
int fmgpu_channelizer_sample_format(const fmgpu_channelizer *z);
/* the prototype's L = D * taps_per_phase taps, at rate U * wide_rate */
size_t fmgpu_channelizer_taps(const fmgpu_channelizer *z, float *out, size_t cap);
/* outputs per row that the next process call with n_in pairs per capture writes. Host state only:
 * no device synchronisation. */
size_t fmgpu_channelizer_outputs(const fmgpu_channelizer *z, size_t n_in);
/* iq_dev: n_in uint8 I,Q pairs (n_in a multiple of the decimation) continuing the stream of the
 * previous call; out_cf32_dev [ch_count][out_stride_samples] complex float for channels
 * ch_first .. ch_first + ch_count - 1 (a rank of a sharded job extracts only its own channels from
 * the capture every rank reads). Asynchronous on `stream`. FMGPU_EINVAL on an object with more
 * than one capture or another format than FMGPU_IQ_CU8. */
int fmgpu_channelizer_process(fmgpu_channelizer *z, const uint8_t *iq_dev, size_t n_in,
                              int ch_first, int ch_count, float *out_cf32_dev,
                              size_t out_stride_samples, void *stream);
/* iq_dev [n_captures][iq_stride_bytes] (stride even, >= 2 * n_in): n_in pairs per capture,
 * continuing each capture's stream. out_cf32_dev [n_captures][ch_count][out_stride_samples]: row
 * w * ch_count + kk is carrier ch_first + kk of capture w, so the buffer is an
 * fmgpu_process_batch_cf32 input of n_captures * ch_count channels as it stands. A rank of a
 * sharded job channelizes either its own captures (its own object) or its ch_first / ch_count share
 * of every capture. Asynchronous on `stream`. It is fmgpu_channelizer_process_iq for FMGPU_IQ_CU8
 * objects, and FMGPU_EINVAL on any other format. */
int fmgpu_channelizer_process_multi(fmgpu_channelizer *z, const uint8_t *iq_dev,
                                    size_t iq_stride_bytes, size_t n_in, int ch_first,
                                    int ch_count, float *out_cf32_dev, size_t out_stride_samples,
                                    void *stream);
/* Any format, any number of captures: iq_dev [n_captures][iq_stride_bytes] holds n_in pairs of the
 * object's format per capture (pair size 2 bytes for cu8 and cs8, 4 for cs16). FMGPU_EINVAL when the
 * stride is not a multiple of the pair size or shorter than pair size * n_in, or iq_dev is not
 * aligned to the pair size; otherwise as fmgpu_channelizer_process_multi. FMGPU_EINVAL on an object
 * with U > 1: it is fmgpu_channelizer_process_stream restricted to U = 1 and n_in a multiple of D. */
int fmgpu_channelizer_process_iq(fmgpu_channelizer *z, const void *iq_dev, size_t iq_stride_bytes,
                                 size_t n_in, int ch_first, int ch_count, float *out_cf32_dev,
                                 size_t out_stride_samples, void *stream);
/* Any object, any n_in >= 1 pairs per capture (a multiple of D or not): writes outputs
 * [0, fmgpu_channelizer_outputs(z, n_in)) of every row of out_cf32_dev
 * [n_captures][ch_count][out_stride_samples] and stores that count in *n_out (n_out may be NULL).
 * A call that completes no output only carries the history. FMGPU_EINVAL when out_stride_samples is
 * less than that count; the input stride, alignment and channel checks are process_iq's.
 * Asynchronous on `stream`. */
int fmgpu_channelizer_process_stream(fmgpu_channelizer *z, const void *iq_dev, size_t iq_stride_bytes,
                                     size_t n_in, int ch_first, int ch_count, float *out_cf32_dev,
                                     size_t out_stride_samples, size_t *n_out, void *stream);

/* fmgpu_process_batch with complex-float input at the DSP rate (engine created with
 * decimation = 1): x_cf32_dev [C][stride_samples] interleaved re,im; base and stride 16-byte
 * aligned. FMDemod::processSplitComplex for every channel (clip flag: |I| or |Q| >= 0.995). */
int fmgpu_process_batch_cf32(fmgpu_engine *e, const float *x_cf32_dev, size_t stride_samples,
                             int n_blocks, float *audio_dev, size_t audio_cap,
                             uint32_t *n_audio_dev, fmgpu_rds_group *groups_dev, size_t group_cap,
                             uint32_t *n_groups_dev, fmgpu_block_status *status_dev, void *stream);

/* Split the channels into `groups` (1..16) ranges that run the pipeline on separate streams:
 * one range's serial (one-lane-per-channel) kernels then overlap another range's FIR kernels
 * and, in fmgpu_process_host, its host<->device copies. Results do not depend on it. */
int fmgpu_set_pipeline_groups(fmgpu_engine *e, int groups);

/* ---- stage-level entry points, one per reference method; HOST buffers, synchronous ----
 * They run the same kernels as the batch path on one channel's state. */
/* ComplexDecimator::executeComplex  liquid_primitives.cpp:461-499 ; out = interleaved re,im */
size_t fmgpu_decimate(fmgpu_engine *e, int channel, const uint8_t *iq, size_t in_samples,
                      float *out_cf32, size_t out_capacity);
/* ComplexDecimator::execute  liquid_primitives.cpp:422-459 ; uint8 I,Q pairs out (re-quantised on
 * the device: clamp(y * 127.5 + 127.5, 0, 255), truncated) */
size_t fmgpu_decimate_u8(fmgpu_engine *e, int channel, const uint8_t *iq, size_t in_samples,
                         uint8_t *out_u8, size_t out_capacity);
/* FMDemod::processSplit (uint8 IQ at the DSP rate)  fm_demod.cpp:245-259 */
size_t fmgpu_demod_u8(fmgpu_engine *e, int channel, const uint8_t *iq, float *mpx_out,
                      float *mono_out, size_t n);
/* FMDemod::processSplitComplex  fm_demod.cpp:261-274 */
size_t fmgpu_demod_cf32(fmgpu_engine *e, int channel, const float *iq_cf32, float *mpx_out,
                        float *mono_out, size_t n);
/* FMDemod::downsampleAudio  fm_demod.cpp:210-226 (mono chain on caller-supplied MPX) */
size_t fmgpu_downsample_mono(fmgpu_engine *e, int channel, const float *mpx, float *audio_out,
                             size_t n);
/* StereoDecoder::processAudio  stereo_decoder.cpp:92-286 */
size_t fmgpu_stereo(fmgpu_engine *e, int channel, const float *mpx, float *left, float *right,
                    size_t n);
/* AFPostProcessor::process  af_post_processor.cpp:47-78 */
size_t fmgpu_afpost(fmgpu_engine *e, int channel, const float *in_left, const float *in_right,
                    size_t n, float *out_left, float *out_right, size_t out_capacity);
/* RDSDecoder::process  rds_decoder.cpp:74-93 ; returns the number of groups (written up to cap) */
size_t fmgpu_rds(fmgpu_engine *e, int channel, const float *mpx, size_t n, fmgpu_rds_group *out,
                 size_t cap);

/* ---- introspection used by tests/ ---------------------------------------------- */
/* Filter designs the engine computed for itself (compared against the oracle's).
 * which: 0 decimator taps, 1 channel filter of `channel`, 2 pilot band-pass,
 * 3 audio low-pass, 4 audio resampler bank [32][24], 5 RDS low-pass,
 * 6 symsync MF bank, 7 symsync dMF bank, 8 RDS resampler bank [32][26].
 * *scale receives the filter's output scale (which 4/8: the phase step). */
size_t fmgpu_get_design(fmgpu_engine *e, int which, int channel, float *out, size_t cap,
                        float *scale);
/* The same designs computed WITHOUT a device or an engine (host only): `which` as above,
 * with 1 = the channel filter FMDemod(cfg rate) holds after setW0BandwidthHz(cfg->w0_bandwidth_hz)
 * and setBandwidthHz(bw_hz). */
size_t fmgpu_design_host(const fmgpu_config *cfg, int which, int bw_hz, float *out, size_t cap,
                         float *scale);
/* HOST-ONLY model of the tensor-core FIR's arithmetic (fmgpu_set_fir_mode 1; fir_tc.cu), evaluated
 * from the same tables the kernel uses: taps (design order, n_taps of them, padded like the engine
 * pads them) as 24-bit integers in three signed digits read back out of the operand image, samples as
 * 24-bit fixed point with quantum 2^-data_shift, 64-bit limb sums, the epilogue's float
 * recombination. x holds n_hist history samples followed by n samples (n a multiple of 32, n_hist
 * at least the filter's reach rounded up to 32); y receives n outputs. Returns n, or 0 when the
 * arguments do not fit or an int32 accumulator of the kernel would have overflowed. Needs no device:
 * the CPU test-suite uses it to check the table builder and the error bound against a float64 FIR. */
size_t fmgpu_fir_tc_host_model(const float *taps, int n_taps, float scale, int data_shift, const float *x,
                               size_t n_hist, size_t n, float *y);
/* The same for the tensor-core decimator (fmgpu_set_decimator_mode 1; decim_tc.cu): taps in design
 * order (fmgpu_design_host, which = 0) and their scale; iq = valid_history sample pairs of history
 * (0 .. n_taps - 1; what is missing of the window counts as byte 0, as after a reset) followed by
 * n_out * decimation pairs; out receives n_out complex floats. Returns n_out, or 0 when the factor /
 * tap count / n_out has no tensor-core form. Host only. */
size_t fmgpu_decim_tc_host_model(int decimation, const float *taps, int n_taps, float scale,
                                 const unsigned char *iq, int valid_history, int n_out, float *out);
/* Intermediate device buffers of the last fmgpu_process_* call, copied to the host:
 * which: 0 decimated cf32 (2 floats/sample), 1 MPX, 2 stereo left at the DSP rate,
 * 3 stereo right, 4 pilot band-pass output, 5 / 6 the matrix outputs L / R in front of the 15 kHz
 * low-pass. Returns floats written. */
size_t fmgpu_debug_read(fmgpu_engine *e, int which, int channel, float *out, size_t cap);
/* Every RDS bit demodulated by `channel` during the last call (before block sync). */
size_t fmgpu_debug_rds_bits(fmgpu_engine *e, int channel, uint8_t *out, size_t cap);
/* Number of kernels this engine has launched so far. */
uint64_t fmgpu_launch_count(const fmgpu_engine *e);
/* Measurement aid: with on = 0 every stage of the block pipeline is queued on ONE stream, so no two
 * stages overlap and the per-stage times of fmgpu_get_stage_times are those of the kernels running
 * alone. Results do not depend on it. Default: on (stages overlap). */
int fmgpu_set_stage_overlap(fmgpu_engine *e, int on);
/* With stage timing enabled and batches queued by fmgpu_process_batch_async: every stage span
 * recorded since the last call (name, pipeline group, start and end in ms after the earliest
 * span). Synchronises the device. Returns the number of spans. */
int fmgpu_debug_timeline(fmgpu_engine *e, const char **names, int *groups, float *t0_ms,
                         float *t1_ms, int cap);
/* Device time (ms) spent per pipeline stage during the last fmgpu_process_batch when
 * stage timing was enabled with fmgpu_enable_stage_timing; names[i] are static strings. */
int fmgpu_enable_stage_timing(fmgpu_engine *e, int on);
int fmgpu_get_stage_times(fmgpu_engine *e, const char **names, float *ms, int cap);

/* Measurement aid (bench.py): the FP32 FMA rate of `device` in TFLOP/s (2 flop per FMA), measured
 * with a register-resident packed-FMA loop on every SM — the roof the FIR kernels are held against. */
int fmgpu_measure_fp32_tflops(int device, double *tflops_out);

/* ---- on-device synthetic multiplex generator (bench.py input; SURVEY Appendix C) ---- */
typedef struct fmgpu_synth_params {
  float deviation_hz;   /* 22500..75000 */
  float tone_l_hz, tone_l_amp, tone_r_hz, tone_r_amp;
  float pilot_amp, rds_amp, iq_amp;
  float snr_db;         /* >= 200 => no noise */
  uint32_t seed;
  uint16_t pi;          /* RDS PI; PS is "CHnnnn  " from the low 16 bits of seed */
  uint16_t pad;
} fmgpu_synth_params;
/* params_host [C]; writes n_samples IQ pairs per channel into iq_dev [C][iq_stride_bytes]. */
int fmgpu_synth_iq(int device, const fmgpu_synth_params *params_host, int n_channels,
                   double fs_iq, size_t n_samples, uint8_t *iq_dev, size_t iq_stride_bytes,
                   void *stream);

#ifdef __cplusplus
}
#endif

#endif /* FMGPU_H_ */
