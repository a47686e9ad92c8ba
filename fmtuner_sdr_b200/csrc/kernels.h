// kernels.h — host-callable launchers of the engine's kernels (kernels.cu).
#ifndef FMGPU_KERNELS_H_
#define FMGPU_KERNELS_H_

#include <vector>

#include "engine.h"

namespace fmgpu {

struct FirRealJob {
  const float *in[2];
  float *out[2];
  size_t in_pitch, out_pitch;
  int in_off, out_off;
  int n_total;
  int Lp;
  float scale;
  int ch0;
};

cudaError_t initRdsTables();

void launchDecim(int M, const uint8_t *iq, size_t iq_stride, const uint8_t *hist,
                 const int *hist_valid, float2 *x1, size_t x1_pitch, int n_out, int ch0, int nch, int Pp, int L, float scale,
                 const TapsParam &taps, const TapsParam &taps_unpadded, cudaStream_t stream);
// decim_tc.cu: the same FIR as an integer contraction on the tensor cores (tcgen05.mma kind::i8,
// TMA-fed, accumulators in TMEM). Not bit-identical to launchDecim: one float rounding of the exact
// sum instead of a 280-term float chain.
bool decimTcSupported(int M, int L, int n_out);
void decimTcBuildTables(int M, const std::vector<float> &hrev, std::vector<uint8_t> *b_image,
                        std::vector<int32_t> *offs);
size_t decimTcHostModel(int M, const std::vector<float> &hrev, float scale, const uint8_t *iq, int valid,
                        int n_out, float *out);
cudaError_t launchDecimTc(int M, int L, const uint8_t *iq, size_t iq_stride, size_t iq_row_bytes,
                          const uint8_t *hist, const int *hist_valid, int total_rows, float2 *x1,
                          size_t x1_pitch, int n_out, int ch0, int nch, float scale,
                          const uint8_t *b_image_dev, const int32_t *offs_dev, int sm_count,
                          cudaStream_t stream);
// fir_tc.cu: the real-tap FIRs of the stereo decoder (pilot band-pass, L/R low-pass) as exact integer
// contractions on the tensor cores: samples as 24-bit fixed point in three byte planes (A operand in
// TMEM), taps as three signed base-256 digits (banded B matrix in shared memory), int32 accumulators
// in TMEM. Not bit-identical to launchFirReal: the exact sum of quantised terms, rounded at the end.
struct FirTcTables {
  std::vector<uint8_t> b_image;
  int32_t off[3];   // 2^23 * sum(integer taps), limbs 2..4
  int shift;        // taps are quantised to 2^-shift
  int ksteps;       // 32-sample sub-chunks per tile window
};
int firTcKsteps(const float *h, int Lp);
bool firTcSupported(const float *h, int Lp, int in_off);
void firTcBuildTables(const float *h, int Lp, FirTcTables *t);
// data_shift: samples are quantised to 2^-data_shift and must satisfy |x| < 2^(23 - data_shift)
// (larger values saturate)
cudaError_t launchFirTc(const FirRealJob &job, int nsig, int nch, const FirTcTables &t,
                        const uint8_t *b_image_dev, int data_shift, int sm_count, cudaStream_t stream);
size_t firTcHostModel(const float *taps, int n_taps, int lp, float scale, int data_shift, const float *x,
                      size_t n_hist, size_t n, float *y);
// channel filter + discriminator fused (complex rows; the AGC between them cannot change the
// discriminator's output and is left out); see fir_tc.cu
bool chanTcSupported(const float *h, int Lp, int in_off);
cudaError_t launchChanDemodTc(const float2 *x2, size_t x2_pitch, int in_off, float2 *y_io, size_t y_pitch,
                              float *mpx, size_t mpx_pitch, int mpx_off, int n_total, int ch0, int nch,
                              float chan_scale, float fd_ref, const FirTcTables &t, const uint8_t *b_image_dev,
                              int data_shift, int sm_count, cudaStream_t stream);
void launchConvertU8(const uint8_t *iq, size_t iq_stride, float2 *x1, size_t x1_pitch, int n,
                     int ch0, int nch, cudaStream_t stream);
void launchRequantU8(const float2 *x1, size_t x1_pitch, uint8_t *out, size_t out_stride, int n, int ch0,
                     int nch, cudaStream_t stream);
void launchCarryIq(uint8_t *hist, int *hist_valid, const uint8_t *iq, size_t iq_stride, long n_in,
                   int ch0, int nch, cudaStream_t stream);
void launchCarryF32(float *buf, size_t pitch, int H, size_t n, int ch0, int nch,
                    cudaStream_t stream);
void launchCarryF2(float2 *buf, size_t pitch, int H, size_t n, int ch0, int nch,
                   cudaStream_t stream);
void launchSaveTail(const float *src, size_t src_pitch, int src_off, float *hist, int hist_pitch,
                    int H, long n, int ch0, int nch, cudaStream_t stream);
void launchDcBlock(const float2 *x1, size_t x1_pitch, const uint8_t *iq_u8, size_t iq_stride,
                   float2 *x2, size_t x2_pitch, DemodState *st, fmgpu_block_status *status,
                   int status_pitch, int n_total, int ch0, int nch, float a1, cudaStream_t stream);
// the I/Q DC blockers of one logical block as a warp-shuffle scan (float input; fast arithmetic)
void launchDcBlockScan(const float2 *x1, size_t x1_pitch, float2 *x2, size_t x2_pitch, DemodState *st,
                       fmgpu_block_status *status, int status_pitch, int n_total, int ch0, int nch,
                       float a1, cudaStream_t stream);
void launchChanFir(const float2 *x2, size_t x2_pitch, float2 *ybuf, size_t y_pitch,
                   const float *chan_taps, const int *chan_lp, const float *chan_scale,
                   const ChanParams *cp, int n_total, int ch0, int nch, cudaStream_t stream);
void launchAgc(float2 *ybuf, size_t y_pitch, DemodState *st, const ChanParams *cp, int n_total,
               int ch0, int nch, cudaStream_t stream);
void launchFreqDem(const float2 *ybuf, size_t y_pitch, float *mpx, size_t mpx_pitch, int n_total,
                   int ch0, int nch, float ref, cudaStream_t stream);
void launchFirReal(const FirRealJob &job, int nsig, int nch, const TapsParam &taps,
                   cudaStream_t stream);
void launchStereo(const float *mpx, size_t mpx_pitch, const float *pilot, size_t pilot_pitch,
                  float *lraw, float *rraw, size_t lr_pitch, StereoState *st, const ChanParams *cp,
                  fmgpu_block_status *status, int status_pitch, int n_total, int ch0, int nch,
                  const EngineConst &k, cudaStream_t stream);
// k_prepare's RDS work (do_rds): the 171 kHz resampler's bookkeeping (the resampler stage), or, on the
// first block of a call, zeroing the call's group / bit counters (the demodulator stage)
enum { PREPARE_RDS_NONE = 0, PREPARE_RDS_RESAMPLER = 1, PREPARE_RDS_COUNTERS = 2 };
void launchPrepare(AudioState *au, RdsState *rds, fmgpu_block_status *status, int status_pitch,
                   int n_total, int ch0, int nch, uint32_t aud_step, uint32_t rds_step, int do_audio,
                   int do_mono, int do_rds, int first, RdsRsRef rr, cudaStream_t stream);
void launchCommit(AudioState *au, RdsState *rds, int ch0, int nch, int do_audio, int do_mono,
                  int do_rds, RdsRsRef rr, cudaStream_t stream);
void launchResample(const float *in0, const float *in1, size_t in_pitch, int in_off,
                    const float *hist, int hist_pitch, float *out, size_t acap, const float *bank,
                    uint32_t step, const AudioState *au, int mono, int max_out, int ch0, int nch,
                    cudaStream_t stream);
void launchAudioIir(float *audio, size_t acap, AudioState *au, const ChanParams *cp, int ch0,
                    int nch, float dc_a1, int mono, int clamp, int mono_dup, cudaStream_t stream);
// de-emphasis + DC blocker of the stereo rows as a warp-shuffle affine scan (fast arithmetic)
void launchAudioIirScan(float *audio, size_t acap, AudioState *au, const ChanParams *cp, int ch0,
                        int nch, float dc_a1, int clamp, cudaStream_t stream);
void launchStoreCounts(const AudioState *au, const RdsState *rds, uint32_t *n_audio,
                       uint32_t *n_groups, int ch0, int nch, int mono, uint32_t acap, uint32_t gcap,
                       cudaStream_t stream);
// MPX -> 171 kHz (tile kernel) -> serial demodulator (lane kernel); max_171 >= every channel's
// n171 of this call, r171 rows padded to whole 32-sample tiles
void launchRdsResample(const float *mpx, size_t mpx_pitch, const float *hist, int hist_pitch,
                       RdsRsRef rr, const float *bank, float *r171, size_t r_pitch,
                       int max_171, int ch0, int nch, const EngineConst &k, cudaStream_t stream);
void launchRdsDemod(RdsState *st, float2 *ring, const float *lpf, const float *mf, const float *dmf,
                    const float *r171, size_t r_pitch, uint8_t *bits_out, uint32_t bits_cap, int ch0,
                    int nch, const EngineConst &k, RdsRsRef rr, cudaStream_t stream);
// blk: the block number the groups found are tagged with
void launchBlockSync(const uint8_t *bits, uint32_t bits_cap, RdsState *st, unsigned long long *words,
                     fmgpu_rds_group *groups, uint32_t gcap, fmgpu_block_status *status,
                     int status_pitch, int blk, int ch0, int nch, cudaStream_t stream);

void launchSigLevel(const uint8_t *iq, size_t iq_stride, fmgpu_level_sums *sums, int nblk,
                    long samples_per_block, int ch0, int nch, cudaStream_t stream);

void launchPackPcm16(const float *audio, size_t acap, const uint32_t *n_audio, float volume,
                     int16_t *pcm, int C, int max_frames, cudaStream_t stream);

// synth.cu
cudaError_t launchSynth(const fmgpu_synth_params *params_dev, const int8_t *chips_dev,
                        int chips_per_channel, int n_channels, double fs_iq, size_t n_samples,
                        uint8_t *iq_dev, size_t iq_stride_bytes, cudaStream_t stream);

}  // namespace fmgpu

#endif  // FMGPU_KERNELS_H_
