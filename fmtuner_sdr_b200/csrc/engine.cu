// engine.cu — host side of the engine and the C ABI (include/fmgpu.h).
//
// Owns the device buffers described in engine.h, the per-channel settings the
// reference keeps inside its objects (FMDemod / StereoDecoder / AFPostProcessor /
// RDSDecoder members), and the launch sequence that restates the per-block body of
// the reference's main loop (src/main.cpp:1232-1308) for C channels at once.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <tuple>
#include <vector>

#include "cuda_handle.h"
#include "design.h"
#include "kernels.h"

using namespace fmgpu;

namespace {

std::string g_create_error;

size_t roundUp(size_t v, size_t m) { return (v + m - 1) / m * m; }

}  // namespace

struct fmgpu_engine {
  fmgpu_config cfg{};
  int C = 0, device = 0, fs = 0, N = 0, M = 1, maxBlocks = 1;
  size_t nmax = 0;    // DSP-rate samples per call
  size_t pitch = 0;   // nmax rounded up
  size_t iqPitch = 0; // bytes per channel in the internal IQ staging buffer
  size_t acap = 0;    // audio frames per channel per call
  size_t gcap = 0;    // groups per channel per call
  size_t bitsCap = 0;
  EngineConst k{};
  std::recursive_mutex mu;  // reset() may arrive from another host thread (SURVEY §8(b))

  // designs
  std::vector<float> decTaps;
  TapsParam decParam{}, decParamRaw{}, pilParam{}, audParam{};
  int decPp = 0, decL = 0, pilLp = 0, pilL = 0, audLp = 0, audL = 0;
  float decScale = 1.0f;
  // decimator arithmetic: 0 = FP32 FFMA2 kernel (bit-identical to the oracle's float chain),
  // 1 = integer contraction on the tensor cores (decim_tc.cu; one rounding of the exact sum)
  int decimMode = 0;
  // linear first-order recursions of the batched path (I/Q DC blockers; de-emphasis + DC blocker at
  // 32 kHz): 0 = serial lane recursions (bit-identical to the oracle), 1 = warp-shuffle parallel
  // scans (k_dcblock_scan, k_audio_iir_scan; float rounding differs)
  int scanMode = 0;
  // real-tap FIRs of the stereo decoder (pilot band-pass, L/R low-pass): 0 = FP32 FFMA2 chains
  // (bit-identical to the oracle), 1 = exact integer contractions on the tensor cores (fir_tc.cu)
  int firMode = 0;
  // channel filter -> AGC -> discriminator: 0 = three kernels in the reference's arithmetic
  // (bit-identical to the oracle), 1 = one tensor-core kernel (fir_tc.cu: integer channel filter,
  // discriminator in its epilogue; the AGC cannot change the discriminator's output and is left out)
  int demodMode = 0;
  bool decimTcOk = false, pilTcOk = false, audTcOk = false;
  FirTcTables pilTc{}, audTc{};
  DeviceArray<uint8_t> dPilB, dAudB;
  int smCount = 148;
  DeviceArray<uint8_t> dDecB;
  DeviceArray<int32_t> dDecOffs;
  std::vector<float> pilTaps, audTaps, rdsLpf;
  fmdesign::ResamplerDesign audRs, rdsRs;
  fmdesign::SymSyncDesign ss;

  // channel filter table
  struct ChanFilter {
    std::vector<float> taps;
    float scale;
    int lp;
    // tensor-core form (fir_tc.cu): integer taps' digits as a B image on the device
    FirTcTables tc{};
    DeviceArray<uint8_t> dB;
    bool tcOk = false;
  };
  std::vector<ChanFilter> filters;
  std::map<std::tuple<unsigned, float, float>, int> filterIndex;
  std::vector<ChanParams> hParams;
  bool paramsDirty = true;

  // device memory
  DeviceArray<uint8_t> dIq, dHistIq;
  DeviceArray<int> dHistValid;
  DeviceArray<float2> dX1, dX2, dY, dRing;
  DeviceArray<float> dR171;  // MPX resampled to 171 kHz (RDS branch): two buffers, by block parity
  size_t r171Pitch = 0;
  DeviceArray<float> dMpx, dPilot, dLraw, dRraw, dLf, dRf, dRdsHist, dMonoHist;
  DeviceArray<float> dChanTaps, dChanScale, dAudBank, dRdsBank, dRdsLpf, dMf, dDmf;
  DeviceArray<int> dChanLp;
  DeviceArray<ChanParams> dParams;
  DeviceArray<DemodState> dDemod;
  DeviceArray<StereoState> dStereo;
  DeviceArray<AudioState> dAudioSt;
  DeviceArray<RdsState> dRds;
  DeviceArray<RdsRsState> dRdsRs;  // 171 kHz resampler bookkeeping (apart from RdsState, see engine.h)
  // device result buffers, two sets: consecutive host submissions alternate between them; the
  // batched and stage-level calls use set 0 when the caller gives no buffers of its own
  struct Results {
    DeviceArray<float> audio;               // [C][2][acap]
    DeviceArray<fmgpu_rds_group> groups;    // [C][gcap]
    DeviceArray<fmgpu_block_status> status; // [C][maxBlocks]
    DeviceArray<uint32_t> nAudio, nGroups;  // [C]
  } res[2];
  DeviceArray<uint8_t> dBits;
  DeviceArray<unsigned long long> dWords;
  size_t x2Pitch = 0, yPitch = 0, mpxPitch = 0, lrPitch = 0, lfPitch = 0;
  Stream stream;  // stage-level (single-channel) entry points, resets, reads

  // ---- block pipeline ---------------------------------------------------------------------
  // The batched path runs ONE LOGICAL BLOCK AT A TIME through per-stage streams: every stage
  // (decimate, DC block, channel FIR, AGC, discriminator, pilot FIR, PLL/matrix, low-pass,
  // resample/de-emphasis, RDS) owns a stream and handles block after block in order (its
  // carried state demands that order anyway), and an event per (stage, block) releases the
  // consumer stage. Stage s of block q therefore runs beside stage s+1 of block q-1: the serial
  // one-lane-per-channel kernels of successive blocks overlap each other and the FIR kernels, and
  // the latency of a block is the slowest stage, not the sum of the stages.
  // Scratch buffers are rings of K = max(3, max_blocks) block slots laid out contiguously in
  // time behind the halo, [H | slot 0 | slot 1 | ...]: block q lives in slot q % K, its FIR halo
  // is simply the tail of the previous slot, and only slot 0 needs the tail of slot K-1 copied
  // in front of it. A producer about to overwrite slot q % K first waits for the consumers of
  // block q - K + 1: they are the last readers of that slot (its tail is their halo).
  enum Stage {
    ST_H2D = 0, ST_DECIM, ST_DC, ST_CHAN, ST_AGC, ST_FD, ST_PILOT, ST_STEREO, ST_LPF, ST_AF, ST_RDS,
    ST_D2H, ST_RDSRS /* MPX -> 171 kHz, one block ahead of the RDS demodulator */, ST_COUNT
  };
  struct Pipe {
    Stream st[ST_COUNT];              // the streams as created
    cudaStream_t run[ST_COUNT] = {};  // the streams in use (all the same one when serialStages)
    std::vector<Event> done[ST_COUNT];  // ring of ER events per stage
    Event callDone;                     // everything of the last batch call of this pipe
    Event hostDone[2];                  // per host ticket: results are in the host buffers
  };
  static constexpr int kMaxGroups = 2;        // channel ranges with their own pipe (streams)
  int nGroups = 1;
  Pipe pipes[kMaxGroups];
  int K = 3;             // ring slots
  int ER = 4;            // events per stage (> K)
  uint64_t seq = 0;      // logical blocks queued so far (slot = seq % K)
  bool headFresh = true; // the halo in front of slot 0 is already in place (start, reset, realign)
  bool asyncPending = false;
  bool serialStages = false;  // measurement aid: every stage on ONE stream, no overlap
  Event evStart;
  // streaming host path: two tickets in flight (submit k+1 before waiting for k)
  struct HostTicket {
    bool pending = false;
    uint32_t *nGroupsHost = nullptr;
    size_t groupCap = 0;
    bool clampGroups = false;
  } tickets[2];
  int nextTicket = 0;
  uint64_t lastSeq0 = 0;  // first block of the last batch call (debug reads)
  int lastBlocks = 0;

  int lastN = 0;  // DSP-rate samples of the last call (debug reads)
  uint64_t launches = 0;
  std::string lastError;

  bool timing = false;
  struct SpanRecord {
    const char *name;
    int group;  // pipeline group
    Event start, end;
  };
  std::vector<SpanRecord> spans;
  int curGroup = 0;
  bool timeline = false;        // keep the raw spans (fmgpu_debug_timeline) instead of merging
  std::vector<std::pair<const char *, float>> lastTimes;
};

namespace {

#define CK(expr)                                                                         \
  do {                                                                                   \
    cudaError_t err__ = (expr);                                                          \
    if (err__ != cudaSuccess) {                                                          \
      cudaGetLastError(); /* reported here: not left for the next call to find */       \
      e->lastError = std::string(#expr) + ": " + cudaGetErrorString(err__);              \
      return (err__ == cudaErrorMemoryAllocation) ? FMGPU_ENOMEM : FMGPU_ENODEV;         \
    }                                                                                    \
  } while (0)

TapsParam padFront(const std::vector<float> &hrev, int lp) {
  TapsParam t{};
  const int L = static_cast<int>(hrev.size());
  for (int i = 0; i < L; i++) {
    t.h[lp - L + i] = hrev[i];
  }
  return t;
}

std::vector<float> reversed(const std::vector<float> &h) {
  return std::vector<float>(h.rbegin(), h.rend());
}

DemodState defaultDemod() {
  DemodState s{};
  s.agc_g = 1.0f;
  s.agc_y2 = 1.0f;
  return s;
}

StereoState defaultStereo(const EngineConst &k) {
  StereoState s{};
  s.dtheta = k.pll_dtheta0;
  s.pll_freq = k.nominal_pll;
  return s;
}

void resetRdsLoops(RdsState &s, const EngineConst &k) {
  // SubcarrierSet::reset (subcarrier.cpp:108-114) + fresh BlockStream (rds_decoder.cpp:23-27)
  for (auto &w : s.wmf) {
    w = make_float2(0.0f, 0.0f);
  }
  s.tau = 0.0f;
  s.rate = 3.0f;
  s.del = 3.0f;
  s.q_hat = 0.0f;
  s.sos_v1 = 0.0f;
  s.b = 0;
  s.decim_counter = 0;
  s.theta = 0;
  s.dtheta = k.rds_dtheta0;
  s.since_reset = 0;
  s.realign = 1;
  s.bitcount = 0;
  s.until = 1;
  s.reg = 0;
  s.bits_since_lost = 0;
  s.expected = 0;
  s.in_sync = 0;
  s.err_ptr = 0;
  s.err_mask = 0;
  s.cur_recv = 0;
  s.cur_err = 0;
  for (int i = 0; i < 4; i++) {
    s.cur_data[i] = 0;
    s.pulse_pos[i] = 0;
    s.pulse_off[i] = 5;
  }
}

RdsState defaultRds(const EngineConst &k) {
  RdsState s{};
  s.agc_g = 0.08f;
  s.agc_y2 = 1.0f;
  resetRdsLoops(s, k);
  s.realign = 0;
  return s;
}

// The channel filter table's slot of a filter design (added on first use), or a negative FMGPU_E*
// code with lastError set.
int filterSlot(fmgpu_engine *e, unsigned len, float cutoff, float atten) {
  const auto key = std::make_tuple(len, cutoff, atten);
  auto it = e->filterIndex.find(key);
  if (it != e->filterIndex.end()) {
    return it->second;
  }
  if (static_cast<int>(e->filters.size()) >= MAX_CHAN_FILTERS) {
    e->lastError = "channel filter table full";
    return FMGPU_ENOMEM;
  }
  fmgpu_engine::ChanFilter f;
  f.taps = fmdesign::kaiserLowpass(len, cutoff, atten, 0.0f);
  f.scale = 2.0f * cutoff;
  f.lp = static_cast<int>(roundUp(len, 8));
  const int slot = static_cast<int>(e->filters.size());
  std::vector<float> row(CHAN_TAPS_PITCH, 0.0f);
  const std::vector<float> hrev = reversed(f.taps);
  for (unsigned i = 0; i < len; i++) {
    row[CHAN_TAPS_PITCH - len + i] = hrev[i];
  }
  CK(cudaMemcpy(e->dChanTaps + static_cast<size_t>(slot) * CHAN_TAPS_PITCH, row.data(),
                CHAN_TAPS_PITCH * sizeof(float), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(e->dChanLp + slot, &f.lp, sizeof(int), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(e->dChanScale + slot, &f.scale, sizeof(float), cudaMemcpyHostToDevice));
  {
    const float *h = row.data() + (CHAN_TAPS_PITCH - f.lp);   // the padded taps as k_chanfir reads them
    if (chanTcSupported(h, f.lp, H_X2)) {
      firTcBuildTables(h, f.lp, &f.tc);
      if (devAlloc(&f.dB, f.tc.b_image.size()) == cudaSuccess &&
          cudaMemcpy(f.dB, f.tc.b_image.data(), f.tc.b_image.size(), cudaMemcpyHostToDevice) == cudaSuccess) {
        f.tcOk = true;
      } else {
        cudaGetLastError();  // no tensor-core image: the three-kernel path runs this filter
      }
    }
  }
  e->filters.push_back(std::move(f));
  e->filterIndex[key] = slot;
  return slot;
}

void syncPipes(fmgpu_engine *e);

int uploadParams(fmgpu_engine *e) {
  if (!e->paramsDirty) {
    return FMGPU_OK;
  }
  syncPipes(e);  // blocks already queued keep the parameters they were queued with
  CK(cudaMemcpyAsync(e->dParams, e->hParams.data(), e->hParams.size() * sizeof(ChanParams),
                     cudaMemcpyHostToDevice, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  e->paramsDirty = false;
  return FMGPU_OK;
}

void deemphCoeffs(int tau_us, int rate, int *on, float *b0, float *a1) {
  // fm_demod.cpp:50-62 / af_post_processor.cpp:31-45
  if (tau_us <= 0) {
    *on = 0;
    return;
  }
  *on = 1;
  const float tau = static_cast<float>(tau_us) * 1e-6f;
  const float dt = 1.0f / static_cast<float>(rate);
  const float alpha = dt / (tau + dt);
  *b0 = alpha / 1.0f;
  *a1 = (-(1.0f - alpha)) / 1.0f;
}

template <typename F> int forChannels(fmgpu_engine *e, int channel, F &&f) {
  if (!e || channel < -1 || channel >= e->C) {
    return FMGPU_EINVAL;
  }
  const int lo = (channel < 0) ? 0 : channel;
  const int hi = (channel < 0) ? e->C : channel + 1;
  for (int c = lo; c < hi; c++) {
    const int rc = f(c);
    if (rc != FMGPU_OK) {
      return rc;
    }
  }
  return FMGPU_OK;
}

struct Span {
  fmgpu_engine *e;
  cudaStream_t s;
  cudaEvent_t b = nullptr;
  Span(fmgpu_engine *e_, const char *name, cudaStream_t s_) : e(e_), s(s_) {
    if (e->timing) {
      e->spans.push_back({name, e->curGroup, {}, {}});
      fmgpu_engine::SpanRecord &r = e->spans.back();
      cudaEventCreate(r.start.out());
      cudaEventCreate(r.end.out());
      cudaEventRecord(r.start, s);
      b = r.end;
    }
  }
  ~Span() {
    if (e->timing) {
      cudaEventRecord(b, s);
    }
  }
};

// zero a [C][pitch] region [0, count) of channel c (or all)
template <typename T>
void zeroPrefix(const DeviceArray<T> &buf, size_t pitch, size_t count, int lo, int hi, cudaStream_t s) {
  cudaMemset2DAsync(buf + static_cast<size_t>(lo) * pitch, pitch * sizeof(T), 0, count * sizeof(T),
                    static_cast<size_t>(hi - lo), s);
}

// One strided copy of the same `bytes` to `field` of every state struct of channels [lo, hi).
template <typename S>
int fillStateField(fmgpu_engine *e, const DeviceArray<S> &base, size_t fieldOffset, const void *value,
                          size_t bytes, int lo, int hi) {
  const size_t cnt = static_cast<size_t>(hi - lo);
  std::vector<uint8_t> rows(cnt * bytes);
  for (size_t i = 0; i < cnt; i++) {
    std::memcpy(rows.data() + i * bytes, value, bytes);
  }
  CK(cudaMemcpy2DAsync(reinterpret_cast<uint8_t *>(base + lo) + fieldOffset, sizeof(S), rows.data(),
                       bytes, bytes, cnt, cudaMemcpyHostToDevice, e->stream));
  CK(cudaStreamSynchronize(e->stream));  // `rows` is pageable and about to go out of scope
  return FMGPU_OK;
}

// ---------------------------------------------------------------------------
// pipeline stages: one logical block of channels [ch0, ch0 + nch) on stream s
// ---------------------------------------------------------------------------
// the decimating FIR of n_out outputs per channel into x1 (history in dHistIq), either flavour
void runDecim(fmgpu_engine *e, const uint8_t *iq, size_t stride, float2 *x1, int n_out, int ch0,
              int nch, cudaStream_t s) {
  if (e->decimMode == 1 && e->decimTcOk && n_out % 16 == 0 && (stride & 15u) == 0 &&
      (reinterpret_cast<uintptr_t>(iq) & 15u) == 0) {
    const cudaError_t err =
        launchDecimTc(e->M, e->decL, iq, stride, static_cast<size_t>(n_out) * e->M * 2, e->dHistIq,
                      e->dHistValid, e->C, x1, e->pitch, n_out, ch0, nch, e->decScale, e->dDecB,
                      e->dDecOffs, e->smCount, s);
    if (err == cudaSuccess) {
      return;
    }
    e->lastError = std::string("tensor-core decimator: ") + cudaGetErrorString(err);
  }
  launchDecim(e->M, iq, stride, e->dHistIq, e->dHistValid, x1, e->pitch, n_out, ch0, nch, e->decPp,
              e->decL, e->decScale, e->decParam, e->decParamRaw, s);
}

// a real-tap FIR of the stereo decoder, either flavour. data_shift: fixed-point scale of the
// tensor-core form (the multiplex is bounded by pi * fd_ref < 2; the matrix outputs by 3x that)
void runFirReal(fmgpu_engine *e, const FirRealJob &j, int nsig, int nch, const TapsParam &taps, bool tc_ok,
                const FirTcTables &t, const uint8_t *b_dev, int data_shift, cudaStream_t s) {
  if (e->firMode == 1 && tc_ok && j.n_total % 32 == 0) {
    const cudaError_t err = launchFirTc(j, nsig, nch, t, b_dev, data_shift, e->smCount, s);
    if (err == cudaSuccess) {
      return;
    }
    e->lastError = std::string("tensor-core FIR: ") + cudaGetErrorString(err);
  }
  launchFirReal(j, nsig, nch, taps, s);
}

// Measurement variant (build_variant with -DFMGPU_EXP_SKIP, never the shipped library): leave the
// main kernel of the stages named in FMGPU_SKIP out of the block pipeline, to see what each one
// costs the step beside the others. Results are WRONG with any stage skipped.
#ifdef FMGPU_EXP_SKIP
static bool expSkip(const char *name) {
  static const std::string v = getenv("FMGPU_SKIP") ? getenv("FMGPU_SKIP") : "";
  return v.find(name) != std::string::npos;
}
#else
constexpr bool expSkip(const char *) { return false; }
#endif

struct BatchOut {
  float *audio = nullptr;  // [C][2][acap]
  size_t acap = 0;
  uint32_t *nAudio = nullptr;
  fmgpu_rds_group *groups = nullptr;
  uint32_t gcap = 0;
  uint32_t *nGroups = nullptr;
  fmgpu_block_status *status = nullptr;  // [C][n_blocks]
};

// the engine's own result buffers of set `set` (the stage-level entry points copy from set 0)
BatchOut engineOut(const fmgpu_engine *e, int set = 0) {
  const fmgpu_engine::Results &r = e->res[set];
  BatchOut out;
  out.audio = r.audio;
  out.acap = e->acap;
  out.nAudio = r.nAudio;
  out.groups = r.groups;
  out.gcap = static_cast<uint32_t>(e->gcap);
  out.nGroups = r.nGroups;
  out.status = r.status;
  return out;
}

// upper bound of the 171 kHz samples n DSP-rate inputs produce (any resampler phase)
int max171(const fmgpu_engine *e, int n) {
  return static_cast<int>((static_cast<unsigned long long>(n) << 24) / e->k.rds_step) + 2;
}

// the 171 kHz rows of block parity par
float *r171Rows(const fmgpu_engine *e, int par) {
  return e->dR171 + static_cast<size_t>(par) * static_cast<size_t>(e->C) * e->r171Pitch;
}

bool anyAgc(const fmgpu_engine *e, int ch0, int nch) {
  for (int c = ch0; c < ch0 + nch; c++) {
    if (e->hParams[c].agc_mode != 0) {
      return true;
    }
  }
  return false;
}

// Ring buffers whose rows begin with a FIR / delay halo: the samples the next block's stage reads in
// front of its own.
enum Halo : unsigned { HALO_X2 = 1, HALO_Y = 2, HALO_MPX = 4, HALO_LR = 8, HALO_LF = 16 };

// Copy the halo of every buffer in `which` from the samples just before position pos of the row (the
// end of the last block written) to the front of the row, for channels [ch0, ch0 + nch).
void carryHalos(fmgpu_engine *e, unsigned which, size_t pos, int ch0, int nch, cudaStream_t s) {
  if (which & HALO_X2) {
    launchCarryF2(e->dX2, e->x2Pitch, H_X2, pos, ch0, nch, s);
    e->launches += 1;
  }
  if (which & HALO_Y) {
    launchCarryF2(e->dY, e->yPitch, Y_OFF, pos, ch0, nch, s);  // slot Y_OFF-1 <- last output
    e->launches += 1;
  }
  if (which & HALO_MPX) {
    launchCarryF32(e->dMpx, e->mpxPitch, H_MPX, pos, ch0, nch, s);
    e->launches += 1;
  }
  if (which & HALO_LR) {
    launchCarryF32(e->dLraw, e->lrPitch, H_LR, pos, ch0, nch, s);
    launchCarryF32(e->dRraw, e->lrPitch, H_LR, pos, ch0, nch, s);
    e->launches += 2;
  }
  if (which & HALO_LF) {
    launchCarryF32(e->dLf, e->lfPitch, H_LF, pos, ch0, nch, s);
    launchCarryF32(e->dRf, e->lfPitch, H_LF, pos, ch0, nch, s);
    e->launches += 2;
  }
}

// One logical block for the stage functions below. The block pipeline (launchBlock) queues them on the
// stage streams; the stage-level entry points call them on the engine's stream with t0 = 0 and carry
// their halos themselves after the call.
struct BlockRef {
  int ch0, nch;
  size_t t0;  // the block's offset in every ring buffer
  int n;      // samples
  fmgpu_block_status *status;  // the block's entry in channel 0's status row (nullptr: none)
  int statusPitch;
  bool carry;  // ring slot 0: bring the tail of the last slot in front of it first
};

BlockRef stageBlock(int channel, int n) { return BlockRef{channel, 1, 0, n, nullptr, 1, false}; }

size_t ringEnd(const fmgpu_engine *e) { return static_cast<size_t>(e->K) * e->N; }

// IQ bytes -> x1: the decimating FIR (M == 1: the conversion to float alone)
void stageDecimate(fmgpu_engine *e, const BlockRef &k, const uint8_t *iq, size_t stride, cudaStream_t s) {
  Span sp(e, "decimate", s);
  if (e->M == 1) {
    launchConvertU8(iq, stride, e->dX1 + k.t0, e->pitch, k.n, k.ch0, k.nch, s);
    e->launches += 1;
    return;
  }
  if (!expSkip("decimate")) runDecim(e, iq, stride, e->dX1 + k.t0, k.n, k.ch0, k.nch, s);
  launchCarryIq(e->dHistIq, e->dHistValid, iq, stride, static_cast<long>(k.n) * e->M, k.ch0, k.nch, s);
  e->launches += 2;
}

// I/Q DC blockers: complex float rows x (else the IQ bytes iq at the DSP rate) -> x2. scan: the
// warp-shuffle form (float input only; fast arithmetic)
void stageDcBlock(fmgpu_engine *e, const BlockRef &k, const float2 *x, size_t xPitch, const uint8_t *iq,
                  size_t iqStride, bool scan, cudaStream_t s) {
  Span sp(e, "dcblock", s);
  if (k.carry) {
    carryHalos(e, HALO_X2, ringEnd(e), k.ch0, k.nch, s);
  }
  if (scan) {
    if (!expSkip("dcblock")) launchDcBlockScan(x, xPitch, e->dX2 + k.t0, e->x2Pitch, e->dDemod, k.status,
                                               k.statusPitch, k.n, k.ch0, k.nch, e->k.dc_a1_iq, s);
  } else {
    launchDcBlock(x, xPitch, iq, iqStride, e->dX2 + k.t0, e->x2Pitch, e->dDemod, k.status, k.statusPitch,
                  k.n, k.ch0, k.nch, e->k.dc_a1_iq, s);
  }
  e->launches += 1;
}

// channel filter + discriminator as one tensor-core kernel, every channel on filter filt: x2 -> MPX (and
// the discriminator's carried sample into the y row). False: refused before anything was launched
// (alignment, pitch).
bool stageChanDemod(fmgpu_engine *e, const BlockRef &k, int filt, cudaStream_t s) {
  Span sp(e, "chan_demod", s);
  if (k.carry) {
    carryHalos(e, HALO_Y | HALO_MPX, ringEnd(e), k.ch0, k.nch, s);
  }
  const auto &f = e->filters[filt];
  const cudaError_t err = expSkip("chan_demod") ? cudaSuccess :
      launchChanDemodTc(e->dX2 + k.t0, e->x2Pitch, H_X2, e->dY + k.t0, e->yPitch, e->dMpx + k.t0, e->mpxPitch,
                        H_MPX, k.n, k.ch0, k.nch, f.scale, e->k.fd_ref, f.tc, f.dB, 21, e->smCount, s);
  e->launches += 1;
  if (err != cudaSuccess) {
    e->lastError = std::string("tensor-core channel filter + discriminator: ") + cudaGetErrorString(err);
    return false;
  }
  return true;
}

// x2 -> y
void stageChanFir(fmgpu_engine *e, const BlockRef &k, cudaStream_t s) {
  Span sp(e, "chanfir", s);
  launchChanFir(e->dX2 + k.t0, e->x2Pitch, e->dY + k.t0, e->yPitch, e->dChanTaps, e->dChanLp, e->dChanScale,
                e->dParams, k.n, k.ch0, k.nch, s);
  e->launches += 1;
}

// y in place
void stageAgc(fmgpu_engine *e, const BlockRef &k, cudaStream_t s) {
  // (running the discriminator inside this lane kernel was tried: its two IEEE divisions per
  // sample do not hide behind the AGC recursion, the stage took 5.6 ms instead of 2.7 + 0.7)
  Span sp(e, "agc", s);
  launchAgc(e->dY + k.t0, e->yPitch, e->dDemod, e->dParams, k.n, k.ch0, k.nch, s);
  e->launches += 1;
}

// y -> MPX
void stageFreqDem(fmgpu_engine *e, const BlockRef &k, cudaStream_t s) {
  Span sp(e, "freqdem", s);
  if (k.carry) {
    carryHalos(e, HALO_Y | HALO_MPX, ringEnd(e), k.ch0, k.nch, s);
  }
  launchFreqDem(e->dY + k.t0, e->yPitch, e->dMpx + k.t0, e->mpxPitch, k.n, k.ch0, k.nch, e->k.fd_ref, s);
  e->launches += 1;
}

// MPX -> 171 kHz rows of parity par (tile kernel; the RDS demodulator of the previous block may run
// beside it on the other parity's rows)
void stageRdsResample(fmgpu_engine *e, const BlockRef &k, int par, cudaStream_t s) {
  const RdsRsRef rr{e->dRdsRs, par};
  Span sp(e, "rds_resample", s);
  launchPrepare(e->dAudioSt, e->dRds, nullptr, 1, k.n, k.ch0, k.nch, e->k.aud_step, e->k.rds_step, 0, 0,
                PREPARE_RDS_RESAMPLER, 0, rr, s);
  if (!expSkip("rds_resample")) launchRdsResample(e->dMpx + k.t0, e->mpxPitch, e->dRdsHist, 32, rr, e->dRdsBank,
                                                  r171Rows(e, par), e->r171Pitch, max171(e, k.n), k.ch0, k.nch,
                                                  e->k, s);
  launchSaveTail(e->dMpx + k.t0, e->mpxPitch, H_MPX, e->dRdsHist, 32, RDS_HIST, k.n, k.ch0, k.nch, s);
  launchCommit(e->dAudioSt, e->dRds, k.ch0, k.nch, 0, 0, 1, rr, s);
  e->launches += 4;
}

// 171 kHz rows of parity par -> bits -> groups into out.groups, tagged with block number b. first: the
// call's first block (its counters start at zero); last: store the call's group counts to out.nGroups.
void stageRdsDemod(fmgpu_engine *e, const BlockRef &k, int par, const BatchOut &out, int b, bool first,
                   bool last, cudaStream_t s) {
  const RdsRsRef rr{e->dRdsRs, par};
  {
    Span sp(e, "rds", s);  // lane kernel: 57 kHz mix ... bits
    if (first) {
      launchPrepare(e->dAudioSt, e->dRds, nullptr, 1, k.n, k.ch0, k.nch, e->k.aud_step, e->k.rds_step, 0, 0,
                    PREPARE_RDS_COUNTERS, 1, rr, s);
      e->launches += 1;
    }
    if (!expSkip("rds_demod")) launchRdsDemod(e->dRds, e->dRing, e->dRdsLpf, e->dMf, e->dDmf, r171Rows(e, par),
                                              e->r171Pitch, e->dBits, static_cast<uint32_t>(e->bitsCap), k.ch0,
                                              k.nch, e->k, rr, s);
  }
  e->launches += 1;
  {
    Span sp(e, "rds_sync", s);  // syndromes at every bit offset + block sync state machine
    if (!expSkip("rds_sync")) launchBlockSync(e->dBits, static_cast<uint32_t>(e->bitsCap), e->dRds, e->dWords,
                                              out.groups, out.gcap, k.status, k.statusPitch, b, k.ch0, k.nch, s);
    if (last) {
      // the call's group counts, from the stream that owns RdsState::n_groups: the next call's
      // first k_prepare on this stream zeroes it again
      launchStoreCounts(e->dAudioSt, e->dRds, nullptr, out.nGroups, k.ch0, k.nch, e->cfg.stereo ? 0 : 1,
                        static_cast<uint32_t>(out.acap), out.gcap, s);
      e->launches += 1;
    }
  }
  e->launches += 1;
}

// MPX -> pilot (band-pass)
void stagePilot(fmgpu_engine *e, const BlockRef &k, cudaStream_t s) {
  Span sp(e, "pilot_fir", s);
  FirRealJob j{};
  j.in[0] = e->dMpx + k.t0;
  j.out[0] = e->dPilot + k.t0;
  j.in_pitch = e->mpxPitch;
  j.out_pitch = e->pitch;
  j.in_off = H_MPX;
  j.out_off = 0;
  j.n_total = k.n;
  j.Lp = e->pilLp;
  j.scale = 1.0f;
  j.ch0 = k.ch0;
  if (!expSkip("pilot_fir")) runFirReal(e, j, 1, k.nch, e->pilParam, e->pilTcOk, e->pilTc, e->dPilB, 22, s);
  e->launches += 1;
}

// MPX + pilot -> L/R before the low-pass (PLL, blend, matrix)
void stageStereo(fmgpu_engine *e, const BlockRef &k, cudaStream_t s) {
  Span sp(e, "stereo_pll", s);
  if (k.carry) {
    carryHalos(e, HALO_LR, ringEnd(e), k.ch0, k.nch, s);
  }
  if (!expSkip("stereo_pll")) launchStereo(e->dMpx + k.t0, e->mpxPitch, e->dPilot + k.t0, e->pitch,
                                           e->dLraw + k.t0, e->dRraw + k.t0, e->lrPitch, e->dStereo, e->dParams,
                                           k.status, k.statusPitch, k.n, k.ch0, k.nch, e->k, s);
  e->launches += 1;
}

// L/R -> 15 kHz low-pass
void stageLpf(fmgpu_engine *e, const BlockRef &k, cudaStream_t s) {
  Span sp(e, "audio_lpf", s);
  if (k.carry) {
    carryHalos(e, HALO_LF, ringEnd(e), k.ch0, k.nch, s);
  }
  FirRealJob j{};
  j.in[0] = e->dLraw + k.t0;
  j.in[1] = e->dRraw + k.t0;
  j.out[0] = e->dLf + k.t0;
  j.out[1] = e->dRf + k.t0;
  j.in_pitch = e->lrPitch;
  j.out_pitch = e->lfPitch;
  j.in_off = H_LR;
  j.out_off = H_LF;
  j.n_total = k.n;
  j.Lp = e->audLp;
  j.scale = e->k.aud_scale;
  j.ch0 = k.ch0;
  if (!expSkip("audio_lpf")) runFirReal(e, j, 2, k.nch, e->audParam, e->audTcOk, e->audTc, e->dAudB, 20, s);
  e->launches += 1;
}

int maxAudioOut(const fmgpu_engine *e, const BatchOut &out, int n) {
  return static_cast<int>(std::min<size_t>(
      out.acap, static_cast<size_t>((static_cast<double>(n) * 16777216.0) / e->k.aud_step) + 2));
}

// low-passed L/R -> out.audio rows (resample, de-emphasis, DC block; clamp: to +-1). first: the call's
// first block (frames start at the row start); scan: the de-emphasis + DC blocker as a warp-shuffle scan
void stageAfPost(fmgpu_engine *e, const BlockRef &k, const BatchOut &out, bool first, bool scan, int clamp,
                 cudaStream_t s) {
  Span sp(e, "afpost", s);
  launchPrepare(e->dAudioSt, e->dRds, k.status, k.statusPitch, k.n, k.ch0, k.nch, e->k.aud_step,
                e->k.rds_step, 1, 0, PREPARE_RDS_NONE, first ? 1 : 0, RdsRsRef{e->dRdsRs, 0}, s);
  if (!expSkip("afpost")) launchResample(e->dLf + k.t0, e->dRf + k.t0, e->lfPitch, H_LF, nullptr, 0, out.audio,
                                         out.acap, e->dAudBank, e->k.aud_step, e->dAudioSt, 0,
                                         maxAudioOut(e, out, k.n), k.ch0, k.nch, s);
  if (scan) {
    launchAudioIirScan(out.audio, out.acap, e->dAudioSt, e->dParams, k.ch0, k.nch, e->k.dc_a1_af, clamp, s);
  } else {
    launchAudioIir(out.audio, out.acap, e->dAudioSt, e->dParams, k.ch0, k.nch, e->k.dc_a1_af, 0, clamp, 0, s);
  }
  launchCommit(e->dAudioSt, e->dRds, k.ch0, k.nch, 1, 0, 0, RdsRsRef{e->dRdsRs, 0}, s);
  e->launches += 4;
}

// FMDemod mono chain (fm_demod.cpp:210-226, main.cpp:1267-1279): MPX -> resample -> de-emphasis -> DC
// block into audio row 0; dup: x0.5 to both rows
void stageMono(fmgpu_engine *e, const BlockRef &k, const BatchOut &out, bool first, int clamp, int dup,
               cudaStream_t s) {
  Span sp(e, "mono", s);
  launchPrepare(e->dAudioSt, e->dRds, k.status, k.statusPitch, k.n, k.ch0, k.nch, e->k.aud_step,
                e->k.rds_step, 0, 1, PREPARE_RDS_NONE, first ? 1 : 0, RdsRsRef{e->dRdsRs, 0}, s);
  launchResample(e->dMpx + k.t0, nullptr, e->mpxPitch, H_MPX, e->dMonoHist, 32, out.audio, out.acap, e->dAudBank,
                 e->k.aud_step, e->dAudioSt, 1, maxAudioOut(e, out, k.n), k.ch0, k.nch, s);
  launchAudioIir(out.audio, out.acap, e->dAudioSt, e->dParams, k.ch0, k.nch, e->k.mono_dc_a1, 1, clamp, dup, s);
  launchSaveTail(e->dMpx + k.t0, e->mpxPitch, H_MPX, e->dMonoHist, 32, AUD_RS_LEN - 1, k.n, k.ch0, k.nch, s);
  launchCommit(e->dAudioSt, e->dRds, k.ch0, k.nch, 0, 1, 0, RdsRsRef{e->dRdsRs, 0}, s);
  e->launches += 5;
}

void collectTimes(fmgpu_engine *e) {
  if (!e->timing) {
    return;
  }
  e->lastTimes.clear();
  for (auto &sp : e->spans) {
    float ms = 0.0f;
    cudaEventSynchronize(sp.end);
    cudaEventElapsedTime(&ms, sp.start, sp.end);
    bool merged = false;
    for (auto &t : e->lastTimes) {
      if (std::strcmp(t.first, sp.name) == 0) {
        t.second += ms;
        merged = true;
      }
    }
    if (!merged) {
      e->lastTimes.emplace_back(sp.name, ms);
    }
  }
  e->spans.clear();
}

// ---------------------------------------------------------------------------
// block pipeline (see fmgpu_engine::Pipe)
// ---------------------------------------------------------------------------
// channel range of pipeline group g (multiples of 32 channels: one warp of lane kernels)
void groupRange(const fmgpu_engine *e, int g, int *ch0, int *nch) {
  const int per = static_cast<int>(roundUp((e->C + e->nGroups - 1) / e->nGroups, 32));
  *ch0 = std::min(e->C, g * per);
  *nch = std::min(e->C, (g + 1) * per) - *ch0;
}

void syncPipes(fmgpu_engine *e) {
  if (!e->asyncPending) {
    return;
  }
  for (auto &P : e->pipes) {
    for (cudaStream_t st : P.st) {
      if (st) {
        cudaStreamSynchronize(st);
      }
    }
  }
  e->asyncPending = false;
}

// Put every FIR halo back in front of slot 0 and restart the block counter at a multiple of K:
// the stage-level entry points and reset() work at buffer offset 0 with in-place carries.
void realign(fmgpu_engine *e) {
  syncPipes(e);
  e->lastBlocks = 0;
  const int slot = static_cast<int>(e->seq % static_cast<uint64_t>(e->K));
  if (slot == 0 && e->headFresh) {
    return;
  }
  const size_t pos = static_cast<size_t>(slot == 0 ? e->K : slot) * e->N;  // end of the last block
  carryHalos(e, HALO_X2 | HALO_Y | HALO_MPX | HALO_LR | HALO_LF, pos, 0, e->C, e->stream);
  cudaStreamSynchronize(e->stream);
  e->seq = roundUp(e->seq, e->K);
  e->headFresh = true;
}

// One logical block (global number q, block b of a call of nb blocks) of channels
// [ch0, ch0 + nch) through the stage streams of pipe P. iq / stride: this block's bytes.
void launchBlock(fmgpu_engine *e, fmgpu_engine::Pipe &P, int ch0, int nch, uint64_t q, int b, int nb,
                 const uint8_t *iq, size_t stride, bool waitH2D, const BatchOut &out,
                 const float2 *xcf = nullptr, size_t xcfStride = 0) {
  using E = fmgpu_engine;
  const int K = e->K, N = e->N;
  const int slot = static_cast<int>(q % static_cast<uint64_t>(K));
  const bool stereo = e->cfg.stereo != 0;
  const bool first = (b == 0), last = (b == nb - 1);
  // slot 0 brings the tail of slot K-1 in front of it
  const BlockRef blk{ch0, nch, static_cast<size_t>(slot) * N, N, out.status ? out.status + b : nullptr, nb,
                     (slot == 0) && !e->headFresh};
  auto ev = [&](int st, uint64_t qq) -> cudaEvent_t { return P.done[st][qq % static_cast<uint64_t>(e->ER)]; };
  // producers: stages of THIS block whose output the stage reads; overwritten: consumer stages
  // of the buffers it writes, which must have finished block q - K (same ring slot)
  auto need = [&](int st, std::initializer_list<int> producers, std::initializer_list<int> readers) {
    for (int p : producers) {
      cudaStreamWaitEvent(P.run[st], ev(p, q), 0);
    }
    // Block q overwrites ring slot q % K. Its last readers are not those of block q - K but of
    // block q - K + 1, whose FIR / delay halo is the TAIL of that slot (only slot 0 reads a copied
    // halo). With K >= 3 this still lets stage s of block q run beside stage s + 1 of block q - 1.
    const uint64_t back = static_cast<uint64_t>(std::max(K - 1, 1));  // K = 1: the halo is a copy
    if (q >= back) {
      for (int r : readers) {
        cudaStreamWaitEvent(P.run[st], ev(r, q - back), 0);
      }
    }
  };
  auto done = [&](int st) { cudaEventRecord(ev(st, q), P.run[st]); };

  const bool decim = (e->M > 1) && !xcf;
  if (decim) {
    if (waitH2D) {
      need(E::ST_DECIM, {E::ST_H2D}, {E::ST_DC});
    } else {
      need(E::ST_DECIM, {}, {E::ST_DC});
    }
    stageDecimate(e, blk, iq, stride, P.run[E::ST_DECIM]);
    done(E::ST_DECIM);
  }
  {
    if (decim) {
      need(E::ST_DC, {E::ST_DECIM}, {E::ST_CHAN});
    } else if (waitH2D) {
      need(E::ST_DC, {E::ST_H2D}, {E::ST_CHAN});
    } else {
      need(E::ST_DC, {}, {E::ST_CHAN});
    }
    // float input (complex-float rows at the DSP rate, read in place, or the decimator's output) may
    // take the scan form; IQ bytes at the DSP rate go to the serial recursions
    const float2 *x = xcf ? xcf : (decim ? e->dX1 + blk.t0 : nullptr);
    stageDcBlock(e, blk, x, xcf ? xcfStride : e->pitch, x ? nullptr : iq, stride, e->scanMode == 1 && x,
                 P.run[E::ST_DC]);
  }
  done(E::ST_DC);
  // fused tensor-core form of channel filter + discriminator: every channel of the range on the same
  // channel filter, and that filter has a tensor-core image
  int fusedFilt = -1;
  if (e->demodMode == 1 && N % 32 == 0) {
    fusedFilt = e->hParams[ch0].filt;
    for (int c = ch0 + 1; c < ch0 + nch && fusedFilt >= 0; c++) {
      if (e->hParams[c].filt != fusedFilt) {
        fusedFilt = -1;
      }
    }
    if (fusedFilt >= 0 && !e->filters[fusedFilt].tcOk) {
      fusedFilt = -1;
    }
  }
  bool fused = false;
  if (fusedFilt >= 0) {
    // one kernel on the channel-filter stream; the AGC and discriminator stages of this block are empty
    if (stereo) {
      need(E::ST_CHAN, {E::ST_DC}, {E::ST_AGC, E::ST_FD, E::ST_PILOT, E::ST_STEREO, E::ST_RDS, E::ST_RDSRS});
    } else {
      need(E::ST_CHAN, {E::ST_DC}, {E::ST_AGC, E::ST_FD, E::ST_RDS, E::ST_RDSRS, E::ST_AF});
    }
    // refused: the three-kernel path takes the block
    fused = stageChanDemod(e, blk, fusedFilt, P.run[E::ST_CHAN]);
  }
  if (!fused) {
    need(E::ST_CHAN, {E::ST_DC}, {E::ST_AGC, E::ST_FD});
    stageChanFir(e, blk, P.run[E::ST_CHAN]);
  }
  done(E::ST_CHAN);
  need(E::ST_AGC, {E::ST_CHAN}, {E::ST_FD});
  if (!fused && anyAgc(e, ch0, nch)) {
    stageAgc(e, blk, P.run[E::ST_AGC]);
  }
  done(E::ST_AGC);
  if (stereo) {
    need(E::ST_FD, {E::ST_AGC}, {E::ST_PILOT, E::ST_STEREO, E::ST_RDS, E::ST_RDSRS});
  } else {
    need(E::ST_FD, {E::ST_AGC}, {E::ST_RDS, E::ST_RDSRS, E::ST_AF /* the mono chain reads MPX */});
  }
  if (!fused) {
    stageFreqDem(e, blk, P.run[E::ST_FD]);
  }
  done(E::ST_FD);
  // ---- RDS branch --------------------------------------------------------------------------
  // two stages: the 171 kHz resampler (tile kernel) of block q + 1 runs beside the demodulator
  // (lane kernel) of block q; the 171 kHz rows and their counts are double-buffered by block parity
  const int par = static_cast<int>(q & 1);
  need(E::ST_RDSRS, {E::ST_FD}, {});
  if (q >= 2) {
    cudaStreamWaitEvent(P.run[E::ST_RDSRS], ev(E::ST_RDS, q - 2), 0);   // the demodulator is done with this parity's rows
  }
  stageRdsResample(e, blk, par, P.run[E::ST_RDSRS]);
  done(E::ST_RDSRS);
  need(E::ST_RDS, {E::ST_RDSRS}, {});
  stageRdsDemod(e, blk, par, out, b, first, last, P.run[E::ST_RDS]);
  done(E::ST_RDS);
  // ---- audio branch ------------------------------------------------------------------------
  cudaStream_t sAf = P.run[E::ST_AF];
  if (stereo) {
    need(E::ST_PILOT, {E::ST_FD}, {E::ST_STEREO});
    stagePilot(e, blk, P.run[E::ST_PILOT]);
    done(E::ST_PILOT);
    need(E::ST_STEREO, {E::ST_PILOT}, {E::ST_LPF});
    stageStereo(e, blk, P.run[E::ST_STEREO]);
    done(E::ST_STEREO);
    need(E::ST_LPF, {E::ST_STEREO}, {E::ST_AF});
    stageLpf(e, blk, P.run[E::ST_LPF]);
    done(E::ST_LPF);
    need(E::ST_AF, {E::ST_LPF}, {});
    stageAfPost(e, blk, out, first, e->scanMode == 1, 1, sAf);
  } else {
    need(E::ST_AF, {E::ST_FD}, {});
    stageMono(e, blk, out, first, 1, 1, sAf);
  }
  if (last) {
    // the call's counts, once both branches have finished its last block
    cudaStreamWaitEvent(sAf, ev(E::ST_RDS, q), 0);
    Span sp(e, "commit", sAf);
    launchStoreCounts(e->dAudioSt, e->dRds, out.nAudio, nullptr, ch0, nch, stereo ? 0 : 1,
                      static_cast<uint32_t>(out.acap), out.gcap, sAf);
    e->launches += 1;
  }
  done(E::ST_AF);
}

int checkBatchArgs(fmgpu_engine *e, const void *iq, size_t stride, int n_blocks, bool device,
                   const float *audio, size_t audio_cap) {
  if (!iq || n_blocks < 1 || n_blocks > e->maxBlocks) {
    e->lastError = "process: n_blocks out of range or null input";
    return FMGPU_EINVAL;
  }
  if (device && ((reinterpret_cast<uintptr_t>(iq) & 15u) || (stride & 15u))) {
    e->lastError = "process: iq buffer and stride must be 16-byte aligned";
    return FMGPU_EINVAL;
  }
  if (stride < static_cast<size_t>(n_blocks) * e->N * e->M * 2) {
    e->lastError = "process: stride smaller than the bytes per channel";
    return FMGPU_EINVAL;
  }
  const size_t n = static_cast<size_t>(n_blocks) * e->N;
  const size_t needAudio = static_cast<size_t>((static_cast<double>(n) * 16777216.0) / e->k.aud_step) + 2;
  if (audio && audio_cap < needAudio) {
    e->lastError = "process: audio capacity too small";
    return FMGPU_ERANGE;
  }
  return FMGPU_OK;
}

// Queue n_blocks logical blocks of every channel. hostIq != nullptr: the bytes come from host
// memory through the H2D stage (block by block into the device ring); else iq_dev is read in place.
int queueBlocks(fmgpu_engine *e, const uint8_t *iq_dev, const uint8_t *iq_host, size_t stride,
                int n_blocks, const BatchOut &out, cudaStream_t caller, bool callerWaits,
                const float2 *xcf = nullptr, size_t xcfStride = 0) {
  using E = fmgpu_engine;
  const size_t blockBytes = static_cast<size_t>(e->N) * e->M * 2;
  const int G = std::max(1, e->nGroups);
  if (!iq_host) {
    cudaEventRecord(e->evStart, caller);  // the IQ (and the output buffers) are ready in stream order
  }
  for (int g = 0; g < G; g++) {
    E::Pipe &P = e->pipes[g];
    int ch0, nch;
    groupRange(e, g, &ch0, &nch);
    if (nch <= 0) {
      continue;
    }
    if (!iq_host) {
      cudaStreamWaitEvent(P.run[(e->M > 1 && !xcf) ? E::ST_DECIM : E::ST_DC], e->evStart, 0);
    }
  }
  for (int b = 0; b < n_blocks; b++) {
    const uint64_t q = e->seq + static_cast<uint64_t>(b);
    const int slot = static_cast<int>(q % static_cast<uint64_t>(e->K));
    for (int g = 0; g < G; g++) {
      E::Pipe &P = e->pipes[g];
      int ch0, nch;
      groupRange(e, g, &ch0, &nch);
      if (nch <= 0) {
        continue;
      }
      e->curGroup = g;
      const uint8_t *iq = nullptr;
      size_t st = stride;
      if (iq_host) {
        // H2D stage: this block's rows into ring slot `slot` of the device staging buffer, once
        // the first compute stage has finished with block q - K
        cudaStream_t s = P.run[E::ST_H2D];
        if (q >= static_cast<uint64_t>(e->K)) {
          cudaStreamWaitEvent(
              s, P.done[e->M > 1 ? E::ST_DECIM : E::ST_DC][(q - e->K) % static_cast<uint64_t>(e->ER)], 0);
        }
        uint8_t *dst = e->dIq + static_cast<size_t>(ch0) * e->iqPitch + slot * blockBytes;
        cudaMemcpy2DAsync(dst, e->iqPitch, iq_host + static_cast<size_t>(ch0) * stride + b * blockBytes,
                          stride, blockBytes, static_cast<size_t>(nch), cudaMemcpyHostToDevice, s);
        cudaEventRecord(P.done[E::ST_H2D][q % static_cast<uint64_t>(e->ER)], s);
        iq = e->dIq + slot * blockBytes;
        st = e->iqPitch;
      } else if (iq_dev) {
        iq = iq_dev + b * blockBytes;
      }
      launchBlock(e, P, ch0, nch, q, b, n_blocks, iq, st, iq_host != nullptr, out,
                  xcf ? xcf + static_cast<size_t>(b) * e->N : nullptr, xcfStride);
    }
    if (slot == 0) {
      e->headFresh = false;
    }
  }
  for (int g = 0; g < G; g++) {
    E::Pipe &P = e->pipes[g];
    int ch0, nch;
    groupRange(e, g, &ch0, &nch);
    if (nch <= 0) {
      continue;
    }
    cudaEventRecord(P.callDone, P.run[E::ST_AF]);
    if (callerWaits) {
      cudaStreamWaitEvent(caller, P.callDone, 0);
    }
  }
  e->lastSeq0 = e->seq;
  e->lastBlocks = n_blocks;
  e->seq += static_cast<uint64_t>(n_blocks);
  e->asyncPending = true;
  e->lastN = n_blocks * e->N;
  const cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) {
    e->lastError = std::string("kernel launch: ") + cudaGetErrorString(err);
    return FMGPU_ENODEV;
  }
  return FMGPU_OK;
}

// iq_dev: IQ bytes, or (cf32) complex floats at the DSP rate; stride in bytes either way
int runBatch(fmgpu_engine *e, const uint8_t *iq_dev, size_t stride, int n_blocks, float *audio_dev,
             size_t audio_cap, uint32_t *n_audio_dev, fmgpu_rds_group *groups_dev, size_t group_cap,
             uint32_t *n_groups_dev, fmgpu_block_status *status_dev, cudaStream_t s,
             bool join = true, bool cf32 = false) {
  int rc = checkBatchArgs(e, iq_dev, stride, n_blocks, true, audio_dev, audio_cap);
  if (rc != FMGPU_OK) {
    return rc;
  }
  rc = uploadParams(e);
  if (rc != FMGPU_OK) {
    return rc;
  }
  const BatchOut own = engineOut(e);
  BatchOut out;
  out.status = status_dev ? status_dev : own.status;
  out.groups = groups_dev ? groups_dev : own.groups;
  out.gcap = groups_dev ? static_cast<uint32_t>(group_cap) : own.gcap;
  out.nAudio = n_audio_dev ? n_audio_dev : own.nAudio;
  out.nGroups = n_groups_dev ? n_groups_dev : own.nGroups;
  // audio is produced straight into the caller's buffer when one is given
  out.audio = audio_dev ? audio_dev : own.audio;
  out.acap = audio_dev ? audio_cap : own.acap;
  if (cf32) {
    return queueBlocks(e, nullptr, nullptr, 0, n_blocks, out, s, join, reinterpret_cast<const float2 *>(iq_dev),
                       stride / sizeof(float2));
  }
  return queueBlocks(e, iq_dev, nullptr, stride, n_blocks, out, s, join);
}

// All design-time work of the reference constructors; touches no CUDA state.
int computeDesigns(fmgpu_engine *e) {
  try {
    EngineConst &k = e->k;
    k.C = e->C;
    k.N = e->N;
    k.M = e->M;
    k.fs = e->fs;
    k.fsf = static_cast<float>(e->fs);
    const int rate = e->fs;
    const int outRate = e->cfg.output_rate;
    // --- ComplexDecimator::init (liquid_primitives.cpp:370-403, main.cpp:670-674)
    if (e->M > 1) {
      const uint32_t f = static_cast<uint32_t>(e->M);
      const uint32_t tppArg = e->cfg.decim_taps_per_phase > 0
                                  ? static_cast<uint32_t>(e->cfg.decim_taps_per_phase)
                                  : ((f >= 8U) ? 28U : ((f >= 4U) ? 20U : 12U));
      const uint32_t tpp = std::max<uint32_t>(4, tppArg);
      const float atten = e->cfg.decim_atten_db > 0 ? static_cast<float>(e->cfg.decim_atten_db) : 80.0f;
      const float cutoff = std::clamp(0.45f / static_cast<float>(f), 0.01f, 0.45f);
      e->decTaps = fmdesign::kaiserLowpass(f * tpp, cutoff, atten, 0.0f);
      e->decL = static_cast<int>(f * tpp);
      e->decPp = static_cast<int>(roundUp(tpp, 4));
      e->decScale = 2.0f * cutoff;
      if (e->decPp * e->M - 1 > H_IQ || e->decPp * e->M > MAX_TAPS) {
        e->lastError = "decimator too long for the IQ history";
        return FMGPU_EINVAL;
      }
      const std::vector<float> hrev = reversed(e->decTaps);
      e->decParam = padFront(hrev, e->decPp * e->M);
      e->decParamRaw = padFront(hrev, e->decL);
      k.dec_lp = e->decPp * e->M;
      k.dec_scale = e->decScale;
    }
    // --- StereoDecoder ctor (stereo_decoder.cpp:25-63)
    int pilotTapCount = static_cast<int>(std::ceil(3.8 * static_cast<double>(rate) / 3000.0));
    pilotTapCount = std::clamp(pilotTapCount, 63, 511);
    if ((pilotTapCount % 2) == 0) {
      pilotTapCount++;
    }
    const float pilotCenterNorm = std::clamp(19000.0f / static_cast<float>(rate), 0.001f, 0.49f);
    const float pilotCutoffNorm = std::clamp(250.0f / static_cast<float>(rate), 0.0005f, 0.45f);
    e->pilTaps = fmdesign::shiftedBandpass(static_cast<unsigned>(pilotTapCount), pilotCutoffNorm,
                                           60.0f, pilotCenterNorm);
    e->pilL = pilotTapCount;
    e->pilLp = static_cast<int>(roundUp(pilotTapCount, 8));
    e->pilParam = padFront(reversed(e->pilTaps), e->pilLp);
    const float audioCutoffNorm = std::clamp(15000.0f / static_cast<float>(rate), 0.01f, 0.45f);
    e->audTaps = fmdesign::kaiserLowpass(121, audioCutoffNorm, 60.0f, 0.0f);
    e->audL = 121;
    e->audLp = 128;
    e->audParam = padFront(reversed(e->audTaps), e->audLp);
    k.pil_lp = e->pilLp;
    k.aud_lp = e->audLp;
    k.aud_scale = 2.0f * audioCutoffNorm;
    k.delay = std::max(0, (pilotTapCount - 1) / 2) + 1;
    constexpr float kPi = 3.14159265358979323846f;
    k.nominal_pll = 2.0f * kPi * 19000.0f / static_cast<float>(rate);
    k.pll_min = 2.0f * kPi * 18750.0f / static_cast<float>(rate);
    k.pll_max = 2.0f * kPi * 19250.0f / static_cast<float>(rate);
    k.pll_alpha = 0.01f;
    k.pll_beta = std::sqrt(0.01f);
    k.pll_dtheta0 = fmdesign::ncoConstrain(k.nominal_pll);
    const float attack[3] = {0.090f, 0.120f, 0.180f};
    const float release[3] = {0.040f, 0.030f, 0.015f};
    const float gate[3] = {0.75f, 0.85f, 0.95f};
    for (int m = 0; m < 3; m++) {
      k.blend_attack[m] = 1.0f - std::exp(-1.0f / (attack[m] * static_cast<float>(rate)));
      k.blend_release[m] = 1.0f - std::exp(-1.0f / (release[m] * static_cast<float>(rate)));
      k.gate[m] = gate[m];
    }
    // --- resamplers (af_post_processor.cpp:7-18, fm_demod.cpp:40-42)
    const float ratio = static_cast<float>(outRate) / static_cast<float>(rate);
    if (ratio < 0.005f || ratio > 8.0f) {
      e->lastError = "resampler ratio is out of supported range";
      return FMGPU_EINVAL;
    }
    e->audRs = fmdesign::resampler(ratio, 12, 0.47f, 60.0f, 32);
    k.aud_step = e->audRs.step;
    k.mono_dc_a1 = -1.0f + 0.0008f;
    k.dc_a1_iq = -1.0f + 0.0005f;
    k.dc_a1_af = -1.0f + 0.005f;
    // --- freqdem (fm_demod.cpp:64-71)
    const float kf = static_cast<float>(75000.0 / static_cast<double>(rate));
    k.fd_ref = static_cast<float>(1.0 / (2.0 * M_PI * static_cast<double>(kf)));
    // --- RDS (subcarrier.cpp:37-45,94-106)
    const float kTarget = 171000.f;
    const float rdsRatio = kTarget / static_cast<float>(rate);
    if (rdsRatio < 0.005f || rdsRatio > 2.0f) {
      e->lastError = "RDS: can't support this sample rate";
      return FMGPU_EINVAL;
    }
    e->rdsRs = fmdesign::resampler(1.f, 13, 0.47f, 60.0f, 32);
    e->rdsRs.step = fmdesign::resamplerStep(rdsRatio);
    k.rds_step = e->rdsRs.step;
    const float lpfFc = 2400.0f / kTarget;
    e->rdsLpf = fmdesign::kaiserLowpass(255, lpfFc, 60.0f, 0.0f);
    k.rds_lpf_scale = 2.0f * lpfFc;
    k.rds_agc_alpha = 500.0f / kTarget;
    e->ss = fmdesign::symsyncRrc(3, 3, 0.8f, 32, 2200.0f / kTarget);
    k.ss_b0 = e->ss.sosB0;
    k.ss_a1 = e->ss.sosA1;
    k.ss_rate_adj = e->ss.rateAdjustment;
    k.rds_dtheta0 = fmdesign::ncoConstrain(57000.f * (2.f * kPi) / kTarget);
    k.rds_pll_alpha = 0.03f / kTarget;
    k.rds_pll_beta = std::sqrt(k.rds_pll_alpha);
    if (e->rdsRs.subLen != RDS_RS_LEN || e->audRs.subLen != AUD_RS_LEN || e->ss.subLen != SS_LEN) {
      e->lastError = "internal: unexpected polyphase sub-filter length";
      return FMGPU_EINVAL;
    }
  } catch (const std::exception &ex) {
    e->lastError = ex.what();
    return FMGPU_EINVAL;
  }

  return FMGPU_OK;
}

}  // namespace

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

int fmgpu_engine_create(const fmgpu_config *cfg, int n_channels, int device, fmgpu_engine **out) {
  if (!cfg || !out || n_channels < 1 || cfg->iq_rate < 1 || cfg->decimation < 1 ||
      cfg->block_samples < 1 || cfg->max_blocks < 1) {
    g_create_error = "fmgpu_engine_create: invalid arguments";
    return FMGPU_EINVAL;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
    g_create_error = "fmgpu_engine_create: no CUDA device (the engine has no CPU fallback)";
    cudaGetLastError();
    return FMGPU_ENODEV;
  }
  fmgpu_engine *e = new (std::nothrow) fmgpu_engine();
  if (!e) {
    return FMGPU_ENOMEM;
  }
  auto fail = [&](int rc) {
    g_create_error = e->lastError;
    fmgpu_engine_destroy(e);
    return rc;
  };
#define CKC(expr)                                                                  \
  do {                                                                             \
    cudaError_t err__ = (expr);                                                    \
    if (err__ != cudaSuccess) {                                                    \
      cudaGetLastError();                                                          \
      e->lastError = std::string(#expr) + ": " + cudaGetErrorString(err__);        \
      return fail(err__ == cudaErrorMemoryAllocation ? FMGPU_ENOMEM : FMGPU_ENODEV); \
    }                                                                              \
  } while (0)

  e->cfg = *cfg;
  if (e->cfg.output_rate <= 0) {
    e->cfg.output_rate = 32000;
  }
  e->C = n_channels;
  e->device = device;
  e->M = cfg->decimation;
  e->fs = cfg->iq_rate / cfg->decimation;
  e->N = cfg->block_samples;
  e->maxBlocks = cfg->max_blocks;
  e->nmax = static_cast<size_t>(e->N) * e->maxBlocks;
  // ring of K block slots per scratch buffer (see fmgpu_engine::Pipe); slots must start on
  // 16-byte boundaries for the cp.async tile loads, else every block goes through slot 0
  // K >= 3: a producer waits for the readers of block q - K + 1 (their halo is the tail of the slot
  // it overwrites), so three slots are what lets neighbouring stages of successive blocks overlap
  e->K = (e->N % 32 == 0) ? std::max(3, e->maxBlocks) : 1;
  if (e->K == 1 && e->maxBlocks > 1) {
    e->lastError = "fmgpu_engine_create: max_blocks > 1 needs block_samples to be a multiple of 32";
    g_create_error = e->lastError;
    delete e;
    return FMGPU_EINVAL;
  }
  e->ER = e->K + 1;
  e->pitch = roundUp(static_cast<size_t>(e->K) * e->N, 32);
  e->x2Pitch = H_X2 + e->pitch;
  e->yPitch = 32 + e->pitch;
  e->mpxPitch = H_MPX + e->pitch;
  e->lrPitch = H_LR + e->pitch;
  e->lfPitch = H_LF + e->pitch;
  e->iqPitch = roundUp(static_cast<size_t>(e->K) * e->N * e->M * 2, 16);
  CKC(cudaSetDevice(device));

  {
    const int drc = computeDesigns(e);
    if (drc != FMGPU_OK) {
      return fail(drc);
    }
  }

  const size_t C = static_cast<size_t>(e->C);
  e->acap = static_cast<size_t>((static_cast<double>(e->nmax) * 16777216.0) / e->k.aud_step) + 8;
  e->gcap = e->nmax * 12 / static_cast<size_t>(std::max(1, e->fs)) + 8;  // 11.4 groups/s
  e->bitsCap = e->nmax / 100 + 64;
  CKC(cudaStreamCreateWithFlags(e->stream.out(), cudaStreamNonBlocking));
  int prLo = 0, prHi = 0;
  CKC(cudaDeviceGetStreamPriorityRange(&prLo, &prHi));  // prHi = numerically smallest = highest
  CKC(cudaEventCreateWithFlags(e->evStart.out(), cudaEventDisableTiming));
  for (auto &P : e->pipes) {
    for (int st = 0; st < fmgpu_engine::ST_COUNT; st++) {
      // The serial one-lane-per-channel stages are the slowest per block: they get the high
      // priority, so their few CTAs are scheduled ahead of the thousands of queued FIR CTAs.
      // (Grading the FIR stages downstream-first as well was measured 3 % slower.)
      const bool lane = st == fmgpu_engine::ST_DC || st == fmgpu_engine::ST_AGC ||
                        st == fmgpu_engine::ST_STEREO || st == fmgpu_engine::ST_RDS ||
                        st == fmgpu_engine::ST_AF;
      const int prio = lane ? prHi : prLo;
      CKC(cudaStreamCreateWithPriority(P.st[st].out(), cudaStreamNonBlocking, prio));
      P.run[st] = P.st[st];
      P.done[st].resize(static_cast<size_t>(e->ER));
      for (auto &ev : P.done[st]) {
        CKC(cudaEventCreateWithFlags(ev.out(), cudaEventDisableTiming));
      }
    }
    CKC(cudaEventCreateWithFlags(P.callDone.out(), cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(P.hostDone[0].out(), cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(P.hostDone[1].out(), cudaEventDisableTiming));
  }
  CKC(initRdsTables());
  CKC(devAlloc(&e->dIq, C * e->iqPitch));
  CKC(devAlloc(&e->dHistIq, C * 2 * H_IQ));
  CKC(devAlloc(&e->dHistValid, C));
  {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) {
      e->smCount = sms;
    }
    e->k.sm_rot = e->smCount;
    if (e->M > 1 && decimTcSupported(e->M, e->decL, e->N)) {
      std::vector<uint8_t> bimg;
      std::vector<int32_t> offs;
      decimTcBuildTables(e->M, reversed(e->decTaps), &bimg, &offs);
      CKC(devAlloc(&e->dDecB, bimg.size()));
      CKC(devAlloc(&e->dDecOffs, offs.size()));
      CKC(cudaMemcpy(e->dDecB, bimg.data(), bimg.size(), cudaMemcpyHostToDevice));
      CKC(cudaMemcpy(e->dDecOffs, offs.data(), offs.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
      e->decimTcOk = true;
    }
    if (firTcSupported(e->pilParam.h, e->pilLp, H_MPX)) {
      firTcBuildTables(e->pilParam.h, e->pilLp, &e->pilTc);
      CKC(devAlloc(&e->dPilB, e->pilTc.b_image.size()));
      CKC(cudaMemcpy(e->dPilB, e->pilTc.b_image.data(), e->pilTc.b_image.size(), cudaMemcpyHostToDevice));
      e->pilTcOk = true;
    }
    if (firTcSupported(e->audParam.h, e->audLp, H_LR)) {
      firTcBuildTables(e->audParam.h, e->audLp, &e->audTc);
      CKC(devAlloc(&e->dAudB, e->audTc.b_image.size()));
      CKC(cudaMemcpy(e->dAudB, e->audTc.b_image.data(), e->audTc.b_image.size(), cudaMemcpyHostToDevice));
      e->audTcOk = true;
    }
    if (const char *fm = getenv("FMGPU_FIR_MODE")) {
      e->firMode = (atoi(fm) == 1 && e->pilTcOk && e->audTcOk) ? 1 : 0;
    }
    if (const char *xm = getenv("FMGPU_DEMOD_MODE")) {
      e->demodMode = (atoi(xm) == 1) ? 1 : 0;
    }
    if (const char *dm = getenv("FMGPU_DECIM_MODE")) {
      e->decimMode = (atoi(dm) == 1 && e->decimTcOk) ? 1 : 0;
    }
    if (const char *im = getenv("FMGPU_SCAN_MODE")) {
      e->scanMode = (atoi(im) == 1) ? 1 : 0;
    }
  }
  CKC(devAlloc(&e->dX1, C * e->pitch));
  CKC(devAlloc(&e->dX2, C * e->x2Pitch));
  CKC(devAlloc(&e->dY, C * e->yPitch));
  CKC(devAlloc(&e->dMpx, C * e->mpxPitch));
  CKC(devAlloc(&e->dPilot, C * e->pitch));
  CKC(devAlloc(&e->dLraw, C * e->lrPitch));
  CKC(devAlloc(&e->dRraw, C * e->lrPitch));
  CKC(devAlloc(&e->dLf, C * e->lfPitch));
  CKC(devAlloc(&e->dRf, C * e->lfPitch));
  e->r171Pitch = roundUp(static_cast<size_t>(max171(e, static_cast<int>(e->nmax))) + 32, 32);
  CKC(devAlloc(&e->dR171, 2 * C * e->r171Pitch));
  CKC(devAlloc(&e->dRdsRs, C));
  CKC(devAlloc(&e->dRing, C * RDS_RING));
  CKC(devAlloc(&e->dRdsHist, C * 32));
  CKC(devAlloc(&e->dMonoHist, C * 32));
  CKC(devAlloc(&e->dChanTaps, static_cast<size_t>(MAX_CHAN_FILTERS) * CHAN_TAPS_PITCH));
  CKC(devAlloc(&e->dChanScale, MAX_CHAN_FILTERS));
  CKC(devAlloc(&e->dChanLp, MAX_CHAN_FILTERS));
  CKC(devAlloc(&e->dAudBank, e->audRs.bank.size()));
  CKC(devAlloc(&e->dRdsBank, e->rdsRs.bank.size()));
  CKC(devAlloc(&e->dRdsLpf, 256));
  CKC(devAlloc(&e->dMf, e->ss.mf.size()));
  CKC(devAlloc(&e->dDmf, e->ss.dmf.size()));
  CKC(devAlloc(&e->dParams, C));
  CKC(devAlloc(&e->dDemod, C));
  CKC(devAlloc(&e->dStereo, C));
  CKC(devAlloc(&e->dAudioSt, C));
  CKC(devAlloc(&e->dRds, C));
  for (auto &r : e->res) {
    CKC(devAlloc(&r.audio, C * 2 * e->acap));
    CKC(devAlloc(&r.groups, C * e->gcap));
    CKC(devAlloc(&r.status, C * static_cast<size_t>(e->maxBlocks)));
    CKC(devAlloc(&r.nAudio, C));
    CKC(devAlloc(&r.nGroups, C));
  }
  CKC(devAlloc(&e->dBits, C * e->bitsCap));
  CKC(devAlloc(&e->dWords, C * e->bitsCap));
  CKC(cudaMemcpy(e->dAudBank, e->audRs.bank.data(), e->audRs.bank.size() * sizeof(float),
                 cudaMemcpyHostToDevice));
  CKC(cudaMemcpy(e->dRdsBank, e->rdsRs.bank.data(), e->rdsRs.bank.size() * sizeof(float),
                 cudaMemcpyHostToDevice));
  {
    const std::vector<float> hrev = reversed(e->rdsLpf);
    CKC(cudaMemcpy(e->dRdsLpf, hrev.data(), hrev.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  CKC(cudaMemcpy(e->dMf, e->ss.mf.data(), e->ss.mf.size() * sizeof(float), cudaMemcpyHostToDevice));
  CKC(cudaMemcpy(e->dDmf, e->ss.dmf.data(), e->ss.dmf.size() * sizeof(float),
                 cudaMemcpyHostToDevice));

  // per-channel defaults: FMDemod ctor filter (fm_demod.cpp:36-37), then the calls main.cpp makes
  const float ctorCut = std::clamp(110000.0f / static_cast<float>(e->fs), 0.01f, 0.45f);
  const int slot0 = filterSlot(e, 81, ctorCut, 60.0f);
  if (slot0 < 0) {
    return fail(slot0);
  }
  ChanParams p{};
  p.filt = slot0;
  p.bandwidth_mode = 0;
  p.w0_hz = 194000;
  p.blend_mode = 1;
  e->hParams.assign(C, p);
  {
    std::vector<DemodState> d(C, defaultDemod());
    std::vector<StereoState> st(C, defaultStereo(e->k));
    std::vector<RdsState> r(C, defaultRds(e->k));
    CKC(cudaMemcpy(e->dDemod, d.data(), C * sizeof(DemodState), cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(e->dStereo, st.data(), C * sizeof(StereoState), cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(e->dRds, r.data(), C * sizeof(RdsState), cudaMemcpyHostToDevice));
  }
  *out = e;
  // constructor defaults of the reference objects, then main.cpp:641-710
  fmgpu_set_deemphasis_us(e, -1, 75);
  fmgpu_set_w0_bandwidth_hz(e, -1, cfg->w0_bandwidth_hz);
  fmgpu_set_agc_mode(e, -1, cfg->dsp_agc);
  fmgpu_set_blend_mode(e, -1, cfg->stereo_blend);
  fmgpu_set_deemphasis_us(e, -1, cfg->deemphasis == 0 ? 50 : (cfg->deemphasis == 1 ? 75 : 0));
  fmgpu_set_force_mono(e, -1, cfg->force_mono);
  fmgpu_set_bandwidth_hz(e, -1, cfg->bandwidth_hz);
  const int rc = uploadParams(e);
  if (rc != FMGPU_OK) {
    *out = nullptr;
    return fail(rc);
  }
  return FMGPU_OK;
#undef CKC
}

void fmgpu_engine_destroy(fmgpu_engine *e) {
  if (!e) {
    return;
  }
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  delete e;  // the handles free every buffer, stream and event
}

const char *fmgpu_last_error(const fmgpu_engine *e) {
  return e ? e->lastError.c_str() : g_create_error.c_str();
}
int fmgpu_n_channels(const fmgpu_engine *e) { return e ? e->C : 0; }
int fmgpu_dsp_rate(const fmgpu_engine *e) { return e ? e->fs : 0; }

// ---- settings --------------------------------------------------------------
int fmgpu_set_w0_bandwidth_hz(fmgpu_engine *e, int channel, int bw_hz) {
  if (!e) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  return forChannels(e, channel, [&](int c) {
    e->hParams[c].w0_hz = std::clamp(bw_hz, 0, 400000);
    return FMGPU_OK;
  });
}

int fmgpu_set_bandwidth_hz(fmgpu_engine *e, int channel, int bw_hz) {
  if (!e || channel < -1 || channel >= e->C) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  const int lo = (channel < 0) ? 0 : channel;
  const int hi = (channel < 0) ? e->C : channel + 1;
  std::vector<int> changed;
  for (int c = lo; c < hi; c++) {
    ChanParams &p = e->hParams[c];
    const fmdesign::ChannelFilterSpec spec = fmdesign::channelFilterSpec(bw_hz, p.w0_hz, e->fs);
    if (spec.index == p.bandwidth_mode) {
      continue;  // fm_demod.cpp:114-116
    }
    const int slot = filterSlot(e, spec.length, spec.cutoff, spec.atten);
    if (slot < 0) {
      return slot;
    }
    p.bandwidth_mode = spec.index;
    p.filt = slot;
    changed.push_back(c);
  }
  if (changed.empty()) {
    return FMGPU_OK;
  }
  e->paramsDirty = true;
  // the FIR is re-created with an empty window (fm_demod.cpp:134); r_prev is kept
  realign(e);  // queued blocks finish; the window (halo) sits in front of ring slot 0
  for (size_t i = 0; i < changed.size();) {  // one memset per run of neighbouring channels
    size_t j = i + 1;
    while (j < changed.size() && changed[j] == changed[j - 1] + 1) {
      j++;
    }
    zeroPrefix(e->dX2, e->x2Pitch, H_X2, changed[i], changed[j - 1] + 1, e->stream);
    i = j;
  }
  CK(cudaStreamSynchronize(e->stream));
  return FMGPU_OK;
}

int fmgpu_set_bandwidth_mode(fmgpu_engine *e, int channel, int mode) {
  return fmgpu_set_bandwidth_hz(e, channel, fmdesign::tefBandwidthHz(mode));
}

int fmgpu_set_agc_mode(fmgpu_engine *e, int channel, int mode) {
  if (!e || mode < 0 || mode > 2 || channel < -1 || channel >= e->C) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  const int lo = (channel < 0) ? 0 : channel;
  const int hi = (channel < 0) ? e->C : channel + 1;
  for (int c = lo; c < hi; c++) {
    ChanParams &p = e->hParams[c];
    p.agc_mode = mode;
    if (mode != 0) {
      p.agc_alpha = (mode == 1) ? 0.01f : 0.001f;
    }
  }
  e->paramsDirty = true;
  if (mode != 0) {
    // AGC::init re-creates the object: gain 1, energy 1 (fm_demod.cpp:146-147). Blocks already
    // queued finish first: an in-flight k_agc would write its own gain back over the reset.
    syncPipes(e);
    static_assert(offsetof(DemodState, agc_y2) == offsetof(DemodState, agc_g) + sizeof(float),
                  "agc_g and agc_y2 are written as one pair");
    const float init[2] = {1.0f, 1.0f};
    return fillStateField(e, e->dDemod, offsetof(DemodState, agc_g), init, sizeof(init), lo, hi);
  }
  return FMGPU_OK;
}

int fmgpu_set_deemphasis_us(fmgpu_engine *e, int channel, int tau_us) {
  if (!e || channel < -1 || channel >= e->C) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  const int lo = (channel < 0) ? 0 : channel;
  const int hi = (channel < 0) ? e->C : channel + 1;
  for (int c = lo; c < hi; c++) {
    ChanParams &p = e->hParams[c];
    deemphCoeffs(tau_us, e->cfg.output_rate, &p.deemph_on, &p.de_b0, &p.de_a1);
    deemphCoeffs(tau_us, e->cfg.output_rate, &p.mono_deemph_on, &p.mono_de_b0, &p.mono_de_a1);
  }
  e->paramsDirty = true;
  if (tau_us > 0) {
    // IIRFilterReal::init creates fresh filters: state cleared — once the queued blocks, whose
    // k_audio_iir writes the state back, have finished
    syncPipes(e);
    const float z[2] = {0.0f, 0.0f};
    int rc = fillStateField(e, e->dAudioSt, offsetof(AudioState, de_v1), z, sizeof(z), lo, hi);
    if (rc == FMGPU_OK) {
      rc = fillStateField(e, e->dAudioSt, offsetof(AudioState, mono_de_v1), z, sizeof(float), lo, hi);
    }
    return rc;
  }
  return FMGPU_OK;
}

int fmgpu_set_deviation_hz(fmgpu_engine *e, double deviation_hz) {
  if (!e || !(deviation_hz > 0.0)) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  // freqdem is re-created: new reference gain, r_prev cleared (fm_demod.cpp:64-71)
  const float kf = static_cast<float>(deviation_hz / static_cast<double>(e->fs));
  e->k.fd_ref = static_cast<float>(1.0 / (2.0 * M_PI * static_cast<double>(kf)));
  realign(e);
  zeroPrefix(e->dY, e->yPitch, Y_OFF, 0, e->C, e->stream);
  CK(cudaStreamSynchronize(e->stream));
  return FMGPU_OK;
}

int fmgpu_set_decimator_mode(fmgpu_engine *e, int mode) {
  if (!e || mode < 0 || mode > 1) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  if (mode == 1 && !e->decimTcOk) {
    e->lastError = "tensor-core decimator: this decimation factor / tap count is not supported";
    return FMGPU_EINVAL;
  }
  syncPipes(e);
  e->decimMode = mode;
  return FMGPU_OK;
}

int fmgpu_get_decimator_mode(const fmgpu_engine *e) { return e ? e->decimMode : FMGPU_EINVAL; }

int fmgpu_set_scan_mode(fmgpu_engine *e, int mode) {
  if (!e || mode < 0 || mode > 1) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  syncPipes(e);
  e->scanMode = mode;
  return FMGPU_OK;
}

int fmgpu_get_scan_mode(const fmgpu_engine *e) { return e ? e->scanMode : FMGPU_EINVAL; }

int fmgpu_set_fir_mode(fmgpu_engine *e, int mode) {
  if (!e || mode < 0 || mode > 1) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  if (mode == 1 && !(e->pilTcOk && e->audTcOk)) {
    e->lastError = "tensor-core FIRs: this pilot / audio filter length is not supported";
    return FMGPU_EINVAL;
  }
  syncPipes(e);
  e->firMode = mode;
  return FMGPU_OK;
}

int fmgpu_get_fir_mode(const fmgpu_engine *e) { return e ? e->firMode : FMGPU_EINVAL; }

int fmgpu_set_demod_mode(fmgpu_engine *e, int mode) {
  if (!e || mode < 0 || mode > 1) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  syncPipes(e);
  e->demodMode = mode;
  return FMGPU_OK;
}

int fmgpu_get_demod_mode(const fmgpu_engine *e) { return e ? e->demodMode : FMGPU_EINVAL; }

int fmgpu_set_blend_mode(fmgpu_engine *e, int channel, int mode) {
  if (!e || mode < 0 || mode > 2) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  return forChannels(e, channel, [&](int c) {
    e->hParams[c].blend_mode = mode;
    e->paramsDirty = true;
    return FMGPU_OK;
  });
}

int fmgpu_set_force_mono(fmgpu_engine *e, int channel, int on) {
  if (!e) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  return forChannels(e, channel, [&](int c) {
    e->hParams[c].force_mono = on ? 1 : 0;
    e->paramsDirty = true;
    return FMGPU_OK;
  });
}

int fmgpu_set_force_stereo(fmgpu_engine *e, int channel, int on) {
  if (!e) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  return forChannels(e, channel, [&](int c) {
    e->hParams[c].force_stereo = on ? 1 : 0;
    e->paramsDirty = true;
    return FMGPU_OK;
  });
}

int fmgpu_reset(fmgpu_engine *e, int channel, unsigned what) {
  if (!e || channel < -1 || channel >= e->C) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  const int lo = (channel < 0) ? 0 : channel;
  const int hi = (channel < 0) ? e->C : channel + 1;
  const size_t cnt = static_cast<size_t>(hi - lo);
  cudaStream_t s = e->stream;
  realign(e);  // queued blocks finish; every halo sits in front of slot 0 again
  CK(cudaStreamSynchronize(s));
  if (what & FMGPU_RESET_DECIM) {
    if (e->M > 1) {
      CK(cudaMemsetAsync(e->dHistIq + static_cast<size_t>(lo) * 2 * H_IQ, 0, cnt * 2 * H_IQ, s));
      CK(cudaMemsetAsync(e->dHistValid + lo, 0, cnt * sizeof(int), s));
    }
  }
  if (what & FMGPU_RESET_DEMOD) {
    // fm_demod.cpp:73-88
    zeroPrefix(e->dX2, e->x2Pitch, H_X2, lo, hi, s);
    zeroPrefix(e->dY, e->yPitch, Y_OFF, lo, hi, s);
    zeroPrefix(e->dMonoHist, 32, 32, lo, hi, s);
    std::vector<DemodState> d(cnt, defaultDemod());
    CK(cudaMemcpyAsync(e->dDemod + lo, d.data(), cnt * sizeof(DemodState), cudaMemcpyHostToDevice, s));
    std::vector<AudioState> a(cnt);
    CK(cudaMemcpyAsync(a.data(), e->dAudioSt + lo, cnt * sizeof(AudioState), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    for (size_t i = 0; i < cnt; i++) {
      if (e->hParams[lo + i].mono_deemph_on) {
        a[i].mono_de_v1 = 0.0f;
      }
      a[i].mono_dc_v1 = 0.0f;
      a[i].mono_phase = 0;
      a[i].mono_phase_next = 0;
    }
    CK(cudaMemcpyAsync(e->dAudioSt + lo, a.data(), cnt * sizeof(AudioState), cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s));
  }
  if (what & FMGPU_RESET_STEREO) {
    // stereo_decoder.cpp:67-86
    zeroPrefix(e->dMpx, e->mpxPitch, H_MPX, lo, hi, s);
    zeroPrefix(e->dLraw, e->lrPitch, H_LR, lo, hi, s);
    zeroPrefix(e->dRraw, e->lrPitch, H_LR, lo, hi, s);
    std::vector<StereoState> st(cnt, defaultStereo(e->k));
    CK(cudaMemcpyAsync(e->dStereo + lo, st.data(), cnt * sizeof(StereoState), cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s));
  }
  if (what & FMGPU_RESET_AFPOST) {
    // af_post_processor.cpp:20-29
    zeroPrefix(e->dLf, e->lfPitch, H_LF, lo, hi, s);
    zeroPrefix(e->dRf, e->lfPitch, H_LF, lo, hi, s);
    std::vector<AudioState> a(cnt);
    CK(cudaMemcpyAsync(a.data(), e->dAudioSt + lo, cnt * sizeof(AudioState), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    for (size_t i = 0; i < cnt; i++) {
      a[i].rs_phase = 0;
      a[i].rs_phase_next = 0;
      a[i].dc_v1[0] = a[i].dc_v1[1] = 0.0f;
      if (e->hParams[lo + i].deemph_on) {
        a[i].de_v1[0] = a[i].de_v1[1] = 0.0f;
      }
    }
    CK(cudaMemcpyAsync(e->dAudioSt + lo, a.data(), cnt * sizeof(AudioState), cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s));
  }
  if (what & FMGPU_RESET_RDS) {
    std::vector<RdsState> r(cnt);
    CK(cudaMemcpyAsync(r.data(), e->dRds + lo, cnt * sizeof(RdsState), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    for (auto &st : r) {
      resetRdsLoops(st, e->k);
    }
    CK(cudaMemcpyAsync(e->dRds + lo, r.data(), cnt * sizeof(RdsState), cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s));
  }
  CK(cudaStreamSynchronize(s));
  return FMGPU_OK;
}

// ---- observables -------------------------------------------------------------
static int readStereo(fmgpu_engine *e, int channel, StereoState *out) {
  if (!e || channel < 0 || channel >= e->C) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  syncPipes(e);
  CK(cudaMemcpyAsync(out, e->dStereo + channel, sizeof(StereoState), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return FMGPU_OK;
}
static int readDemod(fmgpu_engine *e, int channel, DemodState *out) {
  if (!e || channel < 0 || channel >= e->C) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  syncPipes(e);
  CK(cudaMemcpyAsync(out, e->dDemod + channel, sizeof(DemodState), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return FMGPU_OK;
}
int fmgpu_is_stereo(fmgpu_engine *e, int channel) {
  StereoState s{};
  return readStereo(e, channel, &s) == FMGPU_OK ? s.stereo : 0;
}
int fmgpu_pilot_tenths(fmgpu_engine *e, int channel) {
  StereoState s{};
  return readStereo(e, channel, &s) == FMGPU_OK ? s.pilot_tenths : 0;
}
float fmgpu_clip_ratio(fmgpu_engine *e, int channel) {
  DemodState s{};
  return readDemod(e, channel, &s) == FMGPU_OK ? s.clip_ratio : 0.0f;
}
int fmgpu_is_clipping(fmgpu_engine *e, int channel) {
  DemodState s{};
  return readDemod(e, channel, &s) == FMGPU_OK ? s.clipping : 0;
}

// ---- batched paths -------------------------------------------------------------
int fmgpu_process_batch(fmgpu_engine *e, const uint8_t *iq_dev, size_t iq_stride_bytes,
                        int n_blocks, float *audio_dev, size_t audio_cap, uint32_t *n_audio_dev,
                        fmgpu_rds_group *groups_dev, size_t group_cap, uint32_t *n_groups_dev,
                        fmgpu_block_status *status_dev, void *stream) {
  if (!e) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);  // NULL = the legacy default stream
  const int rc = runBatch(e, iq_dev, iq_stride_bytes, n_blocks, audio_dev, audio_cap, n_audio_dev,
                          groups_dev, group_cap, n_groups_dev, status_dev, s);
  if (rc == FMGPU_OK && e->timing) {
    CK(cudaStreamSynchronize(s));
    collectTimes(e);
  }
  return rc;
}

int fmgpu_process_batch_async(fmgpu_engine *e, const uint8_t *iq_dev, size_t iq_stride_bytes,
                              int n_blocks, float *audio_dev, size_t audio_cap,
                              uint32_t *n_audio_dev, fmgpu_rds_group *groups_dev, size_t group_cap,
                              uint32_t *n_groups_dev, fmgpu_block_status *status_dev, void *stream) {
  if (!e) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  return runBatch(e, iq_dev, iq_stride_bytes, n_blocks, audio_dev, audio_cap, n_audio_dev, groups_dev,
                  group_cap, n_groups_dev, status_dev, static_cast<cudaStream_t>(stream), false);
}

int fmgpu_process_batch_cf32(fmgpu_engine *e, const float *x_cf32_dev, size_t stride_samples,
                             int n_blocks, float *audio_dev, size_t audio_cap,
                             uint32_t *n_audio_dev, fmgpu_rds_group *groups_dev, size_t group_cap,
                             uint32_t *n_groups_dev, fmgpu_block_status *status_dev, void *stream) {
  if (!e) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  if (e->M != 1) {
    e->lastError = "process_batch_cf32: the engine must be created with decimation = 1";
    return FMGPU_EINVAL;
  }
  if (!x_cf32_dev || n_blocks < 1 || n_blocks > e->maxBlocks ||
      (reinterpret_cast<uintptr_t>(x_cf32_dev) & 15u) || (stride_samples & 1u) ||
      stride_samples < static_cast<size_t>(n_blocks) * e->N) {
    e->lastError = "process_batch_cf32: bad input pointer, alignment, stride or block count";
    return FMGPU_EINVAL;
  }
  const int rc = runBatch(e, reinterpret_cast<const uint8_t *>(x_cf32_dev), stride_samples * sizeof(float2),
                          n_blocks, audio_dev, audio_cap, n_audio_dev, groups_dev, group_cap, n_groups_dev,
                          status_dev, static_cast<cudaStream_t>(stream), true, true);
  if (rc == FMGPU_OK && e->timing) {
    CK(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    collectTimes(e);
  }
  return rc;
}

int fmgpu_join(fmgpu_engine *e, void *stream) {
  if (!e) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  for (auto &P : e->pipes) {
    // callDone holds the last batch this pipe ran (an event never recorded is complete)
    CK(cudaStreamWaitEvent(s, P.callDone, 0));
  }
  return FMGPU_OK;
}

static int waitHostTicket(fmgpu_engine *e, int ticket) {
  fmgpu_engine::HostTicket &t = e->tickets[ticket];
  if (!t.pending) {
    return FMGPU_OK;
  }
  t.pending = false;
  for (auto &P : e->pipes) {
    CK(cudaEventSynchronize(P.hostDone[ticket]));
  }
  const cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) {
    e->lastError = std::string("process_host: ") + cudaGetErrorString(err);
    return FMGPU_ENODEV;
  }
  if (t.clampGroups) {
    for (int c = 0; c < e->C; c++) {
      t.nGroupsHost[c] = std::min<uint32_t>(t.nGroupsHost[c], static_cast<uint32_t>(t.groupCap));
    }
  }
  return FMGPU_OK;
}

int fmgpu_wait_host(fmgpu_engine *e, int ticket) {
  if (!e || ticket < 0 || ticket > 1) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  const int rc = waitHostTicket(e, ticket);
  if (rc == FMGPU_OK && !e->tickets[0].pending && !e->tickets[1].pending) {
    collectTimes(e);
  }
  return rc;
}

int fmgpu_process_host(fmgpu_engine *e, const uint8_t *iq_host, size_t iq_stride_bytes,
                       int n_blocks, float *audio_host, size_t audio_cap, uint32_t *n_audio_host,
                       fmgpu_rds_group *groups_host, size_t group_cap, uint32_t *n_groups_host,
                       fmgpu_block_status *status_host) {
  const int ticket = fmgpu_submit_host(e, iq_host, iq_stride_bytes, n_blocks, audio_host, audio_cap,
                                       n_audio_host, groups_host, group_cap, n_groups_host,
                                       status_host);
  if (ticket < 0) {
    return ticket;
  }
  return fmgpu_wait_host(e, ticket);
}

int fmgpu_submit_host(fmgpu_engine *e, const uint8_t *iq_host, size_t iq_stride_bytes,
                      int n_blocks, float *audio_host, size_t audio_cap, uint32_t *n_audio_host,
                      fmgpu_rds_group *groups_host, size_t group_cap, uint32_t *n_groups_host,
                      fmgpu_block_status *status_host) {
  if (!e) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  int rc = checkBatchArgs(e, iq_host, iq_stride_bytes, n_blocks, false, audio_host, audio_cap);
  if (rc != FMGPU_OK) {
    return rc;
  }
  rc = uploadParams(e);
  if (rc != FMGPU_OK) {
    return rc;
  }
  const size_t n = static_cast<size_t>(n_blocks) * e->N;
  const size_t frames = std::min(e->acap, static_cast<size_t>((static_cast<double>(n) * 16777216.0) /
                                                               e->k.aud_step) + 2);
  const int G = std::max(1, e->nGroups);
  const int ticket = e->nextTicket;
  rc = waitHostTicket(e, ticket);  // at most two submissions in flight
  if (rc != FMGPU_OK) {
    return rc;
  }
  e->nextTicket ^= 1;
  // H2D stage: block after block into the device ring, each block's kernels released by its own
  // copy; results go back on the D2H stage once the call's last block is done. With a second
  // submission queued behind, its copies overlap this call's kernels.
  // device-side result buffers alternate with the ticket, so the next submission's kernels never
  // wait for this one's device-to-host copies
  const BatchOut out = engineOut(e, ticket);
  rc = queueBlocks(e, nullptr, iq_host, iq_stride_bytes, n_blocks, out, nullptr, false);
  if (rc != FMGPU_OK) {
    return rc;
  }
  for (int g = 0; g < G; g++) {
    int ch0 = 0, nch = e->C;
    groupRange(e, g, &ch0, &nch);
    if (nch <= 0) {
      continue;
    }
    fmgpu_engine::Pipe &P = e->pipes[g];
    cudaStream_t s = P.run[fmgpu_engine::ST_D2H];
    CK(cudaStreamWaitEvent(s, P.callDone, 0));
    const size_t c0 = static_cast<size_t>(ch0), cn = static_cast<size_t>(nch);
    if (audio_host) {
      CK(cudaMemcpy2DAsync(audio_host + c0 * 2 * audio_cap, audio_cap * sizeof(float),
                           out.audio + c0 * 2 * e->acap, e->acap * sizeof(float), frames * sizeof(float),
                           cn * 2, cudaMemcpyDeviceToHost, s));
    }
    if (n_audio_host) {
      CK(cudaMemcpyAsync(n_audio_host + c0, out.nAudio + c0, cn * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    }
    if (groups_host) {
      const size_t gw = std::min(group_cap, e->gcap);
      CK(cudaMemcpy2DAsync(groups_host + c0 * group_cap, group_cap * sizeof(fmgpu_rds_group),
                           out.groups + c0 * e->gcap, e->gcap * sizeof(fmgpu_rds_group),
                           gw * sizeof(fmgpu_rds_group), cn, cudaMemcpyDeviceToHost, s));
    }
    if (n_groups_host) {
      CK(cudaMemcpyAsync(n_groups_host + c0, out.nGroups + c0, cn * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    }
    if (status_host) {
      // the status rows of this call are [C][n_blocks] (pitch = n_blocks)
      CK(cudaMemcpyAsync(status_host + c0 * n_blocks, out.status + c0 * n_blocks,
                         cn * n_blocks * sizeof(fmgpu_block_status), cudaMemcpyDeviceToHost, s));
    }
    CK(cudaEventRecord(P.hostDone[ticket], s));
  }
  const cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) {
    e->lastError = std::string("process_host: ") + cudaGetErrorString(err);
    return FMGPU_ENODEV;
  }
  fmgpu_engine::HostTicket &t = e->tickets[ticket];
  t.pending = true;
  t.nGroupsHost = n_groups_host;
  t.groupCap = group_cap;
  t.clampGroups = n_groups_host && groups_host;
  return ticket;
}

int fmgpu_signal_level_batch(fmgpu_engine *e, const uint8_t *iq_dev, size_t iq_stride_bytes,
                             int n_blocks, fmgpu_level_sums *sums_dev, void *stream) {
  if (!e || !iq_dev || !sums_dev || n_blocks < 1) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const long spb = static_cast<long>(e->N) * e->M;
  if (iq_stride_bytes < static_cast<size_t>(n_blocks) * spb * 2) {
    e->lastError = "signal_level: stride smaller than the bytes per channel";
    return FMGPU_EINVAL;
  }
  CK(cudaMemsetAsync(sums_dev, 0, static_cast<size_t>(e->C) * n_blocks * sizeof(fmgpu_level_sums), s));
  launchSigLevel(iq_dev, iq_stride_bytes, sums_dev, n_blocks, spb, 0, e->C, s);
  e->launches += 1;
  const cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) {
    e->lastError = std::string("signal_level: ") + cudaGetErrorString(err);
    return FMGPU_ENODEV;
  }
  return FMGPU_OK;
}

void fmgpu_signal_level_finish(const fmgpu_level_sums *su, int applied_gain_db,
                               double gain_comp_factor, double signal_bias_db, double floor_dbfs,
                               double ceil_dbfs, fmgpu_signal_level *out) {
  if (!su || !out) {
    return;
  }
  *out = fmgpu_signal_level{0.0f, -120.0, -120.0, 0.0, 0.0};
  if (su->n_samples == 0) {
    return;
  }
  // sum of (v - 127.5)/127.5 and of its square, from the exact integer sums
  const double n = static_cast<double>(su->n_samples);
  const double k = 1.0 / 127.5;
  const double sI = (static_cast<double>(su->sum_i) - 127.5 * n) * k;
  const double sQ = (static_cast<double>(su->sum_q) - 127.5 * n) * k;
  const double sII = (static_cast<double>(su->sum_ii) - 255.0 * static_cast<double>(su->sum_i) +
                      127.5 * 127.5 * n) * k * k;
  const double sQQ = (static_cast<double>(su->sum_qq) - 255.0 * static_cast<double>(su->sum_q) +
                      127.5 * 127.5 * n) * k * k;
  const double meanI = sI / n, meanQ = sQ / n;
  const double varI = std::max(0.0, (sII / n) - (meanI * meanI));
  const double varQ = std::max(0.0, (sQQ / n) - (meanQ * meanQ));
  const double rms = std::sqrt(std::max(1e-15, 0.5 * (varI + varQ)));
  out->dbfs = 20.0 * std::log10(rms + 1e-12);
  out->compensated_dbfs = out->dbfs - (static_cast<double>(applied_gain_db) * gain_comp_factor) +
                          signal_bias_db;
  const double safeCeil = std::max(ceil_dbfs, floor_dbfs + 1.0);
  const double norm = (out->compensated_dbfs - floor_dbfs) / (safeCeil - floor_dbfs);
  out->level120 = std::clamp(static_cast<float>(norm * 120.0), 0.0f, 120.0f);
  const double iqValues = 2.0 * n;
  out->hard_clip_ratio = (2.0 * static_cast<double>(su->hard_clip)) / iqValues;
  out->near_clip_ratio = (2.0 * static_cast<double>(su->near_clip)) / iqValues;
}

int fmgpu_pack_pcm16(fmgpu_engine *e, const float *audio_dev, size_t audio_cap,
                     const uint32_t *n_audio_dev, float volume_scale, int16_t *pcm_dev,
                     void *stream) {
  if (!e || !audio_dev || !n_audio_dev || !pcm_dev || audio_cap == 0) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  launchPackPcm16(audio_dev, audio_cap, n_audio_dev, volume_scale, pcm_dev, e->C,
                  static_cast<int>(std::min(audio_cap, e->acap)), static_cast<cudaStream_t>(stream));
  e->launches += 1;
  return cudaGetLastError() == cudaSuccess ? FMGPU_OK : FMGPU_ENODEV;
}

int fmgpu_set_stage_overlap(fmgpu_engine *e, int on) {
  if (!e) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  syncPipes(e);
  e->serialStages = (on == 0);
  for (auto &P : e->pipes) {
    for (int st = 0; st < fmgpu_engine::ST_COUNT; st++) {
      P.run[st] = e->serialStages ? P.st[fmgpu_engine::ST_DECIM] : P.st[st];
    }
  }
  return FMGPU_OK;
}

int fmgpu_set_pipeline_groups(fmgpu_engine *e, int groups) {
  if (!e || groups < 1 || groups > 16) {
    return FMGPU_EINVAL;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  CK(cudaSetDevice(e->device));
  syncPipes(e);
  // every group owns a full set of stage streams; more than two sets buy nothing (the block
  // pipeline already overlaps the stages) and would exceed the device's hardware queues
  e->nGroups = std::min(groups, fmgpu_engine::kMaxGroups);
  return FMGPU_OK;
}

// ---- stage-level entry points ------------------------------------------------------
#define STAGE_PROLOGUE(cond)                                                    \
  if (!e || channel < 0 || channel >= e->C || !(cond)) {                        \
    return 0;                                                                   \
  }                                                                             \
  std::lock_guard<std::recursive_mutex> lk(e->mu);                              \
  if (cudaSetDevice(e->device) != cudaSuccess || uploadParams(e) != FMGPU_OK) { \
    return 0;                                                                   \
  }                                                                             \
  realign(e); /* the stage-level calls work at ring offset 0, halos in place */ \
  cudaStream_t s = e->stream;

static bool stageFail(fmgpu_engine *e, const char *what) {
  const cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) {
    e->lastError = std::string(what) + ": " + cudaGetErrorString(err);
    return true;
  }
  return false;
}

size_t fmgpu_decimate(fmgpu_engine *e, int channel, const uint8_t *iq, size_t in_samples,
                      float *out_cf32, size_t out_capacity) {
  STAGE_PROLOGUE(iq && out_cf32 && in_samples > 0 && out_capacity > 0)
  const size_t n_out = std::min({in_samples / static_cast<size_t>(e->M), out_capacity});
  if (n_out == 0) {
    return 0;
  }
  if (n_out > e->nmax) {
    e->lastError = "decimate: more samples than the engine was sized for";
    return 0;
  }
  uint8_t *dst = e->dIq + static_cast<size_t>(channel) * e->iqPitch;
  cudaMemcpyAsync(dst, iq, n_out * e->M * 2, cudaMemcpyHostToDevice, s);
  stageDecimate(e, stageBlock(channel, static_cast<int>(n_out)), e->dIq, e->iqPitch, s);
  cudaMemcpyAsync(out_cf32, e->dX1 + static_cast<size_t>(channel) * e->pitch, n_out * sizeof(float2),
                  cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  e->lastN = static_cast<int>(n_out);
  return stageFail(e, "decimate") ? 0 : n_out;
}

size_t fmgpu_decimate_u8(fmgpu_engine *e, int channel, const uint8_t *iq, size_t in_samples,
                         uint8_t *out_u8, size_t out_capacity) {
  STAGE_PROLOGUE(iq && out_u8 && in_samples > 0 && out_capacity > 0)
  const size_t n_out = std::min({in_samples / static_cast<size_t>(e->M), out_capacity});
  if (n_out == 0) {
    return 0;
  }
  if (n_out > e->nmax) {
    e->lastError = "decimate: more samples than the engine was sized for";
    return 0;
  }
  uint8_t *row = e->dIq + static_cast<size_t>(channel) * e->iqPitch;
  cudaMemcpyAsync(row, iq, n_out * e->M * 2, cudaMemcpyHostToDevice, s);
  stageDecimate(e, stageBlock(channel, static_cast<int>(n_out)), e->dIq, e->iqPitch, s);
  // the uint8 result goes back through the front of the channel's (already consumed) input row
  launchRequantU8(e->dX1, e->pitch, e->dIq, e->iqPitch, static_cast<int>(n_out), channel, 1, s);
  e->launches += 1;
  cudaMemcpyAsync(out_u8, row, n_out * 2, cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  e->lastN = static_cast<int>(n_out);
  return stageFail(e, "decimate_u8") ? 0 : n_out;
}

static size_t demodCommon(fmgpu_engine *e, int channel, const uint8_t *iq_u8, const float *iq_cf32,
                          float *mpx_out, float *mono_out, size_t n, cudaStream_t s) {
  if (n > e->nmax) {
    e->lastError = "demod: more samples than the engine was sized for";
    return 0;
  }
  const int ni = static_cast<int>(n);
  if (iq_u8) {
    uint8_t *dst = e->dIq + static_cast<size_t>(channel) * e->iqPitch;
    cudaMemcpyAsync(dst, iq_u8, n * 2, cudaMemcpyHostToDevice, s);
  } else {
    cudaMemcpyAsync(e->dX1 + static_cast<size_t>(channel) * e->pitch, iq_cf32, n * sizeof(float2),
                    cudaMemcpyHostToDevice, s);
  }
  // the serial chain whatever the scan and demodulator modes: DC blocker -> channel FIR -> [AGC] ->
  // discriminator
  const BlockRef blk = stageBlock(channel, ni);
  stageDcBlock(e, blk, iq_u8 ? nullptr : e->dX1.get(), e->pitch, iq_u8 ? e->dIq.get() : nullptr, e->iqPitch,
               false, s);
  stageChanFir(e, blk, s);
  if (anyAgc(e, channel, 1)) {
    stageAgc(e, blk, s);
  }
  stageFreqDem(e, blk, s);
  carryHalos(e, HALO_X2 | HALO_Y, blk.n, channel, 1, s);
  if (mpx_out) {
    cudaMemcpyAsync(mpx_out, e->dMpx + static_cast<size_t>(channel) * e->mpxPitch + H_MPX,
                    n * sizeof(float), cudaMemcpyDeviceToHost, s);
  }
  size_t produced = 0;
  if (mono_out) {
    stageMono(e, blk, engineOut(e), true, 0, 0, s);
    AudioState a{};
    cudaMemcpyAsync(&a, e->dAudioSt + channel, sizeof(a), cudaMemcpyDeviceToHost, s);
    cudaStreamSynchronize(s);
    produced = std::min<size_t>(a.mono_n_out, e->acap);
    cudaMemcpyAsync(mono_out, e->res[0].audio + static_cast<size_t>(channel) * 2 * e->acap,
                    produced * sizeof(float), cudaMemcpyDeviceToHost, s);
  }
  cudaStreamSynchronize(s);
  e->lastN = ni;
  return stageFail(e, "demod") ? 0 : produced;
}

size_t fmgpu_demod_u8(fmgpu_engine *e, int channel, const uint8_t *iq, float *mpx_out,
                      float *mono_out, size_t n) {
  STAGE_PROLOGUE(iq && n > 0)
  return demodCommon(e, channel, iq, nullptr, mpx_out, mono_out, n, s);
}

size_t fmgpu_demod_cf32(fmgpu_engine *e, int channel, const float *iq_cf32, float *mpx_out,
                        float *mono_out, size_t n) {
  STAGE_PROLOGUE(iq_cf32 && n > 0)
  return demodCommon(e, channel, nullptr, iq_cf32, mpx_out, mono_out, n, s);
}

size_t fmgpu_downsample_mono(fmgpu_engine *e, int channel, const float *mpx, float *audio_out,
                             size_t n) {
  STAGE_PROLOGUE(mpx && audio_out && n > 0)
  if (n > e->nmax) {
    e->lastError = "downsample: more samples than the engine was sized for";
    return 0;
  }
  const int ni = static_cast<int>(n);
  cudaMemcpyAsync(e->dMpx + static_cast<size_t>(channel) * e->mpxPitch + H_MPX, mpx,
                  n * sizeof(float), cudaMemcpyHostToDevice, s);
  stageMono(e, stageBlock(channel, ni), engineOut(e), true, 0, 0, s);
  AudioState a{};
  cudaMemcpyAsync(&a, e->dAudioSt + channel, sizeof(a), cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  const size_t produced = std::min<size_t>(a.mono_n_out, e->acap);
  cudaMemcpyAsync(audio_out, e->res[0].audio + static_cast<size_t>(channel) * 2 * e->acap,
                  produced * sizeof(float), cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  return stageFail(e, "downsample") ? 0 : produced;
}

size_t fmgpu_stereo(fmgpu_engine *e, int channel, const float *mpx, float *left, float *right,
                    size_t n) {
  STAGE_PROLOGUE(mpx && left && right && n > 0)
  if (n > e->nmax) {
    e->lastError = "stereo: more samples than the engine was sized for";
    return 0;
  }
  const int ni = static_cast<int>(n);
  cudaMemcpyAsync(e->dMpx + static_cast<size_t>(channel) * e->mpxPitch + H_MPX, mpx,
                  n * sizeof(float), cudaMemcpyHostToDevice, s);
  const BlockRef blk = stageBlock(channel, ni);
  stagePilot(e, blk, s);
  stageStereo(e, blk, s);
  stageLpf(e, blk, s);
  carryHalos(e, HALO_MPX | HALO_LR, blk.n, channel, 1, s);
  cudaMemcpyAsync(left, e->dLf + static_cast<size_t>(channel) * e->lfPitch + H_LF, n * sizeof(float),
                  cudaMemcpyDeviceToHost, s);
  cudaMemcpyAsync(right, e->dRf + static_cast<size_t>(channel) * e->lfPitch + H_LF,
                  n * sizeof(float), cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  e->lastN = ni;
  return stageFail(e, "stereo") ? 0 : n;
}

size_t fmgpu_afpost(fmgpu_engine *e, int channel, const float *in_left, const float *in_right,
                    size_t n, float *out_left, float *out_right, size_t out_capacity) {
  STAGE_PROLOGUE(in_left && in_right && out_left && out_right && n > 0 && out_capacity > 0)
  if (n > e->nmax) {
    e->lastError = "afpost: more samples than the engine was sized for";
    return 0;
  }
  // honour outCapacity as the reference loop does (af_post_processor.cpp:56): stop
  // consuming input once out_capacity frames exist.
  AudioState a{};
  cudaMemcpyAsync(&a, e->dAudioSt + channel, sizeof(a), cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  size_t n_eff = n;
  {
    const unsigned long long num = static_cast<unsigned long long>(n) << 24;
    unsigned long long cnt = 0;
    if (num > a.rs_phase) {
      cnt = (num - a.rs_phase + e->k.aud_step - 1) / e->k.aud_step;
    }
    if (cnt >= out_capacity) {
      // the reference loop also stops when the count EQUALS the capacity: inputs after the one
      // that emitted output #(out_capacity-1) are never pushed
      const unsigned long long P =
          static_cast<unsigned long long>(a.rs_phase) + (out_capacity - 1) * 1ull * e->k.aud_step;
      n_eff = static_cast<size_t>(P >> 24) + 1;
    }
  }
  const int ni = static_cast<int>(n_eff);
  cudaMemcpyAsync(e->dLf + static_cast<size_t>(channel) * e->lfPitch + H_LF, in_left,
                  n_eff * sizeof(float), cudaMemcpyHostToDevice, s);
  cudaMemcpyAsync(e->dRf + static_cast<size_t>(channel) * e->lfPitch + H_LF, in_right,
                  n_eff * sizeof(float), cudaMemcpyHostToDevice, s);
  stageAfPost(e, stageBlock(channel, ni), engineOut(e), true, false, 0, s);
  carryHalos(e, HALO_LF, ni, channel, 1, s);
  cudaMemcpyAsync(&a, e->dAudioSt + channel, sizeof(a), cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  const size_t produced = std::min<size_t>({a.n_out, out_capacity, e->acap});
  cudaMemcpyAsync(out_left, e->res[0].audio + (static_cast<size_t>(channel) * 2 + 0) * e->acap,
                  produced * sizeof(float), cudaMemcpyDeviceToHost, s);
  cudaMemcpyAsync(out_right, e->res[0].audio + (static_cast<size_t>(channel) * 2 + 1) * e->acap,
                  produced * sizeof(float), cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  return stageFail(e, "afpost") ? 0 : produced;
}

size_t fmgpu_rds(fmgpu_engine *e, int channel, const float *mpx, size_t n, fmgpu_rds_group *out,
                 size_t cap) {
  STAGE_PROLOGUE(mpx && n > 0)
  if (n > e->nmax) {
    e->lastError = "rds: more samples than the engine was sized for";
    return 0;
  }
  const int ni = static_cast<int>(n);
  cudaMemcpyAsync(e->dMpx + static_cast<size_t>(channel) * e->mpxPitch + H_MPX, mpx,
                  n * sizeof(float), cudaMemcpyHostToDevice, s);
  // the block pipeline's two RDS stages, as the first block of a call (parity 0)
  const BlockRef blk = stageBlock(channel, ni);
  stageRdsResample(e, blk, 0, s);
  stageRdsDemod(e, blk, 0, engineOut(e), 0, true, false, s);
  RdsState r{};
  cudaMemcpyAsync(&r, e->dRds + channel, sizeof(r), cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  const size_t ng = r.n_groups;
  const size_t copy = std::min({ng, cap, e->gcap});
  if (out && copy > 0) {
    cudaMemcpyAsync(out, e->res[0].groups + static_cast<size_t>(channel) * e->gcap,
                    copy * sizeof(fmgpu_rds_group), cudaMemcpyDeviceToHost, s);
    cudaStreamSynchronize(s);
  }
  e->lastN = ni;
  return stageFail(e, "rds") ? 0 : ng;
}

// ---- introspection ------------------------------------------------------------------
size_t fmgpu_get_design(fmgpu_engine *e, int which, int channel, float *out, size_t cap,
                        float *scale) {
  if (!e) {
    return 0;
  }
  std::vector<float> v;
  float sc = 1.0f;
  switch (which) {
  case 0: v = e->decTaps; sc = e->decScale; break;
  case 1: {
    if (channel < 0 || channel >= e->C) {
      return 0;
    }
    const auto &f = e->filters[e->hParams[channel].filt];
    v = f.taps;
    sc = f.scale;
    break;
  }
  case 2: v = e->pilTaps; sc = 1.0f; break;
  case 3: v = e->audTaps; sc = e->k.aud_scale; break;
  case 4: v = e->audRs.bank; sc = static_cast<float>(e->audRs.step); break;
  case 5: v = e->rdsLpf; sc = e->k.rds_lpf_scale; break;
  case 6: v = e->ss.mf; sc = e->ss.sosB0; break;
  case 7: v = e->ss.dmf; sc = e->ss.sosA1; break;
  case 8: v = e->rdsRs.bank; sc = static_cast<float>(e->rdsRs.step); break;
  default: return 0;
  }
  if (scale) {
    *scale = sc;
  }
  if (out) {
    std::memcpy(out, v.data(), std::min(cap, v.size()) * sizeof(float));
  }
  return v.size();
}

size_t fmgpu_debug_read(fmgpu_engine *e, int which, int channel, float *out, size_t cap) {
  if (!e || !out || channel < 0 || channel >= e->C) {
    return 0;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  cudaSetDevice(e->device);
  syncPipes(e);
  const size_t c = static_cast<size_t>(channel);
  const float *base = nullptr;
  size_t per = 1;  // floats per sample
  switch (which) {
  case 0: base = reinterpret_cast<const float *>(e->dX1 + c * e->pitch); per = 2; break;
  case 1: base = e->dMpx + c * e->mpxPitch + H_MPX; break;
  case 2: base = e->dLf + c * e->lfPitch + H_LF; break;
  case 3: base = e->dRf + c * e->lfPitch + H_LF; break;
  case 4: base = e->dPilot + c * e->pitch; break;
  case 5: base = e->dLraw + c * e->lrPitch + H_LR; break;
  case 6: base = e->dRraw + c * e->lrPitch + H_LR; break;
  default: return 0;
  }
  size_t written = 0;
  if (e->lastBlocks > 0) {
    // a batch call: its blocks sit in ring slots (seq0 + b) % K
    for (int b = 0; b < e->lastBlocks && written < cap; b++) {
      const size_t slot = static_cast<size_t>((e->lastSeq0 + b) % static_cast<uint64_t>(e->K));
      const size_t cnt = std::min(cap - written, per * static_cast<size_t>(e->N));
      cudaMemcpyAsync(out + written, base + per * slot * e->N, cnt * sizeof(float),
                      cudaMemcpyDeviceToHost, e->stream);
      written += cnt;
    }
  } else {
    // a stage-level call: offset 0 (the halos have been carried; the data region is intact)
    written = std::min(per * static_cast<size_t>(e->lastN), cap);
    cudaMemcpyAsync(out, base, written * sizeof(float), cudaMemcpyDeviceToHost, e->stream);
  }
  cudaStreamSynchronize(e->stream);
  return written;
}

size_t fmgpu_debug_rds_bits(fmgpu_engine *e, int channel, uint8_t *out, size_t cap) {
  if (!e || channel < 0 || channel >= e->C) {
    return 0;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  cudaSetDevice(e->device);
  syncPipes(e);
  RdsState r{};
  cudaMemcpyAsync(&r, e->dRds + channel, sizeof(r), cudaMemcpyDeviceToHost, e->stream);
  cudaStreamSynchronize(e->stream);
  const size_t n = std::min<size_t>(r.n_bits, e->bitsCap);
  if (out) {
    cudaMemcpyAsync(out, e->dBits + static_cast<size_t>(channel) * e->bitsCap, std::min(n, cap),
                    cudaMemcpyDeviceToHost, e->stream);
    cudaStreamSynchronize(e->stream);
  }
  return n;
}

uint64_t fmgpu_launch_count(const fmgpu_engine *e) { return e ? e->launches : 0; }

int fmgpu_enable_stage_timing(fmgpu_engine *e, int on) {
  if (!e) {
    return FMGPU_EINVAL;
  }
  e->timing = on != 0;
  return FMGPU_OK;
}

// Debug: with stage timing on, the raw spans (one per stage launch sequence) of every batch
// queued since the last call, as start/end milliseconds after the earliest span. Synchronises.
int fmgpu_debug_timeline(fmgpu_engine *e, const char **names, int *groups, float *t0_ms,
                         float *t1_ms, int cap) {
  if (!e) {
    return 0;
  }
  std::lock_guard<std::recursive_mutex> lk(e->mu);
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  const int n = static_cast<int>(e->spans.size());
  // the earliest start: spans were recorded in launch order, but on different streams
  int first = 0;
  for (int i = 1; i < n; i++) {
    float d = 0.0f;
    if (cudaEventElapsedTime(&d, e->spans[first].start, e->spans[i].start) == cudaSuccess && d < 0.0f) {
      first = i;
    }
  }
  for (int i = 0; i < n && i < cap; i++) {
    names[i] = e->spans[i].name;
    groups[i] = e->spans[i].group;
    cudaEventElapsedTime(&t0_ms[i], e->spans[first].start, e->spans[i].start);
    cudaEventElapsedTime(&t1_ms[i], e->spans[first].start, e->spans[i].end);
  }
  e->spans.clear();
  return n;
}

int fmgpu_get_stage_times(fmgpu_engine *e, const char **names, float *ms, int cap) {
  if (!e) {
    return 0;
  }
  int n = 0;
  for (auto &t : e->lastTimes) {
    if (n < cap) {
      names[n] = t.first;
      ms[n] = t.second;
    }
    n++;
  }
  return n;
}

size_t fmgpu_decim_tc_host_model(int decimation, const float *taps, int n_taps, float scale,
                                 const unsigned char *iq, int valid_history, int n_out, float *out) {
  if (!taps || n_taps < 1) {
    return 0;
  }
  std::vector<float> hrev(taps, taps + n_taps);
  std::reverse(hrev.begin(), hrev.end());
  return decimTcHostModel(decimation, hrev, scale, iq, valid_history, n_out, out);
}

size_t fmgpu_fir_tc_host_model(const float *taps, int n_taps, float scale, int data_shift, const float *x,
                               size_t n_hist, size_t n, float *y) {
  const int lp = static_cast<int>(roundUp(static_cast<size_t>(std::max(n_taps, 1)), 8));
  return firTcHostModel(taps, n_taps, lp, scale, data_shift, x, n_hist, n, y);
}

size_t fmgpu_design_host(const fmgpu_config *cfg, int which, int bw_hz, float *out, size_t cap,
                         float *scale) {
  if (!cfg || cfg->iq_rate < 1 || cfg->decimation < 1) {
    return 0;
  }
  fmgpu_engine tmp;
  tmp.cfg = *cfg;
  if (tmp.cfg.output_rate <= 0) {
    tmp.cfg.output_rate = 32000;
  }
  tmp.M = cfg->decimation;
  tmp.fs = cfg->iq_rate / cfg->decimation;
  if (computeDesigns(&tmp) != FMGPU_OK) {
    return 0;
  }
  std::vector<float> v;
  float sc = 1.0f;
  switch (which) {
  case 0: v = tmp.decTaps; sc = tmp.decScale; break;
  case 1: {
    // FMDemod ctor filter, then setW0BandwidthHz(cfg->w0), setBandwidthHz(bw_hz)
    unsigned len = 81;
    float cut = std::clamp(110000.0f / static_cast<float>(tmp.fs), 0.01f, 0.45f);
    float as = 60.0f;
    const fmdesign::ChannelFilterSpec spec =
        fmdesign::channelFilterSpec(bw_hz, std::clamp(cfg->w0_bandwidth_hz, 0, 400000), tmp.fs);
    if (spec.index != 0) {
      len = spec.length;
      cut = spec.cutoff;
      as = spec.atten;
    }
    v = fmdesign::kaiserLowpass(len, cut, as, 0.0f);
    sc = 2.0f * cut;
    break;
  }
  case 2: v = tmp.pilTaps; sc = 1.0f; break;
  case 3: v = tmp.audTaps; sc = tmp.k.aud_scale; break;
  case 4: v = tmp.audRs.bank; sc = static_cast<float>(tmp.audRs.step); break;
  case 5: v = tmp.rdsLpf; sc = tmp.k.rds_lpf_scale; break;
  case 6: v = tmp.ss.mf; sc = tmp.ss.sosB0; break;
  case 7: v = tmp.ss.dmf; sc = tmp.ss.sosA1; break;
  case 8: v = tmp.rdsRs.bank; sc = static_cast<float>(tmp.rdsRs.step); break;
  default: return 0;
  }
  if (scale) {
    *scale = sc;
  }
  if (out) {
    std::memcpy(out, v.data(), std::min(cap, v.size()) * sizeof(float));
  }
  return v.size();
}

}  // extern "C"
