// channelizer.cu — wideband front end for BASELINE config 4: one IQ capture (24 MS/s) ->
// C carriers at a fixed spacing, each mixed to baseband, low-pass filtered and decimated to the
// engine's DSP rate (240 kS/s), ready for fmgpu_process_batch_cf32.
//
// There is NO reference counterpart (SURVEY §8(f) row 3): the reference tunes one carrier in
// hardware. The parity target is therefore this file's own definition, evaluated in float64 by
// tests/test_gpu_channelizer.py:
//
//   y_k[m] = sum_{n=0}^{L-1} h[n] * x[m*D - n] * exp(-j 2 pi nu_k (m*D - n)),   nu_k = f_k / Fs
//          = exp(-j 2 pi nu_k m D) * sum_n W[n][k] * x[m*D - n],   W[n][k] = h[n] exp(+j 2 pi nu_k n)
//
// with x[s] the input pair converted by the object's sample format (toX below; for uint8,
// (u8 - 127.5) / 127.5, the convention of ComplexDecimator, liquid_primitives.cpp:461-499), h a
// Kaiser-windowed sinc of L = D * taps_per_phase taps scaled to unity pass-band gain, and the input before the first call equal to zero. m counts outputs since creation, so
// consecutive calls continue the same stream (the last L-1 inputs are carried).
//
// Two evaluations of that definition:
//
// * k_channelize_pp — the polyphase form, used whenever the carriers sit on a uniform grid
//   nu_k = (k + c0) / P with P = Fs / spacing an integer (P = 120 for 24 MS/s and 200 kHz; the output
//   rate Fs / D = 240 kS/s is 1.2x the spacing, so this is an oversampled bank, D = 100 != P):
//       x'[s]  = x[s] exp(-j 2 pi c0 s / P)                 (c0 = first_center / spacing = -49.5:
//                                                            a table of period 2P)
//       u_r[m] = sum_{n : (mD - n) mod P = r} h[n] x'[mD - n]     (L MACs per output instant in all)
//       y_k[m] = sum_{r=0}^{P-1} exp(-j 2 pi k r / P) u_r[m]      (a P-point DFT row per channel)
//   One CTA takes 32 output instants: input tile (rotated on the fly) -> the P partial sums of every
//   instant -> the DFT rows of this call's channels, everything in shared memory. Per output instant
//   that is L + 2 P C real-times-complex / complex MACs instead of the L C of the direct form:
//   13x fewer for the whole band, and the stage drops from 0.94 ms to well under 0.1 ms per 68 ms of
//   signal (bench.py config4.channelizer). It stays in FP32: the DFT is a [C][P] x [P][32] complex
//   contraction per CTA, 0.8 GFMA per step for the whole band — a tensor-core (tf32 / split-bf16)
//   form would have to buy back its own operand conversion to save microseconds and would not
//   hold the 2e-5 parity of the float64 model.
// * k_channelize — the direct form (one complex tap table per channel), kept for carrier sets that
//   are not a uniform grid. Lanes of a warp are 32 CHANNELS at the same output instant: the input
//   sample is a shared-memory broadcast, the taps W[n][k..k+31] one coalesced 256-byte line, and
//   every thread keeps 8 output instants so a tap is reused 8 times.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <new>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/fmgpu.h"
#include "cuda_handle.h"
#include "design.h"
#include "device_once.h"

// Captures. One object may serve n_captures captures that advance together (same rate, decimation,
// spacing and filter; capture w's carrier k sits first_center_hz[w] + k * spacing from ITS centre).
// Every kernel takes the capture from one grid dimension (k_chan_carry: one CTA per capture); each
// capture has its own input row, history row and carrier frequencies (direct form: tap table and
// phase steps; polyphase form: rotation table). The prototype taps and the DFT twiddles are shared.
// One capture is the single-capture channelizer, with the same arithmetic.
struct fmgpu_channelizer {
  int device = 0;
  int nCap = 1;                    // captures
  int wideRate = 0, D = 0, C = 0, Cpad = 0, L = 0;
  double spacingHz = 0.0;
  std::vector<float> taps;         // prototype h[n]
  fmgpu::DeviceArray<float2> dW;      // [nCap][L][Cpad]
  fmgpu::DeviceArray<double> dNuD;    // [nCap][Cpad] frac(nu_k * D): phase advance per output, in turns
  int format = FMGPU_IQ_CU8;       // sample format, shared by every capture
  int pairBytes = 2;               // bytes of one I,Q pair of that format
  fmgpu::DeviceArray<uint8_t> dHist;  // [nCap][pairBytes (L-1)]: last L-1 input pairs of the previous call
  // polyphase form (uniform grid): nu_k = (k + c0_w) / P
  bool polyphase = false;
  int P = 0;
  fmgpu::DeviceArray<float> dTaps;    // [L]
  fmgpu::DeviceArray<float2> dRot;    // capture w: [rotOff[w], rotOff[w+1]) exp(-j 2 pi c0_w s / P)
  fmgpu::DeviceArray<int> dRotOff;    // [nCap + 1]; the period of capture w's table is P * T_w
  fmgpu::DeviceArray<float2> dTw;     // [P] exp(-j 2 pi i / P)
  unsigned long long outCount = 0; // outputs produced so far (m of the next output)
  long histValid = 0;              // how many of the carried samples are real input (rest = 0)
  std::string lastError;
};

namespace {

// Sample formats (include/fmgpu.h FMGPU_IQ_*): the pair type a kernel is instantiated on decides only
// how a pair becomes x; everything after the load is the same for every format.
__device__ __forceinline__ float2 toX(uchar2 b) {  // FMGPU_IQ_CU8: offset binary
  constexpr float kScale = 1.0f / 127.5f;
  return make_float2(((float)b.x - 127.5f) * kScale, ((float)b.y - 127.5f) * kScale);
}
__device__ __forceinline__ float2 toX(char2 b) {   // FMGPU_IQ_CS8: exact
  return make_float2((float)b.x * (1.0f / 128.0f), (float)b.y * (1.0f / 128.0f));
}
__device__ __forceinline__ float2 toX(short2 b) {  // FMGPU_IQ_CS16: exact
  return make_float2((float)b.x * (1.0f / 32768.0f), (float)b.y * (1.0f / 32768.0f));
}

constexpr int TMW = 8;            // output instants per thread
constexpr int WARPS = 4;          // warps per CTA: 4 groups of TMW instants
constexpr int TM = TMW * WARPS;   // output instants per CTA

template <typename Pair>
__global__ void __launch_bounds__(32 * WARPS)
k_channelize(const uint8_t *__restrict__ iq, size_t iq_stride, const uint8_t *__restrict__ hist,
             long hist_valid, long n_in,
             const float2 *__restrict__ W, const double *__restrict__ nuD, int L, int D, int Cpad,
             int ch_first, int ch_count, unsigned long long m_base, long n_out,
             float2 *__restrict__ out, size_t out_stride) {
  extern __shared__ float2 cx[];  // tile element a <-> input sample m0*D - (L-1) + a
  const unsigned cap = blockIdx.z;  // capture: its input, history, taps, phase steps and output rows
  iq += cap * iq_stride;
  hist += (size_t)cap * sizeof(Pair) * (L - 1);
  W += (size_t)cap * L * Cpad;
  nuD += (size_t)cap * Cpad;
  out += (size_t)cap * ch_count * out_stride;
  const long m0 = (long)blockIdx.x * TM;
  const int tile_len = (TM - 1) * D + L;
  const long s0 = m0 * D - (L - 1);
  const Pair *in2 = reinterpret_cast<const Pair *>(iq);
  const Pair *hist2 = reinterpret_cast<const Pair *>(hist);
  for (int a = threadIdx.x; a < tile_len; a += blockDim.x) {
    const long s = s0 + a;
    float2 v = make_float2(0.0f, 0.0f);
    if (s >= n_in || s < -hist_valid) {
      // beyond this call (only outputs past n_out would use it) or before the first input ever
      v = make_float2(0.0f, 0.0f);
    } else {
      v = toX((s >= 0) ? in2[s] : hist2[(L - 1) + s]);
    }
    cx[a] = v;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int wq = threadIdx.x >> 5;
  const int kk = blockIdx.y * 32 + lane;          // channel within the selection
  const int k = ch_first + kk;                    // channel of the bank
  const bool valid = kk < ch_count;
  const float2 *Wk = W + (valid ? k : ch_first);  // column k, row pitch Cpad
  float2 acc[TMW];
#pragma unroll
  for (int i = 0; i < TMW; i++) {
    acc[i] = make_float2(0.0f, 0.0f);
  }
  // output instant m0 + wq*TMW + i reads x[m*D - n] = cx[(L-1) + (wq*TMW + i)*D - n]
  const float2 *xb = cx + (L - 1) + wq * TMW * D;
  for (int n = 0; n < L; n++) {
    const float2 w = Wk[(size_t)n * Cpad];
#pragma unroll
    for (int i = 0; i < TMW; i++) {
      const float2 x = xb[i * D - n];  // the same address in every lane: a broadcast
      acc[i].x = fmaf(w.x, x.x, acc[i].x);
      acc[i].x = fmaf(-w.y, x.y, acc[i].x);
      acc[i].y = fmaf(w.x, x.y, acc[i].y);
      acc[i].y = fmaf(w.y, x.x, acc[i].y);
    }
  }
  if (!valid) {
    return;
  }
  const double step = nuD[k];
#pragma unroll
  for (int i = 0; i < TMW; i++) {
    const long m = m0 + wq * TMW + i;
    if (m < n_out) {
      // exp(-j 2 pi nu_k m D): the turn count modulo one, in double
      const unsigned long long mabs = m_base + (unsigned long long)m;
      const double turns = step * (double)(mabs & 0xffffffffull) +
                           step * 4294967296.0 * (double)(mabs >> 32);
      const double fr = turns - floor(turns);
      double sn, cs;
      sincospi(-2.0 * fr, &sn, &cs);
      const float c = (float)cs, s = (float)sn;
      out[(size_t)kk * out_stride + m] =
          make_float2(acc[i].x * c - acc[i].y * s, acc[i].x * s + acc[i].y * c);
    }
  }
}

constexpr int PP_TM = 32;         // output instants per CTA of the polyphase kernel
constexpr int PP_THREADS = 256;

template <typename Pair>
__global__ void __launch_bounds__(PP_THREADS)
k_channelize_pp(const uint8_t *__restrict__ iq, size_t iq_stride, const uint8_t *__restrict__ hist,
                long hist_valid, long n_in, const float *__restrict__ taps,
                const float2 *__restrict__ rot, const int *__restrict__ rot_off,
                const float2 *__restrict__ tw, int L, int D, int P, int ch_first,
                int ch_count, unsigned long long m_base, long n_out, float2 *__restrict__ out,
                size_t out_stride) {
  extern __shared__ float2 pp_smem[];
  const unsigned cap = blockIdx.y;  // capture: its input, history, rotation table and output rows
  iq += cap * iq_stride;
  hist += (size_t)cap * sizeof(Pair) * (L - 1);
  rot += rot_off[cap];
  const int rot_period = rot_off[cap + 1] - rot_off[cap];
  out += (size_t)cap * ch_count * out_stride;
  const int tile_len = (PP_TM - 1) * D + L;
  float2 *xs = pp_smem;                       // [tile_len] rotated input, element a <-> sample m0*D-(L-1)+a
  float2 *u = xs + tile_len;                  // [P][PP_TM + 1]
  float2 *tws = u + (size_t)P * (PP_TM + 1);  // [P]
  float *hs = reinterpret_cast<float *>(tws + P);   // [L]
  const long m0 = (long)blockIdx.x * PP_TM;
  const long s0 = m0 * D - (L - 1);           // call-relative sample index of tile element 0
  const Pair *in2 = reinterpret_cast<const Pair *>(iq);
  const Pair *hist2 = reinterpret_cast<const Pair *>(hist);
  // absolute sample index of call-relative sample 0, modulo the rotation period
  const unsigned long long abs0 = (m_base % (unsigned long long)rot_period) * (unsigned long long)D;
  for (int a = threadIdx.x; a < tile_len; a += PP_THREADS) {
    const long s = s0 + a;
    float2 v = make_float2(0.0f, 0.0f);
    if (s < n_in && s >= -hist_valid) {
      const float2 x = toX((s >= 0) ? in2[s] : hist2[(L - 1) + s]);
      const float xr = x.x, xi = x.y;
      // (abs0 + s) mod period, s may be negative: add a multiple of the period first
      const unsigned long long ai = abs0 + (unsigned long long)(s + (long)rot_period * (long)(L / rot_period + 2));
      const float2 w = rot[ai % (unsigned long long)rot_period];
      v = make_float2(xr * w.x - xi * w.y, xr * w.y + xi * w.x);
    }
    xs[a] = v;
  }
  for (int i = threadIdx.x; i < P; i += PP_THREADS) {
    tws[i] = tw[i];
  }
  for (int i = threadIdx.x; i < L; i += PP_THREADS) {
    hs[i] = taps[i];
  }
  __syncthreads();
  // partial sums: item (m, r), r fastest -> consecutive lanes read consecutive samples and taps
  for (int item = threadIdx.x; item < PP_TM * P; item += PP_THREADS) {
    const int m = item / P, r = item - m * P;
    const unsigned long long mabs = m_base + (unsigned long long)(m0 + m);
    const int mdp = (int)(((mabs % (unsigned long long)P) * (unsigned long long)D) % (unsigned long long)P);
    int n = mdp - r;                    // taps n = n0, n0 + P, ... see (mD - n) mod P = r
    if (n < 0) {
      n += P;
    }
    const float2 *xb = xs + (L - 1) + m * D;
    float ar = 0.0f, ai = 0.0f;
    for (; n < L; n += P) {
      const float h = hs[n];
      const float2 x = xb[-n];
      ar = fmaf(h, x.x, ar);
      ai = fmaf(h, x.y, ai);
    }
    u[(size_t)r * (PP_TM + 1) + m] = make_float2(ar, ai);
  }
  __syncthreads();
  // DFT rows of this call's channels: item (kk, m), m fastest
  for (int item = threadIdx.x; item < ch_count * PP_TM; item += PP_THREADS) {
    const int kk = item / PP_TM, m = item - kk * PP_TM;
    const int k = (ch_first + kk) % P;
    float yr = 0.0f, yi = 0.0f;
    int ti = 0;                          // (k * r) mod P
    for (int r = 0; r < P; r++) {
      const float2 w = tws[ti];
      const float2 v = u[(size_t)r * (PP_TM + 1) + m];
      yr = fmaf(w.x, v.x, yr);
      yr = fmaf(-w.y, v.y, yr);
      yi = fmaf(w.x, v.y, yi);
      yi = fmaf(w.y, v.x, yi);
      ti += k;
      if (ti >= P) {
        ti -= P;
      }
    }
    if (m0 + m < n_out) {
      out[(size_t)kk * out_stride + m0 + m] = make_float2(yr, yi);
    }
  }
}

// hist <- last H pairs of (hist ++ in[0..n_in)), one CTA per capture. It only moves pairs, so it
// is instantiated per pair size (uchar2: cu8 and cs8; short2: cs16), not per format.
template <typename Pair>
__global__ void k_chan_carry(uint8_t *hist, const uint8_t *iq, size_t iq_stride, long n_in, int H) {
  Pair *h = reinterpret_cast<Pair *>(hist) + (size_t)blockIdx.x * H;
  const Pair *in = reinterpret_cast<const Pair *>(iq + blockIdx.x * iq_stride);
  // two phases so the shift is safe when n_in < H
  extern __shared__ __align__(4) unsigned char carry_smem[];
  Pair *tmp = reinterpret_cast<Pair *>(carry_smem);
  for (int e = threadIdx.x; e < H; e += blockDim.x) {
    const long src = n_in - H + e;
    tmp[e] = (src >= 0) ? in[src] : h[e + n_in];
  }
  __syncthreads();
  for (int e = threadIdx.x; e < H; e += blockDim.x) {
    h[e] = tmp[e];
  }
}

// bytes of one I,Q pair of a sample format; 0 for an unknown format
int formatPairBytes(int format) {
  switch (format) {
    case FMGPU_IQ_CU8:
    case FMGPU_IQ_CS8:
      return 2;
    case FMGPU_IQ_CS16:
      return 4;
    default:
      return 0;
  }
}

// The one launch sequence of a call, instantiated on the format's pair type (Carry: the pair type
// of the same size that k_chan_carry moves).
template <typename Pair, typename Carry>
void launchChannelize(fmgpu_channelizer *z, const uint8_t *iq_dev, size_t iq_stride_bytes, size_t n_in,
                      int ch_first, int ch_count, float2 *out, size_t out_stride_samples,
                      size_t smem, size_t pp_smem, cudaStream_t s) {
  const unsigned nCap = static_cast<unsigned>(z->nCap);
  const long n_out = static_cast<long>(n_in / static_cast<size_t>(z->D));
  if (z->polyphase && pp_smem <= 200 * 1024) {
    static fmgpu::DeviceOnce pp_attrs;  // per device and instantiation: device_once.h
    pp_attrs.run([] { return cudaFuncSetAttribute(k_channelize_pp<Pair>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); });
    dim3 grid(static_cast<unsigned>((n_out + PP_TM - 1) / PP_TM), nCap);
    k_channelize_pp<Pair><<<grid, PP_THREADS, pp_smem, s>>>(
        iq_dev, iq_stride_bytes, z->dHist, z->histValid, static_cast<long>(n_in), z->dTaps, z->dRot, z->dRotOff,
        z->dTw, z->L, z->D, z->P, ch_first, ch_count, z->outCount, n_out, out, out_stride_samples);
  } else {
    static fmgpu::DeviceOnce attrs;
    attrs.run([] { return cudaFuncSetAttribute(k_channelize<Pair>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); });
    dim3 grid(static_cast<unsigned>((n_out + TM - 1) / TM), static_cast<unsigned>((ch_count + 31) / 32), nCap);
    k_channelize<Pair><<<grid, 32 * WARPS, smem, s>>>(
        iq_dev, iq_stride_bytes, z->dHist, z->histValid, static_cast<long>(n_in), z->dW, z->dNuD, z->L, z->D,
        z->Cpad, ch_first, ch_count, z->outCount, n_out, out, out_stride_samples);
  }
  const int H = z->L - 1;
  k_chan_carry<Carry><<<nCap, 512, static_cast<size_t>(H) * sizeof(Carry), s>>>(z->dHist, iq_dev, iq_stride_bytes,
                                                                               static_cast<long>(n_in), H);
}

}  // namespace

extern "C" {

int fmgpu_channelizer_create(int device, int wide_rate, int decimation, int n_channels,
                             double first_center_hz, double spacing_hz, int taps_per_phase,
                             double cutoff_hz, float atten_db, fmgpu_channelizer **out) {
  return fmgpu_channelizer_create_multi(device, 1, wide_rate, decimation, n_channels, &first_center_hz,
                                        spacing_hz, taps_per_phase, cutoff_hz, atten_db, out);
}

int fmgpu_channelizer_create_multi(int device, int n_captures, int wide_rate, int decimation,
                                   int n_channels, const double *first_center_hz, double spacing_hz,
                                   int taps_per_phase, double cutoff_hz, float atten_db,
                                   fmgpu_channelizer **out) {
  return fmgpu_channelizer_create_format(device, FMGPU_IQ_CU8, n_captures, wide_rate, decimation, n_channels,
                                         first_center_hz, spacing_hz, taps_per_phase, cutoff_hz, atten_db, out);
}

int fmgpu_channelizer_create_format(int device, int sample_format, int n_captures, int wide_rate,
                                    int decimation, int n_channels, const double *first_center_hz,
                                    double spacing_hz, int taps_per_phase, double cutoff_hz,
                                    float atten_db, fmgpu_channelizer **out) {
  // the capture is a grid dimension: y of k_channelize_pp, z of k_channelize (at most 65535 each)
  if (!out || formatPairBytes(sample_format) == 0 || !first_center_hz || n_captures < 1 || n_captures > 65535 || wide_rate < 1 ||
      decimation < 1 || n_channels < 1 || taps_per_phase < 1 || !(cutoff_hz > 0.0) ||
      cutoff_hz * 2.0 > static_cast<double>(wide_rate)) {
    return FMGPU_EINVAL;
  }
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
    cudaGetLastError();
    return FMGPU_ENODEV;  // no CPU fallback
  }
  fmgpu_channelizer *z = new (std::nothrow) fmgpu_channelizer();
  if (!z) {
    return FMGPU_ENOMEM;
  }
  z->device = device;
  z->nCap = n_captures;
  z->format = sample_format;
  z->pairBytes = formatPairBytes(sample_format);
  z->wideRate = wide_rate;
  z->D = decimation;
  z->C = n_channels;
  z->Cpad = (n_channels + 31) / 32 * 32;
  z->L = decimation * taps_per_phase;
  z->spacingHz = spacing_hz;
  const size_t nCap = static_cast<size_t>(n_captures);
  std::vector<float2> W, rotTab, twTab;
  std::vector<double> nuD;
  std::vector<int> rotOff;
  try {
    const float fc = static_cast<float>(cutoff_hz / static_cast<double>(wide_rate));
    z->taps = fmdesign::kaiserLowpass(static_cast<unsigned>(z->L), fc, atten_db, 0.0f);
    for (float &t : z->taps) {
      t *= 2.0f * fc;  // unity gain in the pass band
    }
    const size_t wRow = static_cast<size_t>(z->L) * z->Cpad;
    W.assign(nCap * wRow, make_float2(0.0f, 0.0f));
    nuD.assign(nCap * z->Cpad, 0.0);
    for (size_t w = 0; w < nCap; w++) {
      for (int k = 0; k < z->C; k++) {
        const double nu = (first_center_hz[w] + spacing_hz * k) / static_cast<double>(wide_rate);
        const double adv = nu * static_cast<double>(decimation);
        nuD[w * z->Cpad + k] = adv - std::floor(adv);
        for (int n = 0; n < z->L; n++) {
          const double turns = nu * static_cast<double>(n);
          const double ph = 2.0 * M_PI * (turns - std::floor(turns));
          W[w * wRow + static_cast<size_t>(n) * z->Cpad + k] =
              make_float2(static_cast<float>(z->taps[n] * std::cos(ph)),
                          static_cast<float>(z->taps[n] * std::sin(ph)));
        }
      }
    }
    // uniform grid? P = Fs / spacing integer, and for every capture c0 = first / spacing with
    // c0 * T integer for a small T; otherwise every capture takes the direct form
    const double pd = static_cast<double>(wide_rate) / spacing_hz;
    const int P = static_cast<int>(std::llround(pd));
    bool uniform = spacing_hz > 0.0 && P >= 2 && P <= 1024 && std::fabs(pd - P) < 1e-9 && n_channels <= P &&
                   getenv("FMGPU_CHANNELIZER_DIRECT") == nullptr;
    std::vector<int> T(nCap, 0);
    for (size_t w = 0; w < nCap && uniform; w++) {
      const double c0 = first_center_hz[w] / spacing_hz;
      for (int t = 1; t <= 8 && T[w] == 0; t++) {
        if (std::fabs(c0 * t - std::round(c0 * t)) < 1e-9) {
          T[w] = t;
        }
      }
      uniform = T[w] > 0;
    }
    if (uniform) {
      z->polyphase = true;
      z->P = P;
      rotOff.assign(nCap + 1, 0);
      for (size_t w = 0; w < nCap; w++) {
        rotOff[w + 1] = rotOff[w] + P * T[w];
      }
      rotTab.resize(rotOff[nCap]);
      for (size_t w = 0; w < nCap; w++) {
        const double c0 = first_center_hz[w] / spacing_hz;
        const int rotPeriod = P * T[w];
        for (int i = 0; i < rotPeriod; i++) {
          // exp(-j 2 pi c0 i / P), the turn count reduced exactly: c0 * T is an integer
          const long long num = std::llround(c0 * T[w]) * static_cast<long long>(i);   // turns * (P T)
          const long long red = ((num % rotPeriod) + rotPeriod) % rotPeriod;
          const double ph = -2.0 * M_PI * static_cast<double>(red) / static_cast<double>(rotPeriod);
          rotTab[rotOff[w] + i] = make_float2(static_cast<float>(std::cos(ph)), static_cast<float>(std::sin(ph)));
        }
      }
      twTab.resize(P);
      for (int i = 0; i < P; i++) {
        const double ph = -2.0 * M_PI * static_cast<double>(i) / static_cast<double>(P);
        twTab[i] = make_float2(static_cast<float>(std::cos(ph)), static_cast<float>(std::sin(ph)));
      }
    }
  } catch (const std::bad_alloc &) {
    delete z;
    return FMGPU_ENOMEM;
  }
  bool ok = cudaSetDevice(device) == cudaSuccess;
  if (z->polyphase) {
    ok = ok && fmgpu::devAlloc(&z->dTaps, z->taps.size()) == cudaSuccess;
    ok = ok && fmgpu::devAlloc(&z->dRot, rotTab.size()) == cudaSuccess;
    ok = ok && fmgpu::devAlloc(&z->dRotOff, rotOff.size()) == cudaSuccess;
    ok = ok && fmgpu::devAlloc(&z->dTw, twTab.size()) == cudaSuccess;
    ok = ok && cudaMemcpy(z->dTaps, z->taps.data(), z->taps.size() * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemcpy(z->dRot, rotTab.data(), rotTab.size() * sizeof(float2), cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemcpy(z->dRotOff, rotOff.data(), rotOff.size() * sizeof(int), cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemcpy(z->dTw, twTab.data(), twTab.size() * sizeof(float2), cudaMemcpyHostToDevice) == cudaSuccess;
  }
  ok = ok && fmgpu::devAlloc(&z->dW, W.size()) == cudaSuccess;
  ok = ok && fmgpu::devAlloc(&z->dNuD, nuD.size()) == cudaSuccess;
  // the input before the first call is ZERO: no uint8 pair maps to 0.0, so for every format the
  // kernel clears the part of the window older than histValid samples
  ok = ok && fmgpu::devAlloc(&z->dHist, nCap * z->pairBytes * static_cast<size_t>(z->L - 1)) == cudaSuccess;
  ok = ok && cudaMemcpy(z->dW, W.data(), W.size() * sizeof(float2), cudaMemcpyHostToDevice) ==
                 cudaSuccess;
  ok = ok && cudaMemcpy(z->dNuD, nuD.data(), nuD.size() * sizeof(double), cudaMemcpyHostToDevice) ==
                 cudaSuccess;
  if (!ok) {
    cudaGetLastError();
    fmgpu_channelizer_destroy(z);
    return FMGPU_ENOMEM;
  }
  *out = z;
  return FMGPU_OK;
}

void fmgpu_channelizer_destroy(fmgpu_channelizer *z) {
  if (!z) {
    return;
  }
  cudaSetDevice(z->device);
  cudaDeviceSynchronize();
  delete z;  // the handles free the device buffers
}

int fmgpu_channelizer_output_rate(const fmgpu_channelizer *z) { return z ? z->wideRate / z->D : 0; }

int fmgpu_channelizer_n_captures(const fmgpu_channelizer *z) { return z ? z->nCap : 0; }

int fmgpu_channelizer_sample_format(const fmgpu_channelizer *z) { return z ? z->format : FMGPU_EINVAL; }

size_t fmgpu_channelizer_taps(const fmgpu_channelizer *z, float *out, size_t cap) {
  if (!z) {
    return 0;
  }
  if (out) {
    for (size_t i = 0; i < z->taps.size() && i < cap; i++) {
      out[i] = z->taps[i];
    }
  }
  return z->taps.size();
}

int fmgpu_channelizer_process(fmgpu_channelizer *z, const uint8_t *iq_dev, size_t n_in,
                              int ch_first, int ch_count, float *out_cf32_dev,
                              size_t out_stride_samples, void *stream) {
  if (z && z->nCap != 1) {
    return FMGPU_EINVAL;
  }
  return fmgpu_channelizer_process_multi(z, iq_dev, 2 * n_in, n_in, ch_first, ch_count, out_cf32_dev,
                                         out_stride_samples, stream);
}

int fmgpu_channelizer_process_multi(fmgpu_channelizer *z, const uint8_t *iq_dev,
                                    size_t iq_stride_bytes, size_t n_in, int ch_first,
                                    int ch_count, float *out_cf32_dev, size_t out_stride_samples,
                                    void *stream) {
  if (z && z->format != FMGPU_IQ_CU8) {
    return FMGPU_EINVAL;
  }
  return fmgpu_channelizer_process_iq(z, iq_dev, iq_stride_bytes, n_in, ch_first, ch_count, out_cf32_dev,
                                      out_stride_samples, stream);
}

int fmgpu_channelizer_process_iq(fmgpu_channelizer *z, const void *iq_dev, size_t iq_stride_bytes,
                                 size_t n_in, int ch_first, int ch_count, float *out_cf32_dev,
                                 size_t out_stride_samples, void *stream) {
  if (!z || !iq_dev || !out_cf32_dev || n_in == 0 || n_in % static_cast<size_t>(z->D) != 0) {
    return FMGPU_EINVAL;
  }
  const size_t pb = static_cast<size_t>(z->pairBytes);
  if (iq_stride_bytes % pb != 0 || iq_stride_bytes < pb * n_in ||
      reinterpret_cast<uintptr_t>(iq_dev) % pb != 0 ||
      ch_first < 0 || ch_count < 1 || ch_first + ch_count > z->C ||
      out_stride_samples < n_in / static_cast<size_t>(z->D)) {
    return FMGPU_EINVAL;
  }
  if (cudaSetDevice(z->device) != cudaSuccess) {
    return FMGPU_ENODEV;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t smem = static_cast<size_t>((TM - 1) * z->D + z->L) * sizeof(float2);
  if (smem > 200 * 1024) {
    z->lastError = "channelizer: filter too long for the shared-memory tile";
    return FMGPU_ERANGE;
  }
  const size_t pp_smem = (static_cast<size_t>((PP_TM - 1) * z->D + z->L) + static_cast<size_t>(z->P) * (PP_TM + 1) +
                          static_cast<size_t>(z->P)) * sizeof(float2) + static_cast<size_t>(z->L) * sizeof(float);
  const uint8_t *iq = static_cast<const uint8_t *>(iq_dev);
  float2 *out = reinterpret_cast<float2 *>(out_cf32_dev);
  switch (z->format) {
    case FMGPU_IQ_CU8:
      launchChannelize<uchar2, uchar2>(z, iq, iq_stride_bytes, n_in, ch_first, ch_count, out, out_stride_samples,
                                       smem, pp_smem, s);
      break;
    case FMGPU_IQ_CS8:
      launchChannelize<char2, uchar2>(z, iq, iq_stride_bytes, n_in, ch_first, ch_count, out, out_stride_samples,
                                      smem, pp_smem, s);
      break;
    default:  // FMGPU_IQ_CS16: create accepts no other format
      launchChannelize<short2, short2>(z, iq, iq_stride_bytes, n_in, ch_first, ch_count, out, out_stride_samples,
                                       smem, pp_smem, s);
      break;
  }
  const long n_out = static_cast<long>(n_in / static_cast<size_t>(z->D));
  z->outCount += static_cast<unsigned long long>(n_out);
  z->histValid = std::min<long>(z->L - 1, z->histValid + static_cast<long>(n_in));
  return cudaGetLastError() == cudaSuccess ? FMGPU_OK : FMGPU_ENODEV;
}

}  // extern "C"
