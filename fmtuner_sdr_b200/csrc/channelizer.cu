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
// Rational rates (fmgpu_channelizer_create_rate): with U/D the reduced ratio output / wide rate, h
// has L = D * taps_per_phase taps designed at rate U * Fs (cut-off cutoff / (U Fs), gain 2 fc U) and
//
//   y_k[m] = sum_{n = 0..L-1, (mD - n) = 0 mod U} h[n] x[(mD - n)/U] exp(-j 2 pi nu_k (mD - n)/U)
//          = sum_i g_q[i] x[s_m - i] exp(-j 2 pi nu_k (s_m - i)),   s_m = floor(mD / U), q = mD mod U,
//
// g_q[i] = h[q + iU] the phase filters of Lin = ceil(L / U) taps. U = 1 is the definition above.
// The host keeps T, the pairs received per capture; outputs 0 .. ceil(T U / D) - 1 exist, so the
// outputs of a call follow from T and n_in, and the last Lin - 1 inputs are carried.
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
#include <numeric>
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
  int wideRate = 0, U = 1, D = 0, C = 0, Cpad = 0, L = 0;
  int Lin = 0;                     // ceil(L / U): taps of one phase table, inputs one output reads
  double spacingHz = 0.0;
  std::vector<float> taps;         // prototype h[n], at rate U * wideRate
  fmgpu::DeviceArray<float2> dW;      // [nCap][U][Lin][Cpad]
  // [nCap][Cpad] phase step in turns: frac(nu_k * D) per output for U = 1, frac(nu_k) per input for U > 1
  fmgpu::DeviceArray<double> dNuD;
  int format = FMGPU_IQ_CU8;       // sample format, shared by every capture
  int pairBytes = 2;               // bytes of one I,Q pair of that format
  fmgpu::DeviceArray<uint8_t> dHist;  // [nCap][pairBytes (Lin-1)]: last Lin-1 input pairs of the previous call
  // polyphase form (uniform grid): nu_k = (k + c0_w) / P
  bool polyphase = false;
  int P = 0;
  fmgpu::DeviceArray<float> dTaps;    // [U][Lin] phase tables g_q[i] = h[q + iU]
  fmgpu::DeviceArray<float2> dRot;    // capture w: [rotOff[w], rotOff[w+1]) exp(-j 2 pi c0_w s / P)
  fmgpu::DeviceArray<int> dRotOff;    // [nCap + 1]; the period of capture w's table is P * T_w
  fmgpu::DeviceArray<float2> dTw;     // [P] exp(-j 2 pi i / P)
  unsigned long long inCount = 0;  // T: pairs per capture received so far; ceil(T U / D) outputs exist
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

constexpr int kMaxInterpolation = 64;  // largest U of fmgpu_channelizer_create_rate

constexpr int TMW = 8;            // output instants per thread
constexpr int WARPS = 4;          // warps per CTA: 4 groups of TMW instants
constexpr int TM = TMW * WARPS;   // output instants per CTA

// Direct form. A CTA takes TM output instants of one phase class: call-relative instants
// o + (g*TM + j)*U, j < TM, with o = blockIdx.x / groups and g = blockIdx.x % groups. They share the
// phase q and their newest samples are exactly D apart, so one tile and one tap table g_q serve all.
// For U = 1 there is one class and the CTA's instants are g*TM + j, as in the integer-decimation form.
template <typename Pair>
__global__ void __launch_bounds__(32 * WARPS)
k_channelize(const uint8_t *__restrict__ iq, size_t iq_stride, const uint8_t *__restrict__ hist,
             long hist_valid, long n_in,
             const float2 *__restrict__ W, const double *__restrict__ nuD, int Lin, int U, int D, int Cpad,
             int ch_first, int ch_count, unsigned long long m_base, unsigned long long t_base, long n_out,
             int groups, float2 *__restrict__ out, size_t out_stride) {
  extern __shared__ float2 cx[];  // tile element a <-> input sample s_first - (Lin-1) + a
  const unsigned cap = blockIdx.z;  // capture: its input, history, taps, phase steps and output rows
  const int o = blockIdx.x / groups;             // phase class: call-relative instant o, o + U, ...
  const long g = blockIdx.x - o * groups;
  const unsigned long long mo = (m_base + o) * (unsigned long long)D;
  const unsigned long long sa = (U == 1) ? mo : mo / (unsigned)U;
  const int q = (int)(mo - sa * (unsigned)U);    // phase of every instant of this CTA
  const long so = (long)(sa - t_base);           // call-relative newest sample of instant o
  iq += cap * iq_stride;
  hist += (size_t)cap * sizeof(Pair) * (Lin - 1);
  W += ((size_t)cap * U + q) * Lin * Cpad;
  nuD += (size_t)cap * Cpad;
  out += (size_t)cap * ch_count * out_stride;
  const long j0 = g * TM;                        // the CTA's first instant is o + j0 * U
  const int tile_len = (TM - 1) * D + Lin;
  const long s0 = so + j0 * D - (Lin - 1);
  const Pair *in2 = reinterpret_cast<const Pair *>(iq);
  const Pair *hist2 = reinterpret_cast<const Pair *>(hist);
  for (int a = threadIdx.x; a < tile_len; a += blockDim.x) {
    const long s = s0 + a;
    float2 v = make_float2(0.0f, 0.0f);
    if (s >= n_in || s < -hist_valid) {
      // beyond this call (only outputs past n_out would use it) or before the first input ever
      v = make_float2(0.0f, 0.0f);
    } else {
      v = toX((s >= 0) ? in2[s] : hist2[(Lin - 1) + s]);
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
  // instant j0 + wq*TMW + i of the class reads x[s - n] = cx[(Lin-1) + (wq*TMW + i)*D - n]
  const float2 *xb = cx + (Lin - 1) + wq * TMW * D;
  for (int n = 0; n < Lin; n++, Wk += Cpad) {
    const float2 w = *Wk;
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
    const long j = j0 + wq * TMW + i;
    const long m = o + j * U;
    if (m < n_out) {
      // exp(-j 2 pi nu_k s_m), the turn count modulo one, in double. U = 1: step = frac(nu_k D)
      // times m; U > 1: step = frac(nu_k) times the absolute newest sample s_m.
      const unsigned long long idx = (U == 1) ? m_base + (unsigned long long)m
                                              : t_base + (unsigned long long)(so + j * D);
      const double turns = step * (double)(idx & 0xffffffffull) +
                           step * 4294967296.0 * (double)(idx >> 32);
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

// Polyphase form. Instant m of the CTA has its own newest sample s_m and phase q_m; the phase
// tables g_q[i] = h[q + iU] are [U][Lin] (zero past the prototype's end), which is h for U = 1.
template <typename Pair>
__global__ void __launch_bounds__(PP_THREADS)
k_channelize_pp(const uint8_t *__restrict__ iq, size_t iq_stride, const uint8_t *__restrict__ hist,
                long hist_valid, long n_in, const float *__restrict__ taps,
                const float2 *__restrict__ rot, const int *__restrict__ rot_off,
                const float2 *__restrict__ tw, int Lin, int U, int D, int P, int ch_first,
                int ch_count, unsigned long long m_base, unsigned long long t_base, long n_out,
                float2 *__restrict__ out, size_t out_stride) {
  extern __shared__ float2 pp_smem[];
  const unsigned cap = blockIdx.y;  // capture: its input, history, rotation table and output rows
  iq += cap * iq_stride;
  hist += (size_t)cap * sizeof(Pair) * (Lin - 1);
  rot += rot_off[cap];
  const int rot_period = rot_off[cap + 1] - rot_off[cap];
  out += (size_t)cap * ch_count * out_stride;
  const long m0 = (long)blockIdx.x * PP_TM;
  // instant m0 + m: (m0 + m) D = sa0 U + q0 + m D, so s_m = s_m0 + (q0 + m D) / U and its phase is
  // (q0 + m D) mod U, in 32 bits
  const unsigned long long md0 = (m_base + (unsigned long long)m0) * (unsigned long long)D;
  const unsigned long long sa0 = (U == 1) ? md0 : md0 / (unsigned)U;   // absolute newest sample of instant m0
  const int q0 = (int)(md0 - sa0 * (unsigned)U);
  const int sp0 = (int)(sa0 % (unsigned)P);
  const long sf = (long)(sa0 - t_base);               // call-relative
  const int tile_len = (q0 + (PP_TM - 1) * D) / U + Lin;
  const int tile_cap = (int)(((PP_TM - 1) * (long)D + U - 1) / U) + Lin;  // the host's tile size
  float2 *xs = pp_smem;                       // [tile_cap] rotated input, element a <-> sample sf-(Lin-1)+a
  float2 *u = xs + tile_cap;                  // [P][PP_TM + 1]
  float2 *tws = u + (size_t)P * (PP_TM + 1);  // [P]
  float *hs = reinterpret_cast<float *>(tws + P);   // [U][Lin]
  const long s0 = sf - (Lin - 1);             // call-relative sample index of tile element 0
  const Pair *in2 = reinterpret_cast<const Pair *>(iq);
  const Pair *hist2 = reinterpret_cast<const Pair *>(hist);
  // absolute sample index of call-relative sample 0, modulo the rotation period
  const unsigned long long abs0 = t_base % (unsigned long long)rot_period;
  for (int a = threadIdx.x; a < tile_len; a += PP_THREADS) {
    const long s = s0 + a;
    float2 v = make_float2(0.0f, 0.0f);
    if (s < n_in && s >= -hist_valid) {
      const float2 x = toX((s >= 0) ? in2[s] : hist2[(Lin - 1) + s]);
      const float xr = x.x, xi = x.y;
      // (abs0 + s) mod period, s may be negative: add a multiple of the period first
      const unsigned long long ai = abs0 + (unsigned long long)(s + (long)rot_period * (long)(Lin / rot_period + 2));
      const float2 w = rot[ai % (unsigned long long)rot_period];
      v = make_float2(xr * w.x - xi * w.y, xr * w.y + xi * w.x);
    }
    xs[a] = v;
  }
  for (int i = threadIdx.x; i < P; i += PP_THREADS) {
    tws[i] = tw[i];
  }
  for (int i = threadIdx.x; i < U * Lin; i += PP_THREADS) {
    hs[i] = taps[i];
  }
  __syncthreads();
  // partial sums: item (m, r), r fastest -> consecutive lanes read consecutive samples and taps
  for (int item = threadIdx.x; item < PP_TM * P; item += PP_THREADS) {
    const int m = item / P, r = item - m * P;
    const int e = q0 + m * D;
    const int ds = (U == 1) ? e : e / U;   // s_m - s_m0
    int i = (sp0 + ds) % P - r;         // taps i = i0, i0 + P, ... see (s_abs_m - i) mod P = r
    if (i < 0) {
      i += P;
    }
    const float2 *xp = xs + (Lin - 1) + ds - i;
    const float *gp = hs + (e - ds * U) * Lin + i;
    float ar = 0.0f, ai = 0.0f;
    for (; i < Lin; i += P, gp += P, xp -= P) {
      const float h = *gp;
      const float2 x = *xp;
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

// outputs that exist once T pairs per capture have been received: ceil(T U / D)
unsigned long long outputsAfter(const fmgpu_channelizer *z, unsigned long long T) {
  return (T * static_cast<unsigned long long>(z->U) + static_cast<unsigned long long>(z->D) - 1) /
         static_cast<unsigned long long>(z->D);
}

// The one launch sequence of a call, instantiated on the format's pair type (Carry: the pair type
// of the same size that k_chan_carry moves).
template <typename Pair, typename Carry>
void launchChannelize(fmgpu_channelizer *z, const uint8_t *iq_dev, size_t iq_stride_bytes, size_t n_in,
                      int ch_first, int ch_count, float2 *out, size_t out_stride_samples, long n_out,
                      size_t smem, size_t pp_smem, cudaStream_t s) {
  const unsigned nCap = static_cast<unsigned>(z->nCap);
  const unsigned long long m_base = outputsAfter(z, z->inCount);
  if (n_out == 0) {
    // no output instant completes in this call: only the history moves
  } else if (z->polyphase && pp_smem <= 200 * 1024) {
    static fmgpu::DeviceOnce pp_attrs;  // per device and instantiation: device_once.h
    pp_attrs.run([] { return cudaFuncSetAttribute(k_channelize_pp<Pair>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); });
    dim3 grid(static_cast<unsigned>((n_out + PP_TM - 1) / PP_TM), nCap);
    k_channelize_pp<Pair><<<grid, PP_THREADS, pp_smem, s>>>(
        iq_dev, iq_stride_bytes, z->dHist, z->histValid, static_cast<long>(n_in), z->dTaps, z->dRot, z->dRotOff,
        z->dTw, z->Lin, z->U, z->D, z->P, ch_first, ch_count, m_base, z->inCount, n_out, out, out_stride_samples);
  } else {
    static fmgpu::DeviceOnce attrs;
    attrs.run([] { return cudaFuncSetAttribute(k_channelize<Pair>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); });
    // U phase classes of ceil(n_out / U) instants at most, TM instants per CTA
    const long groups = ((n_out + z->U - 1) / z->U + TM - 1) / TM;
    dim3 grid(static_cast<unsigned>(groups * z->U), static_cast<unsigned>((ch_count + 31) / 32), nCap);
    k_channelize<Pair><<<grid, 32 * WARPS, smem, s>>>(
        iq_dev, iq_stride_bytes, z->dHist, z->histValid, static_cast<long>(n_in), z->dW, z->dNuD, z->Lin, z->U, z->D,
        z->Cpad, ch_first, ch_count, m_base, z->inCount, n_out, static_cast<int>(groups), out, out_stride_samples);
  }
  const int H = z->Lin - 1;
  k_chan_carry<Carry><<<nCap, 512, static_cast<size_t>(H) * sizeof(Carry), s>>>(z->dHist, iq_dev, iq_stride_bytes,
                                                                               static_cast<long>(n_in), H);
}

// The one constructor: output rate wide_rate * U / D (create_format: U = 1, D = its decimation).
int createBank(int device, int sample_format, int n_captures, int wide_rate, int U, int decimation,
                      int n_channels, const double *first_center_hz, double spacing_hz, int taps_per_phase,
                      double cutoff_hz, float atten_db, fmgpu_channelizer **out) {
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
  z->U = U;
  z->D = decimation;
  z->C = n_channels;
  z->Cpad = (n_channels + 31) / 32 * 32;
  z->L = decimation * taps_per_phase;
  z->Lin = (z->L + U - 1) / U;
  z->spacingHz = spacing_hz;
  const size_t nCap = static_cast<size_t>(n_captures);
  std::vector<float2> W, rotTab, twTab;
  std::vector<float> phaseTaps;
  std::vector<double> nuD;
  std::vector<int> rotOff;
  try {
    // designed at rate U * wide_rate; the gain 2 fc U is unity in the pass band after the U-fold
    // zero stuffing the definition implies
    const float fc = static_cast<float>(cutoff_hz / (static_cast<double>(wide_rate) * U));
    z->taps = fmdesign::kaiserLowpass(static_cast<unsigned>(z->L), fc, atten_db, 0.0f);
    for (float &t : z->taps) {
      t *= 2.0f * fc * static_cast<float>(U);
    }
    // phase tables g_q[i] = h[q + iU], [U][Lin], zero past h's end
    phaseTaps.assign(static_cast<size_t>(U) * z->Lin, 0.0f);
    for (int n = 0; n < z->L; n++) {
      phaseTaps[static_cast<size_t>(n % U) * z->Lin + n / U] = z->taps[n];
    }
    const size_t wRow = static_cast<size_t>(U) * z->Lin * z->Cpad;
    W.assign(nCap * wRow, make_float2(0.0f, 0.0f));
    nuD.assign(nCap * z->Cpad, 0.0);
    for (size_t w = 0; w < nCap; w++) {
      for (int k = 0; k < z->C; k++) {
        const double nu = (first_center_hz[w] + spacing_hz * k) / static_cast<double>(wide_rate);
        const double adv = (U == 1) ? nu * static_cast<double>(decimation) : nu;
        nuD[w * z->Cpad + k] = adv - std::floor(adv);
        for (size_t qi = 0; qi < static_cast<size_t>(U) * z->Lin; qi++) {
          // W_q[i][k] = g_q[i] exp(+j 2 pi nu_k i)
          const double turns = nu * static_cast<double>(qi % z->Lin);
          const double ph = 2.0 * M_PI * (turns - std::floor(turns));
          W[w * wRow + qi * z->Cpad + k] = make_float2(static_cast<float>(phaseTaps[qi] * std::cos(ph)),
                                                       static_cast<float>(phaseTaps[qi] * std::sin(ph)));
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
    ok = ok && fmgpu::devAlloc(&z->dTaps, phaseTaps.size()) == cudaSuccess;
    ok = ok && fmgpu::devAlloc(&z->dRot, rotTab.size()) == cudaSuccess;
    ok = ok && fmgpu::devAlloc(&z->dRotOff, rotOff.size()) == cudaSuccess;
    ok = ok && fmgpu::devAlloc(&z->dTw, twTab.size()) == cudaSuccess;
    ok = ok && cudaMemcpy(z->dTaps, phaseTaps.data(), phaseTaps.size() * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemcpy(z->dRot, rotTab.data(), rotTab.size() * sizeof(float2), cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemcpy(z->dRotOff, rotOff.data(), rotOff.size() * sizeof(int), cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemcpy(z->dTw, twTab.data(), twTab.size() * sizeof(float2), cudaMemcpyHostToDevice) == cudaSuccess;
  }
  ok = ok && fmgpu::devAlloc(&z->dW, W.size()) == cudaSuccess;
  ok = ok && fmgpu::devAlloc(&z->dNuD, nuD.size()) == cudaSuccess;
  // the input before the first call is ZERO: no uint8 pair maps to 0.0, so for every format the
  // kernel clears the part of the window older than histValid samples
  ok = ok && fmgpu::devAlloc(&z->dHist, nCap * z->pairBytes * static_cast<size_t>(z->Lin - 1)) == cudaSuccess;
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
  return createBank(device, sample_format, n_captures, wide_rate, 1, decimation, n_channels, first_center_hz,
                    spacing_hz, taps_per_phase, cutoff_hz, atten_db, out);
}

int fmgpu_channelizer_create_rate(int device, int sample_format, int n_captures, int wide_rate,
                                  int output_rate, int n_channels, const double *first_center_hz,
                                  double spacing_hz, int taps_per_phase, double cutoff_hz, float atten_db,
                                  fmgpu_channelizer **out) {
  if (output_rate < 1 || output_rate > wide_rate) {
    return FMGPU_EINVAL;
  }
  const int g = std::gcd(output_rate, wide_rate);
  if (output_rate / g > kMaxInterpolation) {
    return FMGPU_EINVAL;
  }
  return createBank(device, sample_format, n_captures, wide_rate, output_rate / g, wide_rate / g, n_channels,
                    first_center_hz, spacing_hz, taps_per_phase, cutoff_hz, atten_db, out);
}

void fmgpu_channelizer_destroy(fmgpu_channelizer *z) {
  if (!z) {
    return;
  }
  cudaSetDevice(z->device);
  cudaDeviceSynchronize();
  delete z;  // the handles free the device buffers
}

int fmgpu_channelizer_output_rate(const fmgpu_channelizer *z) {
  return z ? static_cast<int>(static_cast<long long>(z->wideRate) * z->U / z->D) : 0;
}

int fmgpu_channelizer_interpolation(const fmgpu_channelizer *z) { return z ? z->U : 0; }

int fmgpu_channelizer_decimation(const fmgpu_channelizer *z) { return z ? z->D : 0; }

int fmgpu_channelizer_n_captures(const fmgpu_channelizer *z) { return z ? z->nCap : 0; }

int fmgpu_channelizer_sample_format(const fmgpu_channelizer *z) { return z ? z->format : FMGPU_EINVAL; }

size_t fmgpu_channelizer_outputs(const fmgpu_channelizer *z, size_t n_in) {
  if (!z) {
    return 0;
  }
  return static_cast<size_t>(outputsAfter(z, z->inCount + n_in) - outputsAfter(z, z->inCount));
}

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
  if (z && (z->U != 1 || n_in % static_cast<size_t>(z->D) != 0)) {
    return FMGPU_EINVAL;
  }
  return fmgpu_channelizer_process_stream(z, iq_dev, iq_stride_bytes, n_in, ch_first, ch_count, out_cf32_dev,
                                          out_stride_samples, nullptr, stream);
}

int fmgpu_channelizer_process_stream(fmgpu_channelizer *z, const void *iq_dev, size_t iq_stride_bytes,
                                     size_t n_in, int ch_first, int ch_count, float *out_cf32_dev,
                                     size_t out_stride_samples, size_t *n_out, void *stream) {
  if (!z || !iq_dev || !out_cf32_dev || n_in == 0) {
    return FMGPU_EINVAL;
  }
  const size_t outs = fmgpu_channelizer_outputs(z, n_in);
  const size_t pb = static_cast<size_t>(z->pairBytes);
  if (iq_stride_bytes % pb != 0 || iq_stride_bytes < pb * n_in ||
      reinterpret_cast<uintptr_t>(iq_dev) % pb != 0 ||
      ch_first < 0 || ch_count < 1 || ch_first + ch_count > z->C ||
      out_stride_samples < outs) {
    return FMGPU_EINVAL;
  }
  if (cudaSetDevice(z->device) != cudaSuccess) {
    return FMGPU_ENODEV;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t smem = static_cast<size_t>((TM - 1) * z->D + z->Lin) * sizeof(float2);
  if (smem > 200 * 1024) {
    z->lastError = "channelizer: filter too long for the shared-memory tile";
    return FMGPU_ERANGE;
  }
  // the polyphase tile spans s_m0 - (Lin-1) .. s_m0+31, at most ceil(31 D / U) + Lin samples
  const size_t pp_tile = static_cast<size_t>(((PP_TM - 1) * static_cast<long>(z->D) + z->U - 1) / z->U + z->Lin);
  const size_t pp_smem = (pp_tile + static_cast<size_t>(z->P) * (PP_TM + 1) + static_cast<size_t>(z->P)) * sizeof(float2) +
                         static_cast<size_t>(z->U) * z->Lin * sizeof(float);
  const uint8_t *iq = static_cast<const uint8_t *>(iq_dev);
  float2 *out = reinterpret_cast<float2 *>(out_cf32_dev);
  const long nOut = static_cast<long>(outs);
  switch (z->format) {
    case FMGPU_IQ_CU8:
      launchChannelize<uchar2, uchar2>(z, iq, iq_stride_bytes, n_in, ch_first, ch_count, out, out_stride_samples,
                                       nOut, smem, pp_smem, s);
      break;
    case FMGPU_IQ_CS8:
      launchChannelize<char2, uchar2>(z, iq, iq_stride_bytes, n_in, ch_first, ch_count, out, out_stride_samples,
                                      nOut, smem, pp_smem, s);
      break;
    default:  // FMGPU_IQ_CS16: create accepts no other format
      launchChannelize<short2, short2>(z, iq, iq_stride_bytes, n_in, ch_first, ch_count, out, out_stride_samples,
                                       nOut, smem, pp_smem, s);
      break;
  }
  z->inCount += n_in;
  z->histValid = std::min<long>(z->Lin - 1, z->histValid + static_cast<long>(n_in));
  if (n_out) {
    *n_out = outs;
  }
  return cudaGetLastError() == cudaSuccess ? FMGPU_OK : FMGPU_ENODEV;
}

}  // extern "C"
