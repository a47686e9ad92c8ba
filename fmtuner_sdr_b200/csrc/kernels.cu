// kernels.cu — sm_100a kernels of the FM stereo + RDS engine.
//
// Two kinds of kernels:
//  * "tile" kernels: the FIRs and element-wise stages. One CTA per (tile of
//    outputs, channel); inputs staged in shared memory with their halo, outputs
//    register-tiled so every FFMA has one shared-memory operand at most. Dot
//    products are ONE accumulator per output, oldest sample first, fused
//    multiply-add — the order the CPU oracle uses — so results are bit-identical.
//  * "lane" kernels: the serial recursions (DC blockers, AGC, 19 kHz pilot PLL
//    and blend, de-emphasis, the whole RDS demodulator and block synchroniser).
//    One lane per channel, state in registers, one warp per CTA so channels
//    spread over all SMs.
// Compiled with -fmad=false: only explicit fmaf() fuses.
#include "kernels.h"
#include "device_once.h"

#include <type_traits>

#include <algorithm>
#include <cstdlib>

#include "fm_math.h"

namespace fmgpu {

// ---------------------------------------------------------------------------
// constant tables of the RDS (26,16) code, filled by initRdsTables()
// ---------------------------------------------------------------------------
__constant__ uint32_t c_syn_mask[10];   // syndrome bit r = parity(word & c_syn_mask[r])
__constant__ uint32_t c_err_syn[52];    // syndromes of the correctable error bursts
__constant__ uint32_t c_err_vec[52];    // the bursts themselves (1-bit then 2-bit, shift 0..25)
__constant__ uint32_t c_off_word[5];    // offset words A, B, C, C', D

namespace {

const uint32_t kParity[26] = {
    0b1000000000, 0b0100000000, 0b0010000000, 0b0001000000, 0b0000100000, 0b0000010000,
    0b0000001000, 0b0000000100, 0b0000000010, 0b0000000001, 0b1011011100, 0b0101101110,
    0b0010110111, 0b1010000111, 0b1110011111, 0b1100010011, 0b1101010101, 0b1101110110,
    0b0110111011, 0b1000000001, 0b1111011100, 0b0111101110, 0b0011110111, 0b1010100111,
    0b1110001111, 0b1100011011};

uint32_t hostSyndrome(uint32_t v) {
  uint32_t r = 0;
  for (int k = 0; k < 26; k++) {
    if ((v >> k) & 1u) {
      r ^= kParity[25 - k];
    }
  }
  return r;
}

}  // namespace

cudaError_t initRdsTables() {
  uint32_t mask[10];
  for (int r = 0; r < 10; r++) {
    mask[r] = 0;
    for (int k = 0; k < 26; k++) {
      if ((kParity[25 - k] >> r) & 1u) {
        mask[r] |= (1u << k);
      }
    }
  }
  uint32_t esyn[52], evec[52];
  int n = 0;
  for (uint32_t eb : {1u, 3u}) {
    for (uint32_t sh = 0; sh < 26; sh++) {
      evec[n] = (eb << sh) & 0x3ffffffu;
      esyn[n] = hostSyndrome(evec[n]);
      n++;
    }
  }
  const uint32_t offw[5] = {0b0011111100, 0b0110011000, 0b0101101000, 0b1101010000, 0b0110110100};
  cudaError_t e;
  if ((e = cudaMemcpyToSymbol(c_syn_mask, mask, sizeof(mask))) != cudaSuccess) return e;
  if ((e = cudaMemcpyToSymbol(c_err_syn, esyn, sizeof(esyn))) != cudaSuccess) return e;
  if ((e = cudaMemcpyToSymbol(c_err_vec, evec, sizeof(evec))) != cudaSuccess) return e;
  return cudaMemcpyToSymbol(c_off_word, offw, sizeof(offw));
}

// ---------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------
// liquid's nco_crcf goes through double twice: constrain() evaluates (float)((double)theta / 2pi)
// and get_phase() (float)(2pi * (double)(float)theta / 2^32). A float -> double -> float round trip
// costs ~46 cycles of the PLL's serial chain on B200 (F2F pair 38, DMUL 8; r01 latency microbench).
// Both products are evaluated here in float as a two-term product with the exact error of the
// leading term (p = x*hi; e = fma(x, hi, -p); p + fma(x, lo, e)), which is bit-identical:
// tools/nco_float_form_proof.cpp compares EVERY input — all 3.19e9 finite floats below 2^63 for the
// resulting uint32 of constrain(), all 83,886,081 possible (float)theta for the phase — with the
// double form: 0 mismatches (profiles/r02_nco_float_form_proof.txt).
__device__ __forceinline__ uint32_t ncoConstrainDev(float theta) {
  constexpr float kHi = 0x1.45f306p-3f;   // (float)(1 / 2pi), 0.159154943091895 as liquid writes it
  constexpr float kLo = 0x1.b9390ep-28f;  // (float)(0.159154943091895 - kHi)
  const float p0 = __fmul_rn(theta, kHi);
  const float e = __fmaf_rn(theta, kHi, -p0);
  const float p = __fadd_rn(p0, __fmaf_rn(theta, kLo, e));
  float fpart = p - truncf(p);  // == p - (float)(long)p for every |p| < 2^63
  if (fpart < 0.0f) {
    fpart = fpart + 1.0f;
  }
  const float scaled = fpart * 4294967296.0f;  // in [0, 2^32]
  // (uint32_t)(uint64_t)scaled: 2^32 wraps to 0, everything else fits 32 bits
  return (scaled >= 4294967296.0f) ? 0u : __float2uint_rz(scaled);
}

__device__ __forceinline__ float ncoPhaseDev(uint32_t theta) {
  constexpr float kHi = (float)(6.283185307179586 / 4294967296.0);
  constexpr float kLo = (float)(6.283185307179586 / 4294967296.0 - (double)kHi);
  const float t = __uint2float_rn(theta);
  const float p0 = __fmul_rn(t, kHi);
  const float e = __fmaf_rn(t, kHi, -p0);
  return __fadd_rn(p0, __fmaf_rn(t, kLo, e));
}

__device__ __forceinline__ float unwrapDev(float p) {
  // branch-free (the if / else form compiled to a BSSY / BRA / BSYNC region per call, fourteen of
  // them per sample group of k_rds); same values: each candidate is one IEEE addition
  const float kPi = 3.14159265358979323846f;
  const float k2Pi = 2.f * kPi;
  const float down = p - k2Pi;
  const float up = p + k2Pi;
  return (p > kPi) ? down : ((p < -kPi) ? up : p);
}

// a / 57000 without the IEEE-division sequence (its slow-path call sits in a BSSY / BRA / BSYNC
// region: seven of them per sample group of k_rds): q = a y, r = fma(-q, c, a), q + r y with
// y = RN(1 / c). Bit-identical to a / 57000.f for every finite float except |a| <= 9.39e-38 and -0
// (tools/div_const_proof.cpp compares all 4.28e9 of them); its argument here is 57000 x a difference
// of two NCO phases ((float)uint32 * 2 pi / 2^32): +0 or >= 5.7e-12 in magnitude.
__device__ __forceinline__ float divBy57000(float a) {
  constexpr float c = 57000.0f;
  constexpr float y = 1.0f / c;
  const float q = __fmul_rn(a, y);
  const float r = __fmaf_rn(-q, c, a);
  return __fmaf_rn(r, y, q);
}

// Packed FP32 FMA of sm_100 (fma.rn.f32x2 -> FFMA2): acc.x = fma(h, x.x, acc.x) and
// acc.y = fma(h, x.y, acc.y) in ONE instruction, each half an IEEE round-to-nearest fma, so the
// result is bit-identical to two fmaf() calls. ptxas folds the {h, h} pair into a scalar
// (uniform-register) operand. The FIR kernels are issue-bound (ncu r01: 83 % of issue slots,
// FMA pipe 50 %): halving the FMA instruction count frees the slots for the LDS / LDCU traffic.
__device__ __forceinline__ float2 fma2(float h, float2 x, float2 acc) {
  unsigned long long hh, xx, aa, r;
  asm("mov.b64 %0, {%1, %1};" : "=l"(hh) : "f"(h));
  asm("mov.b64 %0, {%1, %2};" : "=l"(xx) : "f"(x.x), "f"(x.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(aa) : "f"(acc.x), "f"(acc.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(hh), "l"(xx), "l"(aa));
  float2 o;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(o.x), "=f"(o.y) : "l"(r));
  return o;
}

// One uint8 IQ pair (I in byte 0, Q in byte 1) -> ((float)byte - 127.5f) * (1 / 127.5f), the
// conversion of ComplexDecimator::executeComplex (liquid_primitives.cpp:480-484), without the
// int->float converter: PRMT builds the bits 0x47000000 | byte << 8 = 32768 + byte exactly, one
// exact subtraction of 32895.5 leaves byte - 127.5 (a 9-bit number), and the single rounding is the
// final multiplication, as in the scalar formula. Both halves go through the packed f32x2 ALU ops.
__device__ __forceinline__ float2 iqBytesToFloat(uint32_t w) {
  const float vi = __uint_as_float(__byte_perm(w, 0x47000000u, 0x7404));
  const float vq = __uint_as_float(__byte_perm(w, 0x47000000u, 0x7414));
  constexpr float kScale = 1.0f / 127.5f;
  unsigned long long v, r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(vi), "f"(vq));
  asm("{\n\t.reg .b64 c, k;\n\t"
      "mov.b64 c, {%2, %2};\n\t"
      "mov.b64 k, {%3, %3};\n\t"
      "add.rn.f32x2 %0, %1, c;\n\t"
      "mul.rn.f32x2 %0, %0, k;\n\t}"
      : "=l"(r)
      : "l"(v), "f"(-32895.5f), "f"(kScale));
  float2 o;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(o.x), "=f"(o.y) : "l"(r));
  return o;
}

// ---------------------------------------------------------------------------
// warp tiles for the lane kernels. A lane kernel walks one channel per lane, so a
// warp touches 32 rows of a [C][time] buffer at once; reading them lane-by-lane is
// 32 cache lines per instruction. Instead the warp moves a [32 rows][LT samples]
// tile between global and shared memory cooperatively (each instruction covers 128
// contiguous bytes of ONE row; loads are cp.async so the next tile streams in while
// the current one is processed) and every lane then reads its own row from shared
// memory, four samples per 128-bit access: row pitches are multiples of 4 floats, so rows move as
// 16-byte transfers and a warp's 128-bit row access is conflict-free (32-bit accesses of the same
// rows hit only 8 banks).
// ---------------------------------------------------------------------------
// samples per tile row of the lane kernels (LT: k_dcblock, k_agc, k_rds; ST: k_stereo). Measured:
// the shared memory the lane kernels hold does not move the 10,000-channel step (DESIGN.md 4a);
// shorter k_stereo tiles lengthen that kernel by 10 % (one block barrier per tile).
constexpr int LT = 32;
constexpr int STEREO_ST = 16;

__device__ __forceinline__ void cpAsync16(void *smem, const void *gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(
                   (uint32_t)__cvta_generic_to_shared(smem)),
               "l"(gmem)
               : "memory");
}
__device__ __forceinline__ void cpAsyncCommit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N> __device__ __forceinline__ void cpAsyncWait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}
// 128-bit shared-memory accesses through a 32-bit shared-window address computed ONCE: through a
// generic float* the compiler re-derives the CTA's shared window base (S2UR SR_CgaCtaId + ULEA) in
// front of the accesses of every loop iteration — ~20 % of the PLL warp's time in k_stereo.
__device__ __forceinline__ uint32_t sharedAddr(const void *p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ float4 ldsF4(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void stsF4(uint32_t a, const float4 &v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// tile[r][k] <- base[(c0 + r) * pitch + start + k],  r < nrows, k < len, as 16-byte
// cp.async transfers: start, pitch and the row pitch TP are multiples of 4 floats; len is
// rounded up to 4 (the over-read stays inside the row's padding). One warp.
// FULL > 0: the row length of a full tile, known at compile time (its index arithmetic is shifts;
// the generic form divides by a run-time row length, ~25 instructions per transfer, which was half
// of the instructions k_dcblock executed)
template <int TP, int FULL = 0>
__device__ __forceinline__ void tileLoadAsync(float *tile, const float *base, size_t pitch, int c0,
                                              int nrows, long start, int len, int lane) {
  if (FULL > 0 && len == FULL) {
    constexpr int cpr = (FULL + 3) / 4;
    const int total = nrows * cpr;
#pragma unroll 4
    for (int idx = lane; idx < total; idx += 32) {
      const int r = idx / cpr;
      const int q = idx - r * cpr;
      cpAsync16(tile + r * TP + 4 * q, base + (size_t)(c0 + r) * pitch + start + 4 * q);
    }
    return;
  }
  const int cpr = (len + 3) >> 2;  // 16-byte chunks per row
  const int total = nrows * cpr;
  for (int idx = lane; idx < total; idx += 32) {
    const int r = idx / cpr;
    const int q = idx - r * cpr;
    cpAsync16(tile + r * TP + 4 * q, base + (size_t)(c0 + r) * pitch + start + 4 * q);
  }
}

__device__ __forceinline__ void cpAsync4(void *smem, const void *gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(
                   (uint32_t)__cvta_generic_to_shared(smem)),
               "l"(gmem)
               : "memory");
}

// same tile, element by element (4-byte cp.async): for a global start that is not 16-byte aligned
// (the delayed MPX of the stereo matrix), so that the tile still lands aligned in shared memory
template <int TP, int LEN>
__device__ __forceinline__ void tileLoadAsync4(float *tile, const float *base, size_t pitch, int c0,
                                               int nrows, long start, int len, int lane) {
  const int total = nrows * LEN;
  for (int idx = lane; idx < total; idx += 32) {
    const int r = idx / LEN;
    const int q = idx - r * LEN;
    if (q < len) {
      cpAsync4(tile + r * TP + q, base + (size_t)(c0 + r) * pitch + start + q);
    }
  }
}

template <int TP, int FULL = 0>
__device__ __forceinline__ void tileStore(const float *tile, float *base, size_t pitch, int c0,
                                          int nrows, long start, int len, int lane) {
  if (FULL > 0 && len == FULL) {
    constexpr int cpr = (FULL + 3) / 4;
    const int total = nrows * cpr;
#pragma unroll 4
    for (int idx = lane; idx < total; idx += 32) {
      const int r = idx / cpr;
      const int q = idx - r * cpr;
      const float4 v = *reinterpret_cast<const float4 *>(tile + r * TP + 4 * q);
      *reinterpret_cast<float4 *>(base + (size_t)(c0 + r) * pitch + start + 4 * q) = v;
    }
    return;
  }
  const int cpr = (len + 3) >> 2;
  const int total = nrows * cpr;
  for (int idx = lane; idx < total; idx += 32) {
    const int r = idx / cpr;
    const int q = idx - r * cpr;
    const float4 v = *reinterpret_cast<const float4 *>(tile + r * TP + 4 * q);
    *reinterpret_cast<float4 *>(base + (size_t)(c0 + r) * pitch + start + 4 * q) = v;
  }
}

// The same tile movers on a 32-bit shared-window byte address (see sharedAddr): no generic -> shared
// conversion per transfer.
__device__ __forceinline__ void cpAsync16S(uint32_t saddr, const void *gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(saddr), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cpAsync4S(uint32_t saddr, const void *gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(saddr), "l"(gmem) : "memory");
}
template <int TP, int FULL>
__device__ __forceinline__ void tileLoadAsyncS(uint32_t tile, const float *base, size_t pitch, int c0,
                                               int nrows, long start, int len, int lane) {
  if (len == FULL) {
    constexpr int cpr = (FULL + 3) / 4;
    const int total = nrows * cpr;
#pragma unroll 4
    for (int idx = lane; idx < total; idx += 32) {
      const int r = idx / cpr;
      const int q = idx - r * cpr;
      cpAsync16S(tile + 4u * (r * TP + 4 * q), base + (size_t)(c0 + r) * pitch + start + 4 * q);
    }
    return;
  }
  const int cpr = (len + 3) >> 2;  // 16-byte chunks per row
  const int total = nrows * cpr;
  for (int idx = lane; idx < total; idx += 32) {
    const int r = idx / cpr;
    const int q = idx - r * cpr;
    cpAsync16S(tile + 4u * (r * TP + 4 * q), base + (size_t)(c0 + r) * pitch + start + 4 * q);
  }
}
template <int TP, int LEN>
__device__ __forceinline__ void tileLoadAsync4S(uint32_t tile, const float *base, size_t pitch, int c0,
                                                int nrows, long start, int len, int lane) {
  const int total = nrows * LEN;
  for (int idx = lane; idx < total; idx += 32) {
    const int r = idx / LEN;
    const int q = idx - r * LEN;
    if (q < len) {
      cpAsync4S(tile + 4u * (r * TP + q), base + (size_t)(c0 + r) * pitch + start + q);
    }
  }
}
template <int TP, int FULL>
__device__ __forceinline__ void tileStoreS(uint32_t tile, float *base, size_t pitch, int c0, int nrows,
                                           long start, int len, int lane) {
  const int cpr = (len == FULL) ? (FULL + 3) / 4 : (len + 3) >> 2;
  const int total = nrows * cpr;
  for (int idx = lane; idx < total; idx += 32) {
    const int r = idx / cpr;
    const int q = idx - r * cpr;
    const float4 v = ldsF4(tile + 4u * (r * TP + 4 * q));
    *reinterpret_cast<float4 *>(base + (size_t)(c0 + r) * pitch + start + 4 * q) = v;
  }
}

// ---------------------------------------------------------------------------
// history carry: buf[c][0..H) <- buf[c][n..n+H)   (the last H samples of hist ++ new)
// ---------------------------------------------------------------------------
template <typename T>
__global__ void k_carry(T *buf, size_t pitch, int H, size_t n, int ch0) {
  T *row = buf + (size_t)(blockIdx.x + ch0) * pitch;
  const int e = threadIdx.x;
  T v{};
  if (e < H) {
    v = row[n + e];
  }
  __syncthreads();
  if (e < H) {
    row[e] = v;
  }
}

// IQ history: hist[c] <- last H_IQ samples of (hist[c] ++ in[c][0..n_in))
__global__ void k_carry_iq(uchar2 *hist, int *hist_valid, const uint8_t *iq, size_t iq_stride,
                           long n_in, int ch0) {
  const int c = blockIdx.x + ch0;
  if (threadIdx.x == 0) {
    // samples older than `valid` are the zero-initialised window of a fresh firdecim
    hist_valid[c] = (int)min((long)H_IQ, (long)hist_valid[c] + n_in);
  }
  uchar2 *h = hist + (size_t)c * H_IQ;
  const uchar2 *in = reinterpret_cast<const uchar2 *>(iq + (size_t)c * iq_stride);
  const int e = threadIdx.x;  // blockDim == H_IQ
  const long src = n_in - H_IQ + e;
  const uchar2 v = (src >= 0) ? in[src] : h[e + n_in];
  __syncthreads();
  h[e] = v;
}

// hist[c][0..H) <- last H samples of (hist[c] ++ src[c][src_off .. src_off+n)); H <= 32.
// Used for windows that belong to a stage other than the owner of the buffer's own
// halo (RDS resampler and FMDemod mono resampler both read the MPX buffer).
__global__ void k_save_tail(const float *src, size_t src_pitch, int src_off, float *hist,
                            int hist_pitch, int H, long n, int ch0) {
  const int c = blockIdx.x + ch0;
  const int e = threadIdx.x;
  float v = 0.0f;
  if (e < H) {
    const long si = n - H + e;
    v = (si >= 0) ? src[(size_t)c * src_pitch + src_off + si] : hist[(size_t)c * hist_pitch + e + n];
  }
  __syncthreads();
  if (e < H) {
    hist[(size_t)c * hist_pitch + e] = v;
  }
}

// ---------------------------------------------------------------------------
// K1: uint8 IQ -> float, polyphase-ordered decimating FIR (firdecim_crcf)
//   y[n] = scale * sum_i hrev[i] * x[n*M - (L-1) + i]      (newest sample = n*M)
// Taps are front-padded with zeros to Pp*M (Pp multiple of 4). 128 threads x 4
// consecutive outputs; the tile (converted to float2) sits in shared memory with a
// one-word skew per 4*M samples so the per-thread stride is odd (no bank conflicts).
// Input bytes are fetched as 128-bit words from the 16-byte aligned virtual stream
// hist ++ input.
// ---------------------------------------------------------------------------
// loads in flight per thread while the tile is filled (the fill is global-latency-bound)
constexpr int DECIM_FILL_UNROLL = 7;
constexpr int DECIM_NT = 128;  // threads per decimator CTA (4 outputs each)

template <int M>
__global__ void __launch_bounds__(DECIM_NT)
k_decim(const uint8_t *__restrict__ iq, size_t iq_stride, const uint8_t *__restrict__ hist,
        const int *__restrict__ hist_valid, float2 *__restrict__ x1, size_t x1_pitch, int n_out,
        int ch0, int Pp, float scale, const __grid_constant__ TapsParam taps) {
  constexpr int R = 4;
  constexpr int T = DECIM_NT * R;
  constexpr int RM = R * M;
  // skew elements per RM samples: the per-thread stride RM + SK must be odd in units of the access
  // size — 8-byte reads for odd M, 16-byte reads (two samples each) for even M
  constexpr int SK = (M % 2 == 0) ? 2 : 1;
  extern __shared__ float2 xs[];
  const int c = blockIdx.y + ch0;
  const int n0 = blockIdx.x * T;
  const int t = threadIdx.x;
  const long o = (long)(n0 - Pp) * M + 1;  // stream index of tile element 0
  const int tile_len = (T + Pp - 1) * M;
  const long v0 = o + H_IQ;                // virtual index (history first)
  const long n_in = (long)n_out * M;
  const unsigned short *in_c = reinterpret_cast<const unsigned short *>(iq + (size_t)c * iq_stride);
  const unsigned short *hist_c = reinterpret_cast<const unsigned short *>(hist) + (size_t)c * H_IQ;
  const long v_first_valid = H_IQ - hist_valid[c];

  // Tile fill: the lanes of a warp take CONSECUTIVE samples (one 16-bit load each), so every
  // 64-bit store of the converted pair is bank-conflict free and the index arithmetic is three
  // adds per sample. (The earlier form converted the 8 samples of one 128-bit load per thread:
  // lane stride 64 B = 8-way conflicts on the stores — ncu r01: 13.7 M of the 20.6 M store
  // wavefronts were conflicts — and ~30 instructions per sample of bounds logic; the fill then
  // cost as many issue slots as the FMA loop.) Samples older than `valid` are the zero window of a
  // fresh firdecim; samples past the end of the input only feed outputs that are never stored.
  {
    // tile-relative bounds, so the loop itself is 32-bit: [a_lo, a_hi) holds real samples, elements
    // below a_hist come from the history buffer
    const int a_lo = (int)max(0L, min((long)tile_len, v_first_valid - v0));
    const int a_hi = (int)max(0L, min((long)tile_len, n_in + H_IQ - v0));
    const int a_hist = (int)max(0L, min((long)tile_len, (long)H_IQ - v0));
    const unsigned short *p_hist = hist_c + v0;
    const unsigned short *p_in = in_c + (v0 - H_IQ);
    auto fill = [&](auto fast_tag) {
      constexpr bool FAST = decltype(fast_tag)::value;  // whole tile inside the input row
#pragma unroll DECIM_FILL_UNROLL
      for (unsigned a = t; a < (unsigned)tile_len; a += DECIM_NT) {
        uint32_t w = 0;
        bool ok = true;
        if (FAST) {
          w = __ldg(p_in + a);
        } else {
          ok = ((int)a >= a_lo) && ((int)a < a_hi);
          if (ok) {
            w = __ldg((((int)a < a_hist) ? p_hist : p_in) + a);
          }
        }
        float2 f = iqBytesToFloat(w);
        if (!FAST && !ok) {
          f = make_float2(0.0f, 0.0f);
        }
        xs[a + SK * (a / RM)] = f;
      }
    };
    if (a_lo == 0 && a_hist == 0 && a_hi == tile_len) {
      if (M % 2 == 0) {
        // even M: tile_len, RM and the skew are even, so elements (a, a + 1), a even, are one
        // 16-byte aligned pair in shared memory: two 16-bit loads, one 128-bit store per lane
#pragma unroll DECIM_FILL_UNROLL
        for (unsigned a = 2 * t; a < (unsigned)tile_len; a += 2 * DECIM_NT) {
          const float2 f0 = iqBytesToFloat(__ldg(p_in + a));
          const float2 f1 = iqBytesToFloat(__ldg(p_in + a + 1));
          *reinterpret_cast<float4 *>(xs + a + SK * (a / RM)) = make_float4(f0.x, f0.y, f1.x, f1.y);
        }
      } else {
        fill(std::true_type{});
      }
    } else {
      fill(std::false_type{});
    }
  }
  __syncthreads();

  float2 acc[R];
#pragma unroll
  for (int j = 0; j < R; j++) {
    acc[j] = make_float2(0.0f, 0.0f);
  }
  float2 seg[R][M];
  const int tbase = t * (RM + SK);
  auto loadSeg = [&](float2 *dst, int at) {  // M consecutive samples from element `at`
    if (M % 2 == 0) {
#pragma unroll
      for (int r = 0; r < M; r += 2) {
        const float4 v = *reinterpret_cast<const float4 *>(xs + at + r);
        dst[r] = make_float2(v.x, v.y);
        dst[r + 1] = make_float2(v.z, v.w);
      }
    } else {
#pragma unroll
      for (int r = 0; r < M; r++) {
        dst[r] = xs[at + r];
      }
    }
  };
#pragma unroll
  for (int u = 0; u < 3; u++) {
    loadSeg(seg[u], tbase + u * M);  // u < 4: no skew element yet
  }
  for (int pp = 0; pp < Pp; pp += 4) {
#pragma unroll
    for (int ps = 0; ps < 4; ps++) {
      const int u = pp + ps + 3;
      loadSeg(seg[(ps + 3) & 3], tbase + u * M + SK * (u >> 2));
#pragma unroll
      for (int r = 0; r < M; r++) {
        const float h = taps.h[(pp + ps) * M + r];
#pragma unroll
        for (int j = 0; j < R; j++) {
          acc[j] = fma2(h, seg[(j + ps) & 3][r], acc[j]);
        }
      }
    }
  }
  float2 *out = x1 + (size_t)c * x1_pitch;
#pragma unroll
  for (int j = 0; j < R; j++) {
    const int n = n0 + R * t + j;
    if (n < n_out) {
      out[n] = make_float2(acc[j].x * scale, acc[j].y * scale);
    }
  }
}

// ---------------------------------------------------------------------------
// generic fallback for decimation factors without an instantiation
__global__ void k_decim_generic(const uint8_t *__restrict__ iq, size_t iq_stride,
                                const uint8_t *__restrict__ hist,
                                const int *__restrict__ hist_valid, float2 *__restrict__ x1,
                                size_t x1_pitch, int n_out, int ch0, int M, int L, float scale,
                                const __grid_constant__ TapsParam taps) {
  const int c = blockIdx.y + ch0;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_out) {
    return;
  }
  const uchar2 *in_c = reinterpret_cast<const uchar2 *>(iq + (size_t)c * iq_stride);
  const uchar2 *hist_c = reinterpret_cast<const uchar2 *>(hist + (size_t)c * (2 * H_IQ));
  constexpr float kScale = 1.0f / 127.5f;
  float ar = 0.0f, ai = 0.0f;
  for (int i = 0; i < L; i++) {
    const long s = (long)n * M - (L - 1) + i;
    const uchar2 b = (s >= 0) ? in_c[s] : hist_c[H_IQ + s];
    float fi = ((float)b.x - 127.5f) * kScale;
    float fq = ((float)b.y - 127.5f) * kScale;
    if (s < -(long)hist_valid[c]) {
      fi = 0.0f;
      fq = 0.0f;
    }
    ar = fmaf(taps.h[i], fi, ar);
    ai = fmaf(taps.h[i], fq, ai);
  }
  x1[(size_t)c * x1_pitch + n] = make_float2(ar * scale, ai * scale);
}

// M == 1 through ComplexDecimator::executeComplex: a pure convert (liquid_primitives.cpp:468-478)
__global__ void k_convert_u8(const uint8_t *__restrict__ iq, size_t iq_stride,
                             float2 *__restrict__ x1, size_t x1_pitch, int n, int ch0) {
  const int c = blockIdx.y + ch0;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) {
    return;
  }
  constexpr float kScale = 1.0f / 127.5f;
  const uchar2 b = reinterpret_cast<const uchar2 *>(iq + (size_t)c * iq_stride)[i];
  x1[(size_t)c * x1_pitch + i] =
      make_float2(((float)b.x - 127.5f) * kScale, ((float)b.y - 127.5f) * kScale);
}

// ComplexDecimator::execute: the decimated sample back to uint8 (liquid_primitives.cpp:452-456):
// clamp(y * 127.5 + 127.5, 0, 255), truncated
__global__ void k_requant_u8(const float2 *__restrict__ x1, size_t x1_pitch, uint8_t *__restrict__ out,
                             size_t out_stride, int n, int ch0) {
  const int c = blockIdx.y + ch0;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) {
    return;
  }
  const float2 y = x1[(size_t)c * x1_pitch + i];
  const float vi = fminf(fmaxf(__fadd_rn(__fmul_rn(y.x, 127.5f), 127.5f), 0.0f), 255.0f);
  const float vq = fminf(fmaxf(__fadd_rn(__fmul_rn(y.y, 127.5f), 127.5f), 0.0f), 255.0f);
  reinterpret_cast<uchar2 *>(out + (size_t)c * out_stride)[i] =
      make_uchar2((unsigned char)vi, (unsigned char)vq);
}

// ---------------------------------------------------------------------------
// S1: I/Q DC blockers (iirfilt dc_blocker, alpha = 0.0005) + clip statistics.
// One lane per channel; fm_demod.cpp:150-208.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(32)
k_dcblock(const float2 *__restrict__ x1, size_t x1_pitch, const uint8_t *__restrict__ iq_u8,
          size_t iq_stride, float2 *__restrict__ x2, size_t x2_pitch, DemodState *st,
          fmgpu_block_status *status, int status_pitch, int n_total, int ch0, int nch, float a1) {
  // ONE warp per 32 channels, one lane per channel: the warp prefetches its next input tile
  // (cp.async), runs the recursions on the current one and writes the finished tile back itself.
  // (A separate mover warp doubles the registers and warp slots this kernel keeps from the FIR
  // kernels for as long as it runs.)
  constexpr int TP = 2 * LT + 4;  // interleaved re,im; 16-byte aligned rows
  extern __shared__ float sm_dc[];
  auto tin = [&](int k2) { return sm_dc + (k2 & 1) * (32 * TP); };
  float *tout = sm_dc + 2 * 32 * TP;
  const int lane = threadIdx.x;
  const int c0 = ch0 + blockIdx.x * 32;
  const int nrows = min(32, ch0 + nch - c0);
  const bool active = lane < nrows;
  const int c = c0 + min(lane, nrows - 1);
  DemodState s{};
  if (active) {
    s = st[c];
  }
  float vi = s.dc_i, vq = s.dc_q;
  const uchar2 *inb =
      (iq_u8 && active) ? reinterpret_cast<const uchar2 *>(iq_u8 + (size_t)c * iq_stride) : nullptr;
  const float *x1f = reinterpret_cast<const float *>(x1);
  float *x2f = reinterpret_cast<float *>(x2);
  const int nchunks = (n_total + LT - 1) / LT;
  if (!iq_u8 && nchunks > 0) {
    tileLoadAsync<TP, 2 * LT>(tin(0), x1f, 2 * x1_pitch, c0, nrows, 0, 2 * min(LT, n_total), lane);
    cpAsyncCommit();
  }
  int clip = 0;
  for (int ck = 0; ck < nchunks; ck++) {
    const int n0 = ck * LT;
    const int len = min(LT, n_total - n0);
    cpAsyncWait<0>();  // tile ck has landed ...
    __syncwarp();      // ... for every lane; every lane is done with tile ck - 1 and its output
    if (!iq_u8 && ck + 1 < nchunks) {
      tileLoadAsync<TP, 2 * LT>(tin(ck + 1), x1f, 2 * x1_pitch, c0, nrows, 2L * (n0 + LT),
                        2 * min(LT, n_total - n0 - LT), lane);
      cpAsyncCommit();
    }
    if (active) {
      const float *ti = tin(ck) + lane * TP;
      float *to = tout + lane * TP;
      int i = 0;
      if (inb) {
        for (; i < len; i++) {
          const uchar2 v = inb[n0 + i];
          if (v.x == 0 || v.x == 255 || v.y == 0 || v.y == 255) {
            clip++;
          }
          const float ir = ((float)v.x - 127.0f) / 127.5f;
          const float qr = ((float)v.y - 127.0f) / 127.5f;
          const float v0i = ir - (a1 * vi);
          to[2 * i] = v0i - vi;
          vi = v0i;
          const float v0q = qr - (a1 * vq);
          to[2 * i + 1] = v0q - vq;
          vq = v0q;
        }
      } else {
        auto sample = [&](float ir, float qr, float &o_i, float &o_q) {
          if (fabsf(ir) >= 0.995f || fabsf(qr) >= 0.995f) {
            clip++;
          }
          const float v0i = ir - (a1 * vi);
          o_i = v0i - vi;
          vi = v0i;
          const float v0q = qr - (a1 * vq);
          o_q = v0q - vq;
          vq = v0q;
        };
        // two complex samples per 128-bit shared-memory access (conflict-free; the 32-bit
        // form hits 8 banks)
#pragma unroll 2
        for (; i + 2 <= len; i += 2) {
          const float4 v = *reinterpret_cast<const float4 *>(ti + 2 * i);
          float4 o;
          sample(v.x, v.y, o.x, o.y);
          sample(v.z, v.w, o.z, o.w);
          *reinterpret_cast<float4 *>(to + 2 * i) = o;
        }
        for (; i < len; i++) {
          sample(ti[2 * i], ti[2 * i + 1], to[2 * i], to[2 * i + 1]);
        }
      }
    }
    __syncwarp();  // the output tile is complete: write it back, 128 contiguous bytes per row
    tileStore<TP, 2 * LT>(tout, x2f, 2 * x2_pitch, c0, nrows, 2L * (H_X2 + n0), 2 * len, lane);
  }
  if (active) {
    const float clip_ratio = (float)clip / (float)n_total;
    if (status) {
      status[(size_t)c * status_pitch].clip_ratio = clip_ratio;
    }
    // only this stage's fields: the AGC stage of the previous block may be running beside it
    st[c].dc_i = vi;
    st[c].dc_q = vq;
    st[c].clipping = (clip > 0) ? 1 : 0;
    st[c].clip_ratio = clip_ratio;
  }
}

// S1 as a warp-shuffle parallel scan (see k_audio_iir_scan): one WARP per channel, 32 complex
// samples per step, I and Q in one packed FMA. v0[j] = x[j] + r v0[j-1] with r = 1 - alpha is affine
// in the carried state, so five Kogge-Stone rounds (shfl_up + fma with r, r^2, ... r^16) give every
// lane its v0[j]; y[j] = v0[j] - v0[j-1]. Float input only (decimated IQ or the complex-float path),
// one logical block per launch. Fast arithmetic: agrees with k_dcblock to float rounding.
__global__ void __launch_bounds__(128)
k_dcblock_scan(const float2 *__restrict__ x1, size_t x1_pitch, float2 *__restrict__ x2, size_t x2_pitch,
               DemodState *st, fmgpu_block_status *status, int status_pitch, int n_total, int ch0,
               int nch, float a1) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (row >= nch) {
    return;
  }
  const int c = ch0 + row;
  const float r = -a1;
  float pw[5];
  pw[0] = r;
#pragma unroll
  for (int k = 1; k < 5; k++) {
    pw[k] = pw[k - 1] * pw[k - 1];
  }
  float sl = 1.0f;   // r^(lane + 1)
  {
    float q = r;
#pragma unroll
    for (int k = 0; k < 6; k++) {
      if (((lane + 1) >> k) & 1) {
        sl *= q;
      }
      q *= q;
    }
  }
  float2 carry = make_float2(st[c].dc_i, st[c].dc_q);
  const float2 *in = x1 + (size_t)c * x1_pitch;
  float2 *out = x2 + (size_t)c * x2_pitch + H_X2;
  int clip = 0;
  // U chunks of 32 samples per iteration: their loads and scan rounds are independent of each other
  // (instruction-level parallelism against the global-memory latency); only the carried state
  // links them, one fma and one broadcast per chunk
  constexpr int U = 4;
  for (int i0 = 0; i0 < n_total; i0 += 32 * U) {
    float2 v[U];
    bool ok[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int i = i0 + 32 * u + lane;
      ok[u] = i < n_total;
      v[u] = ok[u] ? in[i] : make_float2(0.0f, 0.0f);
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      clip += __popc(__ballot_sync(0xffffffffu, ok[u] && (fabsf(v[u].x) >= 0.995f || fabsf(v[u].y) >= 0.995f)));
    }
#pragma unroll
    for (int k = 0; k < 5; k++) {
#pragma unroll
      for (int u = 0; u < U; u++) {
        float2 t;
        t.x = __shfl_up_sync(0xffffffffu, v[u].x, 1 << k);
        t.y = __shfl_up_sync(0xffffffffu, v[u].y, 1 << k);
        if (lane >= (1 << k)) {
          v[u] = fma2(pw[k], t, v[u]);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int base = i0 + 32 * u;
      if (base < n_total) {   // warp-uniform
        v[u] = fma2(sl, carry, v[u]);   // v0[j] of the serial loop
        float2 p;
        p.x = __shfl_up_sync(0xffffffffu, v[u].x, 1);
        p.y = __shfl_up_sync(0xffffffffu, v[u].y, 1);
        if (lane == 0) {
          p = carry;
        }
        if (ok[u]) {
          out[base + lane] = make_float2(v[u].x - p.x, v[u].y - p.y);
        }
        const int last = min(31, n_total - 1 - base);
        carry.x = __shfl_sync(0xffffffffu, v[u].x, last);
        carry.y = __shfl_sync(0xffffffffu, v[u].y, last);
      }
    }
  }
  if (lane == 0) {
    st[c].dc_i = carry.x;
    st[c].dc_q = carry.y;
    st[c].clipping = (clip > 0) ? 1 : 0;
    const float ratio = (float)clip / (float)n_total;
    st[c].clip_ratio = ratio;
    if (status) {
      status[(size_t)c * status_pitch].clip_ratio = ratio;
    }
  }
}

// ---------------------------------------------------------------------------
// K2: channel filter (firfilt_crcf, 81/121 real taps on complex data, per-channel
// bandwidth). 128 threads x 8 consecutive complex outputs, sliding register window.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_chanfir(const float2 *__restrict__ x2, size_t x2_pitch, float2 *__restrict__ ybuf,
          size_t y_pitch, const float *__restrict__ chan_taps, const int *__restrict__ chan_lp,
          const float *__restrict__ chan_scale, const ChanParams *__restrict__ cp, int n_total,
          int ch0) {
  constexpr int R = 8;
  constexpr int T = 128 * R;
  __shared__ float hs[CHAN_TAPS_PITCH];
  extern __shared__ float2 xs[];
  const int c = blockIdx.y + ch0;
  const int n0 = blockIdx.x * T;
  const int t = threadIdx.x;
  const int f = cp[c].filt;
  const int Lp = chan_lp[f];
  const float scale = chan_scale[f];
  if (t < Lp) {
    hs[t] = chan_taps[f * CHAN_TAPS_PITCH + (CHAN_TAPS_PITCH - Lp) + t];
  }
  const float2 *row = x2 + (size_t)c * x2_pitch + H_X2;
  const int b0 = n0 - (Lp - 1);
  const int tile_len = T + Lp - 1 + R;
  for (int a = t; a < tile_len; a += 128) {
    const int s = b0 + a;
    xs[a + (a >> 3)] = (s < n_total) ? row[s] : make_float2(0.0f, 0.0f);
  }
  __syncthreads();
  float2 acc[R], win[R];
#pragma unroll
  for (int j = 0; j < R; j++) {
    acc[j] = make_float2(0.0f, 0.0f);
    const int a = t * R + j;
    win[j] = xs[a + (a >> 3)];
  }
  const float2 *wp = xs + (R + 1) * (t + 1);  // as in k_fir_pair: immediate-offset window loads
  for (int i = 0; i < Lp; i += R) {
#pragma unroll
    for (int u = 0; u < R; u++) {
      const float h = hs[i + u];
#pragma unroll
      for (int j = 0; j < R; j++) {
        acc[j] = fma2(h, win[(j + u) & (R - 1)], acc[j]);
      }
      win[u] = wp[u];
    }
    wp += R + 1;
  }
  float2 *out = ybuf + (size_t)c * y_pitch + Y_OFF;
#pragma unroll
  for (int j = 0; j < R; j++) {
    const int n = n0 + t * R + j;
    if (n < n_total) {
      out[n] = make_float2(acc[j].x * scale, acc[j].y * scale);
    }
  }
}

// S2: pre-discriminator AGC (agc_crcf; fm_demod.cpp:170-172,196-198), in place, lanes with AGC on
__global__ void __launch_bounds__(32)
k_agc(float2 *ybuf, size_t y_pitch, DemodState *st, const ChanParams *cp, int n_total, int ch0,
      int nch) {
  // ONE warp per 32 channels (see k_dcblock): prefetch the next tile, run the AGC recursion in
  // place on the current one, write it back. Two tiles.
  constexpr int TP = 2 * LT + 4;
  extern __shared__ float sm_agc[];
  auto tb = [&](int k2) { return sm_agc + (k2 & 1) * (32 * TP); };
  const int lane = threadIdx.x;
  const int c0 = ch0 + blockIdx.x * 32;
  const int nrows = min(32, ch0 + nch - c0);
  const int c = c0 + min(lane, nrows - 1);
  const bool has_agc = lane < nrows && cp[c].agc_mode != 0;
  if (__ballot_sync(0xffffffffu, has_agc) == 0u) {
    return;  // no channel of this block runs an AGC
  }
  const bool active = has_agc;
  const float alpha = active ? cp[c].agc_alpha : 0.0f;
  float g = 1.0f, y2 = 1.0f;
  if (active) {
    g = st[c].agc_g;
    y2 = st[c].agc_y2;
  }
  float *yf = reinterpret_cast<float *>(ybuf);
  const int nchunks = (n_total + LT - 1) / LT;
  if (nchunks > 0) {
    tileLoadAsync<TP, 2 * LT>(tb(0), yf, 2 * y_pitch, c0, nrows, 2L * Y_OFF, 2 * min(LT, n_total), lane);
    cpAsyncCommit();
  }
  for (int ck = 0; ck < nchunks; ck++) {
    const int n0 = ck * LT;
    const int len = min(LT, n_total - n0);
    cpAsyncWait<0>();
    __syncwarp();  // tile ck visible to every lane; tile ck - 1 has been written back by every lane
    if (ck + 1 < nchunks) {
      tileLoadAsync<TP, 2 * LT>(tb(ck + 1), yf, 2 * y_pitch, c0, nrows, 2L * (Y_OFF + n0 + LT),
                        2 * min(LT, n_total - n0 - LT), lane);
      cpAsyncCommit();
    }
    if (active) {
      float *t = tb(ck) + lane * TP;
      auto sample = [&](float &x, float &y) {
        const float ox = x * g;
        const float oy = y * g;
        const float e = (ox * ox) + (oy * oy);
        y2 = ((1.0f - alpha) * y2) + (alpha * e);
        if (y2 > 1e-6f) {
          g = g * fm_expf((-0.5f * alpha) * fm_logf(y2));
        }
        if (g > 1e6f) {
          g = 1e6f;
        }
        x = ox;
        y = oy;
      };
      int i = 0;
      for (; i + 2 <= len; i += 2) {  // two complex samples per 128-bit access (conflict-free)
        float4 v = *reinterpret_cast<float4 *>(t + 2 * i);
        sample(v.x, v.y);
        sample(v.z, v.w);
        *reinterpret_cast<float4 *>(t + 2 * i) = v;
      }
      for (; i < len; i++) {
        sample(t[2 * i], t[2 * i + 1]);
      }
    }
    __syncwarp();
    // rows without an AGC are written back unchanged
    tileStore<TP, 2 * LT>(tb(ck), yf, 2 * y_pitch, c0, nrows, 2L * (Y_OFF + n0), 2 * len, lane);
  }
  if (active) {
    st[c].agc_g = g;
    st[c].agc_y2 = y2;
  }
}

// K2b: quadrature discriminator, arg(conj(y[n-1]) * y[n]) / (2 pi kf)   (freqdem). A streaming
// kernel (12 B per sample): four samples per thread, 128-bit loads and stores (the data region of
// a y row starts 16-byte aligned at Y_OFF, the MPX data region at H_MPX).
__global__ void __launch_bounds__(256)
k_freqdem(const float2 *__restrict__ ybuf, size_t y_pitch, float *__restrict__ mpx,
          size_t mpx_pitch, int n_total, int ch0, float ref) {
  const int c = blockIdx.y + ch0;
  const int n = 4 * (blockIdx.x * blockDim.x + threadIdx.x);
  if (n >= n_total) {
    return;
  }
  const float2 *y = ybuf + (size_t)c * y_pitch + Y_OFF;  // y[-1] = r_prev
  float *out = mpx + (size_t)c * mpx_pitch + H_MPX;
  auto one = [&](float2 p, float2 r) {
    const float re = (p.x * r.x) + (p.y * r.y);
    const float im = (p.x * r.y) - (p.y * r.x);
    return fm_atan2f(im, re) * ref;
  };
  if (n + 4 <= n_total) {
    const float2 p = y[n - 1];
    const float4 a = *reinterpret_cast<const float4 *>(y + n);      // y[n], y[n+1]
    const float4 b = *reinterpret_cast<const float4 *>(y + n + 2);  // y[n+2], y[n+3]
    const float2 y0 = make_float2(a.x, a.y), y1 = make_float2(a.z, a.w);
    const float2 y2 = make_float2(b.x, b.y), y3 = make_float2(b.z, b.w);
    *reinterpret_cast<float4 *>(out + n) = make_float4(one(p, y0), one(y0, y1), one(y1, y2), one(y2, y3));
  } else {
    for (int i = n; i < n_total; i++) {
      out[i] = one(y[i - 1], y[i]);
    }
  }
}

// ---------------------------------------------------------------------------
// S4: 19 kHz pilot PLL, quality metrics, blend, L-R matrix, per-block lock logic
// (stereo_decoder.cpp:92-286). One lane per channel, the per-sample work split over a
// four-warp software pipeline, one tile of STEREO_ST samples apart (each warp on its own SM
// sub-partition):
//   warp 0     tile mover  global <-> shared (cp.async in, 128-bit stores out), and behind its
//              copies the blend recursion and the L-R matrix
//   warp 1     PLL + envelopes: pilot -> phase error -> NCO update -> sin/cos of the new phase is
//              the one truly serial chain (~264 cycles per sample on B200, tools/microbench/
//              lat_bench.cu); the four one-pole envelopes ride in its idle issue slots, and the
//              stereo-lock logic runs once, after the block's last sample
//   warps 2,3  blend target from the envelopes (up to six IEEE divisions and two square roots per
//              sample, but element-wise): each takes half of the tile's samples
// Round 1 ran everything behind the PLL in ONE warp; with weak signals (no clean-pilot shortcut)
// that warp, not the PLL chain, set the pace: 720-830 cycles per sample.
// Arithmetic and its order are exactly those of the single-lane loop (and of the CPU oracle).
// ---------------------------------------------------------------------------
constexpr int STEREO_TILES = 23;
constexpr int STEREO_THREADS = 128;
// channels per CTA of the two lane kernels (one lane each; lanes past it idle). These kernels are
// bound by dependent-issue latency, not by lanes: fewer channels per warp = more chains per scheduler.
constexpr int STEREO_CPC = 32;
constexpr int RDS_CPC = 32;
static_assert(STEREO_CPC >= 1 && STEREO_CPC <= 32 && RDS_CPC >= 1 && RDS_CPC <= 32, "one lane per channel");
constexpr int STEREO_MINB = 6;  // at most 85 registers per thread

__global__ void __launch_bounds__(STEREO_THREADS, STEREO_MINB)
k_stereo(const float *__restrict__ mpx, size_t mpx_pitch, const float *__restrict__ pilot,
         size_t pilot_pitch, float *__restrict__ lraw, float *__restrict__ rraw, size_t lr_pitch,
         StereoState *st, const ChanParams *cp, fmgpu_block_status *status, int status_pitch,
         int n_total, int ch0, int nch, EngineConst k) {
  constexpr int ST = STEREO_ST;  // samples per tile row
  // 16-byte aligned rows, read and written by their lane four samples at a time; a pitch of ST + 4
  // floats is odd in 16-byte units, so the 8 lanes of a quarter-warp hit 8 different bank groups
  constexpr int TP = ST + 4;
  constexpr int TS = STEREO_CPC * TP;  // floats per tile
  extern __shared__ float sm_st[];
  // chunk j of a ring of n sits in slot j % n
  float *t_pil = sm_st;             // 2: mover -> PLL
  float *t_mpx = t_pil + 2 * TS;    // 2: mover -> PLL (envelope of |mpx|)
  float *t_dly = t_mpx + 2 * TS;    // 2: mover -> matrix (delayed MPX)
  float *t_c2 = t_dly + 2 * TS;     // 3: PLL -> matrix, cos(2 * phase after the sample)
  float *t_frq = t_c2 + 3 * TS;     // 2: PLL -> target, clamped phase increment (m_pllFreq)
  float *t_pbm = t_frq + 2 * TS;    // 2: PLL -> target, pilot-band envelope
  float *t_mm = t_pbm + 2 * TS;     // 2: PLL -> target, MPX envelope
  float *t_s2 = t_mm + 2 * TS;      // 2: PLL -> target, |coherent pilot|^2, or -1 while mono
  float *t_tgt = t_s2 + 2 * TS;     // 2: target -> matrix
  float *t_l = t_tgt + 2 * TS;      // 2: matrix -> mover
  float *t_r = t_l + 2 * TS;        // 2
  const uint32_t sm_base = sharedAddr(sm_st);   // byte address of sm_st in the shared window
  auto sa = [&](const float *p) { return sm_base + 4u * static_cast<uint32_t>(p - sm_st); };
  const int lane = threadIdx.x & 31;
  // 0 mover + blend + matrix, 1 PLL + envelopes, 2/3 target. Warp w of a CTA sits on SM sub-partition
  // w % 4, and the PLL role is the one that sets the pace: the CTAs that share an SM (block b, b + the
  // SM count, ...) rotate the roles, so that their PLL warps land on different schedulers.
  const int role = ((threadIdx.x >> 5) + (k.sm_rot > 0 ? (int)blockIdx.x / k.sm_rot : 0)) & 3;
  const int c0 = ch0 + blockIdx.x * STEREO_CPC;
  const int nrows = min(STEREO_CPC, ch0 + nch - c0);
  const bool active = lane < nrows;
  const int c = c0 + min(lane, nrows - 1);
  constexpr float kPi = 3.14159265358979323846f;
  constexpr float kMatrixScale = 0.5f;
  constexpr float kPilotRatioAcquire = 0.040f, kPilotRatioHold = 0.022f;
  constexpr float kMpxMinAcquire = 0.005f, kMpxMinHold = 0.0028f;
  constexpr float kPilotCoherenceAcquire = 0.18f, kPilotCoherenceHold = 0.11f;
  constexpr float kPllLockAcquireHz = 180.0f, kPllLockHoldHz = 320.0f;
  constexpr float kSmooth = 0.9995f;
  constexpr float kInject = 1.0f - kSmooth;

  StereoState s = st[c];
  const ChanParams p = cp[c];
  const int mode = p.blend_mode;
  const float blendAttack = k.blend_attack[mode];
  const float blendRelease = k.blend_release[mode];
  const float gate = k.gate[mode];
  const float ratioDen = fmaxf(kPilotRatioAcquire - kPilotRatioHold, 1e-4f);
  const float cohDen = fmaxf(kPilotCoherenceAcquire - kPilotCoherenceHold, 1e-4f);
  const float pllDen = fmaxf(kPllLockHoldHz - kPllLockAcquireHz, 1e-3f);

  // PLL warp: the NCO phase carried in the state, and the envelopes
  uint32_t theta = s.theta, dtheta = s.dtheta;
  float phaseNow = ncoPhaseDev(theta);
  float vcoQ, vcoI;
  fm_sincosf(phaseNow, &vcoQ, &vcoI);
  float pbm = s.pbm, mm = s.mm, pilotI = s.pilot_i, pilotQ = s.pilot_q, blend = s.blend;
  float pllFreq = s.pll_freq;

  const int nchunks = (n_total + ST - 1) / ST;
  auto clen = [&](int ck) { return min(ST, n_total - ck * ST); };
  if (role == 0 && nchunks > 0) {
    tileLoadAsyncS<TP, ST>(sa(t_pil), pilot, pilot_pitch, c0, nrows, 0, clen(0), lane);
    tileLoadAsyncS<TP, ST>(sa(t_mpx), mpx, mpx_pitch, c0, nrows, H_MPX, clen(0), lane);
    cpAsyncCommit();
    cpAsyncWait<0>();
  }
  __syncthreads();
  const bool stereoDetected = s.stereo != 0;  // the lock logic runs once, after the last sample

  // step kk: PLL + envelopes on chunk kk, target on chunk kk-1, blend + matrix on chunk kk-2; the
  // mover loads pilot[kk+1], mpx[kk+1], delayed mpx[kk-1] and stores L/R of chunk kk-3
  for (int kk = 0; kk <= nchunks + 2; kk++) {
    if (role == 0) {
      if (kk + 1 < nchunks) {
        tileLoadAsyncS<TP, ST>(sa(t_pil + ((kk + 1) & 1) * TS), pilot, pilot_pitch, c0, nrows,
                               (long)(kk + 1) * ST, clen(kk + 1), lane);
        tileLoadAsyncS<TP, ST>(sa(t_mpx + ((kk + 1) & 1) * TS), mpx, mpx_pitch, c0, nrows,
                               H_MPX + (long)(kk + 1) * ST, clen(kk + 1), lane);
      }
      if (kk >= 1 && kk - 1 < nchunks) {
        const int j = kk - 1;
        tileLoadAsync4S<TP, ST>(sa(t_dly + (j & 1) * TS), mpx, mpx_pitch, c0, nrows,
                                H_MPX + (long)j * ST - k.delay, clen(j), lane);
      }
      cpAsyncCommit();
      if (kk >= 3) {
        const int j = kk - 3;
        tileStoreS<TP, ST>(sa(t_l + (j & 1) * TS), lraw, lr_pitch, c0, nrows, H_LR + (long)j * ST, clen(j), lane);
        tileStoreS<TP, ST>(sa(t_r + (j & 1) * TS), rraw, lr_pitch, c0, nrows, H_LR + (long)j * ST, clen(j), lane);
      }
      // ... and, while its copies are in flight, the blend recursion and the L-R matrix
      if (active && kk >= 2 && kk - 2 < nchunks) {
        const int j = kk - 2;
        const int len = clen(j);
        const int ro = (j & 1) * TS + lane * TP;
        const float *td = t_dly + ro;
        const float *tc2 = t_c2 + (j % 3) * TS + lane * TP;
        const float *tt = t_tgt + ro;
        float *tl = t_l + ro;
        float *tr = t_r + ro;
        auto matrix = [&](float dm, float cos2, float target, float &o_l, float &o_r) {
          const float monoNorm = dm * kMatrixScale;
          const float lr = 2.0f * dm * cos2;
          const float stereoLeft = (dm + lr) * kMatrixScale;
          const float stereoRight = (dm - lr) * kMatrixScale;
          const float blendAlpha = (target > blend) ? blendAttack : blendRelease;
          blend += (target - blend) * blendAlpha;
          o_l = monoNorm + ((stereoLeft - monoNorm) * blend);
          o_r = monoNorm + ((stereoRight - monoNorm) * blend);
        };
        int i = 0;
        const uint32_t a_td = sa(td), a_c2 = sa(tc2), a_tt = sa(tt), a_tl = sa(tl), a_tr = sa(tr);
        for (; i + 4 <= len; i += 4) {
          const float4 dv = ldsF4(a_td + 4u * i);
          const float4 cv = ldsF4(a_c2 + 4u * i);
          const float4 tv = ldsF4(a_tt + 4u * i);
          float4 lv, rv;
          matrix(dv.x, cv.x, tv.x, lv.x, rv.x);
          matrix(dv.y, cv.y, tv.y, lv.y, rv.y);
          matrix(dv.z, cv.z, tv.z, lv.z, rv.z);
          matrix(dv.w, cv.w, tv.w, lv.w, rv.w);
          stsF4(a_tl + 4u * i, lv);
          stsF4(a_tr + 4u * i, rv);
        }
        for (; i < len; i++) {
          matrix(td[i], tc2[i], tt[i], tl[i], tr[i]);
        }
      }
      cpAsyncWait<0>();
    } else if (role == 1) {
      if (active && kk < nchunks) {
        const int len = clen(kk);
        const int ro = (kk & 1) * TS + lane * TP;
        const float *tp = t_pil + ro;
        const float *tm = t_mpx + ro;
        float *tc2 = t_c2 + (kk % 3) * TS + lane * TP;
        float *tf = t_frq + ro;
        float *tpb = t_pbm + ro;
        float *tmm = t_mm + ro;
        float *ts2 = t_s2 + ro;
        const uint32_t a_tp = sa(tp), a_tm = sa(tm), a_tc2 = sa(tc2), a_tf = sa(tf), a_tpb = sa(tpb),
                       a_tmm = sa(tmm), a_ts2 = sa(ts2);
        // one sample: envelopes with the VCO phase BEFORE this sample's update
        // (stereo_decoder.cpp:176-186), then the PLL step
        auto sample = [&](float pil, float x, float &o_frq, float &o_pbm, float &o_mm, float &o_s2,
                          float &o_c2) {
          pbm = (pbm * kSmooth) + (fabsf(pil) * kInject);
          mm = (mm * kSmooth) + (fabsf(x) * kInject);
          pilotI = (pilotI * kSmooth) + ((pil * vcoI) * kInject);
          pilotQ = (pilotQ * kSmooth) + ((pil * vcoQ) * kInject);
          const float error = pil * vcoQ;
          dtheta += ncoConstrainDev(error * k.pll_alpha);
          theta += ncoConstrainDev(error * k.pll_beta);
          theta += dtheta;
          const float phaseNext = ncoPhaseDev(theta);
          float dphi = phaseNext - phaseNow;
          if (dphi > kPi) {
            dphi -= 2.0f * kPi;
          } else if (dphi < -kPi) {
            dphi += 2.0f * kPi;
          }
          pllFreq = fm_clampf(dphi, k.pll_min, k.pll_max);
          float sn, cs;
          fm_sincosf(phaseNext, &sn, &cs);
          o_frq = pllFreq;
          o_pbm = pbm;
          o_mm = mm;
          o_s2 = stereoDetected ? ((pilotI * pilotI) + (pilotQ * pilotQ)) : -1.0f;
          o_c2 = (cs * cs) - (sn * sn);
          phaseNow = phaseNext;
          vcoQ = sn;
          vcoI = cs;
        };
        int i = 0;
        // four samples per 128-bit shared-memory access: a lane's row is 16-byte aligned, so a
        // warp's access is conflict-free (the 32-bit form hits 8 banks: 4-way conflicts)
        for (; i + 4 <= len; i += 4) {
          const float4 pv = ldsF4(a_tp + 4u * i);
          const float4 xv = ldsF4(a_tm + 4u * i);
          float4 of, ob, om, os, oc;
          sample(pv.x, xv.x, of.x, ob.x, om.x, os.x, oc.x);
          sample(pv.y, xv.y, of.y, ob.y, om.y, os.y, oc.y);
          sample(pv.z, xv.z, of.z, ob.z, om.z, os.z, oc.z);
          sample(pv.w, xv.w, of.w, ob.w, om.w, os.w, oc.w);
          stsF4(a_tf + 4u * i, of);
          stsF4(a_tpb + 4u * i, ob);
          stsF4(a_tmm + 4u * i, om);
          stsF4(a_ts2 + 4u * i, os);
          stsF4(a_tc2 + 4u * i, oc);
        }
        for (; i < len; i++) {  // ragged end of the block
          sample(tp[i], tm[i], tf[i], tpb[i], tmm[i], ts2[i], tc2[i]);
        }
      }
    } else if (role == 2 || role == 3) {
      if (active && kk >= 1 && kk - 1 < nchunks) {
        const int j = kk - 1;
        const int len = clen(j);
        // each target warp takes half of the tile, in groups of four samples (128-bit accesses;
        // elements past len are padding: computed, never used)
        const int half = (((len + 1) >> 1) + 3) & ~3;
        const int i0 = (role == 2) ? 0 : half;
        const int i1 = (role == 2) ? min(half, len) : len;
        const int ro = (j & 1) * TS + lane * TP;
        const float *tf = t_frq + ro;
        const float *tpb = t_pbm + ro;
        const float *tmm = t_mm + ro;
        const float *ts2 = t_s2 + ro;
        float *tt = t_tgt + ro;
        auto targetOf = [&](float s2, float ebm, float emm, float frq) -> float {
          float target = 0.0f;
          if (p.force_mono) {
            target = 0.0f;
          } else if (p.force_stereo) {
            target = 1.0f;
          } else if (!(s2 < 0.0f)) {  // stereo detected (the PLL warp stores -1 while mono)
            const float mx = fmaxf(emm, 1e-3f);
            const float pm = fmaxf(ebm, 1e-4f);
            const float dfs = fabsf(frq - k.nominal_pll) * k.fsf;
            const float tB = 0.1803f * pm;
            if (ebm >= 0.0402f * mx && s2 >= tB * tB && dfs <= 1130.0f) {
              // Clean pilot: with ratio >= 0.0402, coherence >= 0.1803 and |f error| <= 179.9 Hz
              // each of the three quality terms below clamps to exactly 1 (margins >= 1e-4
              // against rounding errors of ~1e-7) and no gate trips, so target == 1.0f in every
              // blend mode. Skipping the six IEEE divisions and the square root changes nothing.
              target = 1.0f;
            } else {
              const float pilotMagNow = FM_SQRT(s2);
              const float pilotRatio = ebm / mx;
              const float pilotCoherence = pilotMagNow / pm;
              const float pllErrHz = dfs / (2.0f * kPi);
              const float ratioQ = fm_clampf((pilotRatio - kPilotRatioHold) / ratioDen, 0.0f, 1.0f);
              const float cohQ =
                  fm_clampf((pilotCoherence - kPilotCoherenceHold) / cohDen, 0.0f, 1.0f);
              const float pllQ = fm_clampf((kPllLockHoldHz - pllErrHz) / pllDen, 0.0f, 1.0f);
              const float quality = fminf(ratioQ, fminf(cohQ, pllQ));
              float shaped = quality * quality;
              if (mode == 0) {
                shaped = FM_SQRT(fmaxf(0.0f, quality));
              } else if (mode == 2) {
                shaped = quality * quality * quality;
              }
              if (pilotRatio < (kPilotRatioHold * gate) ||
                  pilotCoherence < (kPilotCoherenceHold * gate) ||
                  pllErrHz > (kPllLockHoldHz * 1.10f)) {
                target = 0.0f;
              } else {
                target = fm_clampf(0.0f + ((1.0f - 0.0f) * shaped), 0.0f, 1.0f);
              }
            }
          }
          return target;
        };
        const uint32_t a_s2 = sa(ts2), a_pb = sa(tpb), a_mm = sa(tmm), a_f = sa(tf), a_t = sa(tt);
        for (int i = i0; i < i1; i += 4) {
          const float4 sv = ldsF4(a_s2 + 4u * i);
          const float4 bv = ldsF4(a_pb + 4u * i);
          const float4 mv = ldsF4(a_mm + 4u * i);
          const float4 fv = ldsF4(a_f + 4u * i);
          float4 tv;
          tv.x = targetOf(sv.x, bv.x, mv.x, fv.x);
          tv.y = targetOf(sv.y, bv.y, mv.y, fv.y);
          tv.z = targetOf(sv.z, bv.z, mv.z, fv.z);
          tv.w = targetOf(sv.w, bv.w, mv.w, fv.w);
          stsF4(a_t + 4u * i, tv);
        }
      }
    }
    __syncthreads();
  }
  if (active && role == 1) {
    // per-block tail (stereo_decoder.cpp:243-286)
    const float pilotMag = FM_SQRT((pilotI * pilotI) + (pilotQ * pilotQ));
    s.pilot_mag = (s.pilot_mag * 0.9f) + (pilotMag * 0.1f);
    const bool det = s.stereo != 0;
    const float mpxThreshold = det ? kMpxMinHold : kMpxMinAcquire;
    const float pilotRatio = pbm / fmaxf(mm, 1e-3f);
    const float pilotCoherence = s.pilot_mag / fmaxf(pbm, 1e-4f);
    const float ratioThreshold = det ? kPilotRatioHold : kPilotRatioAcquire;
    const float coherenceThreshold = det ? kPilotCoherenceHold : kPilotCoherenceAcquire;
    const float pllErrHz = fabsf(pllFreq - k.nominal_pll) * k.fsf / (2.0f * kPi);
    const float pllThreshold = det ? kPllLockHoldHz : kPllLockAcquireHz;
    const bool pilotPresent = (mm > mpxThreshold) && (pilotRatio > ratioThreshold) &&
                              (pilotCoherence > coherenceThreshold) && (pllErrHz < pllThreshold);
    if (!p.force_stereo) {
      if (!det) {
        if (pilotPresent) {
          s.pilot_count++;
          s.loss_count = 0;
          if (s.pilot_count >= 6) {
            s.stereo = 1;
          }
        } else {
          s.pilot_count = 0;
        }
      } else if (pilotPresent) {
        s.loss_count = 0;
      } else if (++s.loss_count >= 24) {
        s.stereo = 0;
        s.pilot_count = 0;
        s.loss_count = 0;
      }
    }
    const float calibrated = s.pilot_mag * 8.0f;
    s.pilot_tenths = min(750, max(0, (int)fm_roundf(calibrated * 750.0f)));
    if (status) {
      fmgpu_block_status *ob = &status[(size_t)c * status_pitch];
      ob->stereo = s.stereo;
      ob->pilot_tenths = s.pilot_tenths;
    }
    StereoState *o = &st[c];
    o->theta = theta;
    o->dtheta = dtheta;
    o->pbm = pbm;
    o->mm = mm;
    o->pilot_i = pilotI;
    o->pilot_q = pilotQ;
    o->pll_freq = pllFreq;
    o->pilot_mag = s.pilot_mag;
    o->stereo = s.stereo;
    o->pilot_count = s.pilot_count;
    o->loss_count = s.loss_count;
    o->pilot_tenths = s.pilot_tenths;
  } else if (active && role == 0) {
    st[c].blend = blend;
  }
}

// ---------------------------------------------------------------------------
// per-call bookkeeping of the fixed-point resamplers (resamp_rrrf, Appendix A.6):
// outputs produced by n inputs from phase p0:  ceil((n*2^24 - p0) / step)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t resampCount(uint32_t phase0, uint32_t step, long n,
                                                uint32_t *phase_next) {
  const unsigned long long num = (unsigned long long)n << 24;
  unsigned long long cnt = 0;
  if (num > phase0) {
    cnt = (num - phase0 + step - 1) / step;
  }
  *phase_next = (uint32_t)(phase0 + cnt * step - num);
  return (uint32_t)cnt;
}

__global__ void k_prepare(AudioState *au, RdsState *rds, fmgpu_block_status *status,
                          int status_pitch, int n_total, int ch0, int nch, uint32_t aud_step,
                          uint32_t rds_step, int do_audio, int do_mono, int do_rds, int first,
                          RdsRsRef rr) {
  const int lane = blockIdx.x * blockDim.x + threadIdx.x;
  if (lane >= nch) {
    return;
  }
  const int c = ch0 + lane;
  if (do_audio || do_mono) {
    AudioState *a = &au[c];
    uint32_t nx;
    const uint32_t p0 = do_mono ? a->mono_phase : a->rs_phase;
    const uint32_t total = resampCount(p0, aud_step, n_total, &nx);
    if (first) {
      a->out_base = 0;  // first logical block of a call: frames are appended from the row start
    }
    if (do_mono) {
      a->mono_n_out = total;
      a->mono_phase_next = nx;
    } else {
      a->n_out = total;
      a->rs_phase_next = nx;
    }
    if (status) {
      status[(size_t)c * status_pitch].n_audio = (int)total;
    }
  }
  if (do_rds == PREPARE_RDS_RESAMPLER) {
    RdsRsState *q = &rr.st[c];
    uint32_t nx;
    q->n171[rr.par] = resampCount(q->rs_phase, rds_step, n_total, &nx);
    q->rs_phase_next = nx;
  }
  if (do_rds == PREPARE_RDS_COUNTERS) {
    RdsState *r = &rds[c];
    if (first) {
      r->n_groups = 0;  // groups and bits accumulate over the logical blocks of one call
      r->n_bits = 0;
      r->bits_done = 0;
    }
  }
}

__global__ void k_commit(AudioState *au, RdsState *rds, int ch0, int nch, int do_audio, int do_mono,
                         int do_rds, RdsRsRef rr) {
  const int lane = blockIdx.x * blockDim.x + threadIdx.x;
  if (lane >= nch) {
    return;
  }
  const int c = ch0 + lane;
  if (do_audio) {
    au[c].rs_phase = au[c].rs_phase_next;
    au[c].out_base += au[c].n_out;
  }
  if (do_mono) {
    au[c].mono_phase = au[c].mono_phase_next;
    au[c].out_base += au[c].mono_n_out;
  }
  if (do_rds) {
    rr.st[c].rs_phase = rr.st[c].rs_phase_next;
  }
}

// ---------------------------------------------------------------------------
// K5b: arbitrary-rate polyphase resampler to 32 kHz (one thread per output frame)
// ---------------------------------------------------------------------------
// The branch length is known at compile time: the dot products are fully unrolled, the taps of the
// thread's branch are read once (128-bit) and serve both rows. (A run-time length spent ~8
// instructions per tap and row on loop bookkeeping.)
__global__ void k_resample(const float *__restrict__ in0, const float *__restrict__ in1,
                           size_t in_pitch, int in_off, const float *__restrict__ hist,
                           int hist_pitch, float *__restrict__ out, size_t acap,
                           const float *__restrict__ bank, uint32_t step, const AudioState *au,
                           int mono, int ch0) {
  constexpr int SUB = AUD_RS_LEN;
  static_assert(SUB % 4 == 0, "the taps of a branch are read four at a time");
  extern __shared__ __align__(16) float bk[];
  for (int i = threadIdx.x; i < 32 * SUB; i += blockDim.x) {
    bk[i] = bank[i];
  }
  __syncthreads();
  const int c = blockIdx.y + ch0;
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t n_out = mono ? au[c].mono_n_out : au[c].n_out;
  const uint32_t ob = au[c].out_base;  // frames already written by earlier blocks of this call
  if (j >= n_out || ob + j >= acap) {
    return;
  }
  const uint32_t phase0 = mono ? au[c].mono_phase : au[c].rs_phase;
  const unsigned long long P = (unsigned long long)phase0 + (unsigned long long)j * step;
  const long i = (long)(P >> 24);
  const int br = (int)((P & 0xffffffull) >> 19);
  const float *h = bk + br * SUB;
  const float *a = in0 + (size_t)c * in_pitch + in_off + i - (SUB - 1);
  if (!(hist && i < SUB - 1)) {
    float hq[SUB];
#pragma unroll
    for (int q = 0; q < SUB; q += 4) {
      const float4 v = *reinterpret_cast<const float4 *>(h + q);
      hq[q] = v.x;
      hq[q + 1] = v.y;
      hq[q + 2] = v.z;
      hq[q + 3] = v.w;
    }
    float acc0 = 0.0f;
#pragma unroll
    for (int q = 0; q < SUB; q++) {
      acc0 = fmaf(hq[q], a[q], acc0);
    }
    out[((size_t)c * 2 + 0) * acap + ob + j] = acc0;
    if (in1) {
      const float *b = in1 + (size_t)c * in_pitch + in_off + i - (SUB - 1);
      float acc1 = 0.0f;
#pragma unroll
      for (int q = 0; q < SUB; q++) {
        acc1 = fmaf(hq[q], b[q], acc1);
      }
      out[((size_t)c * 2 + 1) * acap + ob + j] = acc1;
    }
    return;
  }
  // window reaches before this call: those samples live in the stage's own history
  const float *hc = hist + (size_t)c * hist_pitch;
  constexpr int H = SUB - 1;
  float acc0 = 0.0f;
  for (int q = 0; q < SUB; q++) {
    const long si = i - (SUB - 1) + q;
    const float x = (si >= 0) ? a[q] : hc[H + si];
    acc0 = fmaf(h[q], x, acc0);
  }
  out[((size_t)c * 2 + 0) * acap + ob + j] = acc0;
  if (in1) {
    const float *b = in1 + (size_t)c * in_pitch + in_off + i - (SUB - 1);
    float acc1 = 0.0f;
    for (int q = 0; q < SUB; q++) {
      acc1 = fmaf(h[q], b[q], acc1);
    }
    out[((size_t)c * 2 + 1) * acap + ob + j] = acc1;
  }
}

// ---------------------------------------------------------------------------
// S6: de-emphasis + DC blocker at 32 kHz (af_post_processor.cpp:66-71), in place;
// optional +-1 clamp (main.cpp:1305-1308). Lanes = (channel, side).
// mono = 1: FMDemod mono chain (fm_demod.cpp:216-222) on row 0, then optionally
// x0.5 duplicated to both rows (main.cpp:1275-1278).
// ---------------------------------------------------------------------------
__global__ void k_audio_iir(float *audio, size_t acap, AudioState *au, const ChanParams *cp,
                            int ch0, int nch, float dc_a1, int mono, int clamp, int mono_dup) {
  const int lane = blockIdx.x * blockDim.x + threadIdx.x;
  const int lanes = mono ? nch : 2 * nch;
  if (lane >= lanes) {
    return;
  }
  const int c = ch0 + (mono ? lane : lane / 2);
  const int side = mono ? 0 : (lane & 1);
  AudioState *a = &au[c];
  const ChanParams p = cp[c];
  const uint32_t ob = min((uint32_t)acap, a->out_base);
  const uint32_t n = min((uint32_t)acap - ob, mono ? a->mono_n_out : a->n_out);
  float *row = audio + ((size_t)c * 2 + side) * acap + ob;
  float *row2 = audio + ((size_t)c * 2 + 1) * acap + ob;
  const bool de = mono ? (p.mono_deemph_on != 0) : (p.deemph_on != 0);
  const float b0 = mono ? p.mono_de_b0 : p.de_b0;
  const float a1 = mono ? p.mono_de_a1 : p.de_a1;
  float dv = mono ? a->mono_de_v1 : a->de_v1[side];
  float cv = mono ? a->mono_dc_v1 : a->dc_v1[side];
  for (uint32_t i = 0; i < n; i++) {
    float x = row[i];
    if (de) {
      const float v0 = x - (a1 * dv);
      x = b0 * v0;
      dv = v0;
    }
    const float v0 = x - (dc_a1 * cv);
    float y = v0 - cv;
    cv = v0;
    if (mono_dup) {
      y = y * 0.5f;
    }
    if (clamp) {
      y = fm_clampf(y, -1.0f, 1.0f);
    }
    row[i] = y;
    if (mono_dup) {
      row2[i] = y;
    }
  }
  if (mono) {
    a->mono_de_v1 = dv;
    a->mono_dc_v1 = cv;
  } else {
    a->de_v1[side] = dv;
    a->dc_v1[side] = cv;
  }
}

// S6 as a warp-shuffle parallel scan (north_star item 5): the same two first-order recursions,
// one WARP per (channel, side) row, 32 frames per step. Both filters are affine in their state,
//     v[j] = x[j] + r v[j-1]     (de-emphasis: r = -a1;  DC blocker: r = 1 - alpha),
// so a Kogge-Stone scan over the lanes (5 rounds of shfl_up + fma with r^1, r^2, ... r^16) gives
// every lane its v[j] from the 32 inputs and the state carried in, and the row is read and
// written with coalesced 128-byte accesses instead of one scattered word per lane. The scan adds
// the terms in a different order than the serial loop: results agree to float rounding (~1e-7),
// not bit for bit, so it is the engine's FAST form (fmgpu_set_audio_iir_mode(1)); the lane
// recursion above stays the bit-exact one. Stereo rows only (the mono chain keeps the recursion).
__global__ void __launch_bounds__(128)
k_audio_iir_scan(float *audio, size_t acap, AudioState *au, const ChanParams *cp, int ch0, int nch,
                 float dc_a1, int clamp) {
  const int lane = threadIdx.x & 31;
  const int row_id = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (row_id >= 2 * nch) {
    return;
  }
  const int c = ch0 + (row_id >> 1);
  const int side = row_id & 1;
  AudioState *a = &au[c];
  const ChanParams p = cp[c];
  const uint32_t ob = min((uint32_t)acap, a->out_base);
  const uint32_t n = min((uint32_t)acap - ob, a->n_out);
  float *row = audio + ((size_t)c * 2 + side) * acap + ob;
  const bool de = p.deemph_on != 0;
  const float b0 = p.de_b0;
  const float r1 = -p.de_a1;   // de-emphasis pole
  const float r2 = -dc_a1;     // DC blocker pole
  // r^(2^k) for the scan rounds and r^(lane+1) for the carried state
  float p1[5], p2[5];
  p1[0] = r1;
  p2[0] = r2;
#pragma unroll
  for (int k = 1; k < 5; k++) {
    p1[k] = p1[k - 1] * p1[k - 1];
    p2[k] = p2[k - 1] * p2[k - 1];
  }
  float s1 = 1.0f, s2 = 1.0f;   // r^(lane+1) by binary exponentiation of lane + 1
  {
    const int e = lane + 1;
    float q1 = r1, q2 = r2;
#pragma unroll
    for (int k = 0; k < 6; k++) {
      if ((e >> k) & 1) {
        s1 *= q1;
        s2 *= q2;
      }
      q1 *= q1;
      q2 *= q2;
    }
  }
  float dv = a->de_v1[side];
  float cv = a->dc_v1[side];
  // U chunks per iteration: independent loads and scan rounds; the carried states link them
  constexpr int U = 4;
  for (uint32_t i0 = 0; i0 < n; i0 += 32 * U) {
    float x[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint32_t i = i0 + 32 * u + lane;
      x[u] = (i < n) ? row[i] : 0.0f;
    }
    if (de) {
#pragma unroll
      for (int k = 0; k < 5; k++) {
#pragma unroll
        for (int u = 0; u < U; u++) {
          const float t = __shfl_up_sync(0xffffffffu, x[u], 1 << k);
          if (lane >= (1 << k)) {
            x[u] = fmaf(p1[k], t, x[u]);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < U; u++) {
        const uint32_t base = i0 + 32 * u;
        if (base < n) {   // warp-uniform
          const float v = fmaf(s1, dv, x[u]);   // v0[j] of the serial loop
          dv = __shfl_sync(0xffffffffu, v, min(31u, n - 1 - base));
          x[u] = b0 * v;
          if (base + lane >= n) {
            x[u] = 0.0f;   // nothing past the row's end enters the second scan
          }
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 5; k++) {
#pragma unroll
      for (int u = 0; u < U; u++) {
        const float t = __shfl_up_sync(0xffffffffu, x[u], 1 << k);
        if (lane >= (1 << k)) {
          x[u] = fmaf(p2[k], t, x[u]);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint32_t base = i0 + 32 * u;
      if (base < n) {   // warp-uniform
        const float w = fmaf(s2, cv, x[u]);
        float wp = __shfl_up_sync(0xffffffffu, w, 1);
        if (lane == 0) {
          wp = cv;
        }
        float y = w - wp;
        if (clamp) {
          y = fm_clampf(y, -1.0f, 1.0f);
        }
        if (base + lane < n) {
          row[base + lane] = y;
        }
        cv = __shfl_sync(0xffffffffu, w, min(31u, n - 1 - base));
      }
    }
  }
  if (lane == 0) {
    a->de_v1[side] = dv;
    a->dc_v1[side] = cv;
  }
}

__global__ void k_store_counts(const AudioState *au, const RdsState *rds, uint32_t *n_audio,
                               uint32_t *n_groups, int ch0, int nch, int mono, uint32_t acap,
                               uint32_t gcap) {
  const int lane = blockIdx.x * blockDim.x + threadIdx.x;
  if (lane >= nch) {
    return;
  }
  const int c = ch0 + lane;
  if (n_audio) {
    n_audio[c] = min(acap, au[c].out_base);  // runs after k_commit of the call's last block
  }
  if (n_groups) {
    n_groups[c] = min(gcap, rds[c].n_groups);
  }
}

// ---------------------------------------------------------------------------
// S7: the RDS branch, one lane per channel (redsea_port subcarrier.cpp:117-235,
// liquid_wrappers.cpp:98-147, block_sync.cpp:235-313, rds_decoder.cpp:29-58):
//   resample to 171 kHz -> 57 kHz NCO mix-down -> 255-tap low-pass evaluated only
//   at the /24 instants (running accumulators, oldest sample first) -> AGC ->
//   polyphase symbol synchroniser -> BPSK PLL -> biphase -> differential decode ->
//   (26,16) block synchroniser with burst error correction -> groups.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t rdsSyndromeDev(uint32_t v) {
  uint32_t r = 0;
#pragma unroll
  for (int q = 0; q < 10; q++) {
    r |= (uint32_t)(__popc(v & c_syn_mask[q]) & 1) << q;
  }
  return r;
}

__device__ __forceinline__ int rdsOffsetForSyndromeDev(uint32_t s) {
  switch (s) {
  case 0b1111011000: return 0;  // A
  case 0b1111010100: return 1;  // B
  case 0b1001011100: return 2;  // C
  case 0b1111001100: return 3;  // C'
  case 0b1001011000: return 4;  // D
  default: return 5;            // invalid
  }
}

__device__ __forceinline__ int rdsBlockNumberDev(int off) {
  return (off == 0) ? 0 : (off == 1) ? 1 : (off == 2 || off == 3) ? 2 : (off == 4) ? 3 : 0;
}

__device__ __forceinline__ int rdsNextOffsetDev(int off) {
  return (off == 0) ? 1 : (off == 1) ? 2 : (off == 2 || off == 3) ? 4 : 0;
}

__device__ __forceinline__ bool rdsCouldFollow(int off, uint32_t pos, int ooff, uint32_t opos) {
  const uint32_t d = pos - opos;
  return d % 26 == 0 && d / 26 <= 6 && off != 5 && ooff != 5 &&
         ((uint32_t)rdsBlockNumberDev(ooff) + d / 26) % 4 == (uint32_t)rdsBlockNumberDev(off);
}

// BlockStream::pushBit with the 26-bit window `raw` ending at this bit and its syndrome `syn`
// already evaluated (k_blocksync phase 1 computes them for every bit offset in parallel).
__device__ void rdsPushWord(RdsState &s, uint32_t raw, uint32_t syn, fmgpu_rds_group *groups,
                            uint32_t gcap, uint32_t block_index) {
  s.reg = (s.reg << 1) + (raw & 1u);
  s.until--;
  s.bitcount++;
  if (s.until != 0) {
    return;
  }
  // findBlockInInputRegister
  int off = rdsOffsetForSyndromeDev(syn);
  if (!s.in_sync) {
    s.bits_since_lost++;
    if (off != 5) {
      for (int i = 0; i < 3; i++) {
        s.pulse_pos[i] = s.pulse_pos[i + 1];
        s.pulse_off[i] = s.pulse_off[i + 1];
      }
      s.pulse_pos[3] = s.bitcount;
      s.pulse_off[3] = off;
      bool found = false;
      for (int i1 = 0; i1 < 2 && !found; i1++) {
        for (int i2 = i1 + 1; i2 < 3 && !found; i2++) {
          if (rdsCouldFollow(s.pulse_off[3], s.pulse_pos[3], s.pulse_off[i2], s.pulse_pos[i2]) &&
              rdsCouldFollow(s.pulse_off[i2], s.pulse_pos[i2], s.pulse_off[i1], s.pulse_pos[i1])) {
            found = true;
          }
        }
      }
      if (found) {
        s.in_sync = 1;
        s.expected = off;
        s.cur_recv = 0;
        s.cur_err = 0;
        s.bits_since_lost = 0;
      }
    }
  }
  if (s.in_sync) {
    if (s.expected == 2 && off == 3) {
      s.expected = 3;
    }
    const bool had_errors = (off != s.expected);
    const unsigned long long bitm = 1ull << s.err_ptr;
    s.err_mask = had_errors ? (s.err_mask | bitm) : (s.err_mask & ~bitm);
    s.err_ptr = (s.err_ptr + 1) % 50;
    if (__popcll(s.err_mask) > 42) {
      s.in_sync = 0;
      s.err_mask = 0;
    } else {
      uint32_t data = raw >> 10;
      if (had_errors) {
        const uint32_t want = syn ^ rdsSyndromeDev(c_off_word[s.expected]);
        for (int q = 0; q < 52; q++) {
          if (c_err_syn[q] == want) {
            data = (raw ^ c_err_vec[q]) >> 10;
            off = s.expected;
            break;
          }
        }
      }
      if (off == s.expected) {
        const int bn = rdsBlockNumberDev(s.expected);
        s.cur_data[bn] = (uint16_t)data;
        s.cur_recv |= (1u << bn);
        s.cur_err = had_errors ? (s.cur_err | (1u << bn)) : (s.cur_err & ~(1u << bn));
      }
      const int next = rdsNextOffsetDev(s.expected);
      if (next == 0) {
        if (groups && s.n_groups < gcap) {
          fmgpu_rds_group g;
          uint8_t e = 0;
          uint16_t w[4];
          for (int q = 0; q < 4; q++) {
            const bool rc = (s.cur_recv >> q) & 1u;
            w[q] = rc ? s.cur_data[q] : 0;
            const uint8_t code = !rc ? 3 : (((s.cur_err >> q) & 1u) ? 1 : 0);
            e = (uint8_t)((e << 2) | code);
          }
          g.a = w[0];
          g.b = w[1];
          g.c = w[2];
          g.d = w[3];
          g.errors = e;
          g.pad[0] = g.pad[1] = g.pad[2] = 0;
          g.block_index = block_index;
          groups[s.n_groups] = g;
        }
        s.n_groups++;
        s.cur_recv = 0;
        s.cur_err = 0;
      }
      s.expected = next;
    }
  }
  s.until = s.in_sync ? 26 : 1;
}

// S7a: MPX -> 171 kHz (resamp_rrrf, m = 13, 32 branches; subcarrier.cpp:117-147). The resampler
// has no feedback, so it runs as a tile kernel, one thread per 171 kHz output: output k of a
// channel sits at fixed-point position P = phase + k * step, reads the 26 inputs ending at
// P >> 24 through branch (P >> 19) & 31 — the same dot product, oldest input first, that the
// serial loop of the reference evaluates. Inputs before this call come from the RDS resampler's
// own window (it is not reset with the stereo path).
constexpr int RDS_RS_OUT = 512;                    // outputs per CTA (4 per thread)
constexpr int RDS_RS_ROW = (RDS_RS_LEN + 3) & ~3;  // branch rows padded to 16 bytes
// inputs one CTA can touch: its outputs advance by step / 2^24 < 2 inputs each
constexpr int RDS_RS_SPAN = 2 * RDS_RS_OUT + RDS_RS_LEN + 8;

__global__ void __launch_bounds__(128)
k_rds_resample(const float *__restrict__ mpx, size_t mpx_pitch, const float *__restrict__ hist,
               int hist_pitch, RdsRsRef rr, const float *__restrict__ g_bank,
               float *__restrict__ r171, size_t r_pitch, uint32_t step, int ch0) {
  // Both operands of the 26-tap dot products come from shared memory: the 32 branch rows (128-bit
  // reads) and the input window of the CTA's 512 outputs, filled once with coalesced loads. (Storing
  // the branches transposed or branch-interleaved removes the tap reads' bank conflicts but was
  // slower: 1.62 / 1.30 instead of 1.23 ms per step.) (The
  // first form read its 26 inputs per output straight from global memory and copied the whole bank
  // per 128 outputs: 215 instructions per output.)
  __shared__ __align__(16) float s_bank[32 * RDS_RS_ROW];
  __shared__ float s_x[RDS_RS_SPAN];
  const int c = blockIdx.y + ch0;
  const uint32_t n171 = rr.st[c].n171[rr.par];
  const uint32_t k0 = blockIdx.x * RDS_RS_OUT;
  if (k0 >= n171) {
    return;
  }
  for (int i = threadIdx.x; i < 32 * RDS_RS_ROW; i += blockDim.x) {
    const int br = i / RDS_RS_ROW;
    const int q = i - br * RDS_RS_ROW;
    s_bank[i] = (q < RDS_RS_LEN) ? g_bank[br * RDS_RS_LEN + q] : 0.0f;
  }
  const unsigned long long phase = rr.st[c].rs_phase;
  const uint32_t k_last = min(n171, k0 + RDS_RS_OUT) - 1;
  const long i_lo = (long)((phase + (unsigned long long)k0 * step) >> 24) - (RDS_RS_LEN - 1);
  const long i_hi = (long)((phase + (unsigned long long)k_last * step) >> 24);
  const long span = i_hi - i_lo + 1;
  const float *row = mpx + (size_t)c * mpx_pitch + H_MPX;
  const float *hc = hist + (size_t)c * hist_pitch + RDS_HIST;  // hc[-1] is the newest old input
  // DSP rates above 2 x 171 kHz advance more than 2 inputs per output: the window does not fit,
  // read the inputs from global memory then (same arithmetic)
  const bool staged = span <= RDS_RS_SPAN;
  if (staged) {
    for (int a = threadIdx.x; a < (int)span; a += blockDim.x) {
      const long si = i_lo + a;
      s_x[a] = (si >= 0) ? row[si] : hc[si];
    }
  }
  __syncthreads();
  if (!staged) {
    for (uint32_t k = k0 + threadIdx.x; k <= k_last; k += blockDim.x) {
      const unsigned long long P = phase + (unsigned long long)k * step;
      const long i = (long)(P >> 24);
      const float *h = s_bank + (int)((P & 0xffffffull) >> 19) * RDS_RS_ROW;
      float smp = 0.0f;
      for (int q = 0; q < RDS_RS_LEN; q++) {
        const long si = i - (RDS_RS_LEN - 1) + q;
        smp = fmaf(h[q], (si >= 0) ? row[si] : hc[si], smp);
      }
      r171[(size_t)c * r_pitch + k] = smp;
    }
    return;
  }
#pragma unroll
  for (int u = 0; u < RDS_RS_OUT / 128; u++) {
    const uint32_t k = k0 + u * 128 + threadIdx.x;
    if (k < n171) {
      const unsigned long long P = phase + (unsigned long long)k * step;
      const int br = (int)((P & 0xffffffull) >> 19);
      const float *h = s_bank + br * RDS_RS_ROW;
      const float *x = s_x + ((long)(P >> 24) - (RDS_RS_LEN - 1) - i_lo);
      float hq[RDS_RS_ROW];
#pragma unroll
      for (int q = 0; q < RDS_RS_ROW; q += 4) {
        const float4 v = *reinterpret_cast<const float4 *>(h + q);
        hq[q] = v.x;
        hq[q + 1] = v.y;
        hq[q + 2] = v.z;
        hq[q + 3] = v.w;
      }
      float smp = 0.0f;
#pragma unroll
      for (int q = 0; q < RDS_RS_LEN; q++) {  // oldest input first, as resamp_rrrf's dot product
        smp = fmaf(hq[q], x[q], smp);
      }
      r171[(size_t)c * r_pitch + k] = smp;
    }
  }
}

// S7b: the serial part, one lane per channel, fed by the 171 kHz stream of k_rds_resample. ONE warp
// per 32 channels: it prefetches its own next tile (cp.async) before walking the current one. A
// separate mover warp would hold this kernel's 160+ registers per thread a second time for the
// whole kernel, and what the lane kernels cost the step is the registers and shared memory they
// keep from the FIR kernels running beside them, not their issue slots.
__global__ void __maxnreg__(255)
k_rds(const float *__restrict__ r171, size_t r_pitch, RdsState *st, float2 *ring,
      const float *__restrict__ g_lpf, const float *__restrict__ g_mf,
      const float *__restrict__ g_dmf, uint8_t *bits_out, uint32_t bits_cap, int ch0, int nch,
      EngineConst k, RdsRsRef rr) {
  __shared__ float s_lpf[RDS_LPF_LEN + 1];
  __shared__ float s_mf[32 * SS_LEN];
  __shared__ float s_dmf[32 * SS_LEN];
  __shared__ float2 s_wmf[SS_LEN][32];
  __shared__ float2 s_wdmf[SS_LEN][32];
  __shared__ uint32_t s_nmax;
  const int tl = threadIdx.x;
  for (int i = threadIdx.x; i < RDS_LPF_LEN; i += 32) {
    s_lpf[i] = g_lpf[i];
  }
  for (int i = threadIdx.x; i < 32 * SS_LEN; i += 32) {
    s_mf[i] = g_mf[i];
    s_dmf[i] = g_dmf[i];
  }
  constexpr int TPR = LT + 4;  // 16-byte aligned rows
  extern __shared__ float sm_rds[];
  float *t_in[2] = {sm_rds, sm_rds + 32 * TPR};
  const int c0 = ch0 + blockIdx.x * RDS_CPC;
  const int nrows = min(RDS_CPC, ch0 + nch - c0);
  const bool active = tl < nrows;
  const int c = c0 + min(tl, nrows - 1);
  constexpr float kPi = 3.14159265358979323846f;
  RdsState s = st[c];
  const uint32_t my171 = rr.st[c].n171[rr.par];
  {
    const uint32_t mine = (tl < nrows) ? my171 : 0u;
    const uint32_t mx = __reduce_max_sync(0xffffffffu, mine);
    if (threadIdx.x == 0) {
      s_nmax = mx;
    }
  }
  __syncthreads();
  for (int q = 0; q < SS_LEN; q++) {
    s_wmf[q][tl] = s.wmf[q];
    s_wdmf[q][tl] = s.wdmf[q];
  }
  int sp = 0;  // ring position of the oldest symsync window element
  float2 *ringc = ring + (size_t)c * RDS_RING;
  uint8_t *bout = bits_out + (size_t)c * bits_cap;

  float2 acc[RDS_NACC];
#pragma unroll
  for (int j = 0; j < RDS_NACC; j++) {
    acc[j] = s.acc[j];
  }
  if (active && s.realign) {
    // SubcarrierSet::reset() moved the /24 phase: rebuild the pending sums from the
    // last 254 mixed samples (the low-pass itself is not reset, subcarrier.cpp:108-114)
    const uint32_t u0 = s.ring_pos;  // absolute index of the next sample
#pragma unroll
    for (int j = 0; j < RDS_NACC; j++) {
      float ar = 0.0f, ai = 0.0f;
      const int dj = 24 * j;  // instant t_j = u0 + 24 j
      for (int back = 254 - dj; back >= 1; back--) {
        // sample u = u0 - back contributes with window index 254 - (t_j - u)
        const int idx = 254 - (dj + back);
        if (idx >= 0) {
          const float2 x = ringc[(u0 - (uint32_t)back) & (RDS_RING - 1)];
          ar = fmaf(s_lpf[idx], x.x, ar);
          ai = fmaf(s_lpf[idx], x.y, ai);
        }
      }
      acc[j] = make_float2(ar, ai);
    }
    s.realign = 0;
  }

  uint32_t produced = 0;
  const uint32_t n171 = active ? my171 : 0u;
  const int nchunks = (int)((s_nmax + LT - 1) / LT);
  // tile element ii of chunk ck <-> 171 kHz sample ck*LT + ii (rows are padded to whole tiles)
  auto prefetch = [&](int ck) {
    constexpr int cpr = LT / 4;
    const int total = nrows * cpr;
    for (int idx = tl; idx < total; idx += 32) {
      const int r = idx / cpr;
      const int q4 = 4 * (idx - r * cpr);
      cpAsync16(t_in[ck & 1] + r * TPR + q4, r171 + (size_t)(c0 + r) * r_pitch + (size_t)ck * LT + q4);
    }
  };
  if (nchunks > 0) {
    prefetch(0);
    cpAsyncCommit();
  }

  for (int ck = 0; ck < nchunks; ck++) {
    cpAsyncWait<0>();  // tile ck has landed ...
    __syncwarp();      // ... for every lane, and every lane is done reading tile ck - 1
    if (ck + 1 < nchunks) {
      prefetch(ck + 1);
      cpAsyncCommit();
    }
    const float *trow = t_in[ck & 1] + tl * TPR;
    // Samples of this lane in the tile. They are walked in groups of up to 8 that end at the lane's
    // next /24 decimation instant (or the end of the tile): inside a group nothing feeds back into
    // the NCO, so the 8 NCO steps, the 8 IEEE divisions and the 8 sincos are independent
    // instruction streams instead of one dependent chain per sample, and the symbol-rate block runs
    // once per group boundary for the whole warp, whatever the lanes' /24 phases are. Per value,
    // operations and their order are those of the per-sample loop (subcarrier.cpp:117-235).
    const uint32_t t0 = (uint32_t)ck * LT;
    const int nvalid = (n171 > t0) ? (int)min((uint32_t)LT, n171 - t0) : 0;
    int ii = 0;
    while (__any_sync(0xffffffffu, ii < nvalid)) {
      const uint32_t ph = s.since_reset % 24u;
      const int d0 = (ph == 0) ? 0 : (int)(24u - ph);  // offset of the next decimation instant
      const int m = (ii < nvalid) ? min(8, min(d0 + 1, nvalid - ii)) : 0;
      const bool heavy_last = (m > 0) && (m == d0 + 1);
      // ---- NCO::step for the first m - 1 samples (liquid_wrappers.cpp:125-139) ----
      float pn[8], ph0[8];
      ph0[0] = s.phase0;
      pn[0] = s.prev_f0_phase;
#pragma unroll
      for (int q = 1; q < 8; q++) {
        pn[q] = ncoPhaseDev(s.theta + (uint32_t)q * s.dtheta);
      }
#pragma unroll
      for (int q = 1; q < 8; q++) {
        const float delta = unwrapDev(pn[q] - pn[q - 1]);
        const float x = divBy57000(delta * 57000.f);
        ph0[q] = x;
      }
#pragma unroll
      for (int q = 1; q < 8; q++) {
        ph0[q] = unwrapDev(ph0[q - 1] + ph0[q]);
      }
#pragma unroll
      for (int q = 1; q < 8; q++) {
        if (q < m) {
          s.theta += s.dtheta;
          s.prev_f0_phase = pn[q];
          s.phase0 = ph0[q];
        }
      }
      // ---- mix down, 57 kHz low-pass sums ----
#pragma unroll
      for (int q = 0; q < 8; q++) {
        if (q < m) {
          const float smp = trow[ii + q];
          float sn, cs;
          fm_sincosf(-ph0[q], &sn, &cs);
          const float2 bb = make_float2(smp * cs, smp * sn);
          if (n171 - produced <= (uint32_t)RDS_RING) {
            ringc[s.ring_pos & (RDS_RING - 1)] = bb;
          }
          s.ring_pos++;
          produced++;
          const int base = 254 - (d0 - q);  // window index of this sample in the next output
#pragma unroll
          for (int j = 0; j < RDS_NACC; j++) {
            // base - 24 j >= 0 for every j < 10 (base >= 231)
            if (j < 10 || base >= 24 * j) {
              const float hh = s_lpf[base - 24 * j];
              acc[j].x = fmaf(hh, bb.x, acc[j].x);
              acc[j].y = fmaf(hh, bb.y, acc[j].y);
            }
          }
        }
      }
      if (heavy_last) {
        const float2 lo = make_float2(acc[0].x * k.rds_lpf_scale, acc[0].y * k.rds_lpf_scale);
#pragma unroll
        for (int j = 0; j < RDS_NACC - 1; j++) {
          acc[j] = acc[j + 1];
        }
        acc[RDS_NACC - 1] = make_float2(0.0f, 0.0f);
        // agc_crcf
        const float2 y = make_float2(lo.x * s.agc_g, lo.y * s.agc_g);
        const float e = (y.x * y.x) + (y.y * y.y);
        s.agc_y2 = ((1.0f - k.rds_agc_alpha) * s.agc_y2) + (k.rds_agc_alpha * e);
        if (s.agc_y2 > 1e-6f) {
          s.agc_g = s.agc_g * fm_expf((-0.5f * k.rds_agc_alpha) * fm_logf(s.agc_y2));
        }
        if (s.agc_g > 1e6f) {
          s.agc_g = 1e6f;
        }
        // symsync_crcf step
        s_wmf[sp][tl] = y;
        s_wdmf[sp][tl] = y;
        sp = (sp + 1 == SS_LEN) ? 0 : sp + 1;
        int n_out = 0;
        float2 sym = make_float2(0.0f, 0.0f);
        while (s.b < 32) {
          float mr = 0.0f, mi = 0.0f;
          const float *hm = s_mf + s.b * SS_LEN;
          int wp = sp;
          for (int q = 0; q < SS_LEN; q++) {
            const float2 wv = s_wmf[wp][tl];
            mr = fmaf(hm[q], wv.x, mr);
            mi = fmaf(hm[q], wv.y, mi);
            wp = (wp + 1 == SS_LEN) ? 0 : wp + 1;
          }
          if (n_out == 0) {
            sym = make_float2(mr / 3.0f, mi / 3.0f);
          }
          if (s.decim_counter == 1u) {
            s.decim_counter = 0;
            float dr = 0.0f, di = 0.0f;
            const float *hd = s_dmf + s.b * SS_LEN;
            wp = sp;
            for (int q = 0; q < SS_LEN; q++) {
              const float2 wv = s_wdmf[wp][tl];
              dr = fmaf(hd[q], wv.x, dr);
              di = fmaf(hd[q], wv.y, di);
              wp = (wp + 1 == SS_LEN) ? 0 : wp + 1;
            }
            float qe = (mr * dr) + (mi * di);
            if (qe > 1.0f) {
              qe = 1.0f;
            } else if (qe < -1.0f) {
              qe = -1.0f;
            }
            const float v0 = qe - (k.ss_a1 * s.sos_v1);
            s.q_hat = k.ss_b0 * v0;
            s.sos_v1 = v0;
            s.rate = s.rate + (k.ss_rate_adj * s.q_hat);
            s.del = s.rate + s.q_hat;
          }
          s.decim_counter++;
          s.tau = s.tau + s.del;
          const float bf = s.tau * 32.0f;
          s.b = (int)fm_roundf(bf);
          n_out++;
        }
        s.tau = s.tau - 1.0f;
        s.b -= 32;
        if (n_out == 1) {
          const float pe_raw = (sym.x > 0.0f) ? sym.y : -sym.y;
          const float pe = fm_clampf(pe_raw, -kPi, kPi);
          const float dphi = pe * 12.0f;
          s.dtheta += ncoConstrainDev(dphi * k.rds_pll_alpha);
          s.theta += ncoConstrainDev(dphi * k.rds_pll_beta);
          // biphase
          const float bre = (sym.x - s.bi_prev_re) * 0.5f;
          const bool bval = bre >= 0.0f;
          const bool has = ((s.bi_clock & 1u) == s.bi_polarity);
          s.bi_prev_re = sym.x;
          if (s.bi_clock & 1u) {
            s.bi_odd += fabsf(bre);
          } else {
            s.bi_even += fabsf(bre);
          }
          s.bi_clock++;
          if (s.bi_clock == 128u) {
            if (s.bi_even > s.bi_odd) {
              s.bi_polarity = 0;
            } else if (s.bi_odd > s.bi_even) {
              s.bi_polarity = 1;
            }
            s.bi_even = 0.0f;
            s.bi_odd = 0.0f;
            s.bi_clock = 0;
          }
          if (has) {
            const bool bit = (bval != (s.delta_prev != 0));
            s.delta_prev = bval ? 1 : 0;
            if (s.n_bits < bits_cap) {
              bout[s.n_bits] = bit ? 1 : 0;
            }
            s.n_bits++;
          }
        }
      }
      if (m > 0) {
        // NCO::step of the group's last sample (after the loop filter moved the NCO)
        s.theta += s.dtheta;
        const float pnl = ncoPhaseDev(s.theta);
        const float delta = unwrapDev(pnl - s.prev_f0_phase);
        s.prev_f0_phase = pnl;
        s.phase0 = unwrapDev(s.phase0 + (divBy57000(delta * 57000.f)));
        s.since_reset += (uint32_t)m;
        ii += m;
      }
    }
    __syncthreads();
  }
  if (!active) {
    return;
  }
#pragma unroll
  for (int j = 0; j < RDS_NACC; j++) {
    s.acc[j] = acc[j];
  }
  for (int q = 0; q < SS_LEN; q++) {
    s.wmf[q] = s_wmf[sp][tl];
    s.wdmf[q] = s_wdmf[sp][tl];
    sp = (sp + 1 == SS_LEN) ? 0 : sp + 1;
  }
  st[c] = s;
}

// ---------------------------------------------------------------------------
// K7c: RDS block synchroniser (block_sync.cpp:235-313). Phase 1 evaluates the (26,16) syndrome
// of the 26-bit window ending at EVERY bit offset, in parallel over (channel, bit); phase 2 is
// the sequential sync / FEC state machine, one lane per channel, consuming those syndromes
// (every bit while searching for sync, every 26th once locked).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_blocksync(const uint8_t *__restrict__ bits, uint32_t bits_cap, RdsState *st, unsigned long long *words,
            fmgpu_rds_group *groups, uint32_t gcap, fmgpu_block_status *status, int status_pitch, int blk,
            int ch0, int nch) {
  __shared__ uint32_t s_reg[32], s_nb[32], s_b0[32];
  const int c0 = ch0 + blockIdx.x * 32;
  const int nrows = min(32, ch0 + nch - c0);
  if (threadIdx.x < 32) {
    const bool valid = (int)threadIdx.x < nrows;
    s_reg[threadIdx.x] = valid ? st[c0 + threadIdx.x].reg : 0u;
    s_nb[threadIdx.x] = valid ? min(st[c0 + threadIdx.x].n_bits, bits_cap) : 0u;
    // bits [0, b0) of this call went through the synchroniser with the earlier logical blocks
    s_b0[threadIdx.x] = valid ? min(st[c0 + threadIdx.x].bits_done, s_nb[threadIdx.x]) : 0u;
  }
  __syncthreads();
  for (int r = 0; r < nrows; r++) {
    const uint32_t nb = s_nb[r];
    const uint32_t b0 = s_b0[r];
    const uint32_t reg = s_reg[r];  // the 26-bit register after bit b0 - 1
    const uint8_t *brow = bits + (size_t)(c0 + r) * bits_cap;
    unsigned long long *wrow = words + (size_t)(c0 + r) * bits_cap;
    for (uint32_t i = b0 + threadIdx.x; i < nb; i += blockDim.x) {
      uint32_t w = 0;
#pragma unroll
      for (int q = 25; q >= 0; q--) {  // bit i-q of the stream; bits before b0 sit in reg
        const int idx = (int)i - q;
        const uint32_t bit = (idx >= (int)b0) ? (uint32_t)brow[idx]
                                              : ((reg >> ((int)b0 - 1 - idx)) & 1u);
        w = (w << 1) | bit;
      }
      wrow[i] = (unsigned long long)w | ((unsigned long long)rdsSyndromeDev(w) << 32);
    }
  }
  __syncthreads();
  if ((int)threadIdx.x >= nrows) {
    return;
  }
  const int c = c0 + threadIdx.x;
  RdsState s = st[c];
  const uint32_t nb = s_nb[threadIdx.x];
  const uint32_t bit0 = s_b0[threadIdx.x];
  const unsigned long long *wrow = words + (size_t)c * bits_cap;
  fmgpu_rds_group *gout = groups ? groups + (size_t)c * gcap : nullptr;
  const uint32_t before = s.n_groups;
  for (uint32_t i = bit0; i < nb; i++) {
    const unsigned long long w = wrow[i];
    rdsPushWord(s, (uint32_t)w & 0x3ffffffu, (uint32_t)(w >> 32), gout, gcap, (uint32_t)blk);
  }
  if (status) {
    status[(size_t)c * status_pitch].n_groups = (int)(s.n_groups - before);
  }
  // only the block-synchroniser fields changed
  RdsState *o = &st[c];
  o->bitcount = s.bitcount;
  o->until = s.until;
  o->reg = s.reg;
  o->bits_since_lost = s.bits_since_lost;
  o->expected = s.expected;
  o->in_sync = s.in_sync;
  o->err_ptr = s.err_ptr;
  o->err_mask = s.err_mask;
  for (int q = 0; q < 4; q++) {
    o->cur_data[q] = s.cur_data[q];
    o->pulse_pos[q] = s.pulse_pos[q];
    o->pulse_off[q] = s.pulse_off[q];
  }
  o->cur_recv = s.cur_recv;
  o->cur_err = s.cur_err;
  o->n_groups = s.n_groups;
  o->bits_done = nb;
}

// ---------------------------------------------------------------------------
// RF level meter (signal_level.cpp:145-178): exact integer sums of the IQ bytes of every
// logical block. HBM-bound by design (2 B per IQ sample in, 48 B per block out), so the per-sample
// instruction count is what has to stay small: 128-bit loads; the four sums through dp4a (two
// samples per instruction: I0*m0 + Q0*m1 + I1*m2 + Q1*m3 with byte masks or the word itself as the
// second operand); the two clip counters behind a branch-free any-byte test per word — a byte is
// near clip (<= 8 or >= 247) iff (byte + 9) mod 256 < 18 — so the per-sample comparisons only run
// for the rare words that hold such a byte (hard clip, <= 1 or >= 254, is a subset of near clip).
// uint32 partials per thread (a thread sees a few hundred samples), one 64-bit atomic per warp.
__global__ void __launch_bounds__(256)
k_siglevel(const uint8_t *__restrict__ iq, size_t iq_stride, fmgpu_level_sums *sums, int nblk,
           long samples_per_block, int slices, int ch0) {
  const int c = blockIdx.y + ch0;
  const int b = blockIdx.x / slices;
  const int sl = blockIdx.x - b * slices;
  const long per = (samples_per_block + slices - 1) / slices;
  const long s0 = sl * per;
  const long s1 = min(samples_per_block, s0 + per);
  const uint8_t *base = iq + (size_t)c * iq_stride + 2 * (size_t)b * samples_per_block;
  uint32_t si = 0, sq = 0, sii = 0, sqq = 0;
  uint32_t hard = 0, nearc = 0, cnt = 0;
  auto one = [&](uint32_t vi, uint32_t vq) {
    si += vi;
    sq += vq;
    sii += vi * vi;
    sqq += vq * vq;
    hard += (vi <= 1u || vi >= 254u || vq <= 1u || vq >= 254u) ? 1u : 0u;
    nearc += (vi <= 8u || vi >= 247u || vq <= 8u || vq >= 247u) ? 1u : 0u;
    cnt++;
  };
  auto word = [&](uint32_t w) {  // two samples: bytes I0, Q0, I1, Q1
    si = __dp4a(w, 0x00010001u, si);
    sq = __dp4a(w, 0x01000100u, sq);
    sii = __dp4a(w, w & 0x00ff00ffu, sii);
    sqq = __dp4a(w, w & 0xff00ff00u, sqq);
    // byte + 9 (mod 256) in every lane of the word, then "any byte < 18"
    const uint32_t t = ((w & 0x7f7f7f7fu) + 0x09090909u) ^ (w & 0x80808080u);
    if ((t - 0x12121212u) & ~t & 0x80808080u) {
      const uint32_t i0 = w & 0xffu, q0 = (w >> 8) & 0xffu, i1 = (w >> 16) & 0xffu, q1 = w >> 24;
      hard += (i0 <= 1u || i0 >= 254u || q0 <= 1u || q0 >= 254u) ? 1u : 0u;
      hard += (i1 <= 1u || i1 >= 254u || q1 <= 1u || q1 >= 254u) ? 1u : 0u;
      nearc += (i0 <= 8u || i0 >= 247u || q0 <= 8u || q0 >= 247u) ? 1u : 0u;
      nearc += (i1 <= 8u || i1 >= 247u || q1 <= 8u || q1 >= 247u) ? 1u : 0u;
    }
    cnt += 2;
  };
  // 16-byte chunks (8 IQ pairs); block starts are 16-byte aligned when samples_per_block % 8 == 0
  const long c0 = (s0 + 7) >> 3, c1 = s1 >> 3;
  const bool aligned = ((reinterpret_cast<uintptr_t>(base) & 15u) == 0);
  if (aligned && c1 > c0) {
    for (long s = s0 + threadIdx.x; s < (c0 << 3); s += blockDim.x) {  // head
      one(base[2 * s], base[2 * s + 1]);
    }
    for (long ck = c0 + threadIdx.x; ck < c1; ck += blockDim.x) {       // 128-bit body
      const uint4 raw = __ldg(reinterpret_cast<const uint4 *>(base + 16 * ck));
      word(raw.x);
      word(raw.y);
      word(raw.z);
      word(raw.w);
    }
    for (long s = (c1 << 3) + threadIdx.x; s < s1; s += blockDim.x) {   // tail
      one(base[2 * s], base[2 * s + 1]);
    }
  } else {
    for (long s = s0 + threadIdx.x; s < s1; s += blockDim.x) {
      one(base[2 * s], base[2 * s + 1]);
    }
  }
  unsigned long long wi = si, wq = sq, wii = sii, wqq = sqq;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    wi += __shfl_down_sync(0xffffffffu, wi, o);
    wq += __shfl_down_sync(0xffffffffu, wq, o);
    wii += __shfl_down_sync(0xffffffffu, wii, o);
    wqq += __shfl_down_sync(0xffffffffu, wqq, o);
    hard += __shfl_down_sync(0xffffffffu, hard, o);
    nearc += __shfl_down_sync(0xffffffffu, nearc, o);
    cnt += __shfl_down_sync(0xffffffffu, cnt, o);
  }
  if ((threadIdx.x & 31) == 0) {
    fmgpu_level_sums *o = &sums[(size_t)c * nblk + b];
    atomicAdd(reinterpret_cast<unsigned long long *>(&o->sum_i), wi);
    atomicAdd(reinterpret_cast<unsigned long long *>(&o->sum_q), wq);
    atomicAdd(reinterpret_cast<unsigned long long *>(&o->sum_ii), wii);
    atomicAdd(reinterpret_cast<unsigned long long *>(&o->sum_qq), wqq);
    atomicAdd(&o->hard_clip, hard);
    atomicAdd(&o->near_clip, nearc);
    atomicAdd(&o->n_samples, cnt);
  }
}

// ---------------------------------------------------------------------------
// K8: float audio -> interleaved int16 PCM (audio_output.cpp:1386-1391,1458-1459). Streaming,
// HBM-bound: 8 B in, 4 B out per frame.
// ---------------------------------------------------------------------------
__global__ void k_pack_pcm16(const float *__restrict__ audio, size_t acap,
                             const uint32_t *__restrict__ n_audio, float volume,
                             short2 *__restrict__ pcm, int C) {
  const int c = blockIdx.y;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C || i >= n_audio[c] || i >= acap) {
    return;
  }
  const float l = audio[((size_t)c * 2 + 0) * acap + i] * volume;
  const float r = audio[((size_t)c * 2 + 1) * acap + i] * volume;
  const float lc = fmaxf(-1.0f, fminf(1.0f, l));
  const float rc = fmaxf(-1.0f, fminf(1.0f, r));
  pcm[(size_t)c * acap + i] = make_short2((short)(lc * 32767.0f), (short)(rc * 32767.0f));
}

// ---------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------
#define FMGPU_DECIM_CASE(MM)                                                                     \
  case MM: {                                                                                     \
    constexpr int T = 4 * DECIM_NT;                                                              \
    const int tile_len = (T + Pp - 1) * MM;                                                      \
    const size_t smem = (size_t)(tile_len + 2 * (tile_len / (4 * MM)) + 4) * sizeof(float2);     \
    static DeviceOnce attrs; /* per device: device_once.h */                                     \
    attrs.run([] {                                                                               \
      return cudaFuncSetAttribute(k_decim<MM>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                                  160 * 1024);                                                   \
    });                                                                                          \
    dim3 grid((n_out + T - 1) / T, nch);                                                         \
    k_decim<MM><<<grid, DECIM_NT, smem, stream>>>(iq, iq_stride, hist, hist_valid, x1, x1_pitch, \
                                                  n_out, ch0, Pp, scale, taps);                  \
    break;                                                                                       \
  }

void launchDecim(int M, const uint8_t *iq, size_t iq_stride, const uint8_t *hist,
                 const int *hist_valid, float2 *x1, size_t x1_pitch, int n_out, int ch0, int nch, int Pp, int L, float scale,
                 const TapsParam &taps, const TapsParam &taps_unpadded, cudaStream_t stream) {
  switch (M) {
    FMGPU_DECIM_CASE(2)
    FMGPU_DECIM_CASE(4)
    FMGPU_DECIM_CASE(5)
    FMGPU_DECIM_CASE(8)
    FMGPU_DECIM_CASE(10)
    FMGPU_DECIM_CASE(16)
  default: {
    dim3 grid((n_out + 127) / 128, nch);
    k_decim_generic<<<grid, 128, 0, stream>>>(iq, iq_stride, hist, hist_valid, x1, x1_pitch, n_out,
                                              ch0, M, L, scale, taps_unpadded);
    break;
  }
  }
}

void launchConvertU8(const uint8_t *iq, size_t iq_stride, float2 *x1, size_t x1_pitch, int n,
                     int ch0, int nch, cudaStream_t stream) {
  dim3 grid((n + 255) / 256, nch);
  k_convert_u8<<<grid, 256, 0, stream>>>(iq, iq_stride, x1, x1_pitch, n, ch0);
}

void launchRequantU8(const float2 *x1, size_t x1_pitch, uint8_t *out, size_t out_stride, int n, int ch0,
                     int nch, cudaStream_t stream) {
  dim3 grid((n + 255) / 256, nch);
  k_requant_u8<<<grid, 256, 0, stream>>>(x1, x1_pitch, out, out_stride, n, ch0);
}

void launchCarryIq(uint8_t *hist, int *hist_valid, const uint8_t *iq, size_t iq_stride, long n_in,
                   int ch0, int nch, cudaStream_t stream) {
  k_carry_iq<<<nch, H_IQ, 0, stream>>>(reinterpret_cast<uchar2 *>(hist), hist_valid, iq, iq_stride,
                                       n_in, ch0);
}

void launchCarryF32(float *buf, size_t pitch, int H, size_t n, int ch0, int nch,
                    cudaStream_t stream) {
  k_carry<float><<<nch, 512, 0, stream>>>(buf, pitch, H, n, ch0);
}

void launchCarryF2(float2 *buf, size_t pitch, int H, size_t n, int ch0, int nch,
                   cudaStream_t stream) {
  k_carry<float2><<<nch, 512, 0, stream>>>(buf, pitch, H, n, ch0);
}

void launchDcBlock(const float2 *x1, size_t x1_pitch, const uint8_t *iq_u8, size_t iq_stride,
                   float2 *x2, size_t x2_pitch, DemodState *st, fmgpu_block_status *status,
                   int status_pitch, int n_total, int ch0, int nch, float a1, cudaStream_t stream) {
  constexpr size_t smem = 3 * 32 * (2 * LT + 4) * sizeof(float);
  static DeviceOnce attrs;  // per device: device_once.h
  attrs.run([] { return cudaFuncSetAttribute(k_dcblock, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); });
  k_dcblock<<<(nch + 31) / 32, 32, smem, stream>>>(x1, x1_pitch, iq_u8, iq_stride, x2, x2_pitch, st,
                                               status, status_pitch, n_total, ch0, nch, a1);
}

void launchDcBlockScan(const float2 *x1, size_t x1_pitch, float2 *x2, size_t x2_pitch, DemodState *st,
                       fmgpu_block_status *status, int status_pitch, int n_total, int ch0, int nch,
                       float a1, cudaStream_t stream) {
  k_dcblock_scan<<<(nch + 3) / 4, 128, 0, stream>>>(x1, x1_pitch, x2, x2_pitch, st, status, status_pitch,
                                                   n_total, ch0, nch, a1);
}

void launchChanFir(const float2 *x2, size_t x2_pitch, float2 *ybuf, size_t y_pitch,
                   const float *chan_taps, const int *chan_lp, const float *chan_scale,
                   const ChanParams *cp, int n_total, int ch0, int nch, cudaStream_t stream) {
  constexpr int T = 1024;
  const int tile_len = T + CHAN_TAPS_PITCH - 1 + 8;
  const size_t smem = (size_t)(tile_len + (tile_len >> 3) + 2) * sizeof(float2);
  dim3 grid((n_total + T - 1) / T, nch);
  k_chanfir<<<grid, 128, smem, stream>>>(x2, x2_pitch, ybuf, y_pitch, chan_taps, chan_lp, chan_scale, cp,
                                         n_total, ch0);
}

void launchAgc(float2 *ybuf, size_t y_pitch, DemodState *st, const ChanParams *cp, int n_total,
               int ch0, int nch, cudaStream_t stream) {
  constexpr size_t smem = 2 * 32 * (2 * LT + 4) * sizeof(float);
  static DeviceOnce attrs;  // per device: device_once.h
  attrs.run([] { return cudaFuncSetAttribute(k_agc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); });
  k_agc<<<(nch + 31) / 32, 32, smem, stream>>>(ybuf, y_pitch, st, cp, n_total, ch0, nch);
}

void launchFreqDem(const float2 *ybuf, size_t y_pitch, float *mpx, size_t mpx_pitch, int n_total,
                   int ch0, int nch, float ref, cudaStream_t stream) {
  dim3 grid((n_total + 1023) / 1024, nch);  // 256 threads x 4 samples
  k_freqdem<<<grid, 256, 0, stream>>>(ybuf, y_pitch, mpx, mpx_pitch, n_total, ch0, ref);
}

// K3 / K5: real FIR with taps in the kernel-parameter constant bank (pilot band-pass 305/325 taps;
// 2 x 121-tap 15 kHz low-pass). Two real signals that share the taps ride in the two halves of
// FFMA2 — the L and R rows of one channel (15 kHz low-pass), or the same row of two neighbouring
// channels (pilot band-pass; with an odd channel count the last CTA computes one row, has_b =
// false). The tile is interleaved into float2 {a, b} in shared memory; the inner loop is the
// complex FIR's (8 outputs x 2 signals per thread, one LDS.64 and 8 FFMA2 per tap, taps as
// uniform-register scalars). Each half is the oldest-first fmaf chain of a scalar FIR.
__global__ void __launch_bounds__(128)
k_fir_pair(FirRealJob job, int pair_channels, int nch, const __grid_constant__ TapsParam taps) {
  constexpr int R = 8;
  constexpr int T = 128 * R;
  extern __shared__ float2 fp_x[];
  const int n0 = blockIdx.x * T;
  const int t = threadIdx.x;
  const int Lp = job.Lp;
  // rows a and b of this CTA
  const int ca = job.ch0 + (pair_channels ? 2 * blockIdx.y : blockIdx.y);
  const bool has_b = pair_channels ? (2 * (int)blockIdx.y + 1 < nch) : true;
  const int cb = pair_channels ? (has_b ? ca + 1 : ca) : ca;
  const float *rowa = job.in[0] + (size_t)ca * job.in_pitch + job.in_off;
  const float *rowb = (pair_channels ? job.in[0] : job.in[1]) + (size_t)cb * job.in_pitch + job.in_off;
  const int b0 = n0 - (Lp - 1);
  const int tile_len = T + Lp - 1 + R;
  for (int a = t; a < tile_len; a += 128) {
    const int s = b0 + a;
    float2 v = make_float2(0.0f, 0.0f);
    if (s < job.n_total) {
      v = make_float2(rowa[s], rowb[s]);
    }
    fp_x[a + (a >> 3)] = v;
  }
  __syncthreads();
  float2 acc[R], win[R];
#pragma unroll
  for (int j = 0; j < R; j++) {
    acc[j] = make_float2(0.0f, 0.0f);
    const int a = t * R + j;
    win[j] = fp_x[a + (a >> 3)];
  }
  // element a = t*R + i + u + R sits at a + (a >> 3) = (R + 1) * (t + 1 + i / R) + u: one pointer
  // that advances by R + 1 per round, so every LDS has an immediate offset (the index arithmetic
  // per load was 12 % of this kernel's instructions)
  const float2 *wp = fp_x + (R + 1) * (t + 1);
  for (int i = 0; i < Lp; i += R) {
#pragma unroll
    for (int u = 0; u < R; u++) {
      const float h = taps.h[i + u];
#pragma unroll
      for (int j = 0; j < R; j++) {
        acc[j] = fma2(h, win[(j + u) & (R - 1)], acc[j]);
      }
      win[u] = wp[u];
    }
    wp += R + 1;
  }
  float *outa = job.out[0] + (size_t)ca * job.out_pitch + job.out_off;
  float *outb = (pair_channels ? job.out[0] : job.out[1]) + (size_t)cb * job.out_pitch + job.out_off;
#pragma unroll
  for (int j = 0; j < R; j++) {
    const int n = n0 + t * R + j;
    if (n < job.n_total) {
      outa[n] = acc[j].x * job.scale;
      if (has_b) {
        outb[n] = acc[j].y * job.scale;
      }
    }
  }
}

void launchFirReal(const FirRealJob &job, int nsig, int nch, const TapsParam &taps,
                   cudaStream_t stream) {
  constexpr int T = 1024;
  const int tile_len = T + job.Lp - 1 + 8;
  const size_t smem = (size_t)(tile_len + (tile_len >> 3) + 2) * sizeof(float2);
  const int pair_channels = (nsig == 2) ? 0 : 1;
  dim3 grid((job.n_total + T - 1) / T, pair_channels ? (nch + 1) / 2 : nch);
  k_fir_pair<<<grid, 128, smem, stream>>>(job, pair_channels, nch, taps);
}

void launchStereo(const float *mpx, size_t mpx_pitch, const float *pilot, size_t pilot_pitch,
                  float *lraw, float *rraw, size_t lr_pitch, StereoState *st, const ChanParams *cp,
                  fmgpu_block_status *status, int status_pitch, int n_total, int ch0, int nch,
                  const EngineConst &k, cudaStream_t stream) {
  constexpr size_t smem = STEREO_TILES * STEREO_CPC * (STEREO_ST + 4) * sizeof(float);  // tiles of [CPC][ST + 4]
  static DeviceOnce attrs;  // per device: device_once.h
  attrs.run([] { return cudaFuncSetAttribute(k_stereo, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); });
  k_stereo<<<(nch + STEREO_CPC - 1) / STEREO_CPC, STEREO_THREADS, smem, stream>>>(mpx, mpx_pitch, pilot, pilot_pitch, lraw, rraw,
                                                 lr_pitch, st, cp, status, status_pitch, n_total,
                                                 ch0, nch, k);
}

void launchPrepare(AudioState *au, RdsState *rds, fmgpu_block_status *status, int status_pitch,
                   int n_total, int ch0, int nch, uint32_t aud_step, uint32_t rds_step, int do_audio,
                   int do_mono, int do_rds, int first, RdsRsRef rr, cudaStream_t stream) {
  k_prepare<<<(nch + 127) / 128, 128, 0, stream>>>(au, rds, status, status_pitch, n_total, ch0, nch,
                                                  aud_step, rds_step, do_audio, do_mono, do_rds, first,
                                                  rr);
}

void launchCommit(AudioState *au, RdsState *rds, int ch0, int nch, int do_audio, int do_mono,
                  int do_rds, RdsRsRef rr, cudaStream_t stream) {
  k_commit<<<(nch + 127) / 128, 128, 0, stream>>>(au, rds, ch0, nch, do_audio, do_mono, do_rds, rr);
}

void launchResample(const float *in0, const float *in1, size_t in_pitch, int in_off,
                    const float *hist, int hist_pitch, float *out, size_t acap, const float *bank,
                    uint32_t step, const AudioState *au, int mono, int max_out, int ch0, int nch,
                    cudaStream_t stream) {
  if (max_out <= 0) {
    return;
  }
  dim3 grid((max_out + 127) / 128, nch);
  k_resample<<<grid, 128, 32 * AUD_RS_LEN * sizeof(float), stream>>>(
      in0, in1, in_pitch, in_off, hist, hist_pitch, out, acap, bank, step, au, mono, ch0);
}

void launchSaveTail(const float *src, size_t src_pitch, int src_off, float *hist, int hist_pitch,
                    int H, long n, int ch0, int nch, cudaStream_t stream) {
  k_save_tail<<<nch, 32, 0, stream>>>(src, src_pitch, src_off, hist, hist_pitch, H, n, ch0);
}

void launchAudioIir(float *audio, size_t acap, AudioState *au, const ChanParams *cp, int ch0,
                    int nch, float dc_a1, int mono, int clamp, int mono_dup, cudaStream_t stream) {
  const int lanes = mono ? nch : 2 * nch;
  k_audio_iir<<<(lanes + 31) / 32, 32, 0, stream>>>(audio, acap, au, cp, ch0, nch, dc_a1, mono,
                                                   clamp, mono_dup);
}

void launchAudioIirScan(float *audio, size_t acap, AudioState *au, const ChanParams *cp, int ch0,
                        int nch, float dc_a1, int clamp, cudaStream_t stream) {
  k_audio_iir_scan<<<(2 * nch + 3) / 4, 128, 0, stream>>>(audio, acap, au, cp, ch0, nch, dc_a1, clamp);
}

void launchStoreCounts(const AudioState *au, const RdsState *rds, uint32_t *n_audio,
                       uint32_t *n_groups, int ch0, int nch, int mono, uint32_t acap, uint32_t gcap,
                       cudaStream_t stream) {
  k_store_counts<<<(nch + 127) / 128, 128, 0, stream>>>(au, rds, n_audio, n_groups, ch0, nch, mono,
                                                       acap, gcap);
}

void launchRdsResample(const float *mpx, size_t mpx_pitch, const float *hist, int hist_pitch,
                       RdsRsRef rr, const float *bank, float *r171, size_t r_pitch,
                       int max_171, int ch0, int nch, const EngineConst &k, cudaStream_t stream) {
  dim3 grid((max_171 + RDS_RS_OUT - 1) / RDS_RS_OUT, nch);
  k_rds_resample<<<grid, 128, 0, stream>>>(mpx, mpx_pitch, hist, hist_pitch, rr, bank, r171, r_pitch,
                                           k.rds_step, ch0);
}

void launchRdsDemod(RdsState *st, float2 *ring, const float *lpf, const float *mf, const float *dmf,
                    const float *r171, size_t r_pitch, uint8_t *bits_out, uint32_t bits_cap, int ch0,
                    int nch, const EngineConst &k, RdsRsRef rr, cudaStream_t stream) {
  constexpr size_t smem = 2 * 32 * (LT + 4) * sizeof(float);
  k_rds<<<(nch + RDS_CPC - 1) / RDS_CPC, 32, smem, stream>>>(r171, r_pitch, st, ring, lpf, mf, dmf, bits_out,
                                              bits_cap, ch0, nch, k, rr);
}

void launchBlockSync(const uint8_t *bits, uint32_t bits_cap, RdsState *st, unsigned long long *words,
                     fmgpu_rds_group *groups, uint32_t gcap, fmgpu_block_status *status,
                     int status_pitch, int blk, int ch0, int nch, cudaStream_t stream) {
  k_blocksync<<<(nch + 31) / 32, 128, 0, stream>>>(bits, bits_cap, st, words, groups, gcap, status,
                                                  status_pitch, blk, ch0, nch);
}

void launchSigLevel(const uint8_t *iq, size_t iq_stride, fmgpu_level_sums *sums, int nblk,
                    long samples_per_block, int ch0, int nch, cudaStream_t stream) {
  // enough CTAs to fill the machine even for few channels, ~16K samples per CTA at most
  long slices = std::min<long>(64, std::max<long>(1, samples_per_block / 16384));
  // the kernel's per-thread uint32 partials hold 255^2 * 32768 samples: never give a thread more
  slices = std::max<long>(slices, (samples_per_block + 256L * 32768 - 1) / (256L * 32768));
  dim3 grid((unsigned)(nblk * slices), nch);
  k_siglevel<<<grid, 256, 0, stream>>>(iq, iq_stride, sums, nblk, samples_per_block, (int)slices, ch0);
}

void launchPackPcm16(const float *audio, size_t acap, const uint32_t *n_audio, float volume,
                     int16_t *pcm, int C, int max_frames, cudaStream_t stream) {
  dim3 grid((max_frames + 255) / 256, C);
  k_pack_pcm16<<<grid, 256, 0, stream>>>(audio, acap, n_audio, volume,
                                         reinterpret_cast<short2 *>(pcm), C);
}

}  // namespace fmgpu
