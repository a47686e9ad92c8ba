// fir_tc.cu — the real-tap FIRs of the stereo decoder on the 5th-generation tensor cores: the 19 kHz
// pilot band-pass and the L/R 15 kHz low-pass (/root/reference/src/stereo_decoder.cpp:25-63,172-173,
// 233-239; liquid firfilt_rrrf_execute, one float chain of 305 / 121 terms per output there).
//
//   y_r[n] = scale * sum_i h[i] * x_r[n - (Lp-1) + i]          r = a row (channel, or channel x {L, R})
//
// evaluated as an EXACT INTEGER contraction, like the decimator of decim_tc.cu, but for float data:
//   * the samples become 24-bit offset-binary fixed point, q = rni(x * 2^d) + 2^23 (d = 22 for the
//     multiplex, |x| < 2: one rounding of 1.2e-7, the float ulp at that magnitude; d = 20 for the
//     matrix outputs, |x| < 8), split into three unsigned byte planes;
//   * the taps become round(h * 2^S) (S: the largest tap fills 23 bits), split into three signed
//     base-256 digits; B is the banded (Toeplitz) matrix of those digits, [K = window][N = 3 x 32];
//   * tcgen05.mma kind::i8 (u8 x s8 -> s32), M = 128 rows, N = 96, K = 32 per instruction. Plane a
//     accumulates into columns [32 a, 32 a + 96) of one 160-column accumulator, so that products of
//     equal weight 256^(a + l) share a column: five limb sets of 32 outputs;
//   * the epilogue removes the 2^23 offset limb-wise in integers (2^23 * sum of the integer taps) and
//     recombines the five limbs in float, most significant first.
// The result is the FIR of the quantised samples with taps good to 2^-S, to within three float
// roundings of the exact sum: closer to the real-number answer than the reference's float chain,
// not bit-identical to it (k_fir_pair in kernels.cu stays the bit-exact flavour).
//
// No operand of the data ever sits in shared memory in MMA layout: the A operand lives in TENSOR
// MEMORY. One persistent CTA per SM, fourteen warps:
//   warp 0     TMA producer: [128 rows x 32 floats] boxes of the input rows -> staging ring
//   warp 1     allocates TMEM, issues the MMAs (one elected lane; A from TMEM, B from shared memory)
//   warps 2-5, 10-13  epilogue, two warps per TMEM lane quadrant (outputs 0..15 / 16..31 of the tile):
//              tcgen05.ld the accumulator columns, recombine, stage in 64B-swizzled shared memory, one
//              TMA store of [32 rows x 16 floats] per warp and tile; then zero the columns
//              (tcgen05.st) so that every MMA accumulates
//   warps 6-9  converters: staged floats -> fixed point -> three byte planes -> tcgen05.st into the
//              TMEM ring of 32-sample sub-chunks (lane = row, 8 columns = 32 bytes of K per plane)
// A tile is 32 outputs of 128 rows; its window is KS sub-chunks (KS = WS0/32 + 1, WS0 = the taps'
// reach rounded up to 32), and consecutive tiles of a row tile share all but one of them. Every CTA
// owns one contiguous range of the (row tile, time) tile sequence: perfect balance, and the window
// is primed once per range (and once more where the range crosses into the next row tile).
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "device_once.h"
#include "fm_math.h"
#include "kernels.h"
#include "tc_common.cuh"

namespace fmgpu {

namespace {

using namespace tc;

constexpr int FT_ROWS = 128;          // rows per tile (UMMA M)
constexpr int FT_NO = 32;             // outputs per tile = samples per sub-chunk
constexpr int FT_PLANES = 3;          // data bytes
constexpr int FT_DIGITS = 3;          // tap digits
constexpr int FT_N = FT_DIGITS * FT_NO;                    // 96 (UMMA N)
constexpr int FT_LIMBS = FT_PLANES + FT_DIGITS - 1;        // 5 limb sets
constexpr int FT_ACC_COLS = FT_LIMBS * FT_NO;              // 160 TMEM columns per accumulator
constexpr int FT_SLOT_COLS = FT_PLANES * 8;                // 24 TMEM columns per sub-chunk slot
constexpr int FT_BCHUNK = FT_N * 128;                      // bytes of one 128-byte K chunk of B (12 KB)
constexpr int FT_MAX_KS = 12;
constexpr int ftBBytes(int ks) { return ((ks + 3) / 4) * FT_BCHUNK; }   // 12 KB per 128 bytes of K
constexpr int FT_NSTG_MAX = 4;                             // float staging slots (16 KB each): a launch parameter
constexpr int FT_NSTG_DEFAULT = 3;
constexpr int FT_STG_BYTES = FT_ROWS * FT_NO * 4;
constexpr int FT_HALF = FT_NO / 2;                         // outputs per epilogue warp and tile
constexpr int FT_OUT_BYTES = 32 * FT_HALF * 4;             // one epilogue warp's staging tile (2 KB)
constexpr int FT_THREADS = 448;                            // 14 warps
// shared memory of a CTA: B image, staging ring, 8 epilogue warps x 2 output tiles, barriers. Kept
// small (89 .. 117 KB) so that the lane kernels' CTAs stay resident beside it.
constexpr size_t ftSmemBytes(int ks, int nstg) {
  return 1024 + ftBBytes(ks) + (size_t)nstg * FT_STG_BYTES + 16 * FT_OUT_BYTES + 512;
}

struct FirTcParams {
  int tiles_row;      // tiles per row = n_total / 32
  int row_tiles;      // 128-row tiles per signal
  int nsig;
  int tiles_total;    // nsig * row_tiles * tiles_row
  int in_x0;          // float index inside an input row of tile 0's window start (in_off - WS0)
  int out_x0;         // float index inside an output row of output 0
  int off2, off3, off4;   // 2^23 * sum(hq) as limbs 2..4 (limbs 0, 1 are zero)
  float dscale;       // 2^data_shift: samples are quantised to 2^-data_shift
  float out_scale;    // scale / 2^(S + data_shift)
  // complex form (channel filter + discriminator): rows are (channel, {I, Q}) pairs on adjacent lanes
  int nstg;           // staging slots in use (2 .. FT_NSTG_MAX)
  int nch;            // channels of the call
  float fd_ref;       // discriminator scale 1 / (2 pi kf)
  const float2 *y_prev;   // [c * y_pitch]: the filter output in front of this block (discriminator r_prev)
  float2 *y_last;         // [c * y_pitch]: this block's last filter output, for the next block
  size_t y_pitch;
};

// CTA b owns tiles [lo, hi) of the (signal, row tile, time) sequence
__device__ __forceinline__ void tileRange(const FirTcParams &p, int *lo, int *hi) {
  const long long t = p.tiles_total;
  *lo = static_cast<int>(t * blockIdx.x / gridDim.x);
  *hi = static_cast<int>(t * (blockIdx.x + 1) / gridDim.x);
}
// the run of tiles starting at `cur` that stays inside one row tile: (signal, row tile, first tile, count)
struct Run {
  int sig, rt, t0, nt;
  int own;      // tiles of the CTA's range in this run (cur advances by this)
  int primer;   // complex form: the run starts one tile early; that tile only yields the discriminator's
                // previous sample (its outputs belong to another CTA)
};
template <bool CPLX>
__device__ __forceinline__ Run nextRun(const FirTcParams &p, int cur, int hi) {
  Run r;
  const int row = cur / p.tiles_row;
  r.t0 = cur - row * p.tiles_row;
  r.own = min(hi - cur, p.tiles_row - r.t0);
  r.nt = r.own;
  r.sig = row / p.row_tiles;
  r.rt = row - r.sig * p.row_tiles;
  r.primer = 0;
  if (CPLX && r.t0 > 0) {
    r.primer = 1;
    r.t0 -= 1;
    r.nt += 1;
  }
  return r;
}

// atan2 for the fused discriminator: branch-free, one reciprocal (MUFU.RCP + one Newton step on the
// quotient) instead of fm_atan2f's two IEEE divisions; same Cephes polynomial. |error| <= 3 ulp of
// the result (tests/test_gpu_chan_demod_tc.py compares the multiplex with the three-kernel form).
__device__ __forceinline__ float atan2Fast(float y, float x) {
  const float kPi = 3.14159265358979323846f;
  const float kPi2 = 1.57079632679489661923f;
  const float kPi4 = 0.78539816339744830962f;
  const float ax = fabsf(x), ay = fabsf(y);
  const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
  const bool big = mn > 0.4142135623730950f * mx;
  const float num = big ? mn - mx : mn;
  const float den = fmaxf(big ? mn + mx : mx, 1e-37f);
  float rc;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(den));
  float t = num * rc;
  t = fmaf(fmaf(-den, t, num), rc, t);
  const float z = t * t;
  float pl = fmaf(z, 8.05374449538e-2f, -1.38776856032e-1f);
  pl = fmaf(pl, z, 1.99777106478e-1f);
  pl = fmaf(pl, z, -3.33329491539e-1f);
  float r = (big ? kPi4 : 0.0f) + fmaf(pl * z, t, t);
  r = (ay > ax) ? kPi2 - r : r;
  r = (__float_as_int(x) < 0) ? kPi - r : r;
  return copysignf(r, y);
}

template <int KS, int RING, int NACC, bool CPLX>
__global__ void __launch_bounds__(FT_THREADS, 1)
k_fir_tc(const __grid_constant__ CUtensorMap tm_in0, const __grid_constant__ CUtensorMap tm_in1,
         const __grid_constant__ CUtensorMap tm_out0, const __grid_constant__ CUtensorMap tm_out1,
         const uint4 *__restrict__ b_image, const FirTcParams p) {
  static_assert(NACC * FT_ACC_COLS + RING * FT_SLOT_COLS <= 512, "TMEM budget");
  static_assert(RING >= KS + 1, "ring must hold a window and one sub-chunk in flight");
  constexpr uint32_t A_COL0 = NACC * FT_ACC_COLS;   // accumulators first, the A ring behind them
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smemAddr(smem_raw) + 1023u) & ~1023u;
  const uint32_t sB = base;
  constexpr int B_BYTES = ((KS + 3) / 4) * FT_BCHUNK;
  const uint32_t sStg = sB + B_BYTES;
  const int NSTG = p.nstg;
  const uint32_t sOut = sStg + NSTG * FT_STG_BYTES;
  const uint32_t sBar = sOut + 16 * FT_OUT_BYTES;
  const uint32_t barSFull = sBar, barSEmpty = barSFull + 8 * FT_NSTG_MAX, barAFull = barSEmpty + 8 * FT_NSTG_MAX,
                 barAEmpty = barAFull + 8 * RING, barTFull = barAEmpty + 8 * RING,
                 barTEmpty = barTFull + 8 * NACC, sTmem = barTEmpty + 8 * NACC;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int lo, hi;
  tileRange(p, &lo, &hi);

  // ---- one-time setup ----------------------------------------------------------------------
  {
    uint8_t *gen = smem_raw + (base - smemAddr(smem_raw));
    uint4 *dst = reinterpret_cast<uint4 *>(gen);
    for (int i = threadIdx.x; i < ((KS + 3) / 4) * FT_BCHUNK / 16; i += FT_THREADS) {
      dst[i] = __ldg(b_image + i);
    }
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < FT_NSTG_MAX; i++) {
      mbarInit(barSFull + 8 * i, 1);
      mbarInit(barSEmpty + 8 * i, 4);   // one arrival per converter warp
    }
    for (int i = 0; i < RING; i++) {
      mbarInit(barAFull + 8 * i, 4);    // one arrival per converter warp
      mbarInit(barAEmpty + 8 * i, 1);   // tcgen05.commit
    }
    for (int i = 0; i < NACC; i++) {
      mbarInit(barTFull + 8 * i, 1);    // tcgen05.commit
      mbarInit(barTEmpty + 8 * i, 8);   // one arrival per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(sTmem) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fenceProxyAsync();
  tcFenceBefore();
  __syncthreads();
  tcFenceAfter();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(sTmem));

  if (warp == 0) {
    // ===== TMA producer ======================================================================
    if (lane == 0) {
      uint32_t stg = 0, use = 0;
      for (int cur = lo; cur < hi;) {
        const Run r = nextRun<CPLX>(p, cur, hi);
        const CUtensorMap *map = r.sig ? &tm_in1 : &tm_in0;
        const int nsub = r.nt + KS - 1;
        for (int g = 0; g < nsub; g++) {
          if (use > 0) {
            mbarWait(barSEmpty + 8 * stg, (use - 1) & 1);
          }
          mbarExpectTx(barSFull + 8 * stg, FT_STG_BYTES);
          if (CPLX) {
            // 32 complex samples of 64 channels: two boxes of [64 rows x 32 floats]
            const int x = p.in_x0 + 2 * FT_NO * (r.t0 + g);
            tmaLoad2d(sStg + stg * FT_STG_BYTES, map, barSFull + 8 * stg, x, r.rt * (FT_ROWS / 2));
            tmaLoad2d(sStg + stg * FT_STG_BYTES + FT_STG_BYTES / 2, map, barSFull + 8 * stg, x + FT_NO,
                      r.rt * (FT_ROWS / 2));
          } else {
            tmaLoad2d(sStg + stg * FT_STG_BYTES, map, barSFull + 8 * stg, p.in_x0 + FT_NO * (r.t0 + g),
                      r.rt * FT_ROWS);
          }
          if (++stg == static_cast<uint32_t>(NSTG)) {
            stg = 0;
            use++;
          }
        }
        cur += r.own;
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer ========================================================================
    // u8 x s8 -> s32, K-major B, N = 96, M = 128 (UMMA::InstrDescriptor)
    const uint32_t idesc = (2u << 4) | (0u << 7) | (1u << 10) | ((FT_N >> 3) << 17) | ((FT_ROWS >> 4) << 24);
    const uint32_t desc_hi = static_cast<uint32_t>(smemDesc(0) >> 32);
    const uint32_t b_lo0 = static_cast<uint32_t>(smemDesc(sB));
    uint32_t tile_cnt = 0;
    uint32_t win_slot = 0;        // ring slot of the window's first sub-chunk
    uint32_t wait_slot = 0, wait_use = 0;   // next sub-chunk to wait for
    for (int cur = lo; cur < hi;) {
      const Run r = nextRun<CPLX>(p, cur, hi);
      const int nt = r.nt;
      int landed = 0;             // sub-chunks of this run known to be in TMEM
      for (int i = 0; i < nt; i++, tile_cnt++) {
        const uint32_t acc = tile_cnt % NACC;
        mbarWait(barTEmpty + 8 * acc, (tile_cnt / NACC) & 1);   // zeroed by the epilogue
        while (landed < i + KS) {
          mbarWait(barAFull + 8 * wait_slot, wait_use & 1);
          landed++;
          if (++wait_slot == RING) {
            wait_slot = 0;
            wait_use++;
          }
        }
        tcFenceAfter();
        if (electOne()) {
          const uint32_t d0 = tmem_base + acc * FT_ACC_COLS;
#pragma unroll
          for (int a = 0; a < FT_PLANES; a++) {
            uint32_t slot = win_slot;
#pragma unroll
            for (int k = 0; k < KS; k++) {
              const uint32_t a_col = tmem_base + A_COL0 + slot * FT_SLOT_COLS + a * 8;
              const uint32_t b_lo = b_lo0 + (k >> 2) * (FT_BCHUNK >> 4) + (k & 3) * 2;
              ummaI8Ts(d0 + a * FT_NO, a_col, (static_cast<uint64_t>(desc_hi) << 32) | b_lo, idesc, 1u);
              slot = (slot + 1 == RING) ? 0 : slot + 1;
            }
          }
          ummaCommit(barTFull + 8 * acc);
          // the window moves on by one sub-chunk; the run's last tile releases all of them
          ummaCommit(barAEmpty + 8 * win_slot);
          if (i + 1 == nt) {
            uint32_t slot = win_slot;
#pragma unroll
            for (int k = 1; k < KS; k++) {
              slot = (slot + 1 == RING) ? 0 : slot + 1;
              ummaCommit(barAEmpty + 8 * slot);
            }
          }
        }
        __syncwarp();
        win_slot = (win_slot + 1 == RING) ? 0 : win_slot + 1;
      }
      // the next run starts behind this run's last window
      win_slot += KS - 1;
      if (win_slot >= RING) {
        win_slot -= RING;
      }
      cur += r.own;
    }
  } else if (warp < 6 || warp >= 10) {
    // ===== epilogue (TMEM lanes 32 * (warp % 4) ..; half 0 = outputs 0..15 of a tile, half 1 = 16..31) ====
    const int q = warp & 3;
    const int half = warp >= 10 ? 1 : 0;
    const uint32_t lane_base = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int a = 0; a < NACC; a++) {
      for (int s = 0; s < FT_LIMBS; s++) {
        tmemSt8(tmem_base + lane_base + a * FT_ACC_COLS + s * FT_NO + half * FT_HALF, zero);
        tmemSt8(tmem_base + lane_base + a * FT_ACC_COLS + s * FT_NO + half * FT_HALF + 8, zero);
      }
    }
    tmemWaitSt();
    tcFenceBefore();
    __syncwarp();
    if (lane == 0) {
      for (int i = 0; i < NACC; i++) {
        mbarArrive(barTEmpty + 8 * i);
      }
    }
    const uint32_t my_out = sOut + (half * 4 + q) * 2 * FT_OUT_BYTES;
    uint32_t tile_cnt = 0;
    // complex form: lanes (2 c, 2 c + 1) hold I and Q of channel c of the tile
    const int comp = lane & 1;
    const int ch_row = (q * 32 + lane) >> 1;          // channel inside the 64-channel tile
    float prev_i = 0.0f, prev_q = 0.0f;               // half 0: the filter output in front of the next tile
    // limbs -> float, most significant first (exact while the partial sums are below 2^24)
    auto horner = [&](int d4, int d3, int d2, int d1, int d0) {
      float f = static_cast<float>(d4 - p.off4);
      f = fmaf(f, 256.0f, static_cast<float>(d3 - p.off3));
      f = fmaf(f, 256.0f, static_cast<float>(d2 - p.off2));
      f = fmaf(f, 256.0f, static_cast<float>(d1));
      f = fmaf(f, 256.0f, static_cast<float>(d0));
      return f * p.out_scale;
    };
    // output `col` (0..31) of this lane's row: one column of every limb set
    auto oneOutput = [&](uint32_t taddr, int col) {
      int32_t v[FT_LIMBS];
#pragma unroll
      for (int s = 0; s < FT_LIMBS; s++) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v[s]) : "r"(taddr + s * FT_NO + col));
      }
      tmemWaitLd();
      return horner(v[4], v[3], v[2], v[1], v[0]);
    };
    for (int cur = lo; cur < hi;) {
      const Run r = nextRun<CPLX>(p, cur, hi);
      const CUtensorMap *map = r.sig ? &tm_out1 : &tm_out0;
      const int ch = r.rt * (FT_ROWS / 2) + ch_row;   // complex form: channel of the call
      if (CPLX && !r.primer && half == 0) {
        float2 pv = make_float2(0.0f, 0.0f);
        if (ch < p.nch) {
          pv = p.y_prev[static_cast<size_t>(ch) * p.y_pitch];
        }
        prev_i = pv.x;
        prev_q = pv.y;
      }
      for (int i = 0; i < r.nt; i++, tile_cnt++) {
        const uint32_t acc = tile_cnt % NACC;
        mbarWait(barTFull + 8 * acc, (tile_cnt / NACC) & 1);
        tcFenceAfter();
        // the TMA store that read this staging buffer two tiles ago has to be done with it
        if (lane == 0) {
          bulkWaitRead<1>();
        }
        __syncwarp();
        const uint32_t buf = my_out + (tile_cnt & 1) * FT_OUT_BYTES;
        const uint32_t taddr = tmem_base + lane_base + acc * FT_ACC_COLS;
        const bool skip = CPLX && r.primer && i == 0;   // a primer tile only yields its last output
        float pi = prev_i, pq = prev_q;
        if (CPLX && half == 1 && !skip) {
          // the sample in front of output 16: output 15 of this tile
          const float y15 = oneOutput(taddr, FT_HALF - 1);
          const float o = __shfl_xor_sync(0xffffffffu, y15, 1);
          pi = comp ? o : y15;
          pq = comp ? y15 : o;
        }
        if (!skip) {
          int32_t d[2][FT_LIMBS][8];
#pragma unroll
          for (int g = 0; g < 2; g++) {
#pragma unroll
            for (int s = 0; s < FT_LIMBS; s++) {
              tmemLd8(taddr + s * FT_NO + half * FT_HALF + g * 8, d[g][s]);
            }
          }
          tmemWaitLd();
#pragma unroll
          for (int g = 0; g < 2; g++) {
            float y[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
              y[j] = horner(d[g][4][j], d[g][3][j], d[g][2][j], d[g][1][j], d[g][0][j]);
            }
            if (CPLX) {
              // quadrature discriminator: both lanes of a pair get I and Q of the group's eight samples;
              // the even lane demodulates samples 0..3, the odd lane 4..7
              float vi[9], vq[9];
              vi[0] = pi;
              vq[0] = pq;
#pragma unroll
              for (int j = 0; j < 8; j++) {
                const float o = __shfl_xor_sync(0xffffffffu, y[j], 1);
                vi[j + 1] = comp ? o : y[j];
                vq[j + 1] = comp ? y[j] : o;
              }
              pi = vi[8];
              pq = vq[8];
              float m[4];
#pragma unroll
              for (int jj = 0; jj < 4; jj++) {
                const float ai = comp ? vi[jj + 4] : vi[jj], aq = comp ? vq[jj + 4] : vq[jj];
                const float ri = comp ? vi[jj + 5] : vi[jj + 1], rq = comp ? vq[jj + 5] : vq[jj + 1];
                const float re = (ai * ri) + (aq * rq);
                const float im = (ai * rq) - (aq * ri);
                m[jj] = atan2Fast(im, re) * p.fd_ref;
              }
              // row lane / 2 of the warp's [16 rows x 64 bytes] tile, 16-byte unit 2 g + comp
              const int rr = lane >> 1;
              const uint32_t at = buf + rr * 64 + (static_cast<uint32_t>((2 * g + comp) ^ ((rr >> 1) & 3)) << 4);
              asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(at), "f"(m[0]), "f"(m[1]),
                           "f"(m[2]), "f"(m[3])
                           : "memory");
            } else {
              // row `lane` of the [32 rows x 64 bytes] tile, 16-byte units XOR-swizzled like the tensor map
              const uint32_t row = buf + lane * 64;
              const uint32_t u0 = static_cast<uint32_t>((2 * g) ^ ((lane >> 1) & 3)) << 4;
              const uint32_t u1 = static_cast<uint32_t>((2 * g + 1) ^ ((lane >> 1) & 3)) << 4;
              asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(row + u0), "f"(y[0]), "f"(y[1]),
                           "f"(y[2]), "f"(y[3])
                           : "memory");
              asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(row + u1), "f"(y[4]), "f"(y[5]),
                           "f"(y[6]), "f"(y[7])
                           : "memory");
            }
          }
        }
        if (CPLX && half == 0) {
          // the sample in front of the next tile: output 31 of this one
          const float y31 = oneOutput(taddr, FT_NO - 1);
          const float o = __shfl_xor_sync(0xffffffffu, y31, 1);
          prev_i = comp ? o : y31;
          prev_q = comp ? y31 : o;
        }
        if (CPLX) {
          // each warp of the pair has read one column of the other's half (outputs 15 / 31): nobody
          // zeroes before both are done reading
          asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
        }
        // every MMA accumulates: hand this warp's columns back zeroed
#pragma unroll
        for (int s = 0; s < FT_LIMBS; s++) {
          tmemSt8(taddr + s * FT_NO + half * FT_HALF, zero);
          tmemSt8(taddr + s * FT_NO + half * FT_HALF + 8, zero);
        }
        tmemWaitSt();
        tcFenceBefore();
        fenceProxyAsync();
        __syncwarp();
        if (lane == 0) {
          mbarArrive(barTEmpty + 8 * acc);
          if (!skip) {
            const int x = p.out_x0 + FT_NO * (r.t0 + i) + half * FT_HALF;
            if (CPLX) {
              tmaStore2d(map, buf, x, r.rt * (FT_ROWS / 2) + q * 16);
            } else {
              tmaStore2d(map, buf, x, r.rt * FT_ROWS + q * 32);
            }
          }
          bulkCommit();   // (an empty group when nothing was stored: the wait counts groups)
        }
        if (CPLX && half == 1 && r.t0 + i == p.tiles_row - 1 && comp == 0 && ch < p.nch) {
          p.y_last[static_cast<size_t>(ch) * p.y_pitch] = make_float2(pi, pq);
        }
      }
      cur += r.own;
    }
    if (lane == 0) {
      bulkWait<0>();
    }
  } else {
    // ===== converters (warps 6..9 own TMEM lanes 32 * (warp % 4) ..) =============================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_base = static_cast<uint32_t>(q * 32) << 16;
    const float dscale = p.dscale;
    uint32_t stg = 0, stg_use = 0, slot = 0, slot_use = 0;
    for (int cur = lo; cur < hi;) {
      const Run r = nextRun<CPLX>(p, cur, hi);
      const int nsub = r.nt + KS - 1;
      for (int g = 0; g < nsub; g++) {
        mbarWait(barSFull + 8 * stg, stg_use & 1);
        float x[FT_NO];
        if (CPLX) {
          // my component of my channel's 32 complex samples: two [64 rows x 128 bytes] boxes
          const int chr = row >> 1, cmp = row & 1;
#pragma unroll
          for (int h = 0; h < 2; h++) {
            const uint32_t src = sStg + stg * FT_STG_BYTES + h * (FT_STG_BYTES / 2) + chr * 128;
#pragma unroll
            for (int u = 0; u < 8; u++) {
              const uint32_t at = src + (static_cast<uint32_t>(u ^ (chr & 7)) << 4);
              float a0, a1, a2, a3;
              asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                           : "=f"(a0), "=f"(a1), "=f"(a2), "=f"(a3)
                           : "r"(at));
              x[16 * h + 2 * u] = cmp ? a1 : a0;
              x[16 * h + 2 * u + 1] = cmp ? a3 : a2;
            }
          }
        } else {
          // my row of the [128 rows x 128 bytes] staging tile (128B-swizzled by the TMA)
          const uint32_t src = sStg + stg * FT_STG_BYTES + row * 128;
#pragma unroll
          for (int u = 0; u < 8; u++) {
            const uint32_t at = src + (static_cast<uint32_t>(u ^ (row & 7)) << 4);
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(x[4 * u]), "=f"(x[4 * u + 1]), "=f"(x[4 * u + 2]), "=f"(x[4 * u + 3])
                         : "r"(at));
          }
        }
        __syncwarp();
        if (lane == 0) {
          mbarArrive(barSEmpty + 8 * stg);
        }
        if (++stg == static_cast<uint32_t>(NSTG)) {
          stg = 0;
          stg_use++;
        }
        uint32_t pl[FT_PLANES][8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
          uint32_t qv[4];
#pragma unroll
          for (int e = 0; e < 4; e++) {
            float t = x[4 * u + e] * dscale;
            t = fminf(fmaxf(t, -8388608.0f), 8388607.0f);
            qv[e] = static_cast<uint32_t>(__float2int_rn(t) + 8388608);
          }
          const uint32_t a01 = __byte_perm(qv[0], qv[1], 0x5140);   // q0.b0 q1.b0 q0.b1 q1.b1
          const uint32_t a23 = __byte_perm(qv[2], qv[3], 0x5140);
          const uint32_t c01 = __byte_perm(qv[0], qv[1], 0x0062);   // q0.b2 q1.b2
          const uint32_t c23 = __byte_perm(qv[2], qv[3], 0x0062);
          pl[0][u] = __byte_perm(a01, a23, 0x5410);
          pl[1][u] = __byte_perm(a01, a23, 0x7632);
          pl[2][u] = __byte_perm(c01, c23, 0x5410);
        }
        if (slot_use > 0) {
          mbarWait(barAEmpty + 8 * slot, (slot_use - 1) & 1);
          tcFenceAfter();
        }
        const uint32_t taddr = tmem_base + lane_base + A_COL0 + slot * FT_SLOT_COLS;
#pragma unroll
        for (int a = 0; a < FT_PLANES; a++) {
          tmemSt8(taddr + a * 8, pl[a]);
        }
        tmemWaitSt();
        tcFenceBefore();
        __syncwarp();
        if (lane == 0) {
          mbarArrive(barAFull + 8 * slot);
        }
        if (++slot == RING) {
          slot = 0;
          slot_use++;
        }
      }
      cur += r.own;
    }
  }

  // ---- teardown ------------------------------------------------------------------------------
  tcFenceBefore();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

// float rows [rows][row_floats] with `pitch` floats between rows; boxes of 32 floats x box_rows, 128B swizzle
bool encodeFloatRows(CUtensorMap *map, const float *base, uint64_t row_floats, uint64_t rows, uint64_t pitch,
                     uint32_t box_rows, uint32_t box_floats = FT_NO) {
  EncodeFn fn = encodeFn();
  if (!fn) {
    return false;
  }
  const cuuint64_t dims[2] = {row_floats, rows};
  const cuuint64_t strides[1] = {pitch * sizeof(float)};
  const cuuint32_t box[2] = {box_floats, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE,
            box_floats * 4 == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// first tap that is not zero (the designs are padded in front to a multiple of 8)
int firstTap(const float *h, int Lp) {
  int i0 = 0;
  while (i0 < Lp - 1 && h[i0] == 0.0f) {
    i0++;
  }
  return i0;
}

}  // namespace

int firTcKsteps(const float *h, int Lp) {
  const int reach = Lp - 1 - firstTap(h, Lp);       // oldest sample a tap touches, relative to the output
  const int ws0 = (reach + FT_NO - 1) / FT_NO * FT_NO;
  return ws0 / FT_NO + 1;
}

bool firTcSupported(const float *h, int Lp, int in_off) {
  const int ks = firTcKsteps(h, Lp);
  return (ks == 5 || ks == 11 || ks == 12) && (ks - 1) * FT_NO <= in_off;
}

bool chanTcSupported(const float *h, int Lp, int in_off) {
  const int ks = firTcKsteps(h, Lp);
  return (ks == 4 || ks == 5) && (ks - 1) * FT_NO <= in_off;
}

// Host: integer taps, their digits, and the B image the way tcgen05.mma reads a K-major,
// 128B-swizzled operand: [K chunk of 128 bytes][n = digit * 32 + output j][128 bytes of k].
void firTcBuildTables(const float *h, int Lp, FirTcTables *t) {
  const int ks = firTcKsteps(h, Lp);
  const int ws0 = (ks - 1) * FT_NO;
  float hmax = 0.0f;
  for (int i = 0; i < Lp; i++) {
    hmax = std::max(hmax, std::fabs(h[i]));
  }
  // three balanced base-256 digits hold |v| <= 127 * 65536 + 127 * 256 + 127
  int shift = 0;
  while (shift < 40 && std::ldexp(static_cast<double>(hmax), shift + 1) <= 8355711.0) {
    shift++;
  }
  t->shift = shift;
  t->ksteps = ks;
  t->b_image.assign(static_cast<size_t>((ks + 3) / 4) * FT_BCHUNK, 0);
  long long hsum = 0;
  for (int i = 0; i < Lp; i++) {
    long long v = std::llround(std::ldexp(static_cast<double>(h[i]), shift));
    hsum += v;
    if (v == 0) {
      continue;
    }
    int dg[FT_DIGITS];
    for (int l = 0; l < FT_DIGITS; l++) {   // digit 0 least significant
      long long r = ((v % 256) + 256) % 256;
      if (r >= 128) {
        r -= 256;
      }
      dg[l] = static_cast<int>(r);
      v = (v - r) / 256;
    }
    for (int j = 0; j < FT_NO; j++) {
      const int k = ws0 + j - (Lp - 1) + i;   // byte of the tile's window that tap i of output j reads
      if (k < 0) {
        continue;   // cannot happen: ws0 covers the first non-zero tap
      }
      const int kc = k / 128, kk = k % 128;
      for (int l = 0; l < FT_DIGITS; l++) {
        const int n = l * FT_NO + j;
        const size_t at = static_cast<size_t>(kc) * FT_BCHUNK + static_cast<size_t>(n) * 128 +
                          static_cast<size_t>(((kk >> 4) ^ (n & 7)) << 4) + (kk & 15);
        t->b_image[at] = static_cast<uint8_t>(static_cast<int8_t>(dg[l]));
      }
    }
  }
  // 2^23 * hsum = 256^2 * 128 * hsum, in limbs 2, 3, 4 (digits of hsum in base 256, floor form)
  const long long h0 = ((hsum % 256) + 256) % 256;
  const long long r1 = (hsum - h0) / 256;
  const long long h1 = ((r1 % 256) + 256) % 256;
  const long long h2 = (r1 - h1) / 256;
  t->off[0] = static_cast<int32_t>(128 * h0);
  t->off[1] = static_cast<int32_t>(128 * h1);
  t->off[2] = static_cast<int32_t>(128 * h2);
}

static cudaError_t firTcAttrs() {
  static DeviceOnce attrs;  // per device: device_once.h
  return attrs.run([] {
    const void *fs[] = {(const void *)k_fir_tc<5, 8, 2, false>, (const void *)k_fir_tc<11, 14, 1, false>,
                        (const void *)k_fir_tc<12, 14, 1, false>, (const void *)k_fir_tc<4, 8, 2, true>,
                        (const void *)k_fir_tc<5, 8, 2, true>};
    cudaError_t err = cudaSuccess;
    for (const void *f : fs) {
      if (err == cudaSuccess) {
        err = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(ftSmemBytes(FT_MAX_KS, FT_NSTG_MAX)));
      }
    }
    return err;
  });
}

cudaError_t launchFirTc(const FirRealJob &job, int nsig, int nch, const FirTcTables &t,
                        const uint8_t *b_image_dev, int data_shift, int sm_count, cudaStream_t stream) {
  const cudaError_t attr_err = firTcAttrs();
  if (attr_err != cudaSuccess) {
    return attr_err;
  }
  if (job.n_total % FT_NO != 0 || nsig < 1 || nsig > 2 || nch < 1) {
    return cudaErrorInvalidValue;
  }
  const int ws0 = (t.ksteps - 1) * FT_NO;
  if (ws0 > job.in_off) {
    return cudaErrorInvalidValue;
  }
  FirTcParams p{};
  p.tiles_row = job.n_total / FT_NO;
  p.row_tiles = (nch + FT_ROWS - 1) / FT_ROWS;
  p.nsig = nsig;
  p.tiles_total = nsig * p.row_tiles * p.tiles_row;
  p.in_x0 = job.in_off - ws0;
  p.out_x0 = job.out_off;
  p.off2 = t.off[0];
  p.off3 = t.off[1];
  p.off4 = t.off[2];
  p.dscale = static_cast<float>(std::ldexp(1.0, data_shift));
  p.out_scale = static_cast<float>(std::ldexp(static_cast<double>(job.scale), -(t.shift + data_shift)));
  p.nstg = FT_NSTG_DEFAULT;
  const size_t smem = ftSmemBytes(t.ksteps, p.nstg);
  CUtensorMap tm_in[2], tm_out[2];
  for (int s = 0; s < 2; s++) {
    const int ss = s < nsig ? s : 0;
    const float *in = job.in[ss] + static_cast<size_t>(job.ch0) * job.in_pitch;
    float *out = job.out[ss] + static_cast<size_t>(job.ch0) * job.out_pitch;
    if ((reinterpret_cast<uintptr_t>(in) & 15u) || (reinterpret_cast<uintptr_t>(out) & 15u) ||
        (job.in_pitch & 3u) || (job.out_pitch & 3u)) {
      return cudaErrorInvalidValue;
    }
    if (!encodeFloatRows(&tm_in[s], in, static_cast<uint64_t>(job.in_off + job.n_total),
                         static_cast<uint64_t>(nch), job.in_pitch, FT_ROWS) ||
        !encodeFloatRows(&tm_out[s], out, static_cast<uint64_t>(job.out_off + job.n_total),
                         static_cast<uint64_t>(nch), job.out_pitch, 32, FT_HALF)) {
      return cudaErrorInvalidValue;
    }
  }
  const int grid = std::min(sm_count, p.tiles_total);
  const uint4 *bi = reinterpret_cast<const uint4 *>(b_image_dev);
  switch (t.ksteps) {
    case 5:
      k_fir_tc<5, 8, 2, false><<<grid, FT_THREADS, smem, stream>>>(tm_in[0], tm_in[1], tm_out[0], tm_out[1], bi, p);
      break;
    case 11:
      k_fir_tc<11, 14, 1, false><<<grid, FT_THREADS, smem, stream>>>(tm_in[0], tm_in[1], tm_out[0], tm_out[1], bi, p);
      break;
    case 12:
      k_fir_tc<12, 14, 1, false><<<grid, FT_THREADS, smem, stream>>>(tm_in[0], tm_in[1], tm_out[0], tm_out[1], bi, p);
      break;
    default:
      return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// Host-only model of the kernel's arithmetic, from the SAME tables the kernel uses (include/fmgpu.h:
// fmgpu_fir_tc_host_model): every digit is read back out of the B image through the operand layout,
// the five limb sets are summed in 64-bit integers, and the epilogue's float recombination is
// repeated operation for operation. The CPU test-suite checks it against a float64 FIR: the table
// builder, the digit split, the offset limbs and the bound on the result need no GPU to be tested.
size_t firTcHostModel(const float *taps, int n_taps, int lp, float scale, int data_shift, const float *x,
                      size_t n_hist, size_t n, float *y) {
  if (!taps || !x || !y || n_taps < 1 || lp < n_taps || lp > MAX_TAPS || n % FT_NO != 0) {
    return 0;
  }
  std::vector<float> h(static_cast<size_t>(lp), 0.0f);   // reversed, padded in front (engine.cu: padFront)
  for (int i = 0; i < n_taps; i++) {
    h[lp - n_taps + i] = taps[n_taps - 1 - i];
  }
  FirTcTables t;
  firTcBuildTables(h.data(), lp, &t);
  const int ws0 = (t.ksteps - 1) * FT_NO;
  if (static_cast<size_t>(ws0) > n_hist) {
    return 0;
  }
  const float dscale = static_cast<float>(std::ldexp(1.0, data_shift));
  const float out_scale = static_cast<float>(std::ldexp(static_cast<double>(scale), -(t.shift + data_shift)));
  const float *xs = x + n_hist;   // xs[s], s >= -n_hist
  for (size_t n0 = 0; n0 < n; n0 += FT_NO) {
    long long D[FT_LIMBS][FT_NO] = {};
    for (int k = 0; k < t.ksteps * FT_NO; k++) {
      const float v = xs[static_cast<long>(n0) - ws0 + k];
      float tq = v * dscale;
      tq = std::fmin(std::fmax(tq, -8388608.0f), 8388607.0f);
      const uint32_t q = static_cast<uint32_t>(static_cast<int32_t>(std::nearbyint(tq)) + 8388608);
      const int kc = k / 128, kk = k % 128;
      for (int col = 0; col < FT_N; col++) {
        const size_t at = static_cast<size_t>(kc) * FT_BCHUNK + static_cast<size_t>(col) * 128 +
                          static_cast<size_t>(((kk >> 4) ^ (col & 7)) << 4) + (kk & 15);
        const int dg = static_cast<int8_t>(t.b_image[at]);
        if (dg == 0) {
          continue;
        }
        const int l = col / FT_NO, j = col % FT_NO;
        for (int a = 0; a < FT_PLANES; a++) {
          D[a + l][j] += static_cast<long long>((q >> (8 * a)) & 0xffu) * dg;
        }
      }
    }
    for (int j = 0; j < FT_NO; j++) {
      for (int s2 = 0; s2 < FT_LIMBS; s2++) {
        if (D[s2][j] > 2147483647LL || D[s2][j] < -2147483648LL) {
          return 0;   // an int32 accumulator of the kernel would have overflowed
        }
      }
      float f = static_cast<float>(static_cast<int32_t>(D[4][j]) - t.off[2]);
      f = std::fmaf(f, 256.0f, static_cast<float>(static_cast<int32_t>(D[3][j]) - t.off[1]));
      f = std::fmaf(f, 256.0f, static_cast<float>(static_cast<int32_t>(D[2][j]) - t.off[0]));
      f = std::fmaf(f, 256.0f, static_cast<float>(static_cast<int32_t>(D[1][j])));
      f = std::fmaf(f, 256.0f, static_cast<float>(static_cast<int32_t>(D[0][j])));
      y[n0 + j] = f * out_scale;
    }
  }
  return n;
}

// Channel filter + quadrature discriminator in one kernel (FMDemod::demodulateComplex,
// /root/reference/src/fm_demod.cpp:194-199): x2 rows (DC-blocked complex samples, halo of in_off
// samples in front) -> MPX rows. The pre-discriminator AGC between the two (fm_demod.cpp:196-198)
// multiplies y[n] by a positive real gain, and arg(g y[n] conj(g' y[n-1])) = arg(y[n] conj(y[n-1])):
// it does not change the discriminator's output and is left out. y_io[c * y_pitch + Y_OFF - 1] holds
// the filter output in front of this block, y_io[c * y_pitch + Y_OFF + n_total - 1] receives the last one.
cudaError_t launchChanDemodTc(const float2 *x2, size_t x2_pitch, int in_off, float2 *y_io, size_t y_pitch,
                              float *mpx, size_t mpx_pitch, int mpx_off, int n_total, int ch0, int nch,
                              float chan_scale, float fd_ref, const FirTcTables &t, const uint8_t *b_image_dev,
                              int data_shift, int sm_count, cudaStream_t stream) {
  const cudaError_t attr_err = firTcAttrs();
  if (attr_err != cudaSuccess) {
    return attr_err;
  }
  const int ws0 = (t.ksteps - 1) * FT_NO;
  if (n_total % FT_NO != 0 || nch < 1 || ws0 > in_off || (t.ksteps != 4 && t.ksteps != 5)) {
    return cudaErrorInvalidValue;
  }
  FirTcParams p{};
  p.tiles_row = n_total / FT_NO;
  p.row_tiles = (nch + FT_ROWS / 2 - 1) / (FT_ROWS / 2);
  p.nsig = 1;
  p.tiles_total = p.row_tiles * p.tiles_row;
  p.in_x0 = 2 * (in_off - ws0);
  p.out_x0 = mpx_off;
  p.off2 = t.off[0];
  p.off3 = t.off[1];
  p.off4 = t.off[2];
  p.dscale = static_cast<float>(std::ldexp(1.0, data_shift));
  p.out_scale = static_cast<float>(std::ldexp(static_cast<double>(chan_scale), -(t.shift + data_shift)));
  p.nch = nch;
  p.nstg = FT_NSTG_DEFAULT;
  const size_t smem = ftSmemBytes(t.ksteps, p.nstg);
  p.fd_ref = fd_ref;
  p.y_prev = y_io + static_cast<size_t>(ch0) * y_pitch + Y_OFF - 1;
  p.y_last = y_io + static_cast<size_t>(ch0) * y_pitch + Y_OFF + n_total - 1;
  p.y_pitch = y_pitch;
  const float *in = reinterpret_cast<const float *>(x2 + static_cast<size_t>(ch0) * x2_pitch);
  float *out = mpx + static_cast<size_t>(ch0) * mpx_pitch;
  if ((reinterpret_cast<uintptr_t>(in) & 15u) || (reinterpret_cast<uintptr_t>(out) & 15u) || (x2_pitch & 1u) ||
      (mpx_pitch & 3u)) {
    return cudaErrorInvalidValue;
  }
  CUtensorMap tm_in, tm_out;
  if (!encodeFloatRows(&tm_in, in, 2ull * static_cast<uint64_t>(in_off + n_total), static_cast<uint64_t>(nch),
                       2 * x2_pitch, FT_ROWS / 2) ||
      !encodeFloatRows(&tm_out, out, static_cast<uint64_t>(mpx_off + n_total), static_cast<uint64_t>(nch),
                       mpx_pitch, 16, FT_HALF)) {
    return cudaErrorInvalidValue;
  }
  const int grid = std::min(sm_count, p.tiles_total);
  const uint4 *bi = reinterpret_cast<const uint4 *>(b_image_dev);
  if (t.ksteps == 4) {
    k_fir_tc<4, 8, 2, true><<<grid, FT_THREADS, smem, stream>>>(tm_in, tm_in, tm_out, tm_out, bi, p);
  } else {
    k_fir_tc<5, 8, 2, true><<<grid, FT_THREADS, smem, stream>>>(tm_in, tm_in, tm_out, tm_out, bi, p);
  }
  return cudaGetLastError();
}

}  // namespace fmgpu
