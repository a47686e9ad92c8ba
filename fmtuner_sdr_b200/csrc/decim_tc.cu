// decim_tc.cu — the decimating FIR of ComplexDecimator::executeComplex
// (/root/reference/src/dsp/liquid_primitives.cpp:461-499) on the 5th-generation tensor cores.
//
//   y_c[n] = scale * sum_i hrev[i] * x_c[n*M - (L-1) + i],   x = (byte - 127.5) / 127.5
//
// is evaluated as an INTEGER contraction: the uint8 IQ bytes are the A operand as they are (no
// unpack, no conversion: TMA drops [128 channels x 128 bytes] boxes of the caller's buffer straight
// into 128B-swizzled shared memory), and B is a constant banded (Toeplitz) matrix of the taps,
// quantised to round(hrev * 2^26) and split into four signed base-128 digits ("limbs"):
//
//   D[channel][(limb, j, iq)] = sum_k A[channel][k] * B[(limb, j, iq)][k]       (tcgen05.mma kind::i8,
//                                                                               u8 x s8 -> s32 in TMEM)
//   k = byte offset inside the tile's window, j = 0..15 the tile's outputs, iq = byte parity
//   (N = 128 columns per MMA: sixteen outputs per tile, 28 K-steps for /10 instead of 2 x 23 with
//   eight-output tiles: 0.60 -> 0.565 ms per launch).
//
// The int32 sums are exact; the epilogue recombines the limbs, removes the 127.5 offset in integer
// arithmetic (255 * sum of the taps that see real samples) and rounds ONCE to float. The result is
// the FIR to within one float rounding of the exact sum with taps good to 2^-27 — closer to the
// real-number answer than the 280-term float chain of the reference, but not bit-identical to it
// (the FP32 kernel k_decim in kernels.cu stays the bit-exact flavour).
//
// One CTA per SM, persistent over (128-channel row tile, time segment) work items:
//   warp 0     TMA producer: 16 KB chunks (128 rows x 128 B) into a ring of shared-memory slots
//   warp 1     allocates TMEM and issues the MMAs with the A operand in TMEM (one elected lane)
//   warps 2-5  epilogue: tcgen05.ld the 128 accumulator columns of a tile, recombine, store float2
//   warp 6     copies every chunk from its shared-memory slot into the TMEM A ring (tcgen05.cp)
// mbarrier pairs between them: full / empty (shared-memory ring), A full / A empty (TMEM A ring),
// T full / T empty (accumulators); tcgen05.commit arrives as soon as the operations that read a slot retire.
// Window of tile t (16 outputs): block-relative bytes [ADV*t - WS0, ADV*t - WS0 + 32*KS), ADV = 32*M,
// WS0 = roundup(2L - 2, 32); the bytes in front of the block come from the per-channel history
// buffer (hist tensor map), invalid history is byte 0 and is compensated in the offset term.
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
#include "kernels.h"
#include "tc_common.cuh"

namespace fmgpu {

namespace {

using namespace tc;

constexpr int TC_ROWS = 128;          // channels per tile (UMMA M)
constexpr int TC_NO = 16;             // outputs per tile
constexpr int TC_LIMBS = 4;
constexpr int TC_N = TC_NO * 2 * TC_LIMBS;   // 128 accumulator columns (UMMA N)
constexpr int TC_CHUNK = 128;         // bytes of K per ring slot row (one 128B swizzle atom)
constexpr int TC_CHUNK_BYTES = TC_ROWS * TC_CHUNK;   // 16 KB
constexpr int TC_B_CHUNKS = 7;        // K extent of B: 7 * 128 = 896 bytes >= 32 * KS
constexpr int TC_B_BYTES = TC_B_CHUNKS * TC_N * TC_CHUNK;   // 112 KB
// A ring slots of 16 KB in shared memory: TcParams::ring, a launch parameter. The A operand lives in
// TMEM: a slot is free again as soon as its four tcgen05.cp retire, so the ring only covers the TMA
// latency (five slots; B takes 112 KB of the CTA's 194 KB).
constexpr int TC_RING_TMEM_A = 5;
// TMEM: columns [0, 256) hold a ring of eight chunks (32 columns = 128 bytes of K per lane; a tile's
// window touches up to eight), columns [256, 512) two accumulators of 128 columns
constexpr int TC_A_SLOTS = 8;
constexpr int TC_A_COLS = 32;
constexpr int TC_ACC = 2;
constexpr int TC_COPY_WARP = 6;
constexpr int TC_THREADS = 224;
constexpr int TC_SHIFT = 26;          // taps are quantised to 2^-26
constexpr size_t tcSmemBytes(int ring) { return 1024 + TC_B_BYTES + (size_t)ring * TC_CHUNK_BYTES + 512; }

struct TcParams {
  int M, L, n_out;
  int adv;          // bytes per tile = 2 * M * TC_NO
  int ws0;          // window start in front of the tile's first output sample, bytes
  int ksteps;       // MMAs (32 bytes of K each) per tile
  int halo_chunks;  // chunks in front of the block (from the history buffer)
  int tiles;        // tiles per block = n_out / TC_NO
  int tiles_per_seg;
  int n_seg;
  int row_tiles;
  int ch0, nch;
  int ring;         // shared-memory ring slots
  float out_scale;  // scale / (255 * 2^26)
};

// work item w -> (row tile, first tile of the segment, tiles in it)
__device__ __forceinline__ void workItem(const TcParams &p, int w, int *row, int *t0, int *nt) {
  *row = w / p.n_seg;
  const int s = w - *row * p.n_seg;
  *t0 = s * p.tiles_per_seg;
  *nt = min(p.tiles_per_seg, p.tiles - *t0);
}
// window of tile t in chunk space (chunk g holds block-relative bytes [128 (g - HC), +128))
__device__ __forceinline__ int windowStart(const TcParams &p, int t) {
  return p.adv * t - p.ws0 + TC_CHUNK * p.halo_chunks;   // >= 0
}

constexpr int TC_MAX_KSTEPS = 4 * TC_B_CHUNKS;   // 28
constexpr int TC_WIN_CHUNKS = 8;                 // an 896-byte window starting at a 32-byte phase touches <= 8 chunks

// The MMAs of one tile, fully unrolled for the window's phase PH (its start inside a chunk, in
// 32-byte steps): every operand offset is then an immediate. cb[r] / eb[r]: TMEM column and `A empty`
// barrier of the window's r-th chunk; the first n_free chunks are released right behind the last K
// step that reads them, so that the copy warp can refill their slots while the tile's later K steps run.
// af[r] / ap[r]: `A full` barrier and parity of chunk r. The chunks from n_have on are waited for
// right before the first K step that reads them: the K steps over chunks already in TMEM queue up
// behind the previous tile while the copy warp still brings the new ones.
template <int PH, int KS>
__device__ __forceinline__ void issueTile(int ksteps_rt, int n_free, int n_have, const uint32_t (&af)[TC_WIN_CHUNKS],
                                          const uint32_t (&ap)[TC_WIN_CHUNKS], const uint32_t (&cb)[TC_WIN_CHUNKS],
                                          const uint32_t (&eb)[TC_WIN_CHUNKS], uint32_t b_lo0,
                                          uint32_t desc_hi, uint32_t d_tmem, uint32_t idesc) {
  // KS > 0: the K-step count is a compile-time constant (28 for /10, 22 for /8): no per-step test
  const int ksteps = (KS > 0) ? KS : ksteps_rt;
#pragma unroll
  for (int ks = 0; ks < ((KS > 0) ? KS : TC_MAX_KSTEPS); ks++) {
    if (KS > 0 || ks < ksteps) {
      const int byte = 32 * PH + 32 * ks;
      const int r = byte >> 7;
      const uint32_t b_lo = b_lo0 + (ks >> 2) * ((TC_N * TC_CHUNK) >> 4) + (ks & 3) * 2;
      const uint64_t b_desc = (static_cast<uint64_t>(desc_hi) << 32) | b_lo;
      const uint32_t a_col = cb[r] + ((byte & (TC_CHUNK - 1)) >> 2);   // 4 bytes of K per column
      if ((ks == 0 || (byte & (TC_CHUNK - 1)) == 0) && r >= n_have) {
        mbarWait(af[r], ap[r]);
        tcFenceAfter();
      }
      ummaI8Ts(d_tmem, a_col, b_desc, idesc, ks == 0 ? 0u : 1u);
      const bool chunk_done = (((byte + 32) & (TC_CHUNK - 1)) == 0) || (ks + 1 == ksteps);
      if (chunk_done && r < n_free) {
        ummaCommit(eb[r]);
      }
    }
  }
}

// the chunks a CTA loads, in order, across its work items
struct ChunkCursor {
  int w, stride, n_work, g, g1, y;
  __device__ ChunkCursor(const TcParams &p, int w0, int stride_, int n_work_)
      : w(w0), stride(stride_), n_work(n_work_), g(0), g1(-1), y(0) {
    open(p);
  }
  __device__ void open(const TcParams &p) {
    if (w < n_work) {
      int row, t0, nt;
      workItem(p, w, &row, &t0, &nt);
      g = windowStart(p, t0) / TC_CHUNK;
      g1 = (windowStart(p, t0 + nt - 1) + 32 * p.ksteps - 1) / TC_CHUNK;
      y = p.ch0 + row * TC_ROWS;
    }
  }
  __device__ bool valid() const { return w < n_work; }
  __device__ void next(const TcParams &p) {
    if (++g > g1) {
      w += stride;
      open(p);
    }
  }
  // byte coordinate inside the history rows (chunks in front of the block) or the IQ rows
  __device__ int x(const TcParams &p) const {
    return g < p.halo_chunks ? 2 * H_IQ - TC_CHUNK * (p.halo_chunks - g) : TC_CHUNK * (g - p.halo_chunks);
  }
};

template <int KS>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_decim_tc(const __grid_constant__ CUtensorMap tm_iq, const __grid_constant__ CUtensorMap tm_hist,
           const uint4 *__restrict__ b_image, const int2 *__restrict__ offs, const int *__restrict__ hist_valid,
           float2 *__restrict__ x1, size_t x1_pitch, const TcParams p) {
  constexpr int NACC = TC_ACC;
  constexpr uint32_t ACC_COL0 = TC_A_SLOTS * TC_A_COLS;   // first accumulator column
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smemAddr(smem_raw) + 1023u) & ~1023u;
  const uint32_t sB = base;
  const uint32_t sA = base + TC_B_BYTES;
  const int RING = p.ring;
  const uint32_t sBar = sA + RING * TC_CHUNK_BYTES;
  // barriers: full[RING], empty[RING], tfull[ACC], tempty[ACC], afull[A_SLOTS], aempty[A_SLOTS]; then
  // the TMEM base word
  const uint32_t barFull = sBar, barEmpty = sBar + 8 * RING, barTFull = sBar + 16 * RING,
                 barTEmpty = barTFull + 8 * NACC, barAFull = barTEmpty + 8 * NACC,
                 barAEmpty = barAFull + 8 * TC_A_SLOTS, sTmem = barAEmpty + 8 * TC_A_SLOTS;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_work = p.row_tiles * p.n_seg;

  // ---- one-time setup ----------------------------------------------------------------------
  {  // B image: generic-proxy stores, made visible to the async proxy (UMMA) below
    uint8_t *gen = smem_raw + (base - smemAddr(smem_raw));
    uint4 *dst = reinterpret_cast<uint4 *>(gen);
    for (int i = threadIdx.x; i < TC_B_BYTES / 16; i += TC_THREADS) {
      dst[i] = __ldg(b_image + i);
    }
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < RING; i++) {
      mbarInit(barFull + 8 * i, 1);
      mbarInit(barEmpty + 8 * i, 1);
    }
    for (int i = 0; i < NACC; i++) {
      mbarInit(barTFull + 8 * i, 1);
      mbarInit(barTEmpty + 8 * i, 4);   // one arrival per epilogue warp
    }
    for (int i = 0; i < TC_A_SLOTS; i++) {
      mbarInit(barAFull + 8 * i, 1);    // tcgen05.commit of the copy warp
      mbarInit(barAEmpty + 8 * i, 1);   // tcgen05.commit of the MMA issuer
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(sTmem) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tcFenceBefore();
  __syncthreads();
  tcFenceAfter();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(sTmem));

  if (warp == 0) {
    // ===== TMA producer =====================================================================
    // (An L2 prefetch running 1-3 KB per row ahead of these loads — cp.async.bulk.prefetch.tensor
    // through a 1 KB x 32-row map — was measured and dropped: 1.7x the DRAM reads, same time. The
    // kernel is bound by the tensor cores' shared-memory operand reads, not by these loads.)
    if (lane == 0) {
      uint32_t slot = 0, use = 0;   // ring position of the next chunk
      for (ChunkCursor ld(p, blockIdx.x, gridDim.x, n_work); ld.valid(); ld.next(p)) {
        if (use > 0) {
          mbarWait(barEmpty + 8 * slot, (use - 1) & 1);
        }
        mbarExpectTx(barFull + 8 * slot, TC_CHUNK_BYTES);
        tmaLoad2d(sA + slot * TC_CHUNK_BYTES, ld.g < p.halo_chunks ? &tm_hist : &tm_iq,
                  barFull + 8 * slot, ld.x(p), ld.y);
        if (++slot == static_cast<uint32_t>(RING)) {
          slot = 0;
          use++;
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: the whole warp keeps the (warp-uniform) books, one elected lane issues ======
    // u8 x s8 -> s32, K-major A and B, N = 128, M = 128 (UMMA::InstrDescriptor)
    const uint32_t idesc = (2u << 4) | (0u << 7) | (1u << 10) | ((TC_N >> 3) << 17) | ((TC_ROWS >> 4) << 24);
    const uint32_t desc_hi = static_cast<uint32_t>(smemDesc(0) >> 32);
    const uint32_t b_lo0 = static_cast<uint32_t>(smemDesc(sB));
    uint32_t a_wait = 0, a_wait_use = 0;   // TMEM slot and use count of the next chunk to wait for
    uint32_t gs_slot = 0;                  // TMEM slot of the current window's first chunk
    uint32_t tile_cnt = 0;
    for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
      int row, t0, nt;
      workItem(p, w, &row, &t0, &nt);
      const int g0 = windowStart(p, t0) / TC_CHUNK;
      const int g1 = (windowStart(p, t0 + nt - 1) + 32 * p.ksteps - 1) / TC_CHUNK;
      int have = g0 - 1;   // chunks known to be in TMEM
      int gs = g0;         // first chunk of the current window
      for (int i = 0; i < nt; i++, tile_cnt++) {
        const int ws = windowStart(p, t0 + i);
        const int ge = (ws + 32 * p.ksteps - 1) / TC_CHUNK;
        const uint32_t acc = tile_cnt % NACC;
        const uint32_t ause = tile_cnt / NACC;
        if (ause > 0) {
          mbarWait(barTEmpty + 8 * acc, (ause - 1) & 1);
        }
        // the window's chunks up to `have` were waited for by earlier tiles; the issuing lane waits
        // for the others inside issueTile
        const int n_have = have - gs + 1;
        uint32_t af[TC_WIN_CHUNKS], ap[TC_WIN_CHUNKS];   // A full barrier / parity per window chunk
        {
#pragma unroll
          for (int r = 0; r < TC_WIN_CHUNKS; r++) {
            const uint32_t j = a_wait + static_cast<uint32_t>(max(r - n_have, 0));
            af[r] = barAFull + 8 * (j % TC_A_SLOTS);
            ap[r] = (a_wait_use + j / TC_A_SLOTS) & 1;
          }
          const uint32_t j = a_wait + static_cast<uint32_t>(ge - have);
          a_wait = j % TC_A_SLOTS;
          a_wait_use += j / TC_A_SLOTS;
          have = ge;
        }
        tcFenceAfter();
        // chunks in front of the next tile's window go back to the copy warp as soon as the MMAs
        // that read them are done: a commit right behind the last K step inside them
        const int keep = (i + 1 < nt) ? windowStart(p, t0 + i + 1) / TC_CHUNK : g1 + 1;
        const int n_free = keep - gs;
        uint32_t cb[TC_WIN_CHUNKS], eb[TC_WIN_CHUNKS];   // TMEM column / A empty barrier per window chunk
        {
          uint32_t slot = gs_slot;
#pragma unroll
          for (int r = 0; r < TC_WIN_CHUNKS; r++) {
            cb[r] = tmem_base + slot * TC_A_COLS;
            eb[r] = barAEmpty + 8 * slot;
            slot = (slot + 1 == TC_A_SLOTS) ? 0 : slot + 1;
          }
        }
        const uint32_t d_tmem = tmem_base + ACC_COL0 + acc * TC_N;
        const uint32_t tfull = barTFull + 8 * acc;
        if (electOne()) {
          switch ((ws & (TC_CHUNK - 1)) >> 5) {
            case 0: issueTile<0, KS>(p.ksteps, n_free, n_have, af, ap, cb, eb, b_lo0, desc_hi, d_tmem, idesc); break;
            case 1: issueTile<1, KS>(p.ksteps, n_free, n_have, af, ap, cb, eb, b_lo0, desc_hi, d_tmem, idesc); break;
            case 2: issueTile<2, KS>(p.ksteps, n_free, n_have, af, ap, cb, eb, b_lo0, desc_hi, d_tmem, idesc); break;
            default: issueTile<3, KS>(p.ksteps, n_free, n_have, af, ap, cb, eb, b_lo0, desc_hi, d_tmem, idesc); break;
          }
          ummaCommit(tfull);
        }
        __syncwarp();
        gs = keep;   // the next window starts here
        gs_slot = (gs_slot + n_free) % TC_A_SLOTS;
      }
    }
  } else if (warp == TC_COPY_WARP) {
    // ===== chunk copier: shared-memory ring -> TMEM A ring, in the producer's chunk order ==========
    // Every chunk goes to TMEM once (4 x tcgen05.cp 128x256b = 128 lanes x 32 bytes each) and every MMA
    // that uses it reads it from there. Its shared-memory slot is free as soon as the copies retire
    // (empty); the MMA issuer waits for A full before the first MMA that reads the chunk. A copy into
    // a TMEM slot waits for A empty, which the issuer commits behind the last MMA that reads the slot's
    // previous chunk: cp and mma come from different warps, so the barrier, not issue order, keeps a
    // copy from overtaking those MMAs. A window touches at most all eight slots, so the copies of the
    // next tile's new chunks start as soon as the current tile's first K steps have retired.
    const uint32_t desc_hi = static_cast<uint32_t>(smemDesc(0) >> 32);
    const uint32_t a_lo0 = static_cast<uint32_t>(smemDesc(sA));
    uint32_t ring = 0, ring_use = 0;   // shared-memory slot and use count of the next chunk
    uint32_t a_slot = 0, a_use = 0;    // TMEM slot and use count it goes to
    for (ChunkCursor cc(p, blockIdx.x, gridDim.x, n_work); cc.valid(); cc.next(p)) {
      if (a_use > 0) {
        mbarWait(barAEmpty + 8 * a_slot, (a_use - 1) & 1);
      }
      mbarWait(barFull + 8 * ring, ring_use & 1);
      tcFenceAfter();
      if (electOne()) {
        const uint32_t a_col = tmem_base + a_slot * TC_A_COLS;
        const uint32_t src = a_lo0 + ring * (TC_CHUNK_BYTES >> 4);
#pragma unroll
        for (int sstep = 0; sstep < 4; sstep++) {
          tmemCp128x256(a_col + sstep * 8, (static_cast<uint64_t>(desc_hi) << 32) | (src + 2 * sstep));
        }
        ummaCommit(barEmpty + 8 * ring);
        ummaCommit(barAFull + 8 * a_slot);
      }
      __syncwarp();
      if (++a_slot == TC_A_SLOTS) {
        a_slot = 0;
        a_use++;
      }
      if (++ring == static_cast<uint32_t>(RING)) {
        ring = 0;
        ring_use++;
      }
    }
  } else {
    // ===== epilogue (warps 2..5 own TMEM lanes 32 * (warp % 4) ..) ===============================
    const int q = warp & 3;
    const uint32_t lane_base = static_cast<uint32_t>(q * 32) << 16;
    const int need_hist = p.L - 1;
    const int2 off_all = __ldg(offs);    // every tap sees a real sample
    uint32_t tile_cnt = 0;
    for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
      int row, t0, nt;
      workItem(p, w, &row, &t0, &nt);
      const int c = p.ch0 + row * TC_ROWS + q * 32 + lane;
      const bool live = c < p.ch0 + p.nch;
      const int valid = live ? __ldg(hist_valid + c) : need_hist;
      float2 *out = x1 + static_cast<size_t>(live ? c : p.ch0) * x1_pitch;
      for (int i = 0; i < nt; i++, tile_cnt++) {
        const uint32_t acc = tile_cnt % NACC;
        mbarWait(barTFull + 8 * acc, (tile_cnt / NACC) & 1);
        tcFenceAfter();
        const uint32_t taddr = tmem_base + lane_base + ACC_COL0 + acc * TC_N;
        const int n0 = (t0 + i) * TC_NO;
        // four outputs at a time: the eight columns (j, iq) of each of the four limbs
#pragma unroll 1
        for (int jg = 0; jg < TC_NO / 4; jg++) {
          int32_t d[TC_LIMBS][8];
#pragma unroll
          for (int l = 0; l < TC_LIMBS; l++) {
            tmemLd8(taddr + l * (2 * TC_NO) + 8 * jg, d[l]);
          }
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (jg == TC_NO / 4 - 1) {   // the whole accumulator has been read
            tcFenceBefore();
            __syncwarp();
            if (lane == 0) {
              mbarArrive(barTEmpty + 8 * acc);
            }
          }
          float2 y[4];
#pragma unroll
          for (int jj = 0; jj < 4; jj++) {
            const int j = 4 * jg + jj;
            // taps in front of the first real sample multiply byte 0: leave them out of the offset
            int2 off = off_all;
            const int missing = need_hist - p.M * (n0 + j) - valid;
            if (missing > 0) {
              off = __ldg(offs + min(missing, p.L));
            }
            float v[2];
#pragma unroll
            for (int iq = 0; iq < 2; iq++) {
              const int col = jj * 2 + iq;   // limb 0 = most significant
              const int hi = (d[0][col] << 7) + d[1][col];
              const int lo = (d[2][col] << 7) + d[3][col];
              const int ph = 2 * hi - off.x;   // offset term 255 * sum(hq) split the same way
              const int pl = 2 * lo - off.y;
              v[iq] = fmaf(static_cast<float>(ph), 16384.0f, static_cast<float>(pl)) * p.out_scale;
            }
            y[jj] = make_float2(v[0], v[1]);
          }
          if (live) {
            float4 *o4 = reinterpret_cast<float4 *>(out + n0 + 4 * jg);
            o4[0] = make_float4(y[0].x, y[0].y, y[1].x, y[1].y);
            o4[1] = make_float4(y[2].x, y[2].y, y[3].x, y[3].y);
          }
        }
      }
    }
  }

  // ---- teardown ------------------------------------------------------------------------------
  tcFenceBefore();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

// [rows][row_bytes] uint8 with `pitch` bytes between rows; boxes of 128 bytes x 128 rows, 128B swizzle
bool encodeRows(CUtensorMap *map, const void *base, uint64_t row_bytes, uint64_t rows, uint64_t pitch) {
  EncodeFn fn = encodeFn();
  if (!fn) {
    return false;
  }
  const cuuint64_t dims[2] = {row_bytes, rows};
  const cuuint64_t strides[1] = {pitch};
  const cuuint32_t box[2] = {TC_CHUNK, TC_ROWS};
  const cuuint32_t estr[2] = {1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

bool decimTcSupported(int M, int L, int n_out) {
  if (M < 2 || (M & 1) || L < M || n_out % TC_NO != 0) {
    return false;   // the tile advance 16 * M must be a multiple of the 32-byte MMA K step
  }
  const int ws0 = ((2 * L - 2) + 31) / 32 * 32;
  const int ksteps = (ws0 + 2 * M * (TC_NO - 1) + 2 + 31) / 32;
  const int halo = (ws0 + TC_CHUNK - 1) / TC_CHUNK;
  return ksteps <= 4 * TC_B_CHUNKS && halo * TC_CHUNK <= 2 * H_IQ && L - 1 <= H_IQ;
}

// Host: quantise the reversed taps, split them into limbs and lay the Toeplitz matrix B out the way
// tcgen05.mma reads a K-major 128B-swizzled operand; plus the offset table (entry m: the taps from
// index m on see real samples), each entry 255 * sum(hq) split as {hi, lo} with sum = hi*2^14 + lo.
void decimTcBuildTables(int M, const std::vector<float> &hrev, std::vector<uint8_t> *b_image,
                        std::vector<int32_t> *offs) {
  const int L = static_cast<int>(hrev.size());
  const int ws0 = ((2 * L - 2) + 31) / 32 * 32;
  std::vector<long long> hq(L);
  for (int i = 0; i < L; i++) {
    hq[i] = std::llround(static_cast<double>(hrev[i]) * static_cast<double>(1 << TC_SHIFT));
  }
  b_image->assign(TC_B_BYTES, 0);
  auto digit = [](long long v, int limb) {   // balanced base-128 digits, limb 0 most significant
    int dg[TC_LIMBS];
    for (int l = TC_LIMBS - 1; l >= 0; l--) {
      long long r = ((v % 128) + 128) % 128;
      if (r >= 64) {
        r -= 128;
      }
      dg[l] = static_cast<int>(r);
      v = (v - r) / 128;
    }
    return dg[limb];
  };
  for (int j = 0; j < TC_NO; j++) {
    for (int i = 0; i < L; i++) {
      for (int iq = 0; iq < 2; iq++) {
        // sample i of output j's window is block-relative byte 2 (M (8 t + j) - (L - 1) + i) + iq
        const int k = ws0 + 2 * (M * j - (L - 1) + i) + iq;   // byte inside the tile's window
        for (int l = 0; l < TC_LIMBS; l++) {
          const int n = l * (2 * TC_NO) + j * 2 + iq;
          const int kc = k / TC_CHUNK, kk = k % TC_CHUNK;
          const size_t at = static_cast<size_t>(kc) * TC_N * TC_CHUNK + static_cast<size_t>(n) * TC_CHUNK +
                            static_cast<size_t>(((kk >> 4) ^ (n & 7)) << 4) + (kk & 15);
          (*b_image)[at] = static_cast<uint8_t>(static_cast<int8_t>(digit(hq[i], l)));
        }
      }
    }
  }
  offs->assign(2 * (L + 1), 0);
  long long suffix = 0;
  for (int m = L; m >= 0; m--) {
    if (m < L) {
      suffix += hq[m];
    }
    const long long hi = suffix >> 14, lo = suffix & 16383;   // floor split, lo in [0, 2^14)
    (*offs)[2 * m] = static_cast<int32_t>(255 * hi);
    (*offs)[2 * m + 1] = static_cast<int32_t>(255 * lo);
  }
}

// Host-only model of the kernel's arithmetic from the SAME tables (include/fmgpu.h:
// fmgpu_decim_tc_host_model): digits read back out of the B image through the operand layout, exact
// 64-bit limb sums, the epilogue's integer offset removal and single float rounding. `valid` = real
// sample pairs in front of the block (the rest of the window is byte 0, as after a reset).
size_t decimTcHostModel(int M, const std::vector<float> &hrev, float scale, const uint8_t *iq, int valid,
                        int n_out, float *out) {
  const int L = static_cast<int>(hrev.size());
  if (!decimTcSupported(M, L, n_out) || !iq || !out || valid < 0 || valid > L - 1) {
    return 0;
  }
  std::vector<uint8_t> b_image;
  std::vector<int32_t> offs;
  decimTcBuildTables(M, hrev, &b_image, &offs);
  const int ws0 = ((2 * L - 2) + 31) / 32 * 32;
  const int ksteps = (ws0 + 2 * M * (TC_NO - 1) + 2 + 31) / 32;
  const int adv = 2 * M * TC_NO;
  const float out_scale = static_cast<float>(static_cast<double>(scale) / (255.0 * static_cast<double>(1 << TC_SHIFT)));
  // iq: `valid` pairs of history, then n_out * M pairs; byte b of the block sits at iq[2 * valid + b]
  auto byteAt = [&](long b) -> int {   // block-relative byte; in front of the history: 0
    const long at = 2L * valid + b;
    return at < 0 ? 0 : iq[at];
  };
  for (int t = 0; t < n_out / TC_NO; t++) {
    long long D[TC_N] = {};
    for (int k = 0; k < 32 * ksteps; k++) {
      const int a = byteAt(static_cast<long>(adv) * t - ws0 + k);
      if (a == 0) {
        continue;
      }
      const int kc = k / TC_CHUNK, kk = k % TC_CHUNK;
      for (int n = 0; n < TC_N; n++) {
        const size_t at = static_cast<size_t>(kc) * TC_N * TC_CHUNK + static_cast<size_t>(n) * TC_CHUNK +
                          static_cast<size_t>(((kk >> 4) ^ (n & 7)) << 4) + (kk & 15);
        D[n] += static_cast<long long>(a) * static_cast<int8_t>(b_image[at]);
      }
    }
    for (int j = 0; j < TC_NO; j++) {
      const int missing = (L - 1) - M * (t * TC_NO + j) - valid;
      const int m = missing > 0 ? std::min(missing, L) : 0;
      for (int q = 0; q < 2; q++) {
        const int col = j * 2 + q;
        const int hi = static_cast<int>((D[col] << 7) + D[2 * TC_NO + col]);
        const int lo = static_cast<int>((D[4 * TC_NO + col] << 7) + D[6 * TC_NO + col]);
        const int ph = 2 * hi - offs[2 * m];
        const int pl = 2 * lo - offs[2 * m + 1];
        out[2 * (t * TC_NO + j) + q] = std::fmaf(static_cast<float>(ph), 16384.0f, static_cast<float>(pl)) * out_scale;
      }
    }
  }
  return static_cast<size_t>(n_out);
}

cudaError_t launchDecimTc(int M, int L, const uint8_t *iq, size_t iq_stride, size_t iq_row_bytes,
                          const uint8_t *hist, const int *hist_valid, int total_rows, float2 *x1,
                          size_t x1_pitch, int n_out, int ch0, int nch, float scale,
                          const uint8_t *b_image_dev, const int32_t *offs_dev, int sm_count,
                          cudaStream_t stream) {
  static DeviceOnce attrs;  // per device: device_once.h
  const cudaError_t attr_err = attrs.run([] {
    const void *fs[] = {(const void *)k_decim_tc<28>, (const void *)k_decim_tc<22>, (const void *)k_decim_tc<0>};
    cudaError_t err = cudaSuccess;
    for (const void *f : fs) {
      if (err == cudaSuccess) {
        err = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(tcSmemBytes(TC_RING_TMEM_A)));
      }
    }
    return err;
  });
  if (attr_err != cudaSuccess) {
    return attr_err;
  }
  TcParams p{};
  p.M = M;
  p.L = L;
  p.n_out = n_out;
  p.adv = 2 * M * TC_NO;
  p.ws0 = ((2 * L - 2) + 31) / 32 * 32;
  p.ksteps = (p.ws0 + 2 * M * (TC_NO - 1) + 2 + 31) / 32;
  p.halo_chunks = (p.ws0 + TC_CHUNK - 1) / TC_CHUNK;
  p.tiles = n_out / TC_NO;
  p.row_tiles = (nch + TC_ROWS - 1) / TC_ROWS;
  // segments: enough work items to fill the SMs several times over, at least 32 tiles each
  int n_seg = std::max(1, (8 * sm_count + p.row_tiles - 1) / p.row_tiles);
  n_seg = std::min(n_seg, std::max(1, p.tiles / 32));
  p.tiles_per_seg = (p.tiles + n_seg - 1) / n_seg;
  p.n_seg = (p.tiles + p.tiles_per_seg - 1) / p.tiles_per_seg;
  p.ch0 = ch0;
  p.nch = nch;
  p.out_scale = static_cast<float>(static_cast<double>(scale) / (255.0 * static_cast<double>(1 << TC_SHIFT)));
  CUtensorMap tm_iq, tm_hist;
  if (!encodeRows(&tm_iq, iq, iq_row_bytes, static_cast<uint64_t>(total_rows), iq_stride) ||
      !encodeRows(&tm_hist, hist, 2 * H_IQ, static_cast<uint64_t>(total_rows), 2 * H_IQ)) {
    return cudaErrorInvalidValue;
  }
  const int grid = std::min(sm_count, p.row_tiles * p.n_seg);
  p.ring = TC_RING_TMEM_A;
  const size_t smem_bytes = tcSmemBytes(TC_RING_TMEM_A);
  const uint4 *bi = reinterpret_cast<const uint4 *>(b_image_dev);
  const int2 *of = reinterpret_cast<const int2 *>(offs_dev);
#define FMGPU_TC_LAUNCH(KSV)                                                                              \
  k_decim_tc<KSV><<<grid, TC_THREADS, smem_bytes, stream>>>(tm_iq, tm_hist, bi, of, hist_valid, x1, x1_pitch, p)
  if (p.ksteps == 28) {          // /10 at 2.4 MS/s
    FMGPU_TC_LAUNCH(28);
  } else if (p.ksteps == 22) {   // /8 at 2.048 MS/s
    FMGPU_TC_LAUNCH(22);
  } else {
    FMGPU_TC_LAUNCH(0);
  }
#undef FMGPU_TC_LAUNCH
  return cudaGetLastError();
}

}  // namespace fmgpu
