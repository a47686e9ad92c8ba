// tc_common.cuh — device helpers shared by the tensor-core kernels (decim_tc.cu, fir_tc.cu):
// mbarrier, TMA, tcgen05 (MMA / commit / cp / ld / st / fences), shared-memory descriptors, and the
// host-side cuTensorMapEncodeTiled entry point. Everything is sm_100a inline PTX.
#ifndef FMGPU_TC_COMMON_CUH_
#define FMGPU_TC_COMMON_CUH_

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

namespace fmgpu {
namespace tc {

__device__ __forceinline__ uint32_t smemAddr(const void *p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbarInit(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbarWait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void mbarArrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbarExpectTx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tmaLoad2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int x,
                                          int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void ummaCommit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
__device__ __forceinline__ void tcFenceBefore() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcFenceAfter() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, 128B swizzle, 8-row groups 1024 bytes apart (UMMA::SmemDescriptor, version 1)
__device__ __forceinline__ uint64_t smemDesc(uint32_t addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((addr >> 4) & 0x3FFF);          // start address
  d |= static_cast<uint64_t>(1024 >> 4) << 32;               // stride byte offset
  d |= static_cast<uint64_t>(1) << 46;                       // descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;                       // SWIZZLE_128B
  return d;
}

// one lane of a converged warp; the region it guards is single-threaded and ptxas keeps its
// warp-uniform operands in uniform registers (no waterfall loop around UTCIMMA / UTCBAR)
__device__ __forceinline__ bool electOne() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// A operand from TMEM (128 lanes x 8 columns = 128 rows x 32 bytes of K), B from shared memory
__device__ __forceinline__ void ummaI8Ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// shared memory (128 rows x 256 bits, described like an MMA operand) -> TMEM (128 lanes x 8 columns)
__device__ __forceinline__ void tmemCp128x256(uint32_t tmem_dst, uint64_t s_desc) {
  asm volatile("tcgen05.cp.cta_group::1.128x256b [%0], %1;" ::"r"(tmem_dst), "l"(s_desc) : "memory");
}

__device__ __forceinline__ void tmemLd16(uint32_t taddr, int32_t *v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, "
      "%14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
        "=r"(v[15])
      : "r"(taddr));
}


// registers -> TMEM, 32 lanes x 8 columns (lane = the thread's lane inside its warp's quadrant)
__device__ __forceinline__ void tmemSt8(uint32_t taddr, const uint32_t *v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmemLd8(uint32_t taddr, int32_t *v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmemWaitLd() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmemWaitSt() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// shared memory -> global through a tensor map (bulk async group of the issuing thread)
__device__ __forceinline__ void tmaStore2d(const CUtensorMap *map, uint32_t src, int x, int y) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(src), "r"(x), "r"(y)
               : "memory");
}
__device__ __forceinline__ void bulkCommit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulkWaitRead() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulkWait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fenceProxyAsync() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

using EncodeFn = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                              const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                              CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                              CUtensorMapFloatOOBfill);

inline EncodeFn encodeFn() {
  static EncodeFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess) {
      fn = reinterpret_cast<EncodeFn>(p);
    }
  });
  return fn;
}


}  // namespace tc
}  // namespace fmgpu

#endif  // FMGPU_TC_COMMON_CUH_
