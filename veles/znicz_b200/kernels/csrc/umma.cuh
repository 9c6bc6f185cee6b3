// sm_100a primitives: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld).
// Hand-written inline PTX (no CUTLASS); descriptor bit layouts follow the PTX ISA
// "tcgen05 shared memory descriptor" / "instruction descriptor" tables.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace zn { namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
// Bounded wait: a protocol bug traps instead of hanging the GPU. The bound is WALL time
// (%globaltimer, ZN_MBAR_TIMEOUT_NS, default 20 s): a cycle-count bound fired under
// compute-sanitizer / ncu replay, where a kernel legitimately runs 100-1000x slower.
// -DZN_MBAR_TIMEOUT_NS=0 compiles the check out (release builds that prefer a hang to a trap).
#ifndef ZN_MBAR_TIMEOUT_NS
#define ZN_MBAR_TIMEOUT_NS 20000000000ULL
#endif
__device__ __forceinline__ unsigned long long mbar_now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
#if ZN_MBAR_TIMEOUT_NS > 0
  const unsigned long long t0 = mbar_now_ns();
  unsigned spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 255u) == 0 && mbar_now_ns() - t0 > ZN_MBAR_TIMEOUT_NS) { __trap(); }
  }
#else
  while (!mbar_try_wait(bar, parity)) {}
#endif
}
// 16-byte asynchronous global -> shared copy (LDGSTS); src_bytes = 0 zero-fills the destination
__device__ __forceinline__ void cp_async_16(uint32_t smem_dst, const void* gsrc, uint32_t src_bytes) {
  // .ca: keep the line in L1 - an implicit-GEMM gather re-reads every input element once per
  // filter tap (25x for 5x5), and the tile's halo (<= 20 KB) fits L1; with .cg all of those
  // re-reads went to L2 and the conv kernels were L2-bandwidth bound
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(smem_dst), "l"(gsrc),
               "r"(src_bytes)
               : "memory");
}
// the mbarrier receives one (pre-counted) arrival once all prior cp.async of this thread landed
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// generic-proxy smem writes -> visible to the async proxy (TMA / tensor core reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// im2col-mode TMA (NHWC activation tensor, map built by cuTensorMapEncodeIm2col): loads
// `pixelsPerColumn` consecutive filter-window positions starting at base coordinate (w, h, n) -
// the window's top-left corner in input coordinates, i.e. q * stride - pad - walking W, then H,
// then N inside the bounding box, `channelsPerPixel` channels from c of the pixel at
// base + (off_w, off_h) each; out-of-image pixels arrive as zeros. One instruction replaces the
// 128-thread LDGSTS gather of a [128 pixels x 64 channels] operand block.
__device__ __forceinline__ void tma_load_im2col_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                                   int c, int w, int h, int n, uint16_t off_w,
                                                   uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};" ::"r"(smem_u32(smem_dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
      : "memory");
}

// shared -> global tile store (async proxy); smem must stay valid until wait_group.read
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0,
                                             int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}

// ------------------------------------------------------------------ tcgen05
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16/fp16 inputs, fp32 accumulate
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], 8-bit float inputs (formats in the instruction descriptor),
// fp32 accumulate; one instruction consumes K = 32 elements = 32 bytes of each operand row
__device__ __forceinline__ void mma_f8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                       uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread arrive on `bar` when complete
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread = lane/row)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor, SWIZZLE_128B, version 1 (Blackwell):
//   [0,14)  start address >> 4     [16,30) leading-dim byte offset >> 4
//   [32,46) stride-dim byte offset >> 4     [46,48) version = 1     [61,64) layout = 2 (SW128)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor for kind::f16 with BF16 A/B and FP32 accumulate:
//   [4,6) c_format=1 (F32)  [7,10) a_format=1 (BF16)  [10,13) b_format=1 (BF16)
//   [15] a_major (0=K,1=MN)  [16] b_major  [17,23) N>>3  [24,29) M>>4
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// kind::f8f6f4 with E4M3 x E4M3 (format code 0 for both operands), K-major operands
__host__ __device__ constexpr uint32_t make_idesc_e4m3(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

}}  // namespace zn::umma
