// tc_common.cuh -- PTX wrappers shared by the tcgen05 kernels (flow_t4.cu, flow_row.cu): mbarrier, TMA bulk copy,
// tcgen05.mma / commit / ld / st, UMMA descriptors, the 3-product split GEMM issue, and the packed-image constants.
#pragma once
#include <cuda_fp16.h>

#include "mobius_fast.cuh"
#include "rnf_common.cuh"

namespace rnf {

// Packed global image of one Mobius conditioner (== the shared-memory pieces, one bulk copy each):
//   W1 | W2 | W3 : each [hi 64x64 | lo 64x64] fp16 K-major SWIZZLE_128B, then the bias block [64 x 16] fp16 (no swizzle)
//   W4           : [hi 256x64 | lo 256x64] fp16 SW128 (outputs permuted: component c owns columns 4c..4c+3), bias block [256 x 16]
//   aux          : first[64][4] fp32  (W0[:, :3] and b0 of fc_first), then the fc_first block [64 x 16] fp16 (no swizzle)
// A bias block holds (b_hi, b_lo) in its K columns 0 and 1; multiplied by a constant [128 x 16] tile with ones in those two
// columns it initialises the accumulator with the bias, so the CUDA cores never touch a bias or a scale factor.
constexpr int kBiasBlkHid = 64 * 32;
constexpr int kBiasBlkLast = 256 * 32;
constexpr int kW1Bytes = 2 * 8192 + kBiasBlkHid;  // 18432
constexpr int kHidW = 3 * kW1Bytes;               // 55296
constexpr int kLastW = 2 * 32768 + kBiasBlkLast;  // 73728
constexpr int kAuxFirst = 1024;                   // first[64][4] fp32
constexpr int kAuxBytes = kAuxFirst + kBiasBlkHid; // + fc_first block [64 x 16] fp16 (flow_t4.cu)
constexpr int kAuxStride = kAuxBytes;             // 3072
constexpr int kTcImageBytes = kHidW + kLastW + kAuxBytes;   // 132096

// ------------------------------------------------ PTX wrappers ---------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void named_bar(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_arrive(int id, int nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] . B[smem desc]^T, kind::f16 (fp16 operands, fp32 accumulate).  The 64-bit shared-memory
// descriptors are passed as (low word, common high word): only the low word (start address) changes between MMAs, so
// the single issuing thread spends ~5 instructions per MMA instead of rebuilding both descriptors.
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint32_t a_lo32, uint32_t b_lo32, uint32_t desc_hi32, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 da, db;\n"
      "setp.ne.b32 p, %5, 0;\n"
      "mov.b64 da, {%1, %3};\n"
      "mov.b64 db, {%2, %3};\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_lo32), "r"(b_lo32), "r"(desc_hi32), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float v[32]) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
        "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]), "=r"(u[16]),
        "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]), "=r"(u[24]),
        "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// the inverse: 32 registers -> 32 consecutive fp32 columns of the thread's own TMEM lane (private scratch)
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float v[32]) {
  const uint32_t* u = reinterpret_cast<const uint32_t*>(v);
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]), "r"(u[8]), "r"(u[9]),
      "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15]), "r"(u[16]), "r"(u[17]), "r"(u[18]),
      "r"(u[19]), "r"(u[20]), "r"(u[21]), "r"(u[22]), "r"(u[23]), "r"(u[24]), "r"(u[25]), "r"(u[26]), "r"(u[27]),
      "r"(u[28]), "r"(u[29]), "r"(u[30]), "r"(u[31])
      : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// Asynchronous 16-column TMEM load + a wait that names the destination registers, so that the compiler cannot move
// their consumers above the wait: lets the next chunk's load fly underneath the arithmetic on the current chunk.
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, float v[16]) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
        "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait16(float v[16]) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(u[0]), "+r"(u[1]), "+r"(u[2]), "+r"(u[3]), "+r"(u[4]), "+r"(u[5]), "+r"(u[6]), "+r"(u[7]), "+r"(u[8]),
                 "+r"(u[9]), "+r"(u[10]), "+r"(u[11]), "+r"(u[12]), "+r"(u[13]), "+r"(u[14]), "+r"(u[15])
               :
               : "memory");
}
// stores without the wait (the caller issues one tmem_st_wait() for a batch)
__device__ __forceinline__ void tmem_st16_nowait(uint32_t taddr, const uint32_t u[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]), "r"(u[8]), "r"(u[9]),
      "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// elect.sync: exactly one lane of a converged warp returns true.  Issuing tcgen05.mma under this predicate (inside a
// warp-uniform branch) lets ptxas move the operands to uniform registers with one R2UR each; with an ordinary
// per-thread condition it emits an ELECT / R2UR.BROADCAST / BRA.U.ANY loop per MMA (~15 instructions, ~85 cycles each).
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 rx;\n"
      ".reg .pred px;\n"
      "elect.sync rx|px, 0xFFFFFFFF;\n"
      "@px mov.s32 %0, 1;\n"
      "}\n"
      : "+r"(pred));
  return pred != 0;
}

// UMMA shared-memory descriptor: K-major, SWIZZLE_128B, 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor layout:
// start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) | layout_type=2 (SW128) [61,64)).
constexpr uint32_t kDescHi = 64u | (1u << 14) | (2u << 29);          // bits [32,64): SBO = 1024 B, version 1, SW128
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t saddr) { return ((saddr >> 4) & 0x3FFFu) | (1u << 16); }
// No-swizzle K-major ("interleave") descriptor for the 16-wide bias / ones blocks: 8 x 16 B core matrices, the two K halves
// 128 B apart (LBO), 8-row groups 256 B apart (SBO): element (r, k) at (r/8)*256 + (k/8)*128 + (r%8)*16 + (k%8)*2.
constexpr uint32_t kDescHiNS = 16u | (1u << 14);
__device__ __forceinline__ uint32_t umma_desc_lo_ns(uint32_t saddr) { return ((saddr >> 4) & 0x3FFFu) | (8u << 16); }
// instruction descriptor (cute::UMMA::InstrDescriptor): c=F32 [4,6)=1, a=b=F16 (0), K-major both, N>>3 [17,23), M>>4 [24,29)
__device__ __host__ constexpr uint32_t umma_idesc(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// Issue D[128 x N] = bias + A[128 x 64] . W[N x 64]^T: one K = 16 MMA of the constant ones tile against the bias block
// initialises the accumulator, then the 3-product split  Alo.Whi + Ahi.Wlo + Ahi.Whi  accumulates on top.  a_* / b_* are
// descriptor low words (hi / lo fp16 planes, K-major SW128, 128 B per row); a K step of 16 elements = 32 B = +2.
__device__ __forceinline__ void issue_split_gemm(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                                 uint32_t ones_ns, uint32_t bias_ns, uint32_t idesc) {
  umma_f16(d_tmem, ones_ns, bias_ns, kDescHiNS, idesc, 0);
#pragma unroll
  for (int k = 0; k < 4; ++k) umma_f16(d_tmem, a_lo + 2 * k, b_hi + 2 * k, kDescHi, idesc, 1);
#pragma unroll
  for (int k = 0; k < 4; ++k) umma_f16(d_tmem, a_hi + 2 * k, b_lo + 2 * k, kDescHi, idesc, 1);
#pragma unroll
  for (int k = 0; k < 4; ++k) umma_f16(d_tmem, a_hi + 2 * k, b_hi + 2 * k, kDescHi, idesc, 1);
}

}  // namespace rnf
