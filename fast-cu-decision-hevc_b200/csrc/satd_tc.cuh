// satd_tc.cuh - 8x8 Hadamard SATD on the 5th-generation tensor cores (tcgen05, sm_100a).
//
// SATD(o - p) = sum | (H8 (x) H8) (o - p) |.  The 64x64 matrix H8 (x) H8 has entries +-1, the pixels are
// 8-bit, so  D[r][j] = sum_k o_r[k] * B[j][k] - sum_k p_r[k] * B[j][k]  is an exact int8 x int8 -> int32
// tensor-core product: A = 128 tiles x 64 pixels (u8, K-major, one tile per TMEM lane), B = H8 (x) H8
// (s8), accumulated in TMEM, and the epilogue only has to sum |D[r][0..63]| per lane.
// north_star adopts this path only where ncu shows it beats the integer-ALU butterflies.
//
// Shared-memory operand layout (UMMA K-major, no swizzle, see cute/atom/mma_traits_sm100.hpp
// make_umma_desc<Major::K>): 16-byte chunks; chunk c of row r lives at
//     base + c * LBO + (r / 8) * SBO + (r % 8) * 16      with SBO = 128, LBO = rows * 16
// i.e. [chunk][row-group][8 rows][16 B]; one kind::i8 MMA consumes K = 32 bytes = 2 chunks.
//
// The tcgen05 / mbarrier / bulk-copy wrappers of the tensor-core RMD kernels (rmd_tc2_kernels.cu, rmd_tc3_kernels.cu) live here too.
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

namespace cucd {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major, SWIZZLE_NONE descriptor (version 1 = Blackwell)
__device__ __forceinline__ uint64_t make_desc(uint32_t smemAddr, uint32_t lboBytes, uint32_t sboBytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smemAddr >> 4) & 0x3fffu);
  d |= (uint64_t)((lboBytes >> 4) & 0x3fffu) << 16;
  d |= (uint64_t)((sboBytes >> 4) & 0x3fffu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
// kind::i8 instruction descriptor: D s32, A / B u8 (signed = 0) or s8, both K-major, M x N
__device__ __forceinline__ uint32_t make_idesc_i8(int M, int N, int aSigned, int bSigned) {
  uint32_t d = 0;
  d |= 2u << 4;                       // c_format = S32
  d |= (uint32_t)(aSigned ? 1 : 0) << 7;
  d |= (uint32_t)(bSigned ? 1 : 0) << 10;
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}
// kind::f16 instruction descriptor: D f32, A and B f16 K-major, M x N; aNeg negates the A operand
__device__ __forceinline__ uint32_t make_idesc_f16(int M, int N, int aNeg) {
  uint32_t d = 0;
  d |= 1u << 4;                       // D = F32
  d |= (uint32_t)(aNeg ? 1 : 0) << 13;
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}
__device__ __forceinline__ void mma_i8(uint32_t tmemD, uint64_t descA, uint64_t descB, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
      :: "r"(tmemD), "l"(descA), "l"(descB), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
// A operand in TMEM (lane = row, 4 K-bytes per 32-bit column), B through a shared-memory descriptor
__device__ __forceinline__ void mma_i8_ts(uint32_t tmemD, uint32_t tmemA, uint64_t descB, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
      :: "r"(tmemD), "r"(tmemA), "l"(descB), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void mma_f16_ss(uint32_t tmemD, uint64_t descA, uint64_t descB, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      :: "r"(tmemD), "l"(descA), "l"(descB), "r"(idesc), "r"(accumulate) : "memory");
}
// A operand in TMEM (lane = row, two K elements per 32-bit column)
__device__ __forceinline__ void mma_f16_ts(uint32_t tmemD, uint32_t tmemA, uint64_t descB, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
      :: "r"(tmemD), "r"(tmemA), "l"(descB), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* mbar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" :: "r"(smem_u32(mbar)) : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* mbar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" :: "r"(smem_u32(mbar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* mbar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" :: "r"(smem_u32(mbar)) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* mbar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" :: "r"(smem_u32(mbar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* mbar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}\n"
      :: "r"(smem_u32(mbar)), "r"(parity) : "memory");
}
// global -> shared bulk copy (TMA engine, 1-D); completes `bytes` on the mbarrier
__device__ __forceinline__ void bulk_g2s(void* dstSmem, const void* srcGlobal, uint32_t bytes, uint64_t* mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
               :: "r"(smem_u32(dstSmem)), "l"(srcGlobal), "r"(bytes), "r"(smem_u32(mbar)) : "memory");
}
// one lane of a converged warp
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* slotInSmem, uint32_t cols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" :: "r"(smem_u32(slotInSmem)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {        // the same full warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" :: "r"(addr), "r"(cols) : "memory");
}
// lane = TMEM lane of this thread's warp quarter, 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld16(uint32_t addr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(addr) : "memory");
}
// 32 accumulator columns -> 16 registers: (col 2j & 0xffff) | (col 2j+1 << 16)
__device__ __forceinline__ void tmem_ld16_pack(uint32_t addr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.pack::16b.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(addr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }
__device__ __forceinline__ void tmem_st16(uint32_t addr, const uint32_t* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};\n"
      :: "r"(addr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
         "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t addr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};\n"
      :: "r"(addr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
         "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]),
         "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory"); }

// B = H8 (x) H8 as s8 in the canonical K-major layout for N = 64 rows (coefficients), K = 64 pixels;
// `sign` = +1 or -1.  Called cooperatively by `nthreads` threads.  4 KB.
__device__ __forceinline__ void fill_hadamard64(int8_t* dst, int sign, int tid, int nthreads) {
  for (int i = tid; i < 64 * 64; i += nthreads) {
    const int j = i >> 6, k = i & 63;                 // coefficient j = (u, v), pixel k = (y, x)
    const int u = j >> 3, v = j & 7, y = k >> 3, x = k & 7;
    const int s = (__popc(u & y) + __popc(v & x)) & 1; // natural-ordered Hadamard entry (-1)^(<u,y> + <v,x>)
    const int c = k >> 4;                              // 16-byte chunk along K
    dst[c * (64 * 16) + (j >> 3) * 128 + (j & 7) * 16 + (k & 15)] = (int8_t)((s ? -1 : 1) * sign);
  }
}

}  // namespace tc
}  // namespace cucd
