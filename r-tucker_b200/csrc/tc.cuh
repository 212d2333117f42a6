// tcgen05 / TMEM / mbarrier helpers for sm_100a (inline PTX).  Internal to the library.
//
// Operand staging convention used by every tensor-core kernel here ("interleaved core matrices",
// UMMA SWIZZLE_NONE): a 2-D fp32 array X[rows][cols] (cols contiguous in global memory) is stored as
//     byte_offset(row, col) = (col / 4) * CS + (row / 8) * RS + (row % 8) * 16 + (col % 4) * 4
// i.e. 8 rows x 16 bytes form one contiguous 128-byte core matrix.  The SAME buffer is a valid
//   * K-major operand when the contraction runs along `cols`  (LBO = CS, SBO = RS), and a valid
//   * MN-major operand when the contraction runs along `rows` (LBO = RS, SBO = CS),
// which lets one staged tile feed GEMMs that contract either index (Z = Q O^T, H = G O, dO = G^T Q').
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rt {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- shared-memory matrix descriptor (SWIZZLE_NONE) ----
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);            // bits 0-13: start address >> 4
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;       // bits 16-29: leading dimension byte offset >> 4
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;       // bits 32-45: stride dimension byte offset >> 4
  d |= (uint64_t)1 << 46;                                 // bits 46-47: descriptor version (sm_100)
  return d;                                               // bits 61-63 = 0: no swizzle
}

// ---- instruction descriptor, kind::tf32, fp32 accumulate ----
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4)                       // D format: F32
         | (2u << 7) | (2u << 10)        // A, B format: TF32
         | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16)
         | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
      :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}

// all previously issued MMAs of this thread arrive on the mbarrier when complete
__device__ __forceinline__ void mma_commit(uint64_t* mbar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
               :: "r"(smem_u32(mbar)) : "memory");
}

// ---- TMEM allocation (one full warp) ----
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n"
               :: "r"(smem_u32(smem_slot)), "n"(kCols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" :: "r"(taddr), "n"(kCols) : "memory");
}

__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (tensor core operand reads)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// ---- TMEM -> registers: this warp's 32 lanes x 32 consecutive columns (fp32 bit patterns) ----
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// ---- mbarrier ----
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t}\n"
      :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}

__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;\n" : "=r"(r) : "f"(x));
  return r;
}

// ---- instruction descriptor, kind::f16 with fp16 operands, fp32 accumulate ----
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4)                       // D format: F32
         | (0u << 7) | (0u << 10)        // A, B format: F16
         | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16)
         | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                        bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}

// ---- mbarrier extras ----
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}

// ---- bulk async copies (TMA, non-tensor): global -> shared with mbarrier completion; shared -> global
//      as plain store or as an fp32 add-reduction performed at the L2, tracked by bulk groups ----
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
               :: "r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// a copy of any size as 32 KB bulk copies on one mbarrier
__device__ __forceinline__ void bulk_g2s_split(unsigned char* dst, const unsigned char* src, uint32_t bytes, uint64_t* bar) {
  for (uint32_t o = 0; o < bytes; o += 32768u) bulk_g2s(dst + o, src + o, min(32768u, bytes - o), bar);
}
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n"
               :: "l"(dst), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_s2g_add_f32(void* dst, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;\n"
               :: "l"(dst), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;\n" :: "n"(N) : "memory"); }

// byte offset of element (row, col) of a 16-bit array in the interleaved format: 8 rows x 16 bytes
// (8 columns) per core matrix; CS = byte stride between 8-column blocks (>= rows * 16)
__device__ __forceinline__ uint32_t il16_offset(int row, int col, uint32_t CS) {
  return (uint32_t)(col >> 3) * CS + (uint32_t)(row >> 3) * 128u + (uint32_t)(row & 7) * 16u + (uint32_t)(col & 7) * 2u;
}

// byte offset of element (row, col) in the interleaved staging format (see file header)
__device__ __forceinline__ uint32_t il_offset(int row, int col, uint32_t CS, uint32_t RS) {
  return (uint32_t)(col >> 2) * CS + (uint32_t)(row >> 3) * RS + (uint32_t)(row & 7) * 16u + (uint32_t)(col & 3) * 4u;
}

}  // namespace tc
}  // namespace rt
