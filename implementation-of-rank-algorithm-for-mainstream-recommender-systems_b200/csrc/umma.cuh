// umma.cuh — tcgen05 / TMEM / mbarrier helpers shared by the tensor-core kernels (din.cu, afm.cu, linear.cu).
// sm_100a only.  Operands are bf16 tiles in shared memory in the canonical 128-byte-swizzled layouts (8 lines
// of 128 B form one 1024-byte swizzle atom; the 16-byte chunk index of a line is XORed with line % 8), or, for
// the MN-major tf32 operands of linear.cu, the 128B-base-32B layout described at umma_desc_mn_tf32 (4-line,
// 512-byte atoms; 32-byte granules XORed with line % 4).  Accumulators are fp32 in TMEM, one elected thread
// issues the MMAs.
#pragma once
#include <cuda_bf16.h>
#include "common.cuh"

namespace rk {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// Bounded wait: a faulted MMA must trap, not hang the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    for (uint32_t spin = 0; spin < (1u << 26); ++spin) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
        if (ok) return;
    }
    __trap();
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {   // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {     // same warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols));
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// K-major, 128-byte-swizzled operand: rows of 64 bf16 (128 B), 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3ffff) >> 4);      // start address   [0,14)
    d |= (uint64_t)1 << 16;                           // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;                 // stride byte offset  [32,46)
    d |= (uint64_t)1 << 46;                           // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                           // SWIZZLE_128B
    return d;
}
// kind::f16, A = B = bf16 (K-major), D = f32, M = 128
__host__ __device__ constexpr uint32_t umma_idesc(int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// 16 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// one fp32 column of this thread's TMEM lane (slow paths that walk columns in a loop)
__device__ __forceinline__ float tmem_ld1(uint32_t taddr) {
    uint32_t r;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    return __uint_as_float(r);
}
// 64 consecutive fp32 columns of this thread's TMEM lane in one instruction (one wait instead of two)
__device__ __forceinline__ void tmem_ld64(uint32_t taddr, float (&v)[64]) {
    uint32_t r[64];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 64; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
// Write 8 consecutive K elements (one 16-byte chunk c) of row r into a swizzled operand tile.
__device__ __forceinline__ void store_chunk(uint8_t* tile, int r, int c, const float (&v)[8]) {
    uint4 w;
    w.x = pack_bf16(v[0], v[1]); w.y = pack_bf16(v[2], v[3]);
    w.z = pack_bf16(v[4], v[5]); w.w = pack_bf16(v[6], v[7]);
    *reinterpret_cast<uint4*>(tile + r * 128 + ((c ^ (r & 7)) << 4)) = w;
}

// Split-bf16 operands: x = hi + lo with hi = bf16(x), lo = bf16(x - hi).  A.W is accumulated as
// A_hi.W_hi + A_lo.W_hi + A_hi.W_lo on the tensor core (fp32 accumulation), which keeps ~16 bits
// of every operand: the tensor pipe is nearly idle in this kernel, so the two extra MMAs are free.
__device__ __forceinline__ void store_chunk_split(uint8_t* hi_tile, uint8_t* lo_tile, int r, int c,
                                                  const float (&v)[8]) {
    float lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) lo[j] = v[j] - __bfloat162float(__float2bfloat16_rn(v[j]));
    store_chunk(hi_tile, r, c, v);
    store_chunk(lo_tile, r, c, lo);
}

// 8 consecutive floats (32-byte aligned: every block of the packed weights starts on a multiple of 8)
__device__ __forceinline__ void ld8(const float* __restrict__ p, float (&v)[8]) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// The same tile read with MN as the contiguous dimension (the transposed operand): lines are K
// indices, the 64 elements of a line are consecutive M (or N) indices; `mn_block_bytes` is the
// distance between blocks of 64 MN elements (the leading byte offset), 8-line groups are 1024 B
// apart (the stride byte offset).  Advance K by 16 lines = +2048 bytes on the start address.
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t smem_addr, uint32_t mn_block_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3ffff) >> 4);
    d |= (uint64_t)((mn_block_bytes >> 4) & 0x3fff) << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// ---- kind::tf32 (fp32 operands rounded to tf32 by the caller, fp32 accumulation) ----
// MN-major tf32 operands take only the SWIZZLE_128B_BASE32B layout (type 1; CUTLASS's Layout_MN_SW128_32B_Atom):
// lines of 32 fp32 MN elements (128 bytes), 4 lines form a 512-byte atom in which the 32-byte granule index of
// a line is XORed with line % 4 (address bits [5,7) ^= [7,9)).  4-line groups are 512 bytes apart (the stride
// byte offset), so one MMA's K = 8 is two atoms and K advances by +1024 bytes per MMA; blocks of 32 MN
// elements are `mn_block_bytes` apart (the leading byte offset).
__device__ __forceinline__ uint64_t umma_desc_mn_tf32(uint32_t smem_addr, uint32_t mn_block_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3ffff) >> 4);
    d |= (uint64_t)((mn_block_bytes >> 4) & 0x3fff) << 16;
    d |= (uint64_t)(512 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;                           // SWIZZLE_128B_BASE32B
    return d;
}
// kind::tf32, A = B = tf32 (format 2 at bits 7 and 10), D = f32, M = 128; OR in kUmmaAMn / kUmmaBMn for MN-major
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// 3xTF32 split: x = hi + lo exactly, hi = x rounded to tf32 (low 13 mantissa bits zero, ties away from zero).
// The tensor core reads the top 19 bits of lo, so hi.hi + lo.hi + hi.lo keeps about 22 bits of each operand.
// A finite |x| within 2^-11 relative of FLT_MAX rounds hi to inf (lo = -inf): far outside any gradient.
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
    uint32_t h;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(x));
    hi = __uint_as_float(h);
    lo = x - hi;
}

// asynchronous global -> shared copies (LDGSTS); completion through cp.async.commit_group / wait_group
__device__ __forceinline__ void cp_async8(const void* dst_smem, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(const void* dst_smem, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// One bulk (TMA) copy global -> shared of `bytes` (a multiple of 16, both sides 16-byte aligned), completing on
// an mbarrier: the issuing thread first announces the byte count (arrive.expect_tx), everybody then waits on
// the barrier's phase.  Used for operand tiles that a prologue kernel has already laid out in their swizzled
// shared-memory image: one instruction instead of a convert-and-store loop per CTA.
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// instruction-descriptor bits selecting MN-major A / B
constexpr uint32_t kUmmaAMn = 1u << 15;
constexpr uint32_t kUmmaBMn = 1u << 16;

}  // namespace tc
}  // namespace rk
