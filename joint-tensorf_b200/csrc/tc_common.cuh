// tcgen05 / TMEM / mbarrier helpers (inline PTX, sm_100a) shared by the tensor-core
// shading-head kernels.
//
// Shared-memory operand tiles use the no-swizzle canonical UMMA layout in
// "chunk-major" order: element (r, c) of an R-row tile lives at byte
//     (c / 8) * (R * 16) + r * 16 + (c % 8) * 2                         (bf16)
// i.e. 8x8 core matrices of 128 B, rows contiguous inside a chunk of 8 columns.
//  * read as a K-major operand  (MN = r, K = c):  SBO = 128,    LBO = R * 16
//  * read as an MN-major operand (MN = c, K = r): SBO = R * 16, LBO = 128
// (cute/atom/mma_traits_sm100.hpp canonical INTERLEAVE forms). One thread per row
// writes 16 B per chunk, so a warp writes 512 contiguous bytes: conflict-free.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace jt {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "TC_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra TC_DONE;\n"
        "bra TC_WAIT;\n"
        "TC_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// ---- bulk copies (TMA engine, SASS UBLKCP) -----------------------------------------------------
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 ::"l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- proxies / tcgen05 fences ----------------------------------------------------------------------
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- TMEM ---------------------------------------------------------------------------------------
// one full warp; writes the TMEM base address to *slot (shared memory)
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// 32 lanes x 32 columns of fp32: thread `lane` of warp w reads TMEM lane 32*(w%4)+lane,
// columns [col, col+32) of the accumulator.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float v[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float v[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// ---- descriptors -----------------------------------------------------------------------------
// 64-bit shared-memory matrix descriptor, no swizzle (cute::UMMA::SmemDescriptor):
// [0,14) start>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version = 1, [61,64) layout = 0.
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46);
}
// 32-bit instruction descriptor for kind::f16, bf16 x bf16 -> fp32 (cute::UMMA::InstrDescriptor):
// [4,6) c_format = 1 (F32), [7,10) a_format = 1 (BF16), [10,13) b_format = 1, [15] a_major,
// [16] b_major (0 = K-major, 1 = MN-major), [17,23) N>>3, [24,29) M>>4.
__host__ __device__ constexpr uint32_t idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// general kind::f16 descriptor: operand formats fp16 (0) or bf16 (1). Both operands must use the SAME format on
// B200: a bf16 x fp16 product (tried for "bf16 gradients x fp16 activations" in the weight-gradient GEMMs) faults
// at run time, so the staged tiles stay bf16 (jt_tc_selftest mode 2 covers fp16 x fp16).
__host__ __device__ constexpr uint32_t idesc_f16(int M, int N, int a_mn_major, int b_mn_major, int a_bf16, int b_bf16) {
    return (1u << 4) | ((uint32_t)a_bf16 << 7) | ((uint32_t)b_bf16 << 10) | ((uint32_t)a_mn_major << 15) |
           ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// all previously issued MMAs of this thread arrive on the mbarrier when complete
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- bf16 packing ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_f16(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
// hi/lo split of a float pair with packed conversions only: hi = bf16x2(a, b) (one F2FP), the
// exact fp32 value of each half is a shift / mask of the packed word, lo = bf16x2 of the residuals.
__device__ __forceinline__ void split_pair(float a, float b, uint32_t& hi, uint32_t& lo) {
    hi = pack_bf16(a, b);
    lo = pack_bf16(a - __uint_as_float(hi << 16), b - __uint_as_float(hi & 0xFFFF0000u));
}

// store 8 consecutive columns (one 16 B chunk) of row `r` of an R-row tile; lo != nullptr
// additionally stores the rounding residuals into the second-term tile.
__device__ __forceinline__ void store_chunk(unsigned char* hi, unsigned char* lo, int R, int chunk, int r, const float v[8]) {
    uint4 h, l;
    if (lo) {
        split_pair(v[0], v[1], h.x, l.x); split_pair(v[2], v[3], h.y, l.y);
        split_pair(v[4], v[5], h.z, l.z); split_pair(v[6], v[7], h.w, l.w);
        *reinterpret_cast<uint4*>(lo + (size_t)chunk * R * 16 + r * 16) = l;
    } else {
        h.x = pack_bf16(v[0], v[1]); h.y = pack_bf16(v[2], v[3]); h.z = pack_bf16(v[4], v[5]); h.w = pack_bf16(v[6], v[7]);
    }
    *reinterpret_cast<uint4*>(hi + (size_t)chunk * R * 16 + r * 16) = h;
}

// fp16 variant of store_chunk (single term: 11 significant bits, 8x finer than bf16)
__device__ __forceinline__ void store_chunk_f16(unsigned char* t, int R, int chunk, int r, const float v[8]) {
    uint4 h;
    h.x = pack_f16(v[0], v[1]); h.y = pack_f16(v[2], v[3]); h.z = pack_f16(v[4], v[5]); h.w = pack_f16(v[6], v[7]);
    *reinterpret_cast<uint4*>(t + (size_t)chunk * R * 16 + r * 16) = h;
}

}  // namespace tc
}  // namespace jt
