// Unit test of the tcgen05 plumbing the tensor-core kernels share (tc_common.cuh / head_tc.cuh): one CTA stages
// A and B into shared memory in the canonical UMMA layout, issues the MMAs and reads D back from TMEM, so that the
// shared-memory and instruction descriptors, K-major and MN-major operand reads and fp16 operands can be checked
// against a plain matrix product (jt_tc_selftest, tests/test_gpu_tc.py).
#include "head_tc.cuh"
#include "../../include/jt_vm.h"

namespace jt {
using namespace tc;

// ------------------------------------------------------------------ self test of the MMA plumbing
// mode 0: D[128][N] = A[128][K] * B[N][K]^T          (K-major operands)
// mode 1: D[m][n]   = sum_s X[s][m] * Y[s][n]        (MN-major operands; X [128][Ma], Y [128][N], K = 128 rows)
// mode 2: mode 0 with both operands stored as fp16
__global__ void __launch_bounds__(128) tc_selftest_kernel(int mode, const float* __restrict__ A, int lda,
                                                          const float* __restrict__ B, int ldb, float* __restrict__ D,
                                                          int K, int N, int Ma) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    unsigned char* ta = smem;                       // A / X tile: 128 rows x 128 cols max
    unsigned char* tb = smem + tile_bytes(128, 256);
    if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
    if (warp == 0) tmem_alloc(&tmem_slot, 256);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    if (mode == 0 || mode == 2) {
        for (int c = 0; c < K / 8; ++c) {           // thread = row of A
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = A[(size_t)tid * lda + c * 8 + i];
            if (mode == 2) store_chunk_f16(ta, 128, c, tid, v); else store_chunk(ta, nullptr, 128, c, tid, v);
        }
        if (mode == 2) {
            for (int idx = tid; idx < N * (K / 8); idx += 128) {
                const int chunk = idx / N, n = idx - chunk * N;
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = B[(size_t)n * ldb + chunk * 8 + i];
                store_chunk_f16(tb, N, chunk, n, v);
            }
        } else {
            stage_weight(tb, nullptr, B, ldb, N, K, N, K, nullptr, -1, 0);
        }
    } else {
        for (int c = 0; c < 128 / 8; ++c) {         // X tile padded to 128 columns with zeros
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = (c * 8 + i < Ma) ? A[(size_t)tid * lda + c * 8 + i] : 0.f;
            store_chunk(ta, nullptr, 128, c, tid, v);
        }
        for (int c = 0; c < N / 8; ++c) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = B[(size_t)tid * ldb + c * 8 + i];
            store_chunk(tb, nullptr, 128, c, tid, v);
        }
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
        tc_fence_after();
        if (mode == 0) {
            issue_gemm_kmajor<1>(tmem, ta, nullptr, tb, nullptr, K, N, N);
        } else if (mode == 2) {
            const uint32_t idesc = idesc_f16(128, N, 0, 0, 0, 0);
            for (int ks = 0; ks < K / 16; ++ks)
                mma_bf16(tmem, smem_desc(smem_u32(ta) + ks * 2 * 128 * 16, 128 * 16, 128),
                         smem_desc(smem_u32(tb) + ks * 2 * N * 16, N * 16, 128), idesc, ks > 0);
        } else {
            const uint32_t idesc = idesc_bf16(128, N, 1, 1);
            for (int ks = 0; ks < 128 / 16; ++ks) {             // K = sample rows, 16 per step = 256 B
                const uint64_t ad = smem_desc(smem_u32(ta) + ks * 256, 128, 128 * 16);
                const uint64_t bd = smem_desc(smem_u32(tb) + ks * 256, 128, 128 * 16);
                mma_bf16(tmem, ad, bd, idesc, ks > 0);
            }
        }
        mma_commit(&bar);
    }
    mbar_wait(&bar, 0);
    tc_fence_after();
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
    for (int c0 = 0; c0 < N; c0 += 16) {
        float v[16];
        tmem_ld16(lane_addr + c0, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) if (c0 + i < N) D[(size_t)tid * N + c0 + i] = v[i];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

}  // namespace jt

using namespace jt;

extern "C" int jt_tc_selftest(int mode, const float* A, int lda, const float* B, int ldb, float* D, int K, int N,
                              int Ma, cudaStream_t stream) {
    JT_CHECK_ARG(A && B && D && mode >= 0 && mode <= 2);
    JT_CHECK_ARG(N % 16 == 0 && N >= 16 && N <= 256 && K % 16 == 0 && K >= 16 && K <= 256 && Ma <= 128);
    const int smem = tile_bytes(128, 256) * 2;
    if (int rc = set_smem(tc_selftest_kernel, smem)) return rc;
    g_launches += 1;
    tc_selftest_kernel<<<1, 128, smem, stream>>>(mode, A, lda, B, ldb, D, K, N, Ma);
    JT_RETURN_LAUNCH();
}
