// Shared pieces of the tensor-core shading-head kernels (forward: app_basis_tc.cu +
// head_mlp_tc.cu, backward: shade_tc_bwd.cu): dimensions of the MLP_Fea head, the
// tensor-core column order of layer 1, operand staging and GEMM issue helpers.
#pragma once
#include "jt_common.cuh"
#include "tc_common.cuh"

namespace jt {
using namespace tc;

constexpr int TM = 128;                    // samples per tile == threads per CTA
constexpr int F_ = 27, NB = 32;            // app_dim, padded N of the basis GEMM
constexpr int CT = 144;                    // sum of appearance components
constexpr int IN_ = 150, K1 = 160;         // encoded input (reference order) / padded tensor-core order
constexpr int BIAS1 = 30;                  // tensor-core column order of layer 1 (any K permutation is a valid GEMM):
                                           //   0..26 feat | 27..29 dir | 30 = 1.0 (bias) | 31 = 0 |
                                           //   32+4e..35+4e = [sin x, sin 2x, cos x, cos 2x] of element e
                                           //   (e < 27: feat e, e >= 27: dir e-27) | 152..159 = 0
// reference column (tensorBase.py:116-122 concatenation order) of tensor-core column c; -1 zero, -2 bias
__host__ __device__ constexpr int ref_col_l1(int c) {
    if (c < F_ + 3) return c;
    if (c == BIAS1) return -2;
    if (c < 32 || c >= 152) return -1;
    const int cc = c - 32, e = cc >> 2, r = cc & 3;
    return e < F_ ? (F_ + 3) + 4 * e + r : (F_ + 3) + 4 * F_ + 4 * (e - F_) + r;
}
constexpr int H_ = 64, K2 = 80;            // hidden, padded K of layer 2 (col 64 = 1 -> bias)

__host__ __device__ constexpr int tile_bytes(int rows, int cols) { return rows * cols * 2; }

// ------------------------------------------------------------------ generic staging helpers
// W (n, k) fp32 row-major [N][ldw] -> canonical bf16 tile of NR rows x KP cols. `kmap` selects the
// source column of tile column k: 0 identity (k == bias_col takes bias[n]), 1 layer-1 tensor-core order.
// F16: single-term fp16 tile (inference mode, see issue_gemm_kmajor) instead of bf16 hi (+ lo).
template <bool F16>
__device__ __forceinline__ void store_chunk_t(unsigned char* hi, unsigned char* lo, int R, int chunk, int r, const float v[8]) {
    if (F16) store_chunk_f16(hi, R, chunk, r, v);
    else store_chunk(hi, lo, R, chunk, r, v);
}

template <bool F16 = false>
__device__ inline void stage_weight(unsigned char* hi, unsigned char* lo, const float* __restrict__ W, int ldw, int N, int K,
                             int NR, int KP, const float* __restrict__ bias, int bias_col, int kmap) {
    for (int idx = threadIdx.x; idx < NR * (KP / 8); idx += blockDim.x) {
        const int chunk = idx / NR, n = idx - chunk * NR;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int k = chunk * 8 + i;
            int src = k < K ? k : (k == bias_col ? -2 : -1);
            if (kmap == 1) src = ref_col_l1(k);
            float x = 0.f;
            if (n < N) {
                if (src >= 0) x = W[(size_t)n * ldw + src];
                else if (src == -2 && bias) x = bias[n];
            }
            v[i] = x;
        }
        store_chunk_t<F16>(hi, lo, NR, chunk, n, v);
    }
}

// issue the k-steps of one GEMM: D[128 x N] = A[128 x K] * B[N x K]^T, both K-major tiles.
// The descriptors of k-step ks differ from those of step 0 only in the start-address field
// (+ 2 chunks), so they are one 64-bit add each: the issuing thread's chain stays short.
// SPLIT = 1: bf16 operands; 2: hi + lo bf16 terms, 3 MMAs per product (fp32-class); 3: single-term fp16 operands
// (11 significant bits, 8x finer than bf16: rgb within ~2e-5 of the fp32 head at a third of the MMAs and half the
// shared memory -- used for inference only, because the backward's staged tiles must be bf16 for the range of the
// gradients and a tcgen05 product cannot mix operand formats).
template <int SPLIT>
__device__ __forceinline__ void issue_gemm_kmajor(uint32_t d_tmem, const unsigned char* a_hi, const unsigned char* a_lo,
                                                  const unsigned char* b_hi, const unsigned char* b_lo, int K, int NR,
                                                  int N) {
    const uint32_t idesc = SPLIT == 3 ? idesc_f16(128, N, 0, 0, 0, 0) : idesc_bf16(128, N, 0, 0);
    const uint32_t a_lbo = TM * 16, b_lbo = NR * 16;
    const uint64_t ah0 = smem_desc(smem_u32(a_hi), a_lbo, 128), bh0 = smem_desc(smem_u32(b_hi), b_lbo, 128);
    const uint64_t al0 = SPLIT == 2 ? smem_desc(smem_u32(a_lo), a_lbo, 128) : 0;
    const uint64_t bl0 = SPLIT == 2 ? smem_desc(smem_u32(b_lo), b_lbo, 128) : 0;
    const uint64_t a_inc = (2 * a_lbo) >> 4, b_inc = (2 * b_lbo) >> 4;
#pragma unroll 5
    for (int ks = 0; ks < K / 16; ++ks) {
        const uint64_t ah = ah0 + ks * a_inc, bh = bh0 + ks * b_inc;
        mma_bf16(d_tmem, ah, bh, idesc, ks > 0 ? 1u : 0u);
        if (SPLIT == 2) {
            mma_bf16(d_tmem, ah, bl0 + ks * b_inc, idesc, 1);
            mma_bf16(d_tmem, al0 + ks * a_inc, bh, idesc, 1);
        }
    }
}


// generic tile staging: value(n, k) supplied by a functor
template <class Fn>
__device__ __forceinline__ void stage_tile(unsigned char* hi, unsigned char* lo, int NR, int KP, Fn value) {
    for (int idx = threadIdx.x; idx < NR * (KP / 8); idx += blockDim.x) {
        const int chunk = idx / NR, n = idx - chunk * NR;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = value(n, chunk * 8 + i);
        store_chunk(hi, lo, NR, chunk, n, v);
    }
}

// ------------------------------------------------------------------ encoded-input row (tensorBase.py:43-55,116-122)
// in tensor-core column order (see BIAS1); PE values carry the annealing masks
// clamp(progress*2 - l, 0, 1).
struct PEMask { float f0, f1, v0, v1; };

// sin/cos with a two-constant Cody-Waite reduction to [-pi, pi] and the SFU approximations
// (abs error ~2^-21 there): well below the 2^-17 relative precision of the hi+lo bf16 operands.
__device__ __forceinline__ void fast_sincos(float x, float* s, float* c) {
    const float k = rintf(x * 0.15915494309189535f);
    float r = fmaf(k, -6.2831854820251465f, x);
    r = fmaf(k, 1.7484556000744883e-7f, r);
    *s = __sinf(r);
    *c = __cosf(r);
}

template <bool FAST = false>
__device__ __forceinline__ void encode_chunk(int chunk, const float feat[32], const float dir[3], const PEMask& pm,
                                             float v[8]) {
    if (chunk < 4) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int c = chunk * 8 + i;
            v[i] = c < F_ ? feat[c] : c < F_ + 3 ? dir[c - F_] : c == BIAS1 ? 1.0f : 0.f;
        }
    } else if (chunk < 19) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int e = (chunk - 4) * 2 + h;
            const bool is_view = e >= F_;
            const float src = is_view ? dir[e - F_] : feat[e];
            float s, co;
            if (FAST) fast_sincos(src, &s, &co); else sincosf(src, &s, &co);
            const float m0 = is_view ? pm.v0 : pm.f0, m1 = is_view ? pm.v1 : pm.f1;
            v[4 * h + 0] = s * m0;
            v[4 * h + 1] = (2.f * s * co) * m1;
            v[4 * h + 2] = co * m0;
            v[4 * h + 3] = (1.f - 2.f * s * s) * m1;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = 0.f;
    }
}


// staging block of one 128-sample tile in HBM (bytes): bf16 operand tiles in canonical layout
constexpr int SZ_A0 = tile_bytes(TM, CT), SZ_A1 = tile_bytes(TM, K1), SZ_A2 = tile_bytes(TM, K2), SZ_A3 = SZ_A2;
constexpr int SZ_D2 = tile_bytes(TM, H_), SZ_D1 = SZ_D2, SZ_DF = tile_bytes(TM, NB), SZ_DO = tile_bytes(TM, 8);
constexpr int OFF_A0 = 0, OFF_A1 = OFF_A0 + SZ_A0, OFF_A2 = OFF_A1 + SZ_A1, OFF_A3 = OFF_A2 + SZ_A2;
constexpr int OFF_D2 = OFF_A3 + SZ_A3, OFF_D1 = OFF_D2 + SZ_D2, OFF_DF = OFF_D1 + SZ_D1, OFF_DO = OFF_DF + SZ_DF;
constexpr int STAGE_TILE_BYTES = OFF_DO + SZ_DO;        // 161792

__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read2() { asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory"); }
constexpr int FD = 32;    // floats per feat/dir row written by app_basis_fwd_kernel: feat 0..26 | 27 pad | dir 28..30 | 31 pad

// One row of the dcomps tile [128 x 144] (TMEM columns t_dc ..) -> global, fp32 or bf16 (DC16).
// Two threads per row: hh = 0 writes columns [0,64) + [128,144), hh = 1 columns [64,128).
// `t_dc` already carries the thread's TMEM lane offset.
template <bool DC16>
__device__ __forceinline__ void store_dcomps_row(uint32_t t_dc, int hh, bool live, int row, void* __restrict__ dcomps_out) {
    float* dstf = reinterpret_cast<float*>(dcomps_out) + (size_t)(live ? row : 0) * CT;
    uint4* dsth = reinterpret_cast<uint4*>(reinterpret_cast<unsigned short*>(dcomps_out) + (size_t)(live ? row : 0) * CT);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        float g[32];
        const int c0 = 64 * hh + 32 * k;
        tmem_ld32(t_dc + c0, g);
        if (live) {
            if (DC16) {
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    __stcs(dsth + c0 / 8 + q, make_uint4(pack_bf16(g[8 * q], g[8 * q + 1]), pack_bf16(g[8 * q + 2], g[8 * q + 3]),
                                                         pack_bf16(g[8 * q + 4], g[8 * q + 5]), pack_bf16(g[8 * q + 6], g[8 * q + 7])));
            } else {
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    __stcs(reinterpret_cast<float4*>(dstf) + c0 / 4 + q, make_float4(g[4 * q], g[4 * q + 1], g[4 * q + 2], g[4 * q + 3]));
            }
        }
    }
    if (hh == 0) {
        float g[16];
        tmem_ld16(t_dc + 128, g);
        if (live) {
            if (DC16) {
#pragma unroll
                for (int q = 0; q < 2; ++q)
                    __stcs(dsth + 16 + q, make_uint4(pack_bf16(g[8 * q], g[8 * q + 1]), pack_bf16(g[8 * q + 2], g[8 * q + 3]),
                                                     pack_bf16(g[8 * q + 4], g[8 * q + 5]), pack_bf16(g[8 * q + 6], g[8 * q + 7])));
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    __stcs(reinterpret_cast<float4*>(dstf) + 32 + q, make_float4(g[4 * q], g[4 * q + 1], g[4 * q + 2], g[4 * q + 3]));
            }
        }
    }
}

template <typename K>
static int set_smem(K kernel, int bytes) {
    if (bytes > 48 * 1024)
        if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess) return JT_ERR_LAUNCH;
    return JT_OK;
}

}  // namespace jt
