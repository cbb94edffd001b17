// K3 (tensor-core path) for the LLFF configuration: basis_mat + positional encoding + MLPRender_Fea_WeakView,
// forward and backward, on tcgen05 tensor cores with TMEM accumulators.
//
// Replaces reference `self.basis_mat(...)` (bateRF.py:130, Linear 60 -> 20, no bias), positional_encoding
// (tensorBase.py:43-55) and MLPRender_Fea_WeakView.forward (tensorBase.py:198-214) with the shapes of
// options/bat_llff_VM_MLP.yaml (BASELINE configs[3]): 3 x 20 appearance components, app_dim 20, fea_pe = view_pe = 2,
// hidden 32:
//      in  = [feat 20 | PE(feat) 80]             -> layer1 (100 -> 32) -> relu -> layer2 (32 -> 32) -> relu
//      mid = [PE(viewdir) 12 | h2 32]            -> layer3 (44 -> 3)   -> sigmoid
// and their autograd (inputs of the head are detached from the ray, batBase.py:73-74; the gradient reaches the VM
// factors through the 60 components).
//
// One CTA = one 128-sample tile at a time, thread r = sample row r = TMEM lane r. All four GEMMs of the forward
// take hi + lo bf16 operand terms (3 MMAs per product: fp32-class results, rgb within 1e-4 of the fp32 head); the
// backward GEMMs take bf16 operands like the MLP_Fea backward (shade_tc_bwd.cu). Operand tiles use the no-swizzle
// canonical UMMA layout of tc_common.cuh. Training stages the bf16 tiles the backward needs in HBM with bulk async
// copies (TMA engine): per tile A0 comps [128x64], A1 encoded input [128x112], A2 = relu(h1) [128x48],
// A3 = [relu(h2) 32 | PE(dir) 12 | 1] [128x48]; the backward adds D2, D1 [128x32], DF [128x32], DO [128x8].
// Biases ride in the GEMMs as a 1.0 column. Tile column orders (any K permutation is a valid GEMM):
//      A1: 0..19 feat | 20 = 1 | 21..23 = 0 | 24+4e..27+4e = [sin x, sin 2x, cos x, cos 2x] of feat e | 104..111 = 0
//      A2: 0..31 relu(h1) | 32 = 1 | 0        A3: 0..31 relu(h2) | 32..43 PE(dir) | 44 = 1 | 0
// The appearance sample count of this configuration is small (0.3 - 1.2 M of 4.1 M samples at cfg4: the relu field is
// opaque within a few samples), so the kernels are written for clarity, not for the last 10 %.
#include "head_tc.cuh"
#include "../../include/jt_vm.h"

namespace jt {
namespace wv {
using namespace tc;

constexpr int C60 = 60, KB = 64;            // appearance components, padded K of the basis GEMM
constexpr int FW = 20, NBW = 32;            // app_dim, padded N of the basis GEMM
constexpr int HW = 32;                      // hidden
constexpr int INW = 100, K1W = 112;         // encoded input (reference order) / tile columns
constexpr int BIASW1 = 20;
constexpr int K2W = 48, K3W = 48;
constexpr int MIDW = 44;                    // layer-3 input: PE(dir) 12 | h2 32 (tensorBase.py:209-212)
constexpr int NT = TM;                      // threads per CTA of the backward data kernel (one per row)
constexpr int NTF = 2 * TM;                 // forward: two threads per row (hh = tid >> 7 owns the chunks of its parity)

// reference column (tensorBase.py:199-202 concatenation order) of A1 tile column c; -1 zero, -2 bias
__host__ __device__ constexpr int ref_col_w1(int c) {
    if (c < FW) return c;
    if (c == BIASW1) return -2;
    if (c < 24 || c >= 24 + 4 * FW) return -1;
    return FW + (c - 24);
}

constexpr int SZ_WA0 = tile_bytes(TM, KB), SZ_WA1 = tile_bytes(TM, K1W), SZ_WA2 = tile_bytes(TM, K2W), SZ_WA3 = tile_bytes(TM, K3W);
constexpr int SZ_WD2 = tile_bytes(TM, HW), SZ_WD1 = SZ_WD2, SZ_WDF = tile_bytes(TM, NBW), SZ_WDO = tile_bytes(TM, 8);
constexpr int OFF_WA0 = 0, OFF_WA1 = OFF_WA0 + SZ_WA0, OFF_WA2 = OFF_WA1 + SZ_WA1, OFF_WA3 = OFF_WA2 + SZ_WA2;
constexpr int OFF_WD2 = OFF_WA3 + SZ_WA3, OFF_WD1 = OFF_WD2 + SZ_WD2, OFF_WDF = OFF_WD1 + SZ_WD1, OFF_WDO = OFF_WDF + SZ_WDF;
constexpr int WV_STAGE_TILE_BYTES = OFF_WDO + SZ_WDO;      // 96256

struct FwdSmem {
    static constexpr int WB = tile_bytes(NBW, KB), W1 = tile_bytes(HW, K1W), W2 = tile_bytes(HW, K2W);
    static constexpr int off_wb = 0, off_w1 = off_wb + 2 * WB, off_w2 = off_w1 + 2 * W1;
    static constexpr int off_a0 = off_w2 + 2 * W2, off_a1 = off_a0 + 2 * SZ_WA0, off_a2 = off_a1 + 2 * SZ_WA1;
    static constexpr int off_a3 = off_a2 + 2 * SZ_WA2;
    static constexpr int off_w3 = off_a3 + SZ_WA3;            // fp32 [3][44] + b3[3]
    static constexpr int total = off_w3 + (3 * MIDW + 4) * 4;
};

// PE of one scalar with 2 frequencies (tensorBase.py:43-55): [sin x, sin 2x, cos x, cos 2x] with annealing masks
__device__ __forceinline__ void pe4(float x, float m0, float m1, float v[4]) {
    float s, c;
    fast_sincos(x, &s, &c);              // Cody-Waite reduction + SFU (abs error ~2^-21), as the MLP_Fea head does
    v[0] = s * m0; v[1] = (2.f * s * c) * m1; v[2] = c * m0; v[3] = (1.f - 2.f * s * s) * m1;
}

// comps [A][60] fp32 (jt_vm_gather_fwd app=1) -> rgb [A][4]; featdir [A][32] receives feat 0..19 and the view
// direction at 28..30 (the backward's PE derivative needs the features, the fp32 layer-3 weights the direction).
template <bool SAVE>
__global__ void __launch_bounds__(NTF) wv_head_fwd_kernel(const float* __restrict__ comps, const int* __restrict__ aidx,
                                                         const int* __restrict__ sidx, const float* __restrict__ rays_d,
                                                         int S, int normalize_dir, const float* __restrict__ Wb,
                                                         const float* __restrict__ W1, const float* __restrict__ b1,
                                                         const float* __restrict__ W2, const float* __restrict__ b2,
                                                         const float* __restrict__ W3, const float* __restrict__ b3,
                                                         const int* __restrict__ n_dev, int n_fixed, float fprog, float vprog,
                                                         float* __restrict__ featdir, float* __restrict__ rgb,
                                                         unsigned char* __restrict__ stage) {
    using L = FwdSmem;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, r = tid & (TM - 1), hh = tid >> 7;
    const int n = n_dev ? *n_dev : n_fixed;
    unsigned char* wb_hi = smem + L::off_wb;  unsigned char* wb_lo = wb_hi + L::WB;
    unsigned char* w1_hi = smem + L::off_w1;  unsigned char* w1_lo = w1_hi + L::W1;
    unsigned char* w2_hi = smem + L::off_w2;  unsigned char* w2_lo = w2_hi + L::W2;
    unsigned char* a0_hi = smem + L::off_a0;  unsigned char* a0_lo = a0_hi + SZ_WA0;
    unsigned char* a1_hi = smem + L::off_a1;  unsigned char* a1_lo = a1_hi + SZ_WA1;
    unsigned char* a2_hi = smem + L::off_a2;  unsigned char* a2_lo = a2_hi + SZ_WA2;
    unsigned char* a3 = smem + L::off_a3;
    float* w3s = reinterpret_cast<float*>(smem + L::off_w3);

    if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
    if (warp == 0) tmem_alloc(&tmem_slot, 128);
    stage_tile(wb_hi, wb_lo, NBW, KB, [&](int m, int k) { return (m < FW && k < C60) ? Wb[(size_t)m * C60 + k] : 0.f; });
    stage_tile(w1_hi, w1_lo, HW, K1W, [&](int j, int c) {
        const int rc = ref_col_w1(c);
        return rc >= 0 ? W1[(size_t)j * INW + rc] : (rc == -2 ? b1[j] : 0.f);
    });
    stage_tile(w2_hi, w2_lo, HW, K2W, [&](int j, int k) { return k < HW ? W2[(size_t)j * HW + k] : (k == HW ? b2[j] : 0.f); });
    for (int i = tid; i < 3 * MIDW + 3; i += NTF) w3s[i] = i < 3 * MIDW ? W3[i] : b3[i - 3 * MIDW];
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const uint32_t T_F = 0, T_H1 = 32, T_H2 = 64;
    uint32_t phase = 0;
    const float pf0 = fminf(fmaxf(fprog * 2.f - 0.f, 0.f), 1.f), pf1 = fminf(fmaxf(fprog * 2.f - 1.f, 0.f), 1.f);
    const float pv0 = fminf(fmaxf(vprog * 2.f - 0.f, 0.f), 1.f), pv1 = fminf(fmaxf(vprog * 2.f - 1.f, 0.f), 1.f);

    for (int tile = blockIdx.x; (long long)tile * TM < n; tile += gridDim.x) {
        const int row = tile * TM + r;
        const bool live = row < n;
        unsigned char* st = SAVE ? stage + (size_t)tile * WV_STAGE_TILE_BYTES : nullptr;
        // ---- component row -> A0 (cols 60..63 zero)
        {
            const float4* src = reinterpret_cast<const float4*>(comps + (size_t)(live ? row : 0) * C60);
#pragma unroll
            for (int c = 0; c < KB / 8; ++c) {
                if ((c & 1) != hh) continue;
                float4 x = make_float4(0.f, 0.f, 0.f, 0.f), y = x;
                if (live) {
                    x = __ldcs(src + 2 * c);
                    if (2 * c + 1 < C60 / 4) y = __ldcs(src + 2 * c + 1);
                }
                const float v[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
                store_chunk(a0_hi, a0_lo, TM, c, r, v);
            }
        }
        // view direction of the sample (viewdirs = ray_dir, normalised for NDC rays: batBase.py:63-66)
        float dir[3] = {0.f, 0.f, 0.f};
        if (live) {
            const int ray = sidx[aidx[row]] / S;
            dir[0] = rays_d[3 * ray]; dir[1] = rays_d[3 * ray + 1]; dir[2] = rays_d[3 * ray + 2];
            if (normalize_dir) {
                const float nn = sqrtf(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);
                dir[0] /= nn; dir[1] /= nn; dir[2] /= nn;
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_gemm_kmajor<2>(tmem + T_F, a0_hi, a0_lo, wb_hi, wb_lo, KB, NBW, NBW);
            mma_commit(&bar);
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- features -> global row + encoded input A1
        {
            float f[32];
            tmem_ld32(lane_addr + T_F, f);
            if (live && hh == 0) {
                float4* dst = reinterpret_cast<float4*>(featdir + (size_t)row * FD);
#pragma unroll
                for (int q = 0; q < FW / 4; ++q) __stcs(dst + q, make_float4(f[4 * q], f[4 * q + 1], f[4 * q + 2], f[4 * q + 3]));
                __stcs(dst + 7, make_float4(dir[0], dir[1], dir[2], 0.f));
            }
#pragma unroll
            for (int c = 0; c < K1W / 8; ++c) {
                if ((c & 1) != hh) continue;
                float v[8];
                if (c < 3) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int col = 8 * c + i;
                        v[i] = col < FW ? f[col] : (col == BIASW1 ? 1.f : 0.f);
                    }
                } else if (c < 3 + FW / 2) {
                    pe4(f[2 * (c - 3)], pf0, pf1, v);
                    pe4(f[2 * (c - 3) + 1], pf0, pf1, v + 4);
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = 0.f;
                }
                store_chunk(a1_hi, a1_lo, TM, c, r, v);
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_gemm_kmajor<2>(tmem + T_H1, a1_hi, a1_lo, w1_hi, w1_lo, K1W, HW, HW);
            mma_commit(&bar);
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- relu(h1) -> A2 (col 32 = 1 carries b2)
        {
            float h[32];
            tmem_ld32(lane_addr + T_H1, h);
#pragma unroll
            for (int c = 0; c < K2W / 8; ++c) {
                if ((c & 1) != hh) continue;
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int col = 8 * c + i;
                    v[i] = col < HW ? fmaxf(h[col < HW ? col : 0], 0.f) : (col == HW ? 1.f : 0.f);
                }
                store_chunk(a2_hi, a2_lo, TM, c, r, v);
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_gemm_kmajor<2>(tmem + T_H2, a2_hi, a2_lo, w2_hi, w2_lo, K2W, HW, HW);
            mma_commit(&bar);
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- relu(h2), PE(dir) -> layer 3 in fp32 registers -> sigmoid (+ the A3 tile when training)
        {
            float h[32], pd[12];
            tmem_ld32(lane_addr + T_H2, h);
#pragma unroll
            for (int e = 0; e < 3; ++e) pe4(dir[e], pv0, pv1, pd + 4 * e);
            if (hh == 0) {                            // layer 3 + sigmoid: one thread of the pair
                float o[3];
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    float s = w3s[3 * MIDW + c];
#pragma unroll
                    for (int k = 0; k < 12; ++k) s = fmaf(pd[k], w3s[c * MIDW + k], s);
#pragma unroll
                    for (int j = 0; j < HW; ++j) s = fmaf(fmaxf(h[j], 0.f), w3s[c * MIDW + 12 + j], s);
                    o[c] = 1.f / (1.f + expf(-s));
                }
                if (live) __stcs(reinterpret_cast<float4*>(rgb) + row, make_float4(o[0], o[1], o[2], 0.f));
            }
            if (SAVE && hh == 1) {                    // ... the other one writes the A3 tile
                float row3[K3W];                      // relu(h2) 32 | PE(dir) 12 | 1 | 0 0 0
#pragma unroll
                for (int j = 0; j < HW; ++j) row3[j] = fmaxf(h[j], 0.f);
#pragma unroll
                for (int k = 0; k < 12; ++k) row3[HW + k] = pd[k];
                row3[HW + 12] = 1.f; row3[HW + 13] = row3[HW + 14] = row3[HW + 15] = 0.f;
#pragma unroll
                for (int c = 0; c < K3W / 8; ++c) store_chunk(a3, nullptr, TM, c, r, row3 + 8 * c);
            }
            if (SAVE) fence_async_smem();
        }
        tc_fence_before();               // all tcgen05.ld of this tile are complete before the next tile's MMAs
        __syncthreads();
        if (SAVE && tid == 0) {          // push the bf16 (hi) tiles; the next tile re-writes them only after they drained
            bulk_s2g(st + OFF_WA0, a0_hi, SZ_WA0);
            bulk_s2g(st + OFF_WA1, a1_hi, SZ_WA1);
            bulk_s2g(st + OFF_WA2, a2_hi, SZ_WA2);
            bulk_s2g(st + OFF_WA3, a3, SZ_WA3);
            bulk_commit();
            bulk_wait_read0();
        }
        if (SAVE) __syncthreads();
    }
    if (SAVE && tid == 0) bulk_wait0();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 128);
}

// ------------------------------------------------------------------ backward, data path
struct BwdSmemW {
    static constexpr int W2T = tile_bytes(HW, HW), W1T = tile_bytes(K1W, HW), WBT = tile_bytes(KB, NBW);
    static constexpr int off_w2t = 0, off_w1t = off_w2t + W2T, off_wbt = off_w1t + W1T;
    static constexpr int off_d2 = off_wbt + WBT, off_d1 = off_d2 + SZ_WD2, off_df = off_d1 + SZ_WD1, off_do = off_df + SZ_WDF;
    static constexpr int off_w3 = off_do + SZ_WDO;               // fp32 [3][44]
    static constexpr int total = off_w3 + 3 * MIDW * 4;
};

__device__ __forceinline__ uint32_t chunk_pos_mask(const uint4 q) {     // 8 bf16 -> "is positive" bits
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        m |= ((w[i] & 0x7FFFu) != 0u ? 1u : 0u) << (2 * i);
        m |= ((w[i] & 0x7FFF0000u) != 0u ? 1u : 0u) << (2 * i + 1);
    }
    return m;
}

// dout [A][4] = dL/d(pre-sigmoid) (jt_render_bwd folds the sigmoid derivative in) -> dcomps [A][60] fp32 for the VM
// scatter; stages D2, D1, DF, DO next to the forward's tiles for the weight-gradient kernel (WST = false: a frozen
// head and basis_mat, nothing is staged and dcomps is the same bit for bit).
template <bool WST>
__global__ void __launch_bounds__(NT) wv_head_bwd_data_kernel(const float* __restrict__ dout, const float* __restrict__ featdir,
                                                              const float* __restrict__ Wb, const float* __restrict__ W1,
                                                              const float* __restrict__ W2, const float* __restrict__ W3,
                                                              const int* __restrict__ n_dev, int n_fixed, float fprog,
                                                              float* __restrict__ dcomps, unsigned char* __restrict__ stage) {
    using L = BwdSmemW;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, r = tid;
    const int n = n_dev ? *n_dev : n_fixed;
    unsigned char* w2t = smem + L::off_w2t; unsigned char* w1t = smem + L::off_w1t; unsigned char* wbt = smem + L::off_wbt;
    unsigned char* D2 = smem + L::off_d2;   unsigned char* D1 = smem + L::off_d1;
    unsigned char* DF = smem + L::off_df;   unsigned char* DO = smem + L::off_do;
    float* w3s = reinterpret_cast<float*>(smem + L::off_w3);

    if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
    if (warp == 0) tmem_alloc(&tmem_slot, 256);
    stage_tile(w2t, nullptr, HW, HW, [&](int i, int j) { return W2[(size_t)j * HW + i]; });                  // B(n = i, k = j)
    stage_tile(w1t, nullptr, K1W, HW, [&](int c, int j) { const int rc = ref_col_w1(c); return rc >= 0 ? W1[(size_t)j * INW + rc] : 0.f; });
    stage_tile(wbt, nullptr, KB, NBW, [&](int ic, int m) { return (m < FW && ic < C60) ? Wb[(size_t)m * C60 + ic] : 0.f; });
    for (int i = tid; i < 3 * MIDW; i += NT) w3s[i] = W3[i];
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
    const uint32_t T_DH1 = 0, T_DIN = 32, T_DC = 160;          // 32 + 112 + 64 columns
    uint32_t phase = 0;
    const float pf0 = fminf(fmaxf(fprog * 2.f - 0.f, 0.f), 1.f), pf1 = fminf(fmaxf(fprog * 2.f - 1.f, 0.f), 1.f);

    for (int tile = blockIdx.x; (long long)tile * TM < n; tile += gridDim.x) {
        const int row = tile * TM + r;
        const bool live = row < n;
        unsigned char* st = stage + (size_t)tile * WV_STAGE_TILE_BYTES;
        float go[3] = {0.f, 0.f, 0.f};
        if (live) {
            const float4 g4 = __ldg(reinterpret_cast<const float4*>(dout) + row);
            go[0] = g4.x; go[1] = g4.y; go[2] = g4.z;
        }
        // ---- S0: dh2 = (dout W3[:, 12:]) . [h2 > 0] -> D2 ; dout -> DO
        {
            const float v0[8] = {go[0], go[1], go[2], 0.f, 0.f, 0.f, 0.f, 0.f};
            if (WST) store_chunk(DO, nullptr, TM, 0, r, v0);
#pragma unroll
            for (int c = 0; c < HW / 8; ++c) {
                const uint4 q = __ldg(reinterpret_cast<const uint4*>(st + OFF_WA3 + (size_t)c * TM * 16 + r * 16));
                const uint32_t m = chunk_pos_mask(q);
                float g[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int j = 8 * c + i;
                    g[i] = ((m >> i) & 1u) ? go[0] * w3s[12 + j] + go[1] * w3s[MIDW + 12 + j] + go[2] * w3s[2 * MIDW + 12 + j] : 0.f;
                }
                store_chunk(D2, nullptr, TM, c, r, g);
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_gemm_kmajor<1>(tmem + T_DH1, D2, nullptr, w2t, nullptr, HW, HW, HW);
            mma_commit(&bar);
            if (WST) {
                bulk_s2g(st + OFF_WD2, D2, SZ_WD2);
                bulk_s2g(st + OFF_WDO, DO, SZ_WDO);
                bulk_commit();
            }
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- S1: dh1 = dh1_pre . [h1 > 0] -> D1
        {
            float g[32];
            tmem_ld32(lane_addr + T_DH1, g);
#pragma unroll
            for (int c = 0; c < HW / 8; ++c) {
                const uint4 q = __ldg(reinterpret_cast<const uint4*>(st + OFF_WA2 + (size_t)c * TM * 16 + r * 16));
                const uint32_t m = chunk_pos_mask(q);
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = ((m >> i) & 1u) ? g[8 * c + i] : 0.f;
                store_chunk(D1, nullptr, TM, c, r, v);
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_gemm_kmajor<1>(tmem + T_DIN, D1, nullptr, w1t, nullptr, HW, K1W, K1W);
            mma_commit(&bar);
            if (WST) {
                bulk_s2g(st + OFF_WD1, D1, SZ_WD1);
                bulk_commit();
            }
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- S2: din -> dfeat (chain rule through the encoding) -> DF
        {
            float df[32], raw[32];
            tmem_ld32(lane_addr + T_DIN, raw);                      // cols 0..31: feat 0..19 | bias | 0 | PE of feat 0, 1
#pragma unroll
            for (int e = 0; e < 32; ++e) df[e] = e < FW ? raw[e] : 0.f;
            const float4* fp = reinterpret_cast<const float4*>(featdir + (size_t)(live ? row : 0) * FD);
            float feat[FW];
#pragma unroll
            for (int q = 0; q < FW / 4; ++q) {
                const float4 f4 = live ? __ldg(fp + q) : make_float4(0.f, 0.f, 0.f, 0.f);
                feat[4 * q] = f4.x; feat[4 * q + 1] = f4.y; feat[4 * q + 2] = f4.z; feat[4 * q + 3] = f4.w;
            }
            auto chain = [&](int e, const float* g) {               // g = d/d[sin x, sin 2x, cos x, cos 2x]
                float sn, co;
                fast_sincos(feat[e], &sn, &co);
                const float s2 = 2.f * sn * co, c2 = 1.f - 2.f * sn * sn;
                df[e] += pf0 * (co * g[0] - sn * g[2]) + 2.f * pf1 * (c2 * g[1] - s2 * g[3]);
            };
            chain(0, raw + 24);
            chain(1, raw + 28);
            // PE columns 32..111 hold features 2..19 (4 columns each): 80 columns = 32 + 32 + 16
            {
                float g[32];
                tmem_ld32(lane_addr + T_DIN + 32, g);
#pragma unroll
                for (int q = 0; q < 8; ++q) chain(2 + q, g + 4 * q);
                tmem_ld32(lane_addr + T_DIN + 64, g);
#pragma unroll
                for (int q = 0; q < 8; ++q) chain(10 + q, g + 4 * q);
                float g2[16];
                tmem_ld16(lane_addr + T_DIN + 96, g2);
#pragma unroll
                for (int q = 0; q < 2; ++q) chain(18 + q, g2 + 4 * q);
            }
#pragma unroll
            for (int c = 0; c < NBW / 8; ++c) store_chunk(DF, nullptr, TM, c, r, df + 8 * c);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_gemm_kmajor<1>(tmem + T_DC, DF, nullptr, wbt, nullptr, NBW, KB, KB);
            mma_commit(&bar);
            if (WST) {
                bulk_s2g(st + OFF_WDF, DF, SZ_WDF);
                bulk_commit();
            }
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- S3: dcomps row -> global fp32 [A][60]
        {
            float4* dst = reinterpret_cast<float4*>(dcomps + (size_t)(live ? row : 0) * C60);
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                float g[32];
                tmem_ld32(lane_addr + T_DC + 32 * k, g);
                if (live) {
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        if (8 * k + q < C60 / 4) __stcs(dst + 8 * k + q, make_float4(g[4 * q], g[4 * q + 1], g[4 * q + 2], g[4 * q + 3]));
                }
            }
        }
        if (WST && tid == 0) bulk_wait_read0();       // D2 / D1 / DF / DO have left shared memory
        tc_fence_before();
        __syncthreads();
    }
    if (WST && tid == 0) bulk_wait0();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

// ------------------------------------------------------------------ backward, weight gradients
// TMA -> tcgen05 pipeline over the staged tiles (same scheme as head_bwd_wgrad_kernel in shade_tc_bwd.cu): weight
// gradients are K = samples GEMMs, dW[m][n] = sum_s D[s][m] A[s][n], both operands read MN-major from the staged
// tiles, accumulated in TMEM across all tiles of the CTA and reduced into global memory once.
constexpr int WGW_STAGES = 3;
constexpr int WGW_A_REGION = 32768;            // the M = 128 A descriptor spans 16 groups x 2048 B
constexpr int WGW_STAGE_BYTES = WGW_A_REGION + SZ_WA1;
struct WGroupW { int a_off, a_bytes, b_off, b_bytes, n, col; };
__device__ __forceinline__ WGroupW wgroup_w(int g) {
    switch (g) {
        case 0: return {OFF_WD1, SZ_WD1, OFF_WA1, SZ_WA1, K1W, 0};       // dW1 (+ db1 in column 20)
        case 1: return {OFF_WD2, SZ_WD2, OFF_WA2, SZ_WA2, K2W, 112};     // dW2 (+ db2 in column 32)
        case 2: return {OFF_WDO, SZ_WDO, OFF_WA3, SZ_WA3, K3W, 160};     // dW3 (+ db3 in column 44)
        default: return {OFF_WDF, SZ_WDF, OFF_WA0, SZ_WA0, KB, 208};     // d basis_mat
    }
}

__global__ void __launch_bounds__(TM) wv_head_bwd_wgrad_kernel(const unsigned char* __restrict__ stage, const int* __restrict__ n_dev,
                                                               int n_fixed, float* __restrict__ gWb, float* __restrict__ gW1,
                                                               float* __restrict__ gb1, float* __restrict__ gW2,
                                                               float* __restrict__ gb2, float* __restrict__ gW3,
                                                               float* __restrict__ gb3) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t full[WGW_STAGES], empty[WGW_STAGES], done;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n = n_dev ? *n_dev : n_fixed;
    const int ntiles = (int)(((long long)n + TM - 1) / TM);
    const int my_tiles = blockIdx.x < ntiles ? (ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
    constexpr int NG = 4;

    if (tid == 0) {
        for (int s = 0; s < WGW_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(&done, 1);
        mbar_fence_init();
    }
    // the A region beyond the small gradient tiles is read by the M = 128 descriptor: keep it finite (zero)
    for (int i = tid; i < WGW_STAGES * WGW_STAGE_BYTES / 16; i += TM) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    fence_async_smem();
    if (warp == 0) tmem_alloc(&tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const int items = my_tiles * NG;

    if (warp == 0 && lane == 0) {                 // ---- TMA producer
        for (int i = 0; i < items; ++i) {
            const int s = i % WGW_STAGES, round = i / WGW_STAGES;
            mbar_wait(&empty[s], (round & 1) ^ 1);
            const int tile = blockIdx.x + (i / NG) * gridDim.x;
            const WGroupW g = wgroup_w(i % NG);
            const unsigned char* src = stage + (size_t)tile * WV_STAGE_TILE_BYTES;
            unsigned char* dst = smem + s * WGW_STAGE_BYTES;
            mbar_expect_tx(&full[s], (uint32_t)(g.a_bytes + g.b_bytes));
            bulk_g2s(dst, src + g.a_off, g.a_bytes, &full[s]);
            bulk_g2s(dst + WGW_A_REGION, src + g.b_off, g.b_bytes, &full[s]);
        }
    } else if (warp == 1 && lane == 0) {          // ---- MMA issuer
        for (int i = 0; i < items; ++i) {
            const int s = i % WGW_STAGES, round = i / WGW_STAGES;
            mbar_wait(&full[s], round & 1);
            tc_fence_after();
            const WGroupW g = wgroup_w(i % NG);
            const uint32_t a = smem_u32(smem + s * WGW_STAGE_BYTES), b = a + WGW_A_REGION;
            const uint32_t idesc = idesc_bf16(128, g.n, 1, 1);
#pragma unroll
            for (int ks = 0; ks < TM / 16; ++ks)       // K = 128 sample rows, 16 per MMA = 256 B
                mma_bf16(tmem + g.col, smem_desc(a + ks * 256, 128, TM * 16), smem_desc(b + ks * 256, 128, TM * 16), idesc,
                         (i >= NG || ks > 0) ? 1u : 0u);
            mma_commit(&empty[s]);
        }
        mma_commit(&done);
    }
    __syncwarp();
    if (items > 0) {
        mbar_wait(&done, 0);
        tc_fence_after();
        if (warp == 0) {                               // real rows are all < 32
            const uint32_t lane_addr = tmem;
            const int m = tid;
            for (int c0 = 0; c0 < K1W; c0 += 16) {     // dW1 / db1
                float v[16];
                tmem_ld16(lane_addr + 0 + c0, v);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int rc = ref_col_w1(c0 + i);
                    if (rc >= 0) atomicAdd(gW1 + (size_t)m * INW + rc, v[i]);
                    else if (rc == -2) atomicAdd(gb1 + m, v[i]);
                }
            }
            for (int c0 = 0; c0 < K2W; c0 += 16) {     // dW2 / db2, dW3 / db3
                float v[16], w[16];
                tmem_ld16(lane_addr + 112 + c0, v);
                tmem_ld16(lane_addr + 160 + c0, w);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int c = c0 + i;
                    if (c < HW) { atomicAdd(gW2 + (size_t)m * HW + c, v[i]); if (m < 3) atomicAdd(gW3 + (size_t)m * MIDW + 12 + c, w[i]); }
                    else if (c == HW) { atomicAdd(gb2 + m, v[i]); if (m < 3) atomicAdd(gW3 + (size_t)m * MIDW + 0, w[i]); }
                    else if (c < HW + 12) { if (m < 3) atomicAdd(gW3 + (size_t)m * MIDW + (c - HW), w[i]); }
                    else if (c == HW + 12) { if (m < 3) atomicAdd(gb3 + m, w[i]); }
                }
            }
            for (int c0 = 0; c0 < KB; c0 += 16) {      // d basis_mat
                float v[16];
                tmem_ld16(lane_addr + 208 + c0, v);
                if (m < FW) {
#pragma unroll
                    for (int i = 0; i < 16; ++i)
                        if (c0 + i < C60) atomicAdd(gWb + (size_t)m * C60 + c0 + i, v[i]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

}  // namespace wv
}  // namespace jt

using namespace jt;
using namespace jt::wv;

extern "C" long long jt_wv_stage_bytes(int n_max) {
    return (((long long)n_max + TM - 1) / TM) * WV_STAGE_TILE_BYTES;
}

extern "C" int jt_wv_head_fwd_tc(const float* comps, const int* aidx, const int* sidx, const float* rays_d, int n_samples,
                                 int normalize_dir, const float* Wb, const float* W1, const float* b1, const float* W2,
                                 const float* b2, const float* W3, const float* b3, const int* n_dev, int n_max,
                                 float fea_progress, float view_progress, float* featdir, float* rgb, void* stage,
                                 cudaStream_t stream) {
    JT_CHECK_ARG(comps && aidx && sidx && rays_d && Wb && W1 && b1 && W2 && b2 && W3 && b3 && featdir && rgb && n_samples > 0);
    JT_CHECK_ARG((reinterpret_cast<uintptr_t>(stage) & 127) == 0 && (reinterpret_cast<uintptr_t>(comps) & 15) == 0);
    if (n_max <= 0) return JT_OK;
    long long tiles = ((long long)n_max + TM - 1) / TM;
    int grid = (int)(tiles < kNumSMs ? tiles : kNumSMs);
    g_launches += 1;
    unsigned char* st = static_cast<unsigned char*>(stage);
    if (st) {
        if (int rc = set_smem(wv_head_fwd_kernel<true>, FwdSmem::total)) return rc;
        wv_head_fwd_kernel<true><<<grid, NTF, FwdSmem::total, stream>>>(comps, aidx, sidx, rays_d, n_samples, normalize_dir, Wb, W1, b1,
                                                                      W2, b2, W3, b3, n_dev, n_max, fea_progress, view_progress,
                                                                      featdir, rgb, st);
    } else {
        if (int rc = set_smem(wv_head_fwd_kernel<false>, FwdSmem::total)) return rc;
        wv_head_fwd_kernel<false><<<grid, NTF, FwdSmem::total, stream>>>(comps, aidx, sidx, rays_d, n_samples, normalize_dir, Wb, W1, b1,
                                                                       W2, b2, W3, b3, n_dev, n_max, fea_progress, view_progress,
                                                                       featdir, rgb, nullptr);
    }
    JT_RETURN_LAUNCH();
}

extern "C" int jt_wv_head_bwd_tc(const float* dout, const float* featdir, const float* Wb, const float* W1, const float* W2,
                                 const float* W3, const int* n_dev, int n_max, float fea_progress, float* dcomps, void* stage,
                                 float* gWb, float* gW1, float* gb1, float* gW2, float* gb2, float* gW3, float* gb3,
                                 cudaStream_t stream) {
    JT_CHECK_ARG(dout && featdir && Wb && W1 && W2 && W3 && dcomps && stage);
    const int n_wg = !!gWb + !!gW1 + !!gb1 + !!gW2 + !!gb2 + !!gW3 + !!gb3;
    JT_CHECK_ARG(n_wg == 0 || n_wg == 7);                // all weight gradients, or none (frozen head + basis_mat)
    JT_CHECK_ARG((reinterpret_cast<uintptr_t>(stage) & 127) == 0 && (reinterpret_cast<uintptr_t>(dcomps) & 15) == 0);
    if (n_max <= 0) return JT_OK;
    long long tiles = ((long long)n_max + TM - 1) / TM;
    int grid_d = (int)(tiles < 2 * kNumSMs ? tiles : 2 * kNumSMs);
    int grid_w = (int)(tiles < kNumSMs ? tiles : kNumSMs);
    // each CTA of the data kernel owns 256 of the SM's 512 TMEM columns: ask for enough shared memory that no third
    // CTA becomes resident and waits inside tcgen05.alloc
    const int smem_d = BwdSmemW::total > 100 * 1024 ? BwdSmemW::total : 100 * 1024;
    unsigned char* st = static_cast<unsigned char*>(stage);
    g_launches += 1;
    if (n_wg == 0) {
        if (int rc = set_smem(wv_head_bwd_data_kernel<false>, smem_d)) return rc;
        wv_head_bwd_data_kernel<false><<<grid_d, NT, smem_d, stream>>>(dout, featdir, Wb, W1, W2, W3, n_dev, n_max,
                                                                       fea_progress, dcomps, st);
        JT_RETURN_LAUNCH();
    }
    if (int rc = set_smem(wv_head_bwd_data_kernel<true>, smem_d)) return rc;
    if (int rc = set_smem(wv_head_bwd_wgrad_kernel, WGW_STAGES * WGW_STAGE_BYTES)) return rc;
    g_launches += 1;
    wv_head_bwd_data_kernel<true><<<grid_d, NT, smem_d, stream>>>(dout, featdir, Wb, W1, W2, W3, n_dev, n_max, fea_progress,
                                                                  dcomps, st);
    wv_head_bwd_wgrad_kernel<<<grid_w, TM, WGW_STAGES * WGW_STAGE_BYTES, stream>>>(st, n_dev, n_max, gWb, gW1, gb1, gW2, gb2, gW3, gb3);
    JT_RETURN_LAUNCH();
}
