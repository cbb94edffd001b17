// K3 (tensor-core path), backward of basis_mat + positional encoding + MLP_Fea.
//
// Replaces the autograd of reference basis_mat (tensoRF.py:270), positional_encoding
// (tensorBase.py:43-55) and MLPRender_Fea.forward (tensorBase.py:116-126).
//
// Two kernels, both on tcgen05 tensor cores with TMEM accumulators:
//
//  head_bwd_data_kernel  (two CTAs per SM, thread t = sample row t = TMEM lane t)
//     reads the relu masks from the bf16 tiles A2 = relu(h1), A3 = relu(h2) the training
//     forward saved (so the masks are exactly the forward's) and runs the
//     input-gradient chain
//        dh2 = (dout W3) . [h2>0]         (registers)
//        dh1 = (dh2 W2) . [h1>0]          MMA4   [128x64]  = D2[128x64]  * W2
//        din = dh1 W1                     MMA5   [128x160] = D1[128x64]  * W1
//        dfeat = PE'(din)                 (registers)
//        dcomps = dfeat Wb                MMA6   [128x144] = DF[128x32]  * Wb
//     and writes dcomps (fp32) for the VM scatter kernel. The bf16 operand tiles it
//     builds on the way (D2, D1, DF, DO = dout) are pushed next to the forward's tiles
//     (A0 comps, A1 encoded input, A2, A3) in the HBM staging area with bulk async
//     stores (TMA engine), already in the UMMA canonical layout. Only the wgrad kernel
//     reads them: without weight gradients (WST = false, a frozen head) they stay in
//     shared memory, and dcomps comes out of the same arithmetic bit for bit.
//
//  head_bwd_wgrad_kernel (persistent, one CTA per SM)
//     a TMA -> tcgen05 pipeline over those staged tiles: weight gradients are
//     K = samples GEMMs, dW[m][n] = sum_s A[s][m] B[s][n], i.e. both operands are read
//     MN-major from the same tiles (no transposes), accumulated in TMEM across all
//     tiles of the CTA (464 of the 512 columns), and reduced into global memory once.
//     Bias gradients fall out of the 1.0 columns the forward operands carry.
#include "head_tc.cuh"
#include "../../include/jt_vm.h"

namespace jt {
using namespace tc;

struct BwdSmem {
    static constexpr int W2T = tile_bytes(H_, H_), W1T = tile_bytes(K1, H_), WBT = tile_bytes(CT, NB);
    static constexpr int off_w2t = 0, off_w1t = off_w2t + W2T, off_wbt = off_w1t + W1T;
    static constexpr int off_d2 = off_wbt + WBT, off_d1 = off_d2 + SZ_D2, off_df = off_d1 + SZ_D1, off_do = off_df + SZ_DF;
    static constexpr int off_w3 = off_do + SZ_DO;               // fp32 [3][64]
    static constexpr int total = off_w3 + 3 * H_ * 4;
};

// 8 bf16 of one 16-byte chunk -> "is positive" bits (relu'd activations are >= 0)
__device__ __forceinline__ uint32_t chunk_mask(const uint4 q) {
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        m |= ((w[i] & 0x7FFFu) != 0u ? 1u : 0u) << (2 * i);
        m |= ((w[i] & 0x7FFF0000u) != 0u ? 1u : 0u) << (2 * i + 1);
    }
    return m;
}

constexpr int NTB = 2 * TM;     // two threads per sample row (column halves), as in the forward kernel

template <bool DC16, bool WST>
__global__ void __launch_bounds__(NTB, 2) head_bwd_data_kernel(
    const float* __restrict__ dout, const float* __restrict__ feat_in, int ldf, const float* __restrict__ Wb,
    const float* __restrict__ W1, const float* __restrict__ W2, const float* __restrict__ W3,
    const int* __restrict__ n_dev, int n_fixed, float fprog, void* __restrict__ dcomps_out,
    unsigned char* __restrict__ stage) {
    using L = BwdSmem;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int r = tid & (TM - 1), hh = tid >> 7;
    const int n = n_dev ? *n_dev : n_fixed;

    unsigned char* w2t = smem + L::off_w2t; unsigned char* w1t = smem + L::off_w1t; unsigned char* wbt = smem + L::off_wbt;
    unsigned char* D2 = smem + L::off_d2;   unsigned char* D1 = smem + L::off_d1;
    unsigned char* DF = smem + L::off_df;   unsigned char* DO = smem + L::off_do;
    float* w3s = reinterpret_cast<float*>(smem + L::off_w3);

    if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
    if (warp == 0) tmem_alloc(&tmem_slot, 256);
    stage_tile(w2t, nullptr, H_, H_, [&](int i, int j) { return W2[(size_t)j * H_ + i]; });             // B(n=i,k=j)
    stage_tile(w1t, nullptr, K1, H_, [&](int c, int j) { const int rc = ref_col_l1(c); return rc >= 0 ? W1[(size_t)j * IN_ + rc] : 0.f; });
    stage_tile(wbt, nullptr, CT, NB, [&](int ic, int m) { return m < F_ ? Wb[(size_t)m * CT + ic] : 0.f; });
    for (int i = tid; i < 3 * H_; i += NTB) w3s[i] = W3[i];
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const uint32_t T_DH1 = 0, T_DIN = 64, T_DC = 0;
    uint32_t phase = 0;
    const float pf0 = fminf(fmaxf(fprog * 2.f - 0.f, 0.f), 1.f), pf1 = fminf(fmaxf(fprog * 2.f - 1.f, 0.f), 1.f);

    // the global reads of the NEXT tile (relu-mask chunks of A3 / A2, the feature row, dout) are
    // issued while the current tile computes
    float go[3];
    uint4 q3[4], q2[4];
    float feat[16];
    auto prefetch = [&](long long t) {
        const long long rw = t * TM + r;
        const bool lv = rw < n;
        const bool tv = t * TM < n;
        const unsigned char* stn = stage + (size_t)(tv ? t : 0) * STAGE_TILE_BYTES;
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
            const size_t o = (size_t)(hh * 4 + c4) * TM * 16 + r * 16;
            q3[c4] = tv ? __ldg(reinterpret_cast<const uint4*>(stn + OFF_A3 + o)) : make_uint4(0, 0, 0, 0);
            q2[c4] = tv ? __ldg(reinterpret_cast<const uint4*>(stn + OFF_A2 + o)) : make_uint4(0, 0, 0, 0);
        }
        const float4* fp = reinterpret_cast<const float4*>(feat_in + (size_t)(lv ? rw : 0) * ldf) + 4 * hh;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float4 f4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (lv && (hh == 0 || q < 3)) f4 = __ldg(fp + q);
            feat[4 * q] = f4.x; feat[4 * q + 1] = f4.y; feat[4 * q + 2] = f4.z; feat[4 * q + 3] = f4.w;
        }
        go[0] = go[1] = go[2] = 0.f;
        if (lv) {
            const float4 g4 = __ldg(reinterpret_cast<const float4*>(dout) + rw);
            go[0] = g4.x; go[1] = g4.y; go[2] = g4.z;
        }
    };
    prefetch(blockIdx.x);

    for (int tile = blockIdx.x; (long long)tile * TM < n; tile += gridDim.x) {
        const int row = tile * TM + r;
        const bool live = row < n;
        unsigned char* st = stage + (size_t)tile * STAGE_TILE_BYTES;
        // ---- S0: dh2 = (dout W3) . [h2 > 0] -> D2 (this thread: columns [32 hh, 32 hh + 32)) ; dout -> DO
        if (WST && hh == 0) {
            const float v[8] = {go[0], go[1], go[2], 0.f, 0.f, 0.f, 0.f, 0.f};
            store_chunk(DO, nullptr, TM, 0, r, v);
        }
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
            const int c = hh * 4 + c4;
            const uint32_t m = chunk_mask(q3[c4]);
            float g[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int j = c * 8 + i;
                g[i] = ((m >> i) & 1u) ? go[0] * w3s[j] + go[1] * w3s[H_ + j] + go[2] * w3s[2 * H_ + j] : 0.f;
            }
            store_chunk(D2, nullptr, TM, c, r, g);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_gemm_kmajor<1>(tmem + T_DH1, D2, nullptr, w2t, nullptr, H_, H_, H_);
            mma_commit(&bar);
            if (WST) {
                bulk_s2g(st + OFF_D2, D2, SZ_D2);
                bulk_s2g(st + OFF_DO, DO, SZ_DO);
                bulk_commit();
            }
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- S1: dh1 = dh1_pre . [h1 > 0] -> D1
        {
            float g[32];
            tmem_ld32(lane_addr + T_DH1 + 32 * hh, g);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int cc = hh * 4 + c;
                const uint32_t m = chunk_mask(q2[c]);
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = ((m >> i) & 1u) ? g[c * 8 + i] : 0.f;
                store_chunk(D1, nullptr, TM, cc, r, v);
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_gemm_kmajor<1>(tmem + T_DIN, D1, nullptr, w1t, nullptr, H_, K1, K1);
            mma_commit(&bar);
            if (WST) {
                bulk_s2g(st + OFF_D1, D1, SZ_D1);
                bulk_commit();
            }
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- S2: din -> dfeat (chain rule through the encoding) -> DF; this thread: elements [16 hh, 16 hh + 16)
        {
            float df[16], raw[32];
            tmem_ld32(lane_addr + T_DIN, raw);
#pragma unroll
            for (int e = 0; e < 16; ++e) df[e] = (16 * hh + e < F_) ? (hh == 0 ? raw[e] : raw[16 + e]) : 0.f;
#pragma unroll
            for (int k = 0; k < 2; ++k) {                      // 8 source elements per 32 columns
                float g[32];
                tmem_ld32(lane_addr + T_DIN + 32 + 64 * hh + 32 * k, g);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int el = 8 * k + q;
                    if (16 * hh + el < F_) {
                        float sn, co;
                        fast_sincos(feat[el], &sn, &co);
                        const float s2 = 2.f * sn * co, c2 = 1.f - 2.f * sn * sn;
                        df[el] += pf0 * (co * g[4 * q] - sn * g[4 * q + 2]) + 2.f * pf1 * (c2 * g[4 * q + 1] - s2 * g[4 * q + 3]);
                    }
                }
            }
            store_chunk(DF, nullptr, TM, 2 * hh, r, df);
            store_chunk(DF, nullptr, TM, 2 * hh + 1, r, df + 8);
        }
        prefetch((long long)tile + gridDim.x);   // q3 / q2 / feat / go of this tile are dead from here on
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_gemm_kmajor<1>(tmem + T_DC, DF, nullptr, wbt, nullptr, NB, CT, CT);
            mma_commit(&bar);
            if (WST) {
                bulk_s2g(st + OFF_DF, DF, SZ_DF);
                bulk_commit();
            }
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- S3: dcomps row -> global (fp32, or bf16 when DC16)
        store_dcomps_row<DC16>(lane_addr + T_DC, hh, live, row, dcomps_out);
        if (WST && tid == 0) bulk_wait_read0();       // D2 / D1 / DF / DO have left shared memory
        tc_fence_before();
        __syncthreads();
    }
    if (WST && tid == 0) bulk_wait0();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

// ------------------------------------------------------------------ weight gradients
constexpr int WG_STAGES = 3;
constexpr int WG_A_REGION = 32768;            // the M=128 A descriptor spans 16 groups x 2048 B
constexpr int WG_STAGE_BYTES = WG_A_REGION + SZ_A1;
// basis_mat alone (SH shading): stages of [A region | component tile]
constexpr int WG_SH_STAGES = 3;
constexpr int WG_SH_STAGE_BYTES = WG_A_REGION + SZ_A0;

struct WGroup { int a_off, a_bytes, b_off, b_bytes, n, col; };
__device__ __forceinline__ WGroup wgroup(int g) {
    switch (g) {
        case 0: return {OFF_D1, SZ_D1, OFF_A1, SZ_A1, K1, 0};        // dW1 (+db1 in the bias column)
        case 1: return {OFF_D2, SZ_D2, OFF_A2, SZ_A2, K2, 160};      // dW2 (+db2 in column 64)
        case 2: return {OFF_DO, SZ_DO, OFF_A3, SZ_A3, K2, 240};      // dW3 (+db3 in column 64)
        default: return {OFF_DF, SZ_DF, OFF_A0, SZ_A0, CT, 320};     // d basis_mat
    }
}

// Groups [G0, G0 + NG) of wgroup() are accumulated: <0, 4> is the MLP_Fea head + basis_mat,
// <3, 1> basis_mat alone (SH shading: jt_sh_bwd_tc).
template <int G0, int NG, int STAGES, int STAGE_BYTES>
__global__ void __launch_bounds__(TM) head_bwd_wgrad_kernel(const unsigned char* __restrict__ stage,
                                                            const int* __restrict__ n_dev, int n_fixed,
                                                            float* __restrict__ gWb, float* __restrict__ gW1,
                                                            float* __restrict__ gb1, float* __restrict__ gW2,
                                                            float* __restrict__ gb2, float* __restrict__ gW3,
                                                            float* __restrict__ gb3) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t full[STAGES], empty[STAGES], done;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n = n_dev ? *n_dev : n_fixed;
    const int ntiles = (int)(((long long)n + TM - 1) / TM);
    const int my_tiles = blockIdx.x < ntiles ? (ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(&done, 1);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const int items = my_tiles * NG;

    if (warp == 0 && lane == 0) {                 // ---- TMA producer
        for (int i = 0; i < items; ++i) {
            const int s = i % STAGES, round = i / STAGES;
            mbar_wait(&empty[s], (round & 1) ^ 1);
            const int tile = blockIdx.x + (i / NG) * gridDim.x;
            const WGroup g = wgroup(G0 + i % NG);
            const unsigned char* src = stage + (size_t)tile * STAGE_TILE_BYTES;
            unsigned char* dst = smem + s * STAGE_BYTES;
            mbar_expect_tx(&full[s], (uint32_t)(g.a_bytes + g.b_bytes));
            bulk_g2s(dst, src + g.a_off, g.a_bytes, &full[s]);
            bulk_g2s(dst + WG_A_REGION, src + g.b_off, g.b_bytes, &full[s]);
        }
    } else if (warp == 1 && lane == 0) {          // ---- MMA issuer
        for (int i = 0; i < items; ++i) {
            const int s = i % STAGES, round = i / STAGES;
            mbar_wait(&full[s], round & 1);
            tc_fence_after();
            const WGroup g = wgroup(G0 + i % NG);
            const uint32_t a = smem_u32(smem + s * STAGE_BYTES), b = a + WG_A_REGION;
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
        if (warp < 2) {                               // real rows are all < 64
            const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
            const int m = tid;
            for (int c0 = 0; G0 == 0 && c0 < K1; c0 += 32) {     // dW1 / db1
                float v[32];
                tmem_ld32(lane_addr + 0 + c0, v);
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int r = ref_col_l1(c0 + i);
                    if (r >= 0) atomicAdd(gW1 + (size_t)m * IN_ + r, v[i]);
                    else if (r == -2) atomicAdd(gb1 + m, v[i]);
                }
            }
            for (int c0 = 0; G0 == 0 && c0 < K2; c0 += 16) {     // dW2 / db2, dW3 / db3
                float v[16], w[16];
                tmem_ld16(lane_addr + 160 + c0, v);
                tmem_ld16(lane_addr + 240 + c0, w);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int c = c0 + i;
                    if (c < H_) { atomicAdd(gW2 + (size_t)m * H_ + c, v[i]); if (m < 3) atomicAdd(gW3 + (size_t)m * H_ + c, w[i]); }
                    else if (c == H_) { atomicAdd(gb2 + m, v[i]); if (m < 3) atomicAdd(gb3 + m, w[i]); }
                }
            }
            for (int c0 = 0; c0 < CT; c0 += 16) {     // d basis_mat
                float v[16];
                tmem_ld16(lane_addr + 320 + c0, v);
                if (m < F_) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) atomicAdd(gWb + (size_t)m * CT + c0 + i, v[i]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------ SH shading (SHRender, tensorBase.py:68-72)
// Backward of basis_mat + SHRender on the tensor cores. rgb = relu(sum_k Y_k(dir) feat[c*9+k] + 0.5),
// so dfeat[c*9+k] = dpre[c] * Y_k(dir) needs only the view direction (kept by the forward in the
// feat/dir rows) and dpre = dL/d(pre-activation) (jt_render_bwd folds relu' into it):
//     DF[128x32] (bf16) = dpre (x) Y     ->  MMA  dcomps[128x144] = DF * Wb   (TMEM)  -> bf16 rows
// DF is pushed to the staging area next to the forward's component tile A0, and the
// basis_mat weight gradient is group 3 of the shared TMA -> tcgen05 wgrad pipeline.
// WST = false (frozen basis_mat): no staging area, DF stays in shared memory.
struct ShBwdSmem {
    static constexpr int WBT = tile_bytes(CT, NB);
    static constexpr int OUT = TM * CT * 2;                     // dcomps tile, bf16 row-major = its global image
    static constexpr int off_wbt = 0, off_df = off_wbt + WBT, off_out = off_df + 2 * SZ_DF;
    // 91 KB: two CTAs per SM (each allocates 256 of the SM's 512 TMEM columns)
    static constexpr int total = off_out + 2 * OUT;
};

// dcomps leaves the SM as ONE bulk async store per tile: the 128 rows x 288 B of a tile are contiguous in
// global memory, the threads only write their TMEM columns into a shared-memory image of it (per-thread
// 16-byte global stores at a 288-byte row pitch kept the LSU queues full: lg_throttle, 0.33 ms). DF and
// the output tile are double-buffered; the issuing thread waits for the bulk stores of two tiles ago
// *before* it signals the MMA barrier, so passing that barrier also means both buffers are free.
template <bool WST>
__global__ void __launch_bounds__(NTB, 2) sh_bwd_data_kernel(const float* __restrict__ dout, const float* __restrict__ featdir,
                                                             int ldf, const float* __restrict__ Wb,
                                                             const int* __restrict__ n_dev, int n_fixed,
                                                             unsigned short* __restrict__ dcomps_out,
                                                             unsigned char* __restrict__ stage) {
    using L = ShBwdSmem;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int r = tid & (TM - 1), hh = tid >> 7;
    const int n = n_dev ? *n_dev : n_fixed;
    unsigned char* wbt = smem + L::off_wbt;

    if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
    if (warp == 0) tmem_alloc(&tmem_slot, 256);
    stage_tile(wbt, nullptr, CT, NB, [&](int ic, int m) { return m < F_ ? Wb[(size_t)m * CT + ic] : 0.f; });
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    uint32_t phase = 0;
    int buf = 0;

    float4 g4, d4;                     // dpre and view direction of the NEXT tile's row (prefetched)
    auto prefetch = [&](long long t) {
        const long long rw = t * TM + r;
        g4 = d4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rw < n) {
            g4 = __ldcs(reinterpret_cast<const float4*>(dout) + rw);
            d4 = __ldcs(reinterpret_cast<const float4*>(featdir + (size_t)rw * ldf + 28));
        }
    };
    prefetch(blockIdx.x);

    for (int tile = blockIdx.x; (long long)tile * TM < n; tile += gridDim.x, buf ^= 1) {
        const int rows = min(TM, n - tile * TM);
        unsigned char* DF = smem + L::off_df + buf * SZ_DF;
        unsigned char* OUT = smem + L::off_out + buf * L::OUT;
        // ---- DF row: columns c*9+k = dpre[c] * Y_k, 27..31 = 0; this thread: columns [16 hh, 16 hh + 16)
        {
            const float d[3] = {d4.x, d4.y, d4.z};
            const float go[3] = {g4.x, g4.y, g4.z};
            float y[9], df[16];
            sh9(d, y);
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                const int col = 16 * hh + e;             // hh is warp-uniform: both candidates are compile-time
                const int c0 = e / 9, k0 = e % 9, c1 = (16 + e) / 9, k1 = (16 + e) % 9;
                const float v0 = go[c0] * y[k0];
                const float v1 = (16 + e) < F_ ? go[c1 < 3 ? c1 : 0] * y[k1] : 0.f;
                df[e] = col < F_ ? (hh == 0 ? v0 : v1) : 0.f;
            }
            store_chunk(DF, nullptr, TM, 2 * hh, r, df);
            store_chunk(DF, nullptr, TM, 2 * hh + 1, r, df + 8);
        }
        prefetch((long long)tile + gridDim.x);
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_gemm_kmajor<1>(tmem, DF, nullptr, wbt, nullptr, NB, CT, CT);
            if (WST) {
                bulk_s2g(stage + (size_t)tile * STAGE_TILE_BYTES + OFF_DF, DF, SZ_DF);
                bulk_commit();
                // pending afterwards: at most OUT(t-1) and DF(t) -> DF(t-1) and OUT(t-2), the previous users of the
                // buffers this tile's successor / this tile's epilogue write, have been read out of shared memory
                bulk_wait_read2();
            } else {
                bulk_wait_read1();             // only OUT(t-1) may still be pending: OUT(t-2) has been read
            }
            mma_commit(&bar);
        }
        mbar_wait(&bar, phase); phase ^= 1;
        tc_fence_after();
        // ---- dcomps row -> bf16 -> shared-memory image of the tile; hh = 0: columns [0,64) + [128,144), hh = 1: [64,128)
        {
            uint4* orow = reinterpret_cast<uint4*>(OUT + (size_t)r * (CT * 2));
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                float g[32];
                const int c0 = 64 * hh + 32 * k;
                tmem_ld32(lane_addr + c0, g);
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    orow[c0 / 8 + q] = make_uint4(pack_bf16(g[8 * q], g[8 * q + 1]), pack_bf16(g[8 * q + 2], g[8 * q + 3]),
                                                  pack_bf16(g[8 * q + 4], g[8 * q + 5]), pack_bf16(g[8 * q + 6], g[8 * q + 7]));
            }
            if (hh == 0) {
                float g[16];
                tmem_ld16(lane_addr + 128, g);
#pragma unroll
                for (int q = 0; q < 2; ++q)
                    orow[16 + q] = make_uint4(pack_bf16(g[8 * q], g[8 * q + 1]), pack_bf16(g[8 * q + 2], g[8 * q + 3]),
                                              pack_bf16(g[8 * q + 4], g[8 * q + 5]), pack_bf16(g[8 * q + 6], g[8 * q + 7]));
            }
        }
        fence_async_smem();
        tc_fence_before();                     // all tcgen05.ld of this tile are complete before the next MMAs
        __syncthreads();
        if (tid == 0) {
            bulk_s2g(dcomps_out + (size_t)tile * TM * CT, OUT, (uint32_t)rows * (CT * 2));
            bulk_commit();
        }
    }
    if (tid == 0) bulk_wait0();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

}  // namespace jt

using namespace jt;

extern "C" long long jt_head_tc_stage_bytes(int n_max) {
    return (((long long)n_max + TM - 1) / TM) * STAGE_TILE_BYTES;
}

extern "C" int jt_head_bwd_tc(const float* dout, const float* feat, int ldf, const float* Wb, const float* W1, const float* W2,
                              const float* W3, const int* n_dev, int n_max, float fea_progress, void* dcomps,
                              int dcomps_bf16, void* stage, float* gWb, float* gW1, float* gb1, float* gW2, float* gb2, float* gW3,
                              float* gb3, cudaStream_t stream) {
    JT_CHECK_ARG(dout && feat && Wb && W1 && W2 && W3 && dcomps && stage && ldf >= 28 && ldf % 4 == 0);
    const int n_wg = !!gWb + !!gW1 + !!gb1 + !!gW2 + !!gb2 + !!gW3 + !!gb3;
    JT_CHECK_ARG(n_wg == 0 || n_wg == 7);                // all weight gradients, or none (frozen head + basis_mat)
    JT_CHECK_ARG((reinterpret_cast<uintptr_t>(stage) & 127) == 0);
    if (n_max <= 0) return JT_OK;
    const bool wg = n_wg == 7;
    long long tiles = ((long long)n_max + TM - 1) / TM;
    int grid_d = (int)(tiles < 2 * kNumSMs ? tiles : 2 * kNumSMs);
    int grid_w = (int)(tiles < kNumSMs ? tiles : kNumSMs);
    unsigned char* st = static_cast<unsigned char*>(stage);
#define JT_HBD(DC, WS)                                                                                              \
    {                                                                                                               \
        if (int rc = set_smem(head_bwd_data_kernel<DC, WS>, BwdSmem::total)) return rc;                             \
        head_bwd_data_kernel<DC, WS><<<grid_d, NTB, BwdSmem::total, stream>>>(dout, feat, ldf, Wb, W1, W2, W3, n_dev, \
                                                                            n_max, fea_progress, dcomps, st);       \
    }
    if (dcomps_bf16) { if (wg) JT_HBD(true, true) else JT_HBD(true, false) }
    else { if (wg) JT_HBD(false, true) else JT_HBD(false, false) }
#undef JT_HBD
    g_launches += 1;
    if (wg) {
        if (int rc = set_smem(head_bwd_wgrad_kernel<0, 4, WG_STAGES, WG_STAGE_BYTES>, WG_STAGES * WG_STAGE_BYTES)) return rc;
        g_launches += 1;
        head_bwd_wgrad_kernel<0, 4, WG_STAGES, WG_STAGE_BYTES><<<grid_w, TM, WG_STAGES * WG_STAGE_BYTES, stream>>>(
            st, n_dev, n_max, gWb, gW1, gb1, gW2, gb2, gW3, gb3);
    }
    JT_RETURN_LAUNCH();
}

extern "C" int jt_sh_bwd_tc(const float* dout, const float* featdir, int ldf, const float* Wb, const int* n_dev,
                            int n_max, void* dcomps, int dcomps_bf16, void* stage, float* gWb, cudaStream_t stream) {
    // gWb = NULL (frozen basis_mat): no weight gradient, and `stage` may be NULL (a forward without staging)
    JT_CHECK_ARG(dout && featdir && Wb && dcomps && (stage || !gWb) && ldf >= 32 && ldf % 4 == 0);
    JT_CHECK_ARG(dcomps_bf16 == 1);                     // dcomps rows are bf16 [A][144] (what jt_vm_scatter_rays reads)
    JT_CHECK_ARG((reinterpret_cast<uintptr_t>(stage) & 127) == 0 && (reinterpret_cast<uintptr_t>(dcomps) & 15) == 0);
    if (n_max <= 0) return JT_OK;
    long long tiles = ((long long)n_max + TM - 1) / TM;
    int grid_d = (int)(tiles < 2 * kNumSMs ? tiles : 2 * kNumSMs);
    int grid_w = (int)(tiles < kNumSMs ? tiles : kNumSMs);
    unsigned char* st = static_cast<unsigned char*>(stage);
    unsigned short* dc = static_cast<unsigned short*>(dcomps);
    g_launches += 1;
    if (!gWb) {
        if (int rc = set_smem(sh_bwd_data_kernel<false>, ShBwdSmem::total)) return rc;
        sh_bwd_data_kernel<false><<<grid_d, NTB, ShBwdSmem::total, stream>>>(dout, featdir, ldf, Wb, n_dev, n_max, dc, nullptr);
        JT_RETURN_LAUNCH();
    }
    if (int rc = set_smem(sh_bwd_data_kernel<true>, ShBwdSmem::total)) return rc;
    if (int rc = set_smem(head_bwd_wgrad_kernel<3, 1, WG_SH_STAGES, WG_SH_STAGE_BYTES>, WG_SH_STAGES * WG_SH_STAGE_BYTES)) return rc;
    g_launches += 1;
    sh_bwd_data_kernel<true><<<grid_d, NTB, ShBwdSmem::total, stream>>>(dout, featdir, ldf, Wb, n_dev, n_max, dc, st);
    head_bwd_wgrad_kernel<3, 1, WG_SH_STAGES, WG_SH_STAGE_BYTES><<<grid_w, TM, WG_SH_STAGES * WG_SH_STAGE_BYTES, stream>>>(
        st, n_dev, n_max, gWb, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
    JT_RETURN_LAUNCH();
}
