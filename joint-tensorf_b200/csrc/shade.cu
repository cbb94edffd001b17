// K3 (strict-fp32 path) -- basis_mat projection and the shading heads as plain
// SIMT fp32 GEMMs plus the positional-encoding and SH kernels around them.
//
// Replaces reference basis_mat (tensoRF.py:156,270 / bateRF.py:130),
// positional_encoding (tensorBase.py:43-55), MLPRender_Fea.forward
// (tensorBase.py:116-126), MLPRender_Fea_WeakView.forward (tensorBase.py:198-214),
// SHRender (tensorBase.py:68-72) + eval_sh_bases deg 2 (sh.py:88-113) and their
// autograd. This is the bit-faithful fp32 mode (<= 1e-4 parity class); the tensor-core
// (tcgen05) heads live in app_basis_tc.cu, head_mlp_tc.cu, shade_tc_bwd.cu, weakview_tc.cu.
#include "jt_common.cuh"
#include "../../include/jt_vm.h"

namespace jt {

// ------------------------------------------------------------------ Y = act(X * W^T + b) [* (mask > 0)]
constexpr int BM = 128, BN = 64, KC = 32, XP = BM + 4;

__global__ void __launch_bounds__(256) gemm_nt_kernel(const float* __restrict__ X, int ldx,
                                                      const float* __restrict__ W, int ldw, int w_kn,
                                                      const float* __restrict__ bias, float* __restrict__ Y, int ldy,
                                                      const float* __restrict__ mask, int ldm,
                                                      const int* __restrict__ m_dev, int m_fixed, int N, int K,
                                                      int act) {
    __shared__ __align__(16) float Xs[KC][XP];
    __shared__ __align__(16) float Ws[KC][BN];
    const int M = m_dev ? *m_dev : m_fixed;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int n0 = blockIdx.y * BN;
    for (int tile = blockIdx.x; (long long)tile * BM < M; tile += gridDim.x) {
        const int m0 = tile * BM;
        float acc[8][4];
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
        for (int k0 = 0; k0 < K; k0 += KC) {
#pragma unroll
            for (int it = 0; it < 4; ++it) {
                const int idx = tid + it * 256;
                const int r = idx >> 3, kq = idx & 7;
                const int m = m0 + r, kc = k0 + kq * 4;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (m < M && kc < K) {
                    const float* src = X + (size_t)m * ldx + kc;
                    if (kc + 3 < ldx) {
                        v = *reinterpret_cast<const float4*>(src);
                        if (kc + 1 >= K) v.y = 0.f;
                        if (kc + 2 >= K) v.z = 0.f;
                        if (kc + 3 >= K) v.w = 0.f;
                    } else {
                        v.x = src[0];
                        if (kc + 1 < K) v.y = src[1];
                        if (kc + 2 < K) v.z = src[2];
                    }
                }
                Xs[kq * 4 + 0][r] = v.x; Xs[kq * 4 + 1][r] = v.y;
                Xs[kq * 4 + 2][r] = v.z; Xs[kq * 4 + 3][r] = v.w;
            }
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int idx = tid + it * 256;
                const int kk = idx >> 6, nn = idx & 63;
                const int k = k0 + kk, n = n0 + nn;
                float w = 0.f;
                if (k < K && n < N) w = w_kn ? W[(size_t)k * ldw + n] : W[(size_t)n * ldw + k];
                Ws[kk][nn] = w;
            }
            __syncthreads();
#pragma unroll 8
            for (int kk = 0; kk < KC; ++kk) {
                const float4 xa = *reinterpret_cast<const float4*>(&Xs[kk][ty * 8]);
                const float4 xb = *reinterpret_cast<const float4*>(&Xs[kk][ty * 8 + 4]);
                const float4 w = *reinterpret_cast<const float4*>(&Ws[kk][tx * 4]);
                const float xr[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
                const float wc[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int r = 0; r < 8; ++r)
#pragma unroll
                    for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(xr[r], wc[c], acc[r][c]);
            }
            __syncthreads();
        }
        const int n = n0 + tx * 4;
        const int wy = min(ldy, (N + 3) & ~3);      // writable width: N rounded up to a float4 (pad columns <- 0)
        if (n < wy) {
            float b[4] = {0.f, 0.f, 0.f, 0.f};
            if (bias) {
#pragma unroll
                for (int c = 0; c < 4; ++c) if (n + c < N) b[c] = bias[n + c];
            }
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const int m = m0 + ty * 8 + r;
                if (m >= M) continue;
                float v[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float t = acc[r][c] + b[c];
                    if (act == 1) t = fmaxf(t, 0.f);
                    else if (act == 2) t = 1.0f / (1.0f + expf(-t));
                    if (mask && n + c < N) t = mask[(size_t)m * ldm + n + c] > 0.f ? t : 0.f;
                    v[c] = (n + c < N) ? t : 0.f;
                }
                float* dst = Y + (size_t)m * ldy + n;
                *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
            }
        }
    }
}

// ------------------------------------------------------------------ dW[N][K] += dY^T X ; db[N] += sum dY
// Per chunk of `tbm` sample rows (staged in shared memory) a thread owns one 4 x 8 output tile; when the output
// has fewer than 256 tiles (N = 32, K = 100: 104), the chunk's rows are split into slices and every slice gets its
// own set of threads -- the partial sums meet in the atomics at the end anyway -- so the whole CTA works.
constexpr int TBM_MAX = 64;

__global__ void __launch_bounds__(256) gemm_tn_kernel(const float* __restrict__ dY, int ldy,
                                                      const float* __restrict__ X, int ldx,
                                                      const int* __restrict__ m_dev, int m_fixed, int N, int K,
                                                      float* __restrict__ dW, int ldw, float* __restrict__ db, int tbm,
                                                      int vec4) {
    extern __shared__ __align__(16) float smem[];
    const int NP = (N + 3) & ~3;
    const int KP = (K + 1 + 7) & ~7;          // column K carries 1.0 -> bias gradient
    float* Ys = smem;                          // [tbm][NP]
    float* Xs = smem + tbm * NP;               // [tbm][KP]
    const int M = m_dev ? *m_dev : m_fixed;
    const int tid = threadIdx.x;
    const int ng = NP >> 2, kg = KP >> 3, ntile = ng * kg;
    const int slices = ntile <= 128 ? 256 / ntile : 1;
    const int rps = (tbm + slices - 1) / slices;             // rows per slice
    int tile_of[2], r0_of[2], r1_of[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const int t = tid + s * 256;
        if (slices > 1) {
            const int sl = t / ntile;
            tile_of[s] = (s == 0 && sl < slices) ? t - sl * ntile : -1;
            r0_of[s] = sl * rps;
            r1_of[s] = min(tbm, r0_of[s] + rps);
        } else {
            tile_of[s] = t < ntile ? t : -1;
            r0_of[s] = 0;
            r1_of[s] = tbm;
        }
    }
    float acc[2][4][8];
#pragma unroll
    for (int s = 0; s < 2; ++s)
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 8; ++b) acc[s][a][b] = 0.f;
    for (int chunk = blockIdx.x; (long long)chunk * tbm < M; chunk += gridDim.x) {
        const int m0 = chunk * tbm;
        if (vec4) {                                          // 16-byte staging loads (rows and widths 16 B aligned)
            const int nq = NP >> 2, kq = KP >> 2;
            for (int idx = tid; idx < tbm * nq; idx += 256) {
                const int r = idx / nq, c = (idx - r * nq) * 4;
                const int m = m0 + r;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (m < M) v = *reinterpret_cast<const float4*>(dY + (size_t)m * ldy + c);      // N % 4 == 0
                *reinterpret_cast<float4*>(&Ys[r * NP + c]) = v;
            }
            for (int idx = tid; idx < tbm * kq; idx += 256) {
                const int r = idx / kq, c = (idx - r * kq) * 4;
                const int m = m0 + r;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (m < M) {
                    if (c < K) v = *reinterpret_cast<const float4*>(X + (size_t)m * ldx + c);   // K % 4 == 0
                    else if (c == K) v.x = 1.0f;
                }
                *reinterpret_cast<float4*>(&Xs[r * KP + c]) = v;
            }
        } else {
            for (int idx = tid; idx < tbm * NP; idx += 256) {
                const int r = idx / NP, c = idx - r * NP;
                const int m = m0 + r;
                Ys[idx] = (m < M && c < N) ? dY[(size_t)m * ldy + c] : 0.f;
            }
            for (int idx = tid; idx < tbm * KP; idx += 256) {
                const int r = idx / KP, c = idx - r * KP;
                const int m = m0 + r;
                float v = 0.f;
                if (m < M) v = (c < K) ? X[(size_t)m * ldx + c] : (c == K ? 1.0f : 0.f);
                Xs[idx] = v;
            }
        }
        __syncthreads();
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            if (tile_of[s] >= 0) {
                const int ni = tile_of[s] % ng, ki = tile_of[s] / ng;
#pragma unroll 4
                for (int m = r0_of[s]; m < r1_of[s]; ++m) {
                    const float4 y = *reinterpret_cast<const float4*>(&Ys[m * NP + ni * 4]);
                    const float4 xa = *reinterpret_cast<const float4*>(&Xs[m * KP + ki * 8]);
                    const float4 xb = *reinterpret_cast<const float4*>(&Xs[m * KP + ki * 8 + 4]);
                    const float yv[4] = {y.x, y.y, y.z, y.w};
                    const float xv[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int b = 0; b < 8; ++b) acc[s][a][b] = fmaf(yv[a], xv[b], acc[s][a][b]);
                }
            }
        }
        __syncthreads();
    }
    if (slices > 1) {
        // the row slices of a tile meet in shared memory first (one global atomic per output and CTA, as before)
        float* red = smem;                                   // [ntile][32]
        for (int i = tid; i < ntile * 32; i += 256) red[i] = 0.f;
        __syncthreads();
        if (tile_of[0] >= 0) {
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) atomicAdd(&red[tile_of[0] * 32 + a * 8 + b], acc[0][a][b]);
        }
        __syncthreads();
        if (tid < ntile) {
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) acc[0][a][b] = red[tid * 32 + a * 8 + b];
        } else {
            tile_of[0] = -1;
        }
    }
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        if (tile_of[s] < 0) continue;
        const int ni = tile_of[s] % ng, ki = tile_of[s] / ng;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const int n = ni * 4 + a;
            if (n >= N) continue;
#pragma unroll
            for (int b = 0; b < 8; ++b) {
                const int k = ki * 8 + b;
                const float v = acc[s][a][b];
                if (v == 0.f) continue;
                if (k < K) atomicAdd(dW + (size_t)n * ldw + k, v);
                else if (k == K && db) atomicAdd(db + n, v);
            }
        }
    }
}

// ------------------------------------------------------------------ positional encoding
// Column c of the encoded row (tensorBase.py:43-55): per source element e the
// block [sin(x*2^0..2^(F-1)), cos(x*2^0..2^(F-1))], each scaled by the
// annealing mask clamp(progress*F - l, 0, 1).
struct PEParams {
    int F;            // app_dim
    int fpe, vpe;     // frequency counts
    int mode;         // 0: MLP_Fea  [feat, dir, PE(feat), PE(dir)] -> out
                      // 1: WeakView [feat, PE(feat)] -> out ; [PE(dir)] -> out2 (cols 0..6*vpe)
    float fprog, vprog;
    int S;            // samples per ray (ray = sidx / S)
    int normalize_dir;
};

__device__ __forceinline__ void load_dir(const float* __restrict__ rays_d, int ray, int normalize, float d[3]) {
    d[0] = rays_d[3 * ray]; d[1] = rays_d[3 * ray + 1]; d[2] = rays_d[3 * ray + 2];
    if (normalize) {
        const float n = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
        d[0] /= n; d[1] /= n; d[2] /= n;
    }
}

// One thread per (sample, source element): one sincosf per frequency instead of separate sinf / cosf calls per
// output column, no per-column div/mod chain, and the [sin.., cos..] block of an element is one contiguous
// 2*nf-float run per thread. (The first version -- a warp per sample, a lane per output column -- spent ~600
// warp instructions per sample: 0.31 ms for the 0.31 M appearance samples of the LLFF configuration.)
__global__ void __launch_bounds__(256) pe_fwd_kernel(PEParams P, const float* __restrict__ feat, int ldf,
                                                     const int* __restrict__ aidx, const int* __restrict__ sidx,
                                                     const float* __restrict__ rays_d,
                                                     const int* __restrict__ n_dev, int n_fixed,
                                                     float* __restrict__ out, int ldo, float* __restrict__ out2,
                                                     int ldo2) {
    const int n = n_dev ? *n_dev : n_fixed;
    const int E = P.F + 3;                                     // source elements per sample: features, then direction
    const int nfe = 2 * P.fpe * P.F, nve = 2 * P.vpe * 3;
    const int raw = P.F + (P.mode == 0 ? 3 : 0);
    const int main_cols = raw + nfe + (P.mode == 0 ? nve : 0);
    const long long total = (long long)n * E;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const int a = (int)(idx / E), e = (int)(idx - (long long)a * E);
        float* o = out + (size_t)a * ldo;
        float x, prog;
        float* dst;
        int nf;
        if (e < P.F) {
            x = feat[(size_t)a * ldf + e];
            o[e] = x;
            nf = P.fpe; prog = P.fprog;
            dst = o + raw + e * 2 * P.fpe;
            if (e == 0) for (int c = main_cols; c < ldo; ++c) o[c] = 0.f;       // padding columns
        } else {
            const int k = e - P.F;
            const int ray = sidx[aidx[a]] / P.S;
            float d[3];
            load_dir(rays_d, ray, P.normalize_dir, d);
            x = d[k];
            nf = P.vpe; prog = P.vprog;
            if (P.mode == 0) { o[P.F + k] = x; dst = o + raw + nfe + k * 2 * P.vpe; }
            else dst = out2 + (size_t)a * ldo2 + k * 2 * P.vpe;
        }
        for (int l = 0; l < nf; ++l) {
            const float m = fminf(fmaxf(prog * nf - (float)l, 0.f), 1.f);
            float sn, cs;
            sincosf(x * (float)(1 << l), &sn, &cs);
            dst[l] = sn * m;
            dst[nf + l] = cs * m;
        }
    }
}

__global__ void __launch_bounds__(256) pe_bwd_kernel(PEParams P, const float* __restrict__ feat, int ldf,
                                                     const float* __restrict__ din, int ldi,
                                                     const int* __restrict__ n_dev, int n_fixed,
                                                     float* __restrict__ dfeat, int ldd) {
    const int n = n_dev ? *n_dev : n_fixed;
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    const int raw = P.F + (P.mode == 0 ? 3 : 0);
    for (int a = warp; a < n; a += nwarps) {
        const float* g = din + (size_t)a * ldi;
        for (int e = lane; e < ldd; e += 32) {
            float v = 0.f;
            if (e < P.F) {
                const float x = feat[(size_t)a * ldf + e];
                v = g[e];
                for (int l = 0; l < P.fpe; ++l) {
                    const float m = fminf(fmaxf(P.fprog * P.fpe - (float)l, 0.f), 1.f);
                    const float sc = (float)(1 << l);
                    float s, c;
                    sincosf(x * sc, &s, &c);
                    v += sc * m * (c * g[raw + e * 2 * P.fpe + l] - s * g[raw + e * 2 * P.fpe + P.fpe + l]);
                }
            }
            dfeat[(size_t)a * ldd + e] = v;
        }
    }
}

// ------------------------------------------------------------------ SH (deg 2) shading
// fwd: rgb[a][c] = relu(sum_k Y_k f[a][c*9+k] + 0.5); bwd: dfeat[a][c*9+k] = dout[a][c] * Y_k
__global__ void __launch_bounds__(256) sh_kernel(int bwd, const float* __restrict__ feat, int ldf,
                                                 const int* __restrict__ aidx, const int* __restrict__ sidx,
                                                 const float* __restrict__ rays_d, int S, int normalize_dir,
                                                 const int* __restrict__ n_dev, int n_fixed,
                                                 float* __restrict__ rgb, const float* __restrict__ dout,
                                                 float* __restrict__ dfeat, int ldd) {
    const int n = n_dev ? *n_dev : n_fixed;
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < n; a += gridDim.x * blockDim.x) {
        const int ray = sidx[aidx[a]] / S;
        float d[3], y[9];
        load_dir(rays_d, ray, normalize_dir, d);
        sh9(d, y);
        if (!bwd) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float s = 0.f;
#pragma unroll
                for (int k = 0; k < 9; ++k) s += y[k] * feat[(size_t)a * ldf + c * 9 + k];
                rgb[4 * (size_t)a + c] = fmaxf(s + 0.5f, 0.f);
            }
            rgb[4 * (size_t)a + 3] = 0.f;
        } else {
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int k = 0; k < 9; ++k) dfeat[(size_t)a * ldd + c * 9 + k] = dout[4 * (size_t)a + c] * y[k];
            for (int c = 27; c < ldd; ++c) dfeat[(size_t)a * ldd + c] = 0.f;
        }
    }
}

static int tiles_grid(int m_max, int per, int cap) {
    long long t = ((long long)m_max + per - 1) / per;
    if (t < 1) t = 1;
    return (int)(t < cap ? t : cap);
}

}  // namespace jt

using namespace jt;

extern "C" int jt_gemm_nt(const float* X, int ldx, const float* W, int ldw, int w_kn, const float* bias, float* Y,
                          int ldy, const float* mask, int ldm, const int* m_dev, int m_max, int N, int K, int act,
                          cudaStream_t stream) {
    JT_CHECK_ARG(X && W && Y && N > 0 && K > 0 && ldx >= K && ldy >= N);
    JT_CHECK_ARG((ldx & 3) == 0 && (ldy & 3) == 0 && act >= 0 && act <= 2);
    JT_CHECK_ARG((reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(Y) & 15) == 0);
    if (m_max <= 0) return JT_OK;
    dim3 grid(tiles_grid(m_max, BM, kNumSMs * 4), (N + BN - 1) / BN);
    g_launches += 1;
    gemm_nt_kernel<<<grid, 256, 0, stream>>>(X, ldx, W, ldw, w_kn, bias, Y, ldy, mask, ldm, m_dev, m_max, N, K, act);
    JT_RETURN_LAUNCH();
}

extern "C" int jt_gemm_tn(const float* dY, int ldy, const float* X, int ldx, const int* m_dev, int m_max, int N,
                          int K, float* dW, int ldw, float* db, cudaStream_t stream) {
    JT_CHECK_ARG(dY && X && dW && N > 0 && K > 0 && ldy >= N && ldx >= K && ldw >= K);
    const int NP = (N + 3) & ~3, KP = (K + 1 + 7) & ~7;
    JT_CHECK_ARG((NP >> 2) * (KP >> 3) <= 512);
    if (m_max <= 0) return JT_OK;
    int tbm = TBM_MAX;                                        // rows per chunk: as many as fit 48 KB of shared memory
    while (tbm > 16 && (size_t)tbm * (NP + KP) * sizeof(float) > 48 * 1024) tbm >>= 1;
    size_t smem = (size_t)tbm * (NP + KP) * sizeof(float);
    const size_t red_bytes = (size_t)(NP >> 2) * (KP >> 3) * 32 * sizeof(float);     // slice reduction (<= 128 tiles)
    if ((NP >> 2) * (KP >> 3) <= 128 && smem < red_bytes) smem = red_bytes;
    JT_CHECK_ARG(smem <= 48 * 1024);
    int grid = tiles_grid(m_max, tbm, kNumSMs * 2);
    g_launches += 1;
    const int vec4 = (N % 4 == 0) && (K % 4 == 0) && (ldy % 4 == 0) && (ldx % 4 == 0) &&
                     ((reinterpret_cast<uintptr_t>(dY) | reinterpret_cast<uintptr_t>(X)) & 15) == 0;
    gemm_tn_kernel<<<grid, 256, smem, stream>>>(dY, ldy, X, ldx, m_dev, m_max, N, K, dW, ldw, db, tbm, vec4);
    JT_RETURN_LAUNCH();
}

extern "C" int jt_pe_encode(int bwd, int app_dim, int fea_pe, int view_pe, int mode, float fea_progress,
                            float view_progress, int n_samples, int normalize_dir, const float* feat, int ldf,
                            const int* aidx, const int* sidx, const float* rays_d, const int* n_dev, int n_max,
                            float* out, int ldo, float* out2, int ldo2, const float* din, int ldi,
                            cudaStream_t stream) {
    JT_CHECK_ARG(feat && app_dim > 0 && fea_pe >= 0 && view_pe >= 0 && (mode == 0 || mode == 1));
    JT_CHECK_ARG(fea_pe <= 16 && view_pe <= 5);
    if (n_max <= 0) return JT_OK;
    PEParams P{app_dim, fea_pe, view_pe, mode, fea_progress, view_progress, n_samples, normalize_dir};
    int grid = tiles_grid(n_max, 8, kNumSMs * 8);
    g_launches += 1;
    if (!bwd) {
        JT_CHECK_ARG(aidx && sidx && rays_d && out && (mode == 0 || out2));
        const int cols = app_dim + (mode == 0 ? 3 : 0) + 2 * fea_pe * app_dim + (mode == 0 ? 6 * view_pe : 0);
        JT_CHECK_ARG(ldo >= cols && (mode == 0 || ldo2 >= 6 * view_pe));
        const int grid_f = tiles_grid(n_max, 256 / 32, kNumSMs * 16);       // ~ (app_dim + 3) threads per sample
        pe_fwd_kernel<<<grid_f, 256, 0, stream>>>(P, feat, ldf, aidx, sidx, rays_d, n_dev, n_max, out, ldo, out2, ldo2);
    } else {
        JT_CHECK_ARG(din && out && ldo >= app_dim);
        pe_bwd_kernel<<<grid, 256, 0, stream>>>(P, feat, ldf, din, ldi, n_dev, n_max, out, ldo);
    }
    JT_RETURN_LAUNCH();
}

extern "C" int jt_sh_shade(int bwd, const float* feat, int ldf, const int* aidx, const int* sidx,
                           const float* rays_d, int n_samples, int normalize_dir, const int* n_dev, int n_max,
                           float* rgb, const float* dout, float* dfeat, int ldd, cudaStream_t stream) {
    JT_CHECK_ARG(aidx && sidx && rays_d && ldf >= 27);
    JT_CHECK_ARG(bwd ? (dout && dfeat && ldd >= 27) : (feat && rgb));
    if (n_max <= 0) return JT_OK;
    int grid = tiles_grid(n_max, 256, kNumSMs * 8);
    g_launches += 1;
    sh_kernel<<<grid, 256, 0, stream>>>(bwd, feat, ldf, aidx, sidx, rays_d, n_samples, normalize_dir, n_dev, n_max,
                                        rgb, dout, dfeat, ldd);
    JT_RETURN_LAUNCH();
}
