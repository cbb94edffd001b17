// K4 -- density activation, raw2alpha (transmittance scan), appearance-sample
// selection + compaction, front-to-back compositing, and their backward pass
// as a reverse scan.
//
// Replaces reference feature2density (tensorBase.py:696-700), raw2alpha
// (tensorBase.py:57-65), the app_mask selection + boolean indexing
// (batBase.py:127-139) and the accumulation / background / clamp / depth block
// (batBase.py:142-165), plus the autograd of all of them.
//
// One warp owns one ray and walks its compacted valid samples 32 at a time;
// the running transmittance is a warp product-scan with a carry. Invalid
// samples have sigma = 0 in the reference, i.e. alpha = 0 and a factor
// 1 - 0 + 1e-10 == 1.0f in the cumprod, so skipping them is exact.
#include "jt_common.cuh"
#include "vm_taps.cuh"
#include "../../include/jt_vm.h"

namespace jt {

// ------------------------------------------------------------------ forward, pass A
// per ray: sigma -> alpha -> T (exclusive product scan) -> weight; accumulates acc
// and sum(w*z); counts appearance samples (w > thres).
// Each lane owns KS consecutive samples of a 32*KS-sample block: one warp scan per block instead of one per 32
// samples, and KS independent loads in flight per lane (the kernel is one warp per ray and latency-bound: with KS = 1
// it reached 30 % of the HBM rate of its 40 bytes per sample).
constexpr int KS = 4;       // forward (measured: 0.050 -> 0.046 ms for the three launches of jt_alpha_fwd)
// (the backward keeps one sample per lane: four cost registers (79) and time, 0.056 -> 0.062 ms; it is software-pipelined instead)
__global__ void __launch_bounds__(256) alpha_fwd_kernel(const int* __restrict__ off, int n_rays,
                                                        const float* __restrict__ sigfeat,
                                                        const float* __restrict__ dist,
                                                        const float4* __restrict__ samp, float shift, int act,
                                                        float dscale, float thres, float* __restrict__ weight,
                                                        float* __restrict__ trans, float* __restrict__ acc_out,
                                                        float* __restrict__ wz_out, int* __restrict__ app_cnt) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int r = warp; r < n_rays; r += nwarps) {
        const int b = off[r], e = off[r + 1];
        double carry = 1.0;
        float acc = 0.f, wz = 0.f;
        int cnt = 0;
        // the inputs of the next block are requested before the current one is scanned
        float nsf[KS], ndj[KS], nz[KS];
#pragma unroll
        for (int k = 0; k < KS; ++k) {
            const int j = b + lane * KS + k;
            nsf[k] = ndj[k] = nz[k] = 0.f;
            if (j < e) { nsf[k] = sigfeat[j]; ndj[k] = dist[j]; nz[k] = samp[j].w; }
        }
        for (int j0 = b; j0 < e; j0 += 32 * KS) {
            const int jl = j0 + lane * KS;                   // first sample of this lane
            float q[KS], alpha[KS], z[KS];
            double pl = 1.0;                                 // product of this lane's q (double, see below)
#pragma unroll
            for (int k = 0; k < KS; ++k) {
                q[k] = 1.0f; alpha[k] = 0.f; z[k] = nz[k];
                if (jl + k < e) {
                    const float sigma = density_act(nsf[k] + shift, act);
                    alpha[k] = 1.0f - exp_neg(-sigma * (ndj[k] * dscale));
                    q[k] = 1.0f - alpha[k] + 1e-10f;
                }
                pl *= (double)q[k];
            }
#pragma unroll
            for (int k = 0; k < KS; ++k) {
                const int j = jl + 32 * KS + k;
                if (j < e) { nsf[k] = sigfeat[j]; ndj[k] = dist[j]; nz[k] = samp[j].w; }
            }
            // Inclusive product scan over the warp, in DOUBLE: the reference's torch.cumprod accumulates in double on
            // the CPU (ATen cumprod_cpu_kernel: at::acc_type<float, false>) and rounds every prefix to fp32 once, so
            // T_j carries one rounding instead of j; a float scan here was the largest single difference to the
            // reference's weights / gradients at the front of long opaque rays.
            double p = pl;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                double v = __shfl_up_sync(0xffffffffu, p, o);
                if (lane >= o) p *= v;
            }
            double excl = __shfl_up_sync(0xffffffffu, p, 1);
            if (lane == 0) excl = 1.0;
            double Td = carry * excl;                        // transmittance in front of this lane's first sample
            bool pass[KS];
#pragma unroll
            for (int k = 0; k < KS; ++k) {
                const float T = (float)Td;
                const float w = alpha[k] * T;
                pass[k] = false;
                if (jl + k < e) {
                    weight[jl + k] = w;
                    trans[jl + k] = T;
                    acc += w;
                    wz += w * z[k];
                    pass[k] = w > thres;
                }
                Td *= (double)q[k];
            }
#pragma unroll
            for (int k = 0; k < KS; ++k) cnt += __popc(__ballot_sync(0xffffffffu, pass[k]));
            carry *= __shfl_sync(0xffffffffu, p, 31);
        }
        acc = warp_sum(acc);
        wz = warp_sum(wz);
        if (lane == 0) { acc_out[r] = acc; wz_out[r] = wz; app_cnt[r] = cnt; }
    }
}

// ------------------------------------------------------------------ forward, pass B
// appearance compaction: aidx[a] = sample slot j, app_of[j] = a (or -1).
// app_cap bounds the appearance list: entries a >= app_cap are dropped (app_of = -1, nothing written to aidx) and
// app_used = {min(A, app_cap), A > app_cap} tells the caller -- every later kernel of the appearance stage takes
// app_used[0] as its device-side count, so buffers sized app_cap are never overrun.
__global__ void __launch_bounds__(256) app_fill_kernel(const int* __restrict__ off, const int* __restrict__ aoff,
                                                       int n_rays, const float* __restrict__ weight, float thres,
                                                       int* __restrict__ aidx, int* __restrict__ app_of, int app_cap,
                                                       int* __restrict__ app_used) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    if (app_used && blockIdx.x == 0 && threadIdx.x == 0) {
        const int total = aoff[n_rays];
        app_used[0] = min(total, app_cap);
        app_used[1] = total > app_cap ? 1 : 0;
    }
    for (int r = warp; r < n_rays; r += nwarps) {
        const int b = off[r], e = off[r + 1];
        int base = aoff[r];
        // four 32-sample chunks per iteration: their loads are independent (one warp per ray: latency-bound)
        for (int j0 = b; j0 < e; j0 += 128) {
            float wv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = j0 + 32 * u + lane;
                wv[u] = j < e ? weight[j] : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = j0 + 32 * u + lane;
                const bool ok = (j < e) && (wv[u] > thres);
                const unsigned m = __ballot_sync(0xffffffffu, ok);
                if (j < e) {
                    int a = ok ? base + __popc(m & ((1u << lane) - 1u)) : -1;
                    if (a >= app_cap) a = -1;
                    app_of[j] = a;
                    if (a >= 0) aidx[a] = j;
                }
                base += __popc(m);
            }
        }
    }
}

// ------------------------------------------------------------------ forward, pass C
// batBase.py:160-162: depth = sum w*t + (1 - acc) * ray_dir_z - near + 0.05 (one expression for both compositing kernels,
// so render_normals' depth is bit-identical to forward's)
__device__ __forceinline__ float ray_depth(float wz, float acc, float dir_z, float depth_bias) {
    return wz + (1.0f - acc) * dir_z + depth_bias;
}

// rgb_map = sum w*rgb (+ 1-acc if white) clamped; depth; opacity.
__global__ void __launch_bounds__(256) composite_fwd_kernel(const int* __restrict__ aoff, int n_rays,
                                                            const int* __restrict__ aidx,
                                                            const float* __restrict__ weight,
                                                            const float* __restrict__ rgb,
                                                            const float* __restrict__ acc_in,
                                                            const float* __restrict__ wz_in,
                                                            const float* __restrict__ rays_d, int white_bg,
                                                            float depth_bias, float* __restrict__ rgb_pre,
                                                            float* __restrict__ rgb_map, float* __restrict__ depth,
                                                            float* __restrict__ opacity, int app_cap) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int r = warp; r < n_rays; r += nwarps) {
        const int b = min(aoff[r], app_cap), e = min(aoff[r + 1], app_cap);
        float c0 = 0.f, c1 = 0.f, c2 = 0.f;
        for (int a0 = b + lane; a0 < e; a0 += 128) {        // four entries per lane in flight: index -> weight is a
            int jx[4];                                        // dependent gather, the colours are independent loads
            float4 cv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int a = a0 + 32 * u;
                jx[u] = a < e ? aidx[a] : -1;
                cv[u] = a < e ? __ldcs(reinterpret_cast<const float4*>(rgb) + a) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float w = jx[u] >= 0 ? weight[jx[u]] : 0.f;
                c0 += w * cv[u].x; c1 += w * cv[u].y; c2 += w * cv[u].z;
            }
        }
        c0 = warp_sum(c0); c1 = warp_sum(c1); c2 = warp_sum(c2);
        if (lane == 0) {
            const float acc = acc_in[r];
            const float bg = white_bg ? (1.0f - acc) : 0.0f;
            c0 += bg; c1 += bg; c2 += bg;
            rgb_pre[3 * r + 0] = c0; rgb_pre[3 * r + 1] = c1; rgb_pre[3 * r + 2] = c2;
            rgb_map[3 * r + 0] = fminf(fmaxf(c0, 0.f), 1.f);
            rgb_map[3 * r + 1] = fminf(fmaxf(c1, 0.f), 1.f);
            rgb_map[3 * r + 2] = fminf(fmaxf(c2, 0.f), 1.f);
            depth[r] = ray_depth(wz_in[r], acc, rays_d[3 * r + 2], depth_bias);
            opacity[r] = acc;
        }
    }
}

// Normal map: normal[r] = sum_j w_j n_j over ALL valid samples of ray r (the weights whose sum is opacity), n [V][3] the
// per-sample unit normals of jt_field_density_grad; depth and opacity as composite_fwd_kernel writes them. One warp
// per ray, lane-strided sums then a fixed butterfly: the result does not depend on the batch the ray is rendered in.
__global__ void __launch_bounds__(256) normal_composite_kernel(const int* __restrict__ off, int n_rays,
                                                               const float* __restrict__ weight,
                                                               const float* __restrict__ nrm,
                                                               const float* __restrict__ acc_in,
                                                               const float* __restrict__ wz_in,
                                                               const float* __restrict__ rays_d, float depth_bias,
                                                               float* __restrict__ normal, float* __restrict__ depth,
                                                               float* __restrict__ opacity) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int r = warp; r < n_rays; r += nwarps) {
        const int b = off[r], e = off[r + 1];
        float c0 = 0.f, c1 = 0.f, c2 = 0.f;
        for (int j = b + lane; j < e; j += 32) {
            const float w = weight[j];
            c0 += w * nrm[3 * j]; c1 += w * nrm[3 * j + 1]; c2 += w * nrm[3 * j + 2];
        }
        c0 = warp_sum(c0); c1 = warp_sum(c1); c2 = warp_sum(c2);
        if (lane == 0) {
            const float acc = acc_in[r];
            normal[3 * r + 0] = c0; normal[3 * r + 1] = c1; normal[3 * r + 2] = c2;
            depth[r] = ray_depth(wz_in[r], acc, rays_d[3 * r + 2], depth_bias);
            opacity[r] = acc;
        }
    }
}

// ------------------------------------------------------------------ backward
// Reverse walk over a ray's valid samples: d rgb_map / d opacity ->
//   dout[a]   = dL/d(pre-activation of the shading head)   (shade_act folds sigmoid / relu')
//   dsig[j]   = dL/d sigma_feature
//   dnorm[r]  = dL/d |ray_dir|   (NDC rays only: dists are scaled by the norm)
// Autograd of raw2alpha (tensorBase.py:57-65) gives, with S_j = sum_{i>j} dL/dw_i * w_i,
//   dL/dalpha_j = dL/dw_j * T_j - S_j / q_j,        q_j = 1 - alpha_j + 1e-10.
// In a nearly opaque field with nearly constant colours the two terms cancel to ~1e-4 of their size, and their fp32
// errors do not: T_j and the w_i inside S_j come from differently grouped products (a parallel scan here, a
// sequential cumprod in the reference). The same quantity is therefore evaluated as
//   dL/dalpha_j = T_j * (dL/dw_j - Y_j),   Y_j = S_j / (q_j T_j) = sum_{i>j} dL/dw_i alpha_i prod_{j<k<i} q_k,
// where Y obeys the first-order recurrence Y_{j-1} = dL/dw_j alpha_j + q_j Y_j (a reverse scan of affine maps):
// no transmittance enters the cancelling difference, only local factors do. Identical in exact arithmetic; in fp32
// it is closer to the float64 result than the reference's own autograd is (tests/gpu_common.py slice_parity).
__global__ void __launch_bounds__(256) render_bwd_kernel(const int* __restrict__ off, int n_rays,
                                                         const float* __restrict__ sigfeat,
                                                         const float* __restrict__ dist,
                                                         const float* __restrict__ weight,
                                                         const float* __restrict__ trans,
                                                         const int* __restrict__ app_of,
                                                         const float* __restrict__ rgb,
                                                         const float* __restrict__ rgb_pre,
                                                         const float* __restrict__ g_rgb,
                                                         const float* __restrict__ g_acc, float shift, int act,
                                                         float dscale, int white_bg, int shade_act,
                                                         float* __restrict__ dout, float* __restrict__ dsig,
                                                         float* __restrict__ dnorm) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int r = warp; r < n_rays; r += nwarps) {
        const int b = off[r], e = off[r + 1];
        float gm[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float pre = rgb_pre[3 * r + c];
            gm[c] = (pre >= 0.0f && pre <= 1.0f) ? g_rgb[3 * r + c] : 0.0f;      // clamp backward
        }
        const float dacc = (g_acc ? g_acc[r] : 0.0f) - (white_bg ? (gm[0] + gm[1] + gm[2]) : 0.0f);
        double carry = 0.0;
        float dn = 0.f;
        const int len = e - b;
        // Reverse index i = i0 + lane, sample j = e-1-i. Software pipeline over the 32-sample chunks (one warp per ray:
        // every exposed latency is paid ~20 times in a row): while chunk c is scanned, the per-sample inputs of chunk
        // c+2 and the colours of chunk c+1 (a dependent gather through app_of) are already in flight.
        const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
        auto load_vals = [&](int i, float& w, float& sf, float& dj, float& tj, int& a) {
            w = 0.f; sf = 0.f; dj = 0.f; tj = 0.f; a = -1;
            if (i < len) {
                const int j = e - 1 - i;
                w = weight[j]; sf = sigfeat[j]; dj = dist[j]; tj = trans[j]; a = app_of[j];
            }
        };
        auto load_rgb = [&](int a) -> float4 { return a >= 0 ? *reinterpret_cast<const float4*>(rgb + 4 * (size_t)a) : zero4; };
        float w0, sf0, dj0, tj0, w1, sf1, dj1, tj1;
        int a0, a1;
        load_vals(lane, w0, sf0, dj0, tj0, a0);
        load_vals(32 + lane, w1, sf1, dj1, tj1, a1);
        float4 c0 = load_rgb(a0);
        for (int i0 = 0; i0 < len; i0 += 32) {
            const int i = i0 + lane;
            const float4 c1 = load_rgb(a1);
            float w2, sf2, dj2, tj2;
            int a2;
            load_vals(i + 64, w2, sf2, dj2, tj2, a2);
            const int j = e - 1 - i;
            float dw = 0.f, xx = 0.f, sg = 0.f, dd = 0.f, ex = 1.f, al = 0.f, qf = 1.f;
            if (i < len) {
                dw = dacc;
                if (a0 >= 0) {
                    const float r0 = c0.x, r1 = c0.y, r2 = c0.z;
                    dw += gm[0] * r0 + gm[1] * r1 + gm[2] * r2;
                    float d0 = w0 * gm[0], d1 = w0 * gm[1], d2 = w0 * gm[2];
                    if (shade_act == 1) { d0 *= r0 * (1.f - r0); d1 *= r1 * (1.f - r1); d2 *= r2 * (1.f - r2); }
                    else if (shade_act == 2) { d0 = r0 > 0.f ? d0 : 0.f; d1 = r1 > 0.f ? d1 : 0.f; d2 = r2 > 0.f ? d2 : 0.f; }
                    *reinterpret_cast<float4*>(dout + 4 * (size_t)a0) = make_float4(d0, d1, d2, 0.f);
                }
                xx = sf0 + shift;
                sg = density_act(xx, act);
                dd = dj0 * dscale;
                ex = exp_neg(-sg * dd);
                al = 1.0f - ex;
                qf = 1.0f - al + 1e-10f;
            }
            // this sample's affine map y -> A + Q y, in double like the forward scan (and the reference's CPU cumsum)
            double A = (double)dw * (double)al, Q = (double)qf;
            // inclusive scan over the lanes: (A, Q) o (A', Q') = (A + Q A', Q Q')
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const double a2s = __shfl_up_sync(0xffffffffu, A, o), q2s = __shfl_up_sync(0xffffffffu, Q, o);
                if (lane >= o) { A = fma(Q, a2s, A); Q *= q2s; }
            }
            const double zin = fma(Q, carry, A);     // Y in front of this lane's sample (includes it)
            double y = __shfl_up_sync(0xffffffffu, zin, 1);
            if (lane == 0) y = carry;                // Y_j: everything behind sample j
            if (i < len) {
                const float dalpha = (float)((double)tj0 * ((double)dw - y));
                const float dsigma = dalpha * dd * ex;
                dsig[j] = dsigma * density_act_grad(xx, act);
                dn += dalpha * sg * ex * dd;          // d/d(norm) * norm
            }
            carry = __shfl_sync(0xffffffffu, zin, 31);
            w0 = w1; sf0 = sf1; dj0 = dj1; tj0 = tj1; a0 = a1; c0 = c1;
            w1 = w2; sf1 = sf2; dj1 = dj2; tj1 = tj2; a1 = a2;
        }
        if (dnorm) {
            dn = warp_sum(dn);
            if (lane == 0) dnorm[r] = dn;
        }
    }
}

__global__ void ray_init_kernel(const float* __restrict__ rays_d, const float* __restrict__ dnorm, int n_rays,
                                float* __restrict__ d_o, float* __restrict__ d_d) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rays) return;
    float k = 0.f, x = 0.f, y = 0.f, z = 0.f;
    if (dnorm) {
        x = rays_d[3 * r]; y = rays_d[3 * r + 1]; z = rays_d[3 * r + 2];
        const float n2 = x * x + y * y + z * z;
        k = n2 > 0.f ? dnorm[r] / n2 : 0.f;                        // dnorm holds dL/dnorm * norm
    }
    d_o[3 * r] = 0.f; d_o[3 * r + 1] = 0.f; d_o[3 * r + 2] = 0.f;
    d_d[3 * r] = k * x; d_d[3 * r + 1] = k * y; d_d[3 * r + 2] = k * z;
}

static int ray_grid(int n_rays) {
    int want = (n_rays + 7) / 8;
    int cap = kNumSMs * 8;
    return want < cap ? (want < 1 ? 1 : want) : cap;
}

}  // namespace jt

using namespace jt;

extern "C" int jt_alpha_fwd(const int* ray_off, int n_rays, const float* sigfeat, const float* dist,
                            const float* samp, float density_shift, int act, float distance_scale, float thres,
                            float* weight, float* trans, float* acc, float* wz, int* app_cnt, int* app_off,
                            int* aidx, int* app_of, int app_cap, int* app_used, cudaStream_t stream) {
    JT_CHECK_ARG(ray_off && sigfeat && dist && samp && weight && trans && acc && wz && app_cnt && app_off && aidx && app_of);
    JT_CHECK_ARG(act == 0 || act == 1);
    JT_CHECK_ARG(app_cap > 0);
    if (n_rays <= 0) return JT_OK;
    int grid = ray_grid(n_rays);
    g_launches += 2;
    alpha_fwd_kernel<<<grid, 256, 0, stream>>>(ray_off, n_rays, sigfeat, dist, reinterpret_cast<const float4*>(samp),
                                               density_shift, act, distance_scale, thres, weight, trans, acc, wz,
                                               app_cnt);
    if (int rc = jt_exclusive_scan(app_cnt, app_off, n_rays, stream)) return rc;
    app_fill_kernel<<<grid, 256, 0, stream>>>(ray_off, app_off, n_rays, weight, thres, aidx, app_of, app_cap, app_used);
    JT_RETURN_LAUNCH();
}

extern "C" int jt_composite_fwd(const int* app_off, int n_rays, const int* aidx, const float* weight,
                                const float* rgb, const float* acc, const float* wz, const float* rays_d,
                                int white_bg, float depth_bias, float* rgb_pre, float* rgb_map, float* depth,
                                float* opacity, int app_cap, cudaStream_t stream) {
    JT_CHECK_ARG(app_off && aidx && weight && rgb && acc && wz && rays_d && rgb_pre && rgb_map && depth && opacity);
    if (n_rays <= 0) return JT_OK;
    g_launches += 1;
    composite_fwd_kernel<<<ray_grid(n_rays), 256, 0, stream>>>(app_off, n_rays, aidx, weight, rgb, acc, wz, rays_d,
                                                               white_bg, depth_bias, rgb_pre, rgb_map, depth, opacity,
                                                               app_cap > 0 ? app_cap : 2147483647);
    JT_RETURN_LAUNCH();
}

extern "C" int jt_normal_composite(const int* ray_off, int n_rays, const float* weight, const float* normals,
                                   const float* acc, const float* wz, const float* rays_d, float depth_bias,
                                   float* normal_map, float* depth, float* opacity, cudaStream_t stream) {
    JT_CHECK_ARG(ray_off && weight && normals && acc && wz && rays_d && normal_map && depth && opacity);
    if (n_rays <= 0) return JT_OK;
    g_launches += 1;
    normal_composite_kernel<<<ray_grid(n_rays), 256, 0, stream>>>(ray_off, n_rays, weight, normals, acc, wz, rays_d,
                                                                  depth_bias, normal_map, depth, opacity);
    JT_RETURN_LAUNCH();
}

extern "C" int jt_render_bwd(const int* ray_off, int n_rays, const float* sigfeat, const float* dist,
                             const float* weight, const float* trans, const int* app_of, const float* rgb,
                             const float* rgb_pre, const float* g_rgb, const float* g_acc, float density_shift,
                             int act, float distance_scale, int white_bg, int shade_act, float* dout, float* dsig,
                             float* dnorm, cudaStream_t stream) {
    JT_CHECK_ARG(ray_off && sigfeat && dist && weight && trans && app_of && rgb && rgb_pre && g_rgb && dout && dsig);
    if (n_rays <= 0) return JT_OK;
    g_launches += 1;
    render_bwd_kernel<<<ray_grid(n_rays), 256, 0, stream>>>(ray_off, n_rays, sigfeat, dist, weight, trans, app_of, rgb,
                                                            rgb_pre, g_rgb, g_acc, density_shift, act, distance_scale,
                                                            white_bg, shade_act, dout, dsig, dnorm);
    JT_RETURN_LAUNCH();
}

extern "C" int jt_ray_init(const float* rays_d, const float* dnorm, int n_rays, float* d_o, float* d_d,
                           cudaStream_t stream) {
    JT_CHECK_ARG(rays_d && d_o && d_d);
    if (n_rays <= 0) return JT_OK;
    g_launches += 1;
    ray_init_kernel<<<(n_rays + 255) / 256, 256, 0, stream>>>(rays_d, dnorm, n_rays, d_o, d_d);
    JT_RETURN_LAUNCH();
}
