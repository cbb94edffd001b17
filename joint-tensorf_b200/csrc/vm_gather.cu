// K2 -- plane x line VM feature interpolation, forward and backward.
//
// Replaces reference BAT_VMSplit.compute_densityfeature (bateRF.py:41-94; twin
// tensoRF.py:230-251) and the gather part of compute_appfeature
// (bateRF.py:97-128; twin tensoRF.py:254-268), i.e. the 12 F.grid_sample calls
// per forward and their grid_sampler_2d_backward atomics.
//
// Layout: factors are channel-last ([H][W][C] planes, [L][C] lines) so one
// bilinear tap of all channels is one contiguous vector. Four lanes share a
// sample; lane `sub` owns channel quads sub, sub+4, ... and loads them as
// float4 (16 B), so the four lanes of a sample read 64 contiguous bytes per
// tap and a warp covers 8 consecutive samples of (mostly) one ray, whose taps
// overlap in L1. The backward pass re-reads the taps (for the coordinate
// gradient that drives the pose optimisation, bateRF.py:44-46 does not detach
// coordinates) and scatters factor gradients with 16-byte vector RED
// operations.
#include <stdlib.h>
#include "jt_common.cuh"
#include "vm_taps.cuh"
#include "../../include/jt_vm.h"

namespace jt {

// APP == false: out[e] = sum_i sum_c P_ic * L_ic               (density feature)
// APP == true : out[e][off_i + c] = P_ic * L_ic                (appearance components, before basis_mat)
template <bool APP, bool B16>
__global__ void __launch_bounds__(256, 4) vm_fwd_kernel(Factors F, const float4* __restrict__ samp,
                                                     const int* __restrict__ slot, const int* __restrict__ n_dev,
                                                     int n_fixed, float* __restrict__ out) {
    const int n = n_dev ? *n_dev : n_fixed;
    const int lane = threadIdx.x & 31, sub = lane & 3, grp = lane >> 2;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int base = warp * 8; base < n; base += nwarps * 8) {
        const int e = base + grp;
        const bool act = e < n;
        float acc = 0.f;
        if (act) {
            const int j = slot ? slot[e] : e;
            const float4 u4 = samp[j];
            const float u[3] = {u4.x, u4.y, u4.z};
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const PlaneTaps t = plane_taps(F, i, u);
                const int C = F.C[i];
                for (int q = sub * 4; q < C; q += 16) {
                    float4 a = ld_tap4<B16>(F.plane[i], t.o00 + q), b = ld_tap4<B16>(F.plane[i], t.o10 + q);
                    float4 c = ld_tap4<B16>(F.plane[i], t.o01 + q), d = ld_tap4<B16>(F.plane[i], t.o11 + q);
                    float4 la = ld_tap4<B16>(F.line[i], t.ol0 + q), lb = ld_tap4<B16>(F.line[i], t.ol1 + q);
                    float4 pv = f4_bilin(a, t.w00, b, t.w10, c, t.w01, d, t.w11);
                    float4 lv = f4_lerp2(la, t.tl.w0, lb, t.tl.w1);
                    if (APP) {
                        __stcs(reinterpret_cast<float4*>(out + (size_t)e * F.ctot + F.off[i] + q), f4_mul(pv, lv));
                    } else {
                        acc += f4_dot(pv, lv);
                    }
                }
            }
        }
        if (!APP) {
            acc = quad_sum(acc);
            if (act && sub == 0) out[e] = acc;
        }
    }
}

// Density feature of a field whose three planes all have 16 channels (every shipped config). vm_fwd_kernel<false>
// spends most of its issue slots on per-sample setup -- record load, 3 x 3 tap positions, weights, offsets -- that
// each of the 4 lanes of a sample repeats for one quad of channels. Here 2 lanes share a sample and lane h owns
// quads 2h and 2h + 1 (channels 8h .. 8h + 7), so a warp covers 16 samples for about the same setup work, and the
// offsets are 32-bit (the host checks H W C < 2^31). The sum keeps vm_fwd_kernel's order -- per quad k,
// a_k = ((0 + dot_0k) + dot_1k) + dot_2k over the planes, then (a_0 + a_1) + (a_2 + a_3) -- so the result is
// bit-identical to it. The per-plane step is dens16_plane (vm_taps.cuh).
template <bool B16>
__global__ void __launch_bounds__(256, 4) vm_density16_fwd_kernel(Factors F, const float4* __restrict__ samp,
                                                                const int* __restrict__ slot, const int* __restrict__ n_dev,
                                                                int n_fixed, float* __restrict__ out) {
    const int n = n_dev ? *n_dev : n_fixed;
    const int lane = threadIdx.x & 31, h = lane & 1, grp = lane >> 1;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int base = warp * 16; base < n; base += nwarps * 16) {
        const int e = base + grp;
        const bool act = e < n;
        float a0 = 0.f, a1 = 0.f;                        // quads 2h, 2h + 1
        if (act) {
            const int j = slot ? slot[e] : e;
            const float4 u4 = samp[j];
            const float u[3] = {u4.x, u4.y, u4.z};
#pragma unroll
            for (int i = 0; i < 3; ++i) dens16_plane<B16>(F, i, u, h * 8, a0, a1);
        }
        float acc = a0 + a1;
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        if (act && h == 0) out[e] = acc;
    }
}

// Backward of the above. gin: density -> dL/dsigma_feature [n]; app -> dL/dcomponents [n][ctot].
// dsamp[j] (float4, xyz used) receives dL/du in normalised coordinates; `accumulate`
// selects store (density pass, runs first) or add (appearance pass; each sample
// slot appears at most once in `slot`, so the read-modify-write has one owner).
// QI > 0: every plane has exactly 16*QI channels -> the 7*QI tap loads of a plane are
// issued back to back (memory-level parallelism is what bounds this kernel: ncu shows
// ~70 % of stall samples on the long scoreboard); QI == 0: generic channel loop.
template <bool APP, int QI>
__global__ void __launch_bounds__(256) vm_bwd_kernel(Factors F, FactorGrads G, const float4* __restrict__ samp,
                                                     const int* __restrict__ slot, const int* __restrict__ n_dev,
                                                     int n_fixed, const float* __restrict__ gin,
                                                     float4* __restrict__ dsamp, int accumulate) {
    const int n = n_dev ? *n_dev : n_fixed;
    const int lane = threadIdx.x & 31, sub = lane & 3, grp = lane >> 2;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    constexpr int NQ = QI > 0 ? QI : 1;
    for (int base = warp * 8; base < n; base += nwarps * 8) {
        const int e = base + grp;
        const bool act = e < n;
        float du[3] = {0.f, 0.f, 0.f};
        int j = 0;
        if (act) {
            j = slot ? slot[e] : e;
            const float4 u4 = samp[j];
            const float u[3] = {u4.x, u4.y, u4.z};
            const float gs = APP ? 0.f : gin[e];
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const PlaneTaps t = plane_taps(F, i, u);
                const int C = F.C[i];
                float sx = 0.f, sy = 0.f, sl = 0.f;
                const int q_end = QI > 0 ? sub * 4 + 1 : C;            // QI > 0: one pass of the outer loop
                for (int q0 = sub * 4; q0 < q_end; q0 += 16 * NQ) {
                    float4 a[NQ], b[NQ], c[NQ], d[NQ], la[NQ], lb[NQ], g4[NQ];
#pragma unroll
                    for (int k = 0; k < NQ; ++k) {
                        const int q = q0 + 16 * k;
                        a[k] = ldg4(t.p00 + q); b[k] = ldg4(t.p10 + q); c[k] = ldg4(t.p01 + q); d[k] = ldg4(t.p11 + q);
                        la[k] = ldg4(t.l0 + q); lb[k] = ldg4(t.l1 + q);
                        g4[k] = APP ? __ldcs(reinterpret_cast<const float4*>(gin + (size_t)e * F.ctot + F.off[i] + q))
                                    : make_float4(gs, gs, gs, gs);
                    }
#pragma unroll
                    for (int k = 0; k < NQ; ++k) {
                        const int q = q0 + 16 * k;
                        float4 pv = f4_bilin(a[k], t.w00, b[k], t.w10, c[k], t.w01, d[k], t.w11);
                        float4 lv = f4_lerp2(la[k], t.tl.w0, lb[k], t.tl.w1);
                        float4 gl = f4_mul(g4[k], lv);      // dL/dP (interpolated)
                        float4 gp = f4_mul(g4[k], pv);      // dL/dL (interpolated)
                        if (t.w00 != 0.f) red_add_v4(G.plane[i] + t.o00 + q, f4_scale(gl, t.w00));
                        if (t.w10 != 0.f) red_add_v4(G.plane[i] + t.o10 + q, f4_scale(gl, t.w10));
                        if (t.w01 != 0.f) red_add_v4(G.plane[i] + t.o01 + q, f4_scale(gl, t.w01));
                        if (t.w11 != 0.f) red_add_v4(G.plane[i] + t.o11 + q, f4_scale(gl, t.w11));
                        if (t.tl.w0 != 0.f) red_add_v4(G.line[i] + t.ol0 + q, f4_scale(gp, t.tl.w0));
                        if (t.tl.w1 != 0.f) red_add_v4(G.line[i] + t.ol1 + q, f4_scale(gp, t.tl.w1));
                        // d/d index (ATen grid_sampler_2d_backward: out-of-range taps read as 0)
                        float4 dpx = f4_lerp2(f4_lerp2(b[k], t.tx.m1, a[k], -t.tx.m0), t.ty.w0,
                                              f4_lerp2(d[k], t.tx.m1, c[k], -t.tx.m0), t.ty.w1);
                        float4 dpy = f4_lerp2(f4_lerp2(c[k], t.ty.m1, a[k], -t.ty.m0), t.tx.w0,
                                              f4_lerp2(d[k], t.ty.m1, b[k], -t.ty.m0), t.tx.w1);
                        float4 dl = f4_lerp2(lb[k], t.tl.m1, la[k], -t.tl.m0);
                        sx += f4_dot(gl, dpx);
                        sy += f4_dot(gl, dpy);
                        sl += f4_dot(gp, dl);
                    }
                }
                du[mat0(i)] += sx * t.tx.scale;
                du[mat1(i)] += sy * t.ty.scale;
                du[vecm(i)] += sl * t.tl.scale;
            }
        }
        du[0] = quad_sum(du[0]); du[1] = quad_sum(du[1]); du[2] = quad_sum(du[2]);
        if (act && sub == 0 && dsamp) {
            float4 v = make_float4(du[0], du[1], du[2], 0.f);
            if (accumulate) { float4 o = dsamp[j]; v.x += o.x; v.y += o.y; v.z += o.z; }
            dsamp[j] = v;
        }
    }
}

static int grid_for(int n_hint) {
    long long want = ((long long)n_hint + 63) / 64;            // 64 samples per CTA pass
    long long cap = (long long)kNumSMs * 8;
    long long g = want < cap ? want : cap;
    return (int)(g < 1 ? 1 : g);
}

}  // namespace jt

using namespace jt;

extern "C" int jt_vm_gather_fwd(int app, const void* const* h_factors, const int* h_dims, const float* samp,
                                const int* slot, const int* n_dev, int n_max, float* out, cudaStream_t stream) {
    JT_CHECK_ARG(h_factors && h_dims && samp && out);
    if (n_max <= 0) return JT_OK;
    Factors F;
    if (int rc = fill_factors(F, h_factors, h_dims)) return rc;
    bool dens16 = !app;                            // density, 16 channels per plane: vm_density16_fwd_kernel
    for (int i = 0; i < 3; ++i)
        dens16 = dens16 && F.C[i] == 16 && (long long)F.H[i] * F.W[i] * 16 < 2147483647LL && F.L[i] < (1 << 26);
    // the same CTA passes over the sample list: 16 samples per warp instead of 8
    int grid = dens16 ? grid_for((n_max + 1) / 2) : grid_for(n_max);
    g_launches += 1;
    const float4* sp = reinterpret_cast<const float4*>(samp);
    if (app && F.bf16) vm_fwd_kernel<true, true><<<grid, 256, 0, stream>>>(F, sp, slot, n_dev, n_max, out);
    else if (app) vm_fwd_kernel<true, false><<<grid, 256, 0, stream>>>(F, sp, slot, n_dev, n_max, out);
    else if (dens16 && F.bf16) vm_density16_fwd_kernel<true><<<grid, 256, 0, stream>>>(F, sp, slot, n_dev, n_max, out);
    else if (dens16) vm_density16_fwd_kernel<false><<<grid, 256, 0, stream>>>(F, sp, slot, n_dev, n_max, out);
    else if (F.bf16) vm_fwd_kernel<false, true><<<grid, 256, 0, stream>>>(F, sp, slot, n_dev, n_max, out);
    else vm_fwd_kernel<false, false><<<grid, 256, 0, stream>>>(F, sp, slot, n_dev, n_max, out);
    JT_RETURN_LAUNCH();
}

extern "C" int jt_vm_gather_bwd(int app, const void* const* h_factors, void* const* h_factor_grads,
                                const int* h_dims, const float* samp, const int* slot, const int* n_dev,
                                int n_max, const float* gin, float* dsamp, int accumulate, cudaStream_t stream) {
    JT_CHECK_ARG(h_factors && h_factor_grads && h_dims && samp && gin);
    if (n_max <= 0) return JT_OK;
    Factors F;
    if (int rc = fill_factors(F, h_factors, h_dims)) return rc;
    if (F.bf16) return JT_ERR_UNSUPPORTED;          // the standalone feature ops differentiate the fp32 master factors
    FactorGrads G;
    for (int i = 0; i < 3; ++i) {
        G.plane[i] = static_cast<float*>(h_factor_grads[i]);
        G.line[i] = static_cast<float*>(h_factor_grads[3 + i]);
        JT_CHECK_ARG(G.plane[i] && G.line[i]);
    }
    int grid = grid_for(n_max);
    g_launches += 1;
    const float4* sp = reinterpret_cast<const float4*>(samp);
    float4* dp = reinterpret_cast<float4*>(dsamp);
    int qi = 0;                                   // uniform channel count in {16, 32, 48} -> unrolled variant
    if (F.C[0] == F.C[1] && F.C[1] == F.C[2] && F.C[0] % 16 == 0 && F.C[0] <= 48) qi = F.C[0] / 16;
    static const char* env_qi = getenv("JT_VM_BWD_QI");       // tuning override: 0 forces the generic loop
    if (env_qi && atoi(env_qi) == 0) qi = 0;
#define JT_BWD(APPV, QIV) vm_bwd_kernel<APPV, QIV><<<grid, 256, 0, stream>>>(F, G, sp, slot, n_dev, n_max, gin, dp, accumulate)
    if (app) { if (qi == 3) JT_BWD(true, 3); else if (qi == 2) JT_BWD(true, 2); else if (qi == 1) JT_BWD(true, 1); else JT_BWD(true, 0); }
    else { if (qi == 3) JT_BWD(false, 3); else if (qi == 2) JT_BWD(false, 2); else if (qi == 1) JT_BWD(false, 1); else JT_BWD(false, 0); }
#undef JT_BWD
    JT_RETURN_LAUNCH();
}
