// Density and its spatial gradient at points (forward mode, no atomics): sigma = density_act(feat + shift) and
// d sigma / d x, where feat = sum_i sum_c plane_i,c(u) * line_i,c(u) is the piecewise-multilinear function that
// grid_sample(bilinear, align_corners=True, zeros) evaluates and u = (x - aabb0) * inv - 1 (normalize_coord). Inside a
// cell the derivative of a bilinear tap along its x axis is (size-1)/2 * [(p10 - p00) wy0 + (p11 - p01) wy1], with
// out-of-range taps read as 0 (Tap::m0 / m1), the same for the y axis and the line; per channel the product rule
// d(P L) = dP L + P dL. Used by compute_density_grad / compute_normals (explicit points) and render_normals
// (compacted samples). The feature sums keep field_alpha_kernel's order, so 1 - exp(-sigma * len) is bit-identical
// to jt_field_alpha.
#include "jt_common.cuh"
#include "vm_taps.cuh"
#include "../../include/jt_vm.h"

namespace jt {

struct GradArgs {
    const float* xyz;            // explicit points [n][3], or NULL: samp records
    const float4* samp;          // normalised coordinates (xyz of each record)
    const int* slot;             // element e reads samp[slot[e]] (NULL: samp[e])
    const int* n_dev;
    long long n_max;
    float shift;
    int act, use_mask, normals;
};

// One channel quad of plane / line pair i from its six taps: feature into feat; d/d index along the plane's x, y and
// the line's axis into sx, sy, sl (ATen grid_sampler_2d_backward's form, as vm_bwd_kernel has it). T: PlaneTaps or
// Cell16 (weights and Tap records).
template <class T>
__device__ __forceinline__ void grad_quad(const T& t, float4 a, float4 b, float4 c, float4 d, float4 la, float4 lb,
                                          float& feat, float& sx, float& sy, float& sl) {
    const float4 pv = f4_bilin(a, t.w00, b, t.w10, c, t.w01, d, t.w11);
    const float4 lv = f4_lerp2(la, t.tl.w0, lb, t.tl.w1);
    feat += f4_dot(pv, lv);
    const float4 dpx = f4_lerp2(f4_lerp2(b, t.tx.m1, a, -t.tx.m0), t.ty.w0, f4_lerp2(d, t.tx.m1, c, -t.tx.m0), t.ty.w1);
    const float4 dpy = f4_lerp2(f4_lerp2(c, t.ty.m1, a, -t.ty.m0), t.tx.w0, f4_lerp2(d, t.ty.m1, b, -t.ty.m0), t.tx.w1);
    const float4 dl = f4_lerp2(lb, t.tl.m1, la, -t.tl.m0);
    sx += f4_dot(lv, dpx);
    sy += f4_dot(lv, dpy);
    sl += f4_dot(pv, dl);
}

// Tap setup of a 16-channel plane / line pair with 32-bit element offsets (the host checks H W 16 < 2^31), as
// dens16_plane has it: half the address registers of PlaneTaps.
struct Cell16 {
    Tap tx, ty, tl;
    float w00, w10, w01, w11;
    unsigned o00, o10, o01, o11, ol0, ol1;
};
__device__ __forceinline__ Cell16 cell16(const Factors& F, int i, const float u[3]) {
    Cell16 t;
    t.tx = make_tap(u[mat0(i)], F.W[i]); t.ty = make_tap(u[mat1(i)], F.H[i]); t.tl = make_tap(u[vecm(i)], F.L[i]);
    const unsigned W = (unsigned)F.W[i];
    const unsigned r0 = (unsigned)t.ty.i0 * W, r1 = (unsigned)t.ty.i1 * W;
    t.o00 = (r0 + t.tx.i0) * 16u; t.o10 = (r0 + t.tx.i1) * 16u;
    t.o01 = (r1 + t.tx.i0) * 16u; t.o11 = (r1 + t.tx.i1) * 16u;
    t.ol0 = (unsigned)t.tl.i0 * 16u; t.ol1 = (unsigned)t.tl.i1 * 16u;
    t.w00 = t.tx.w0 * t.ty.w0; t.w10 = t.tx.w1 * t.ty.w0;
    t.w01 = t.tx.w0 * t.ty.w1; t.w11 = t.tx.w1 * t.ty.w1;
    return t;
}

// Point e's normalised coordinate, and whether the occupancy mask keeps it (explicit points only: compacted samples
// were culled by the marcher).
__device__ __forceinline__ bool grad_point(const Geom& G, const MaskGeom& M, const GradArgs& A, long long e, float u[3]) {
    if (A.xyz) {
        const float p[3] = {A.xyz[3 * e], A.xyz[3 * e + 1], A.xyz[3 * e + 2]};
        if (A.use_mask && !mask_keep(M, p)) return false;
#pragma unroll
        for (int a = 0; a < 3; ++a) u[a] = __fsub_rn(__fmul_rn(__fsub_rn(p[a], G.a0[a]), G.inv[a]), 1.0f);
    } else {
        const float4 u4 = A.samp[A.slot ? A.slot[e] : e];
        u[0] = u4.x; u[1] = u4.y; u[2] = u4.z;
    }
    return true;
}

// -g / |g| in a scale-free form (no overflow or underflow of the squares); 0 where g is 0 or not finite.
__device__ __forceinline__ void outward_normal(float g[3]) {
    const float m = fmaxf(fabsf(g[0]), fmaxf(fabsf(g[1]), fabsf(g[2])));
    if (!(m > 0.0f) || !isfinite(m) || !isfinite(g[0]) || !isfinite(g[1]) || !isfinite(g[2])) {
        g[0] = g[1] = g[2] = 0.0f;
        return;
    }
    const float s0 = g[0] / m, s1 = g[1] / m, s2 = g[2] / m;
    const float len = sqrtf(s0 * s0 + s1 * s1 + s2 * s2);
    g[0] = -s0 / len; g[1] = -s1 / len; g[2] = -s2 / len;
}

// The first lane of point e writes sigma and d sigma / dx = act'(feat + shift) * dfeat/du * inv (or the unit normal).
__device__ __forceinline__ void grad_store(const Geom& G, const GradArgs& A, long long e, bool keep, float feat,
                                           const float du[3], float* __restrict__ sigma, float* __restrict__ grad) {
    const float x = feat + A.shift;
    const float dact = keep ? density_act_grad(x, A.act) : 0.0f;
    if (sigma) sigma[e] = keep ? density_act(x, A.act) : 0.0f;
    float g[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) g[a] = dact * du[a] * G.inv[a];
    if (A.normals) outward_normal(g);
    grad[3 * e] = g[0]; grad[3 * e + 1] = g[1]; grad[3 * e + 2] = g[2];
}

// Any channel count: 4 lanes per point (lane `sub` owns quads sub, sub + 4, ..), 8 points per warp -- the layout and
// the summation order of field_alpha_kernel.
__global__ void __launch_bounds__(256) density_grad_kernel(Factors F, Geom G, MaskGeom M, GradArgs A,
                                                           float* __restrict__ sigma, float* __restrict__ grad) {
    const long long n = A.n_dev ? *A.n_dev : A.n_max;
    const int lane = threadIdx.x & 31, sub = lane & 3, grp = lane >> 2;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long base = warp * 8; base < n; base += nwarps * 8) {
        const long long e = base + grp;
        const bool act = e < n;
        float feat = 0.f, du[3] = {0.f, 0.f, 0.f};
        bool keep = false;
        if (act) {
            float u[3];
            keep = grad_point(G, M, A, e, u);
            if (keep) {
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    const PlaneTaps t = plane_taps(F, i, u);
                    float sx = 0.f, sy = 0.f, sl = 0.f;
                    for (int q = sub * 4; q < F.C[i]; q += 16)
                        grad_quad(t, ldg4(t.p00 + q), ldg4(t.p10 + q), ldg4(t.p01 + q), ldg4(t.p11 + q), ldg4(t.l0 + q),
                                  ldg4(t.l1 + q), feat, sx, sy, sl);
                    du[mat0(i)] += sx * t.tx.scale;
                    du[mat1(i)] += sy * t.ty.scale;
                    du[vecm(i)] += sl * t.tl.scale;
                }
            }
        }
        feat = quad_sum(feat);
        du[0] = quad_sum(du[0]); du[1] = quad_sum(du[1]); du[2] = quad_sum(du[2]);
        if (act && sub == 0) grad_store(G, A, e, keep, feat, du, sigma, grad);
    }
}

// 16 channels per plane (every shipped config): 2 lanes per point, lane h owns quads 2h and 2h + 1, 16 points per
// warp -- vm_density16_fwd_kernel's layout. Per quad k the feature is a_k = ((0 + dot_0k) + dot_1k) + dot_2k over the
// planes, then (a_0 + a_1) + (a_2 + a_3): field_alpha_kernel's order, so sigma is bit-identical to it.
__global__ void __launch_bounds__(256, 3) density16_grad_kernel(Factors F, Geom G, MaskGeom M, GradArgs A,
                                                                float* __restrict__ sigma, float* __restrict__ grad) {
    const long long n = A.n_dev ? *A.n_dev : A.n_max;
    const int lane = threadIdx.x & 31, h = lane & 1, grp = lane >> 1;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long base = warp * 16; base < n; base += nwarps * 16) {
        const long long e = base + grp;
        const bool act = e < n;
        float a0 = 0.f, a1 = 0.f, du[3] = {0.f, 0.f, 0.f};
        bool keep = false;
        if (act) {
            float u[3];
            keep = grad_point(G, M, A, e, u);
            if (keep) {
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    const Cell16 t = cell16(F, i, u);
                    const float* P = F.plane[i];
                    const float* Ln = F.line[i];
                    const unsigned q = h * 8;
                    float4 a[2], b[2], c[2], d[2], la[2], lb[2];
#pragma unroll
                    for (int k = 0; k < 2; ++k) {          // all twelve loads of the plane in flight at once
                        a[k] = ldg4(P + t.o00 + q + 4 * k); b[k] = ldg4(P + t.o10 + q + 4 * k);
                        c[k] = ldg4(P + t.o01 + q + 4 * k); d[k] = ldg4(P + t.o11 + q + 4 * k);
                        la[k] = ldg4(Ln + t.ol0 + q + 4 * k); lb[k] = ldg4(Ln + t.ol1 + q + 4 * k);
                    }
                    float sx = 0.f, sy = 0.f, sl = 0.f;
                    grad_quad(t, a[0], b[0], c[0], d[0], la[0], lb[0], a0, sx, sy, sl);
                    grad_quad(t, a[1], b[1], c[1], d[1], la[1], lb[1], a1, sx, sy, sl);
                    du[mat0(i)] += sx * t.tx.scale;
                    du[mat1(i)] += sy * t.ty.scale;
                    du[vecm(i)] += sl * t.tl.scale;
                }
            }
        }
        float feat = a0 + a1;
        feat += __shfl_xor_sync(0xffffffffu, feat, 1);
#pragma unroll
        for (int a = 0; a < 3; ++a) du[a] += __shfl_xor_sync(0xffffffffu, du[a], 1);
        if (act && h == 0) grad_store(G, A, e, keep, feat, du, sigma, grad);
    }
}

}  // namespace jt

using namespace jt;

extern "C" int jt_field_density_grad(const void* const* h_factors, const int* h_dims, const float* h_geom,
                                     const float* xyz, const float* samp, const int* slot, const int* n_dev,
                                     long long n_max, const uint32_t* mask_bits, const int* h_mask_dims,
                                     const float* h_mask_geom, float density_shift, int act, int normals,
                                     float* sigma, float* grad, cudaStream_t stream) {
    JT_CHECK_ARG(h_factors && h_dims && h_geom && grad);
    JT_CHECK_ARG((xyz != nullptr) != (samp != nullptr));
    JT_CHECK_ARG(!xyz || (!slot && !n_dev));                // explicit points: n_max is the count
    JT_CHECK_ARG(!mask_bits || (xyz && h_mask_dims && h_mask_geom));
    JT_CHECK_ARG(act == 0 || act == 1);
    if (n_max <= 0) return JT_OK;
    Factors F;
    if (int rc = fill_factors(F, h_factors, h_dims)) return rc;
    if (F.bf16) return JT_ERR_UNSUPPORTED;          // geometry queries read the fp32 master factors
    GradArgs A{};
    A.xyz = xyz; A.samp = reinterpret_cast<const float4*>(samp); A.slot = slot; A.n_dev = n_dev; A.n_max = n_max;
    A.shift = density_shift; A.act = act; A.use_mask = mask_bits != nullptr; A.normals = normals ? 1 : 0;
    Geom G = make_geom(h_geom);
    MaskGeom M = make_mask(mask_bits, h_mask_dims, h_mask_geom);
    bool c16 = true;
    for (int i = 0; i < 3; ++i) c16 = c16 && F.C[i] == 16 && (long long)F.H[i] * F.W[i] * 16 < 2147483647LL && F.L[i] < (1 << 26);
    const long long per_block = c16 ? 128 : 64;                // points per 256-thread block and pass
    const long long blocks = (n_max + per_block - 1) / per_block;
    const int grid = (int)(blocks < (long long)kNumSMs * 16 ? blocks : (long long)kNumSMs * 16);
    if (c16) density16_grad_kernel<<<grid, 256, 0, stream>>>(F, G, M, A, sigma, grad);
    else density_grad_kernel<<<grid, 256, 0, stream>>>(F, G, M, A, sigma, grad);
    ++g_launches;
    JT_RETURN_LAUNCH();
}
