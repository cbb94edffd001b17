// Device helpers shared by the kernels that evaluate the VM field at a point: bilinear / linear tap setup on the
// channel-last factors (vm_gather.cu, field_maint.cu, field_grad.cu, raycast.cu), the ray sample points (march.cu,
// raycast.cu), the density activation (composite.cu, field_maint.cu) and the occupancy-mask test (march.cu,
// field_maint.cu).
#pragma once
#include "jt_common.cuh"

namespace jt {

__device__ __forceinline__ float4 f4_scale(float4 a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }
__device__ __forceinline__ float4 f4_mul(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float f4_dot(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
__device__ __forceinline__ float4 f4_lerp2(float4 a, float wa, float4 b, float wb) {
    return make_float4(a.x * wa + b.x * wb, a.y * wa + b.y * wb, a.z * wa + b.z * wb, a.w * wa + b.w * wb);
}
__device__ __forceinline__ float4 f4_bilin(float4 a, float wa, float4 b, float wb, float4 c, float wc, float4 d, float wd) {
    return make_float4(a.x * wa + b.x * wb + c.x * wc + d.x * wd, a.y * wa + b.y * wb + c.y * wc + d.y * wd,
                       a.z * wa + b.z * wb + c.z * wc + d.z * wd, a.w * wa + b.w * wb + c.w * wc + d.w * wd);
}

struct PlaneTaps {
    const float *p00, *p10, *p01, *p11, *l0, *l1;
    size_t o00, o10, o01, o11, ol0, ol1;     // element offsets (shared by value and gradient buffers)
    float w00, w10, w01, w11;
    Tap tx, ty, tl;
};

__device__ __forceinline__ PlaneTaps plane_taps(const Factors& F, int i, const float u[3]) {
    PlaneTaps t;
    t.tx = make_tap(u[mat0(i)], F.W[i]);
    t.ty = make_tap(u[mat1(i)], F.H[i]);
    t.tl = make_tap(u[vecm(i)], F.L[i]);
    const size_t C = F.C[i];
    size_t r0 = (size_t)t.ty.i0 * F.W[i], r1 = (size_t)t.ty.i1 * F.W[i];
    t.o00 = (r0 + t.tx.i0) * C; t.o10 = (r0 + t.tx.i1) * C;
    t.o01 = (r1 + t.tx.i0) * C; t.o11 = (r1 + t.tx.i1) * C;
    t.ol0 = (size_t)t.tl.i0 * C; t.ol1 = (size_t)t.tl.i1 * C;
    t.p00 = F.plane[i] + t.o00; t.p10 = F.plane[i] + t.o10;
    t.p01 = F.plane[i] + t.o01; t.p11 = F.plane[i] + t.o11;
    t.l0 = F.line[i] + t.ol0; t.l1 = F.line[i] + t.ol1;
    t.w00 = t.tx.w0 * t.ty.w0; t.w10 = t.tx.w1 * t.ty.w0;     // nw, ne
    t.w01 = t.tx.w0 * t.ty.w1; t.w11 = t.tx.w1 * t.ty.w1;     // sw, se
    return t;
}

// One channel-quad pair of a 16-channel plane / line pair i at normalised coordinate u: lane half q (0 or 8) adds
// quads q/4 and q/4 + 1 of the plane's dot product into a0 and a1, with 32-bit element offsets (the host checks
// H W 16 < 2^31). The density gather's 2-lanes-per-sample layout (vm_density16_fwd_kernel) and the ray caster's.
template <bool B16>
__device__ __forceinline__ void dens16_plane(const Factors& F, const int i, const float u[3], const int q,
                                             float& a0, float& a1) {
    const Tap tx = make_tap(u[mat0(i)], F.W[i]), ty = make_tap(u[mat1(i)], F.H[i]), tl = make_tap(u[vecm(i)], F.L[i]);
    const unsigned W = (unsigned)F.W[i];
    const unsigned r0 = (unsigned)ty.i0 * W, r1 = (unsigned)ty.i1 * W;
    const unsigned o00 = (r0 + tx.i0) * 16u + q, o10 = (r0 + tx.i1) * 16u + q;
    const unsigned o01 = (r1 + tx.i0) * 16u + q, o11 = (r1 + tx.i1) * 16u + q;
    const unsigned ol0 = (unsigned)tl.i0 * 16u + q, ol1 = (unsigned)tl.i1 * 16u + q;
    const float w00 = tx.w0 * ty.w0, w10 = tx.w1 * ty.w0, w01 = tx.w0 * ty.w1, w11 = tx.w1 * ty.w1;
    const float* P = F.plane[i];
    const float* Ln = F.line[i];
    float4 a[2], b[2], c[2], d[2], la[2], lb[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        a[k] = ld_tap4<B16>(P, o00 + 4 * k); b[k] = ld_tap4<B16>(P, o10 + 4 * k);
        c[k] = ld_tap4<B16>(P, o01 + 4 * k); d[k] = ld_tap4<B16>(P, o11 + 4 * k);
        la[k] = ld_tap4<B16>(Ln, ol0 + 4 * k); lb[k] = ld_tap4<B16>(Ln, ol1 + 4 * k);
    }
    a0 += f4_dot(f4_bilin(a[0], w00, b[0], w10, c[0], w01, d[0], w11), f4_lerp2(la[0], tl.w0, lb[0], tl.w1));
    a1 += f4_dot(f4_bilin(a[1], w00, b[1], w10, c[1], w01, d[1], w11), f4_lerp2(la[1], tl.w0, lb[1], tl.w1));
}

// ---- ray sampling (march.cu's marcher and raycast.cu's caster: the same points bit for bit)
struct RaySetup {
    float o[3], d[3];
    float tmin;      // metric rays only
    float norm;      // |d| (NDC rays scale dists by it), 1 for metric rays
};

__device__ __forceinline__ RaySetup load_ray(const float* __restrict__ ro, const float* __restrict__ rd, int r,
                                             const Geom& g, bool ndc) {
    RaySetup s;
#pragma unroll
    for (int a = 0; a < 3; ++a) { s.o[a] = ro[3 * r + a]; s.d[a] = rd[3 * r + a]; }
    s.tmin = 0.f;
    s.norm = 1.f;
    if (!ndc) {
        float tm = -INFINITY;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            float vec = (s.d[a] == 0.0f) ? 1e-6f : s.d[a];
            float ra = __fdiv_rn(__fsub_rn(g.a1[a], s.o[a]), vec);
            float rb = __fdiv_rn(__fsub_rn(g.a0[a], s.o[a]), vec);
            tm = fmaxf(tm, fminf(ra, rb));
        }
        s.tmin = fminf(fmaxf(tm, g.near_), g.far_);
    } else {
        s.norm = sqrtf(s.d[0] * s.d[0] + s.d[1] * s.d[1] + s.d[2] * s.d[2]);
    }
    return s;
}

// depth of sample k. metric: t_min + stepSize * (k + jitter); NDC: table lookup.
__device__ __forceinline__ float sample_depth(const RaySetup& s, const Geom& g, int k, float jit,
                                              const float* __restrict__ ztab, bool ndc) {
    if (ndc) return ztab[k];
    float rng = __fadd_rn((float)k, jit);
    return __fadd_rn(s.tmin, __fmul_rn(g.step, rng));
}

__device__ __forceinline__ bool point_in_box(const RaySetup& s, const Geom& g, float t, float p[3]) {
    bool ok = true;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        p[a] = __fadd_rn(s.o[a], __fmul_rn(s.d[a], t));
        ok = ok && !((g.a0[a] > p[a]) || (p[a] > g.a1[a]));
    }
    return ok;
}

// exp(x) for x <= 0 as the reference's alpha = 1 - exp(-sigma*dist) needs it (tensorBase.py:59): for a thin
// medium (x ~ -1e-4, every sample of a freshly initialised Blender field) alpha is the distance of exp(x) from 1 in
// units of 2^-24, so ONE ulp of exp() is 3e-4 of alpha. CUDA's expf is within 2 ulp but biased by ~0.3 ulp in this
// range (measured: every weight / appearance gradient of the 300^3 field was 1.7e-4 off the CPU reference, whose
// vectorised exp is correctly rounded 96 % of the time). 1 + expm1f(x) is a single rounding of an exact-enough
// increment, i.e. the correctly rounded exp(x), for |x| < 0.1; beyond that the amplification is gone.
__device__ __forceinline__ float exp_neg(float x) { return x > -0.1f ? 1.0f + expm1f(x) : expf(x); }

__device__ __forceinline__ float density_act(float x, int act) {
    // act 0: softplus (beta 1, threshold 20; ATen softplus), act 1: relu. x already includes the shift.
    if (act == 0) return x > 20.0f ? x : log1pf(expf(x));
    return fmaxf(x, 0.0f);
}
__device__ __forceinline__ float density_act_grad(float x, int act) {
    if (act == 0) {
        if (x > 20.0f) return 1.0f;
        float z = expf(x);
        return z / (z + 1.0f);
    }
    return x > 0.0f ? 1.0f : 0.0f;
}

// grid_sample(volume, trilinear, align_corners=True, zeros) > 0 for a {0,1}
// volume  <=>  some in-range corner with a set bit has three positive 1-D
// weights (all 8 terms are non-negative). Index arithmetic follows ATen's
// scalar path ((u + 1) / 2) * (size - 1) with separately rounded ops.
__device__ __forceinline__ bool mask_keep(const MaskGeom& m, const float p[3]) {
    int i0[3];
    bool frac[3];
    const int size[3] = {m.W, m.H, m.D};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        float u = __fsub_rn(__fmul_rn(__fsub_rn(p[a], m.a0[a]), m.inv[a]), 1.0f);
        float x = __fmul_rn(__fdiv_rn(__fadd_rn(u, 1.0f), 2.0f), (float)(size[a] - 1));
        float xf = floorf(x);
        frac[a] = (x - xf) > 0.0f;                 // weight of the +1 corner is positive
        i0[a] = (int)fminf(fmaxf(xf, -2.0f), (float)size[a]);
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        int dx = c & 1, dy = (c >> 1) & 1, dz = c >> 2;
        if ((dx && !frac[0]) || (dy && !frac[1]) || (dz && !frac[2])) continue;
        int x = i0[0] + dx, y = i0[1] + dy, z = i0[2] + dz;
        if (x < 0 || x >= m.W || y < 0 || y >= m.H || z < 0 || z >= m.D) continue;
        long long n = ((long long)z * m.H + y) * m.W + x;
        if ((m.bits[n >> 5] >> (n & 31)) & 1u) return true;
    }
    return false;
}

// host: unpack h_geom / the mask description of the C ABI (include/jt_vm.h "Layouts")
inline Geom make_geom(const float* h) {
    Geom g;
    for (int a = 0; a < 3; ++a) { g.a0[a] = h[a]; g.a1[a] = h[3 + a]; g.inv[a] = h[6 + a]; }
    g.step = h[9]; g.near_ = h[10]; g.far_ = h[11];
    return g;
}
inline MaskGeom make_mask(const uint32_t* bits, const int* dims, const float* hg) {
    MaskGeom m{};
    m.bits = bits;
    if (bits) {
        m.W = dims[0]; m.H = dims[1]; m.D = dims[2];
        for (int a = 0; a < 3; ++a) { m.a0[a] = hg[a]; m.inv[a] = hg[3 + a]; }
    }
    return m;
}

}  // namespace jt
