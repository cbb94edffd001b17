// Ray casting against the field's surface: the first point of each ray where compute_alpha(p, length) >= level
// (the level set extract_mesh contours), on the forward's own sample depths, refined to the first crossing between
// the hit sample and the one before it.
//
// One warp per ray. Sample phase: the warp tests 32 / LPS consecutive samples per iteration (LPS lanes per sample:
// 2 with 16 channels on every plane, vm_density16_fwd_kernel's layout through dens16_plane; 4 otherwise,
// field_alpha_kernel's loop), and a ballot of the predicate gives the first inside sample. Points, the box test and
// the alpha sums are the marcher's and jt_field_alpha's bit for bit (vm_taps.cuh), so the hit sample is the first
// sample of the no-grad forward whose compute_alpha reaches the level. Refinement: the same warp evaluates 32 / LPS - 1
// equally spaced interior points of the bracket [t_{k-1}, t_k] per round and keeps the first inside point and the one
// before it -- the first crossing at a finer resolution, not bisection, which could settle on a later root.
#include "jt_common.cuh"
#include "vm_taps.cuh"
#include "../../include/jt_vm.h"

namespace jt {

struct CastArgs {
    const float* ro;
    const float* rd;
    const float* ztab;           // NDC depth table [S], or NULL: metric rays
    int* ctr;                    // zeroed ray counter (rays handed out by atomics), or NULL: static grid stride
    int n_rays, S, act, use_mask;
    float shift, length, level;
};

constexpr int kMaxRounds = 64;   // a round always shrinks the bracket; fp32 ends it within ~8 rounds

// The predicate at point p for the LPS lanes of one sample (all 32 lanes call it: it shuffles): in the box
// (point_in_box's result `inb`), kept by the occupancy mask and 1 - exp(-sigma * length) >= level with
// jt_field_alpha's taps and summation order. Lanes out of the box or masked issue no tap loads.
template <int LPS>
__device__ __forceinline__ bool cast_inside(const Factors& F, const Geom& G, const MaskGeom& M, const CastArgs& A,
                                            bool inb, const float p[3], int sub) {
    const bool live = inb && (!A.use_mask || mask_keep(M, p));
    float u[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) u[a] = __fsub_rn(__fmul_rn(__fsub_rn(p[a], G.a0[a]), G.inv[a]), 1.0f);
    float acc;
    if (LPS == 2) {
        float a0 = 0.f, a1 = 0.f;
        if (live) {
#pragma unroll
            for (int i = 0; i < 3; ++i) dens16_plane<false>(F, i, u, sub * 8, a0, a1);
        }
        acc = a0 + a1;
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    } else {
        acc = 0.f;
        if (live) {
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const PlaneTaps t = plane_taps(F, i, u);
                const int C = F.C[i];
                for (int q = sub * 4; q < C; q += 16) {
                    float4 a = ldg4(t.p00 + q), b = ldg4(t.p10 + q), c = ldg4(t.p01 + q), d = ldg4(t.p11 + q);
                    float4 la = ldg4(t.l0 + q), lb = ldg4(t.l1 + q);
                    acc += f4_dot(f4_bilin(a, t.w00, b, t.w10, c, t.w01, d, t.w11), f4_lerp2(la, t.tl.w0, lb, t.tl.w1));
                }
            }
        }
        acc = quad_sum(acc);
    }
    const float sigma = live ? density_act(acc + A.shift, A.act) : 0.0f;
    return live && 1.0f - exp_neg(-sigma * A.length) >= A.level;
}

template <int LPS>
__device__ __forceinline__ void cast_ray(const Factors& F, const Geom& G, const MaskGeom& M, const CastArgs& A, int r,
                                         float* __restrict__ t_out, float* __restrict__ xyz_out,
                                         int* __restrict__ k_out, int* __restrict__ rounds_out) {
    constexpr int SPI = 32 / LPS;                                   // samples (or sub-points) per iteration
    constexpr unsigned kLead = LPS == 2 ? 0x55555555u : 0x11111111u;   // the first lane of every sample
    const int lane = threadIdx.x & 31, sub = lane % LPS, grp = lane / LPS;
    const bool ndc = A.ztab != nullptr;
    const RaySetup s = load_ray(A.ro, A.rd, r, G, ndc);
    int hit = -1;
    float hi = 0.f;
    bool entered = false;
    for (int k0 = 0; k0 < A.S; k0 += SPI) {
        const int k = k0 + grp;
        float t = 0.f, p[3] = {0.f, 0.f, 0.f};
        bool inb = false;
        if (k < A.S) {
            t = sample_depth(s, G, k, 0.0f, A.ztab, ndc);
            inb = point_in_box(s, G, t, p);
        }
        const unsigned hb = __ballot_sync(0xffffffffu, cast_inside<LPS>(F, G, M, A, inb, p, sub)) & kLead;
        if (hb) {
            const int L = __ffs(hb) - 1;
            hit = k0 + L / LPS;
            hi = __shfl_sync(0xffffffffu, t, L);
            break;
        }
        // Metric rays: t_k increases with k and every coordinate of o + d t is monotone in t, so the samples in the
        // box are one run. Once the last sample of an iteration is out after one was in, no later sample is in.
        if (!ndc) {
            const unsigned ib = __ballot_sync(0xffffffffu, inb) & kLead;
            entered = entered || ib != 0u;
            const int last = LPS * (min(SPI, A.S - k0) - 1);
            if (entered && !((ib >> last) & 1u)) break;
        }
    }
    int rounds = 0;
    if (hit > 0) {
        float lo = sample_depth(s, G, hit - 1, 0.0f, A.ztab, ndc);
        const float stop = __fmul_rn(__fsub_rn(hi, lo), 0x1p-20f);
        const int j = grp + 1;                                      // interior points 1 .. SPI - 1; slot SPI idles
        while (__fsub_rn(hi, lo) > stop && nextafterf(lo, INFINITY) < hi && rounds < kMaxRounds) {
            const float w = __fmul_rn(__fsub_rn(hi, lo), 1.0f / SPI);
            const float tj = fminf(__fadd_rn(lo, __fmul_rn(w, (float)j)), hi);
            float q[3];
            const bool inb = point_in_box(s, G, tj, q) && j < SPI;
            const unsigned hb = __ballot_sync(0xffffffffu, cast_inside<LPS>(F, G, M, A, inb, q, sub)) & kLead;
            if (hb) {
                const int L = __ffs(hb) - 1;
                const float tp = __shfl_sync(0xffffffffu, tj, L >= LPS ? L - LPS : 0);
                hi = __shfl_sync(0xffffffffu, tj, L);
                if (L >= LPS) lo = tp;
            } else {
                lo = __shfl_sync(0xffffffffu, tj, LPS * (SPI - 2));
            }
            ++rounds;
        }
    }
    if (lane == 0) {
        float p[3] = {0.f, 0.f, 0.f};
        if (hit >= 0) point_in_box(s, G, hi, p);
        t_out[r] = hit >= 0 ? hi : INFINITY;
        xyz_out[3 * r] = p[0]; xyz_out[3 * r + 1] = p[1]; xyz_out[3 * r + 2] = p[2];
        k_out[r] = hit;
        if (rounds_out) rounds_out[r] = rounds;
    }
}

// Persistent grid, one warp per ray; rays come from an atomic counter (A.ctr) or a static grid stride. A ray's
// result depends on nothing but the ray, so the schedule does not change it.
template <int LPS>
__global__ void __launch_bounds__(256) raycast_kernel(Factors F, Geom G, MaskGeom M, CastArgs A,
                                                      float* __restrict__ t_out, float* __restrict__ xyz_out,
                                                      int* __restrict__ k_out, int* __restrict__ rounds_out) {
    const int lane = threadIdx.x & 31;
    const int stride = (gridDim.x * blockDim.x) >> 5;
    int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    for (;;) {
        if (A.ctr) {
            int v = 0;
            if (lane == 0) v = atomicAdd(A.ctr, 1);
            r = __shfl_sync(0xffffffffu, v, 0);
        }
        if (r >= A.n_rays) break;
        cast_ray<LPS>(F, G, M, A, r, t_out, xyz_out, k_out, rounds_out);
        if (!A.ctr) r += stride;
    }
}

template <int LPS>
int launch_raycast(const Factors& F, const Geom& G, const MaskGeom& M, const CastArgs& A, float* t, float* xyz,
                   int* k, int* rounds, cudaStream_t stream) {
    static int per_sm = 0;
    if (per_sm == 0 && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, raycast_kernel<LPS>, 256, 0) != cudaSuccess)
        return JT_ERR_LAUNCH;
    const long long blocks = ((long long)A.n_rays + 7) / 8;         // 8 warps per block
    const long long cap = (long long)kNumSMs * (per_sm > 0 ? per_sm : 1);
    raycast_kernel<LPS><<<(int)(blocks < cap ? blocks : cap), 256, 0, stream>>>(F, G, M, A, t, xyz, k, rounds);
    ++g_launches;
    JT_RETURN_LAUNCH();
}

}  // namespace jt

using namespace jt;

extern "C" int jt_raycast(const void* const* h_factors, const int* h_dims, const float* h_geom,
                          const uint32_t* mask_bits, const int* h_mask_dims, const float* h_mask_geom,
                          float density_shift, int act, float length, float level, const float* rays_o,
                          const float* rays_d, int n_rays, const float* ztab, int n_samples, int* work, float* t,
                          float* xyz, int* k, int* rounds, cudaStream_t stream) {
    JT_CHECK_ARG(h_factors && h_dims && h_geom && rays_o && rays_d && t && xyz && k);
    JT_CHECK_ARG(!mask_bits || (h_mask_dims && h_mask_geom));
    JT_CHECK_ARG(act == 0 || act == 1);
    JT_CHECK_ARG(level > 0.0f && level < 1.0f && n_samples > 0 && n_rays >= 0);
    Factors F;
    if (int rc = fill_factors(F, h_factors, h_dims)) return rc;
    if (F.bf16) return JT_ERR_UNSUPPORTED;          // geometry queries read the fp32 master factors
    if (n_rays == 0) return JT_OK;
    CastArgs A{};
    A.ro = rays_o; A.rd = rays_d; A.ztab = ztab; A.ctr = work;
    A.n_rays = n_rays; A.S = n_samples; A.act = act; A.use_mask = mask_bits != nullptr;
    A.shift = density_shift; A.length = length; A.level = level;
    const Geom G = make_geom(h_geom);
    const MaskGeom M = make_mask(mask_bits, h_mask_dims, h_mask_geom);
    bool c16 = true;
    for (int i = 0; i < 3; ++i) c16 = c16 && F.C[i] == 16 && (long long)F.H[i] * F.W[i] * 16 < 2147483647LL && F.L[i] < (1 << 26);
    return c16 ? launch_raycast<2>(F, G, M, A, t, xyz, k, rounds, stream)
               : launch_raycast<4>(F, G, M, A, t, xyz, k, rounds, stream);
}
