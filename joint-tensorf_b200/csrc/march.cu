// K1 -- ray marching (sample_ray / sample_ray_ndc), AABB + alpha-mask culling and
// warp-level compaction of the valid samples.
//
// Replaces reference TensorBase.sample_ray (tensorBase.py:572-612),
// sample_ray_ndc (tensorBase.py:554-571), the alpha-mask culling block
// (batBase.py:76-82 -> AlphaGridMask.sample_alpha tensorBase.py:91-98), the
// boolean-mask indexing that follows it (batBase.py:104-120) and
// normalize_coord (tensorBase.py:502-503).
//
// Bit-exact class: every operation that feeds the in-box test is issued as a
// separately rounded IEEE fp32 op (__fadd_rn/__fmul_rn/__fdiv_rn are never
// contracted into FMAs), in the reference's order, so the valid mask equals the
// reference's bit for bit. The jitter (torch RNG) and the NDC depth table
// (torch.linspace) are inputs, never recomputed here.
#include "jt_common.cuh"
#include "vm_taps.cuh"
#include "../../include/jt_vm.h"

namespace jt {

// RaySetup, load_ray, sample_depth and point_in_box live in vm_taps.cuh (the ray caster samples the same points).

// ---------------------------------------------------------------- dense variant (API parity)
__global__ void sample_dense_kernel(const float* __restrict__ ro, const float* __restrict__ rd,
                                    const float* __restrict__ aux, int ndc, int n_rays, int S, Geom g,
                                    MaskGeom m, int use_mask, float* __restrict__ pts, float* __restrict__ z,
                                    uint8_t* __restrict__ valid) {
    int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (warp >= n_rays) return;
    RaySetup s = load_ray(ro, rd, warp, g, ndc);
    float jit = (!ndc && aux) ? aux[warp] : 0.0f;
    for (int k = lane; k < S; k += 32) {
        float t = sample_depth(s, g, k, jit, aux, ndc);
        float p[3];
        bool ok = point_in_box(s, g, t, p);
        if (ok && use_mask) ok = mask_keep(m, p);
        size_t e = (size_t)warp * S + k;
        pts[3 * e + 0] = p[0]; pts[3 * e + 1] = p[1]; pts[3 * e + 2] = p[2];
        z[e] = t;
        valid[e] = ok ? 1 : 0;
    }
}

// ---------------------------------------------------------------- compaction, pass 1: count
__global__ void march_count_kernel(const float* __restrict__ ro, const float* __restrict__ rd,
                                   const float* __restrict__ aux, int ndc, int n_rays, int S, Geom g,
                                   MaskGeom m, int use_mask, int* __restrict__ cnt) {
    int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (warp >= n_rays) return;
    RaySetup s = load_ray(ro, rd, warp, g, ndc);
    float jit = (!ndc && aux) ? aux[warp] : 0.0f;
    int c = 0;
    for (int k0 = 0; k0 < S; k0 += 32) {
        int k = k0 + lane;
        bool ok = false;
        if (k < S) {
            float t = sample_depth(s, g, k, jit, aux, ndc);
            float p[3];
            ok = point_in_box(s, g, t, p);
            if (ok && use_mask) ok = mask_keep(m, p);
        }
        c += __popc(__ballot_sync(0xffffffffu, ok));
    }
    if (lane == 0) cnt[warp] = c;
}

// Exclusive scan of n ints by ONE CTA (n is the ray count: 4096 per training
// batch). off has n+1 entries; off[n] is the total.
__global__ void exclusive_scan_kernel(const int* __restrict__ cnt, int* __restrict__ off, int n) {
    __shared__ int part[1024];
    int tid = threadIdx.x;
    int per = (n + blockDim.x - 1) / blockDim.x;
    int b = tid * per, e = min(b + per, n);
    int s = 0;
    for (int i = b; i < e; ++i) s += cnt[i];
    part[tid] = s;
    __syncthreads();
    for (int o = 1; o < blockDim.x; o <<= 1) {         // Hillis-Steele inclusive scan
        int v = (tid >= o) ? part[tid - o] : 0;
        __syncthreads();
        part[tid] += v;
        __syncthreads();
    }
    int run = part[tid] - s;
    for (int i = b; i < e; ++i) { off[i] = run; run += cnt[i]; }
    if (tid == blockDim.x - 1) off[n] = part[tid];
}

// ---------------------------------------------------------------- compaction, pass 2: fill
// One warp per ray; ballot + popc give each valid sample its slot, so the list
// is ray-major and depth-ordered (deterministic, equal to nonzero(mask)).
__global__ void march_fill_kernel(const float* __restrict__ ro, const float* __restrict__ rd,
                                  const float* __restrict__ aux, int ndc, int n_rays, int S, Geom g,
                                  MaskGeom m, int use_mask, const int* __restrict__ off,
                                  int* __restrict__ sidx, float4* __restrict__ samp, float* __restrict__ dist) {
    int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (warp >= n_rays) return;
    RaySetup s = load_ray(ro, rd, warp, g, ndc);
    float jit = (!ndc && aux) ? aux[warp] : 0.0f;
    int base = off[warp];
    for (int k0 = 0; k0 < S; k0 += 32) {
        int k = k0 + lane;
        bool ok = false;
        float t = 0.f, p[3] = {0.f, 0.f, 0.f};
        if (k < S) {
            t = sample_depth(s, g, k, jit, aux, ndc);
            ok = point_in_box(s, g, t, p);
            if (ok && use_mask) ok = mask_keep(m, p);
        }
        unsigned b = __ballot_sync(0xffffffffu, ok);
        if (ok) {
            int j = base + __popc(b & ((1u << lane) - 1u));
            float4 v;
            v.x = __fsub_rn(__fmul_rn(__fsub_rn(p[0], g.a0[0]), g.inv[0]), 1.0f);   // normalize_coord
            v.y = __fsub_rn(__fmul_rn(__fsub_rn(p[1], g.a0[1]), g.inv[1]), 1.0f);
            v.z = __fsub_rn(__fmul_rn(__fsub_rn(p[2], g.a0[2]), g.inv[2]), 1.0f);
            v.w = t;
            float dz = 0.0f;                               // last sample: dist = 0 (batBase.py:69)
            if (k + 1 < S) dz = __fsub_rn(sample_depth(s, g, k + 1, jit, aux, ndc), t);
            sidx[j] = warp * S + k;
            samp[j] = v;
            dist[j] = dz * s.norm;
        }
        base += __popc(b);
    }
}

}  // namespace jt

using namespace jt;

extern "C" int jt_sample_ray_dense(const float* rays_o, const float* rays_d, const float* aux, int ndc,
                                   int n_rays, int n_samples, const float* h_geom, const uint32_t* mask_bits,
                                   const int* h_mask_dims, const float* h_mask_geom, float* pts, float* z,
                                   uint8_t* valid, cudaStream_t stream) {
    JT_CHECK_ARG(rays_o && rays_d && h_geom && pts && z && valid && n_samples > 0);
    JT_CHECK_ARG(!ndc || aux);
    JT_CHECK_ARG(!mask_bits || (h_mask_dims && h_mask_geom));
    if (n_rays <= 0) return JT_OK;
    Geom g = make_geom(h_geom);
    MaskGeom m = make_mask(mask_bits, h_mask_dims, h_mask_geom);
    int blocks = (n_rays + 7) / 8;
    g_launches += 1;
    sample_dense_kernel<<<blocks, 256, 0, stream>>>(rays_o, rays_d, aux, ndc, n_rays, n_samples, g, m,
                                                    mask_bits != nullptr, pts, z, valid);
    JT_RETURN_LAUNCH();
}

extern "C" int jt_march_compact(const float* rays_o, const float* rays_d, const float* aux, int ndc, int n_rays,
                                int n_samples, const float* h_geom, const uint32_t* mask_bits,
                                const int* h_mask_dims, const float* h_mask_geom, int* ray_cnt, int* ray_off,
                                int* sidx, float* samp, float* dist, cudaStream_t stream) {
    JT_CHECK_ARG(rays_o && rays_d && h_geom && ray_cnt && ray_off && sidx && samp && dist && n_samples > 0);
    JT_CHECK_ARG(!ndc || aux);
    JT_CHECK_ARG(!mask_bits || (h_mask_dims && h_mask_geom));
    JT_CHECK_ARG((long long)n_rays * n_samples < 2147483647LL);
    if (n_rays <= 0) return JT_OK;
    Geom g = make_geom(h_geom);
    MaskGeom m = make_mask(mask_bits, h_mask_dims, h_mask_geom);
    int blocks = (n_rays + 7) / 8;
    int um = mask_bits != nullptr;
    g_launches += 3;
    march_count_kernel<<<blocks, 256, 0, stream>>>(rays_o, rays_d, aux, ndc, n_rays, n_samples, g, m, um, ray_cnt);
    exclusive_scan_kernel<<<1, 1024, 0, stream>>>(ray_cnt, ray_off, n_rays);
    march_fill_kernel<<<blocks, 256, 0, stream>>>(rays_o, rays_d, aux, ndc, n_rays, n_samples, g, m, um, ray_off,
                                                  sidx, reinterpret_cast<float4*>(samp), dist);
    JT_RETURN_LAUNCH();
}

extern "C" int jt_exclusive_scan(const int* cnt, int* off, int n, cudaStream_t stream) {
    JT_CHECK_ARG(cnt && off && n > 0);
    g_launches += 1;
    exclusive_scan_kernel<<<1, 1024, 0, stream>>>(cnt, off, n);
    JT_RETURN_LAUNCH();
}
