// K2 backward, ray-walking form -- factor-gradient scatter with per-cell run merging.
//
// Replaces the 12 grid_sampler_2d_backward calls of one training step (autograd of
// bateRF.py:81-82,124-127 / tensoRF.py:245-248,263-266) plus the autograd of
// `rays_pts = o + d * t` / normalize_coord (tensorBase.py:502-503,597) that turns the
// coordinate gradients into d/d rays_o, d/d rays_d for the pose optimisation.
//
// Why a second scatter kernel: vm_bwd_kernel (vm_gather.cu) issues one 16-byte RED per
// (sample, tap, channel quad) and is bound by the LSU's RED rate (~1.3 cycles per lane-op
// per SM; 216 lane-ops per appearance sample). The marcher steps half a voxel
// (step_ratio 0.5, tensorBase.py:483-484), so consecutive samples of a ray stay in the
// same bilinear cell of a plane for ~2.1 samples and in the same line cell for ~3.9
// (measured on the cfg2 batch). Here a *walker* (C/4 lanes, one channel quad each) walks a
// segment of consecutive samples of the compacted, ray-major list, keeps the four corner
// gradients and the two line gradients of the current cell in registers, and flushes
// them with REDs only when the cell changes: 2.6 instead of 6 RED units per sample and
// plane, and the tap values are re-loaded only on a cell change as well.
// The coordinate gradient is reduced per ray in registers (sum_j du_j and sum_j du_j t_j
// are all the pose gradient needs) and flushed once per ray segment, so no per-sample
// dL/du array is written and no separate ray_bwd pass is needed.
#include <limits.h>
#include <stdlib.h>
#include <type_traits>
#include "jt_common.cuh"
#include "../../include/jt_vm.h"

namespace jt {

// Packed fp32 arithmetic (sm_100 FFMA2 / FMUL2: two IEEE fp32 operations per instruction and per fma-pipe
// slot). The walker is bound by instruction issue at ~2 warps per scheduler, and scalar FFMA occupies the fma
// pipe for two cycles per warp: pairing the channel math halves both. A float4 is two aligned register pairs.
__device__ __forceinline__ float2 lo2(float4 v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 hi2(float4 v) { return make_float2(v.z, v.w); }
__device__ __forceinline__ float4 cat4(float2 l, float2 h) { return make_float4(l.x, l.y, h.x, h.y); }
__device__ __forceinline__ float2 dup2(float s) { return make_float2(s, s); }
__device__ __forceinline__ float4 f4z() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ void f4_fma(float4& acc, float4 a, float2 s) {          // acc += a * s
    acc = cat4(__ffma2_rn(lo2(a), s, lo2(acc)), __ffma2_rn(hi2(a), s, hi2(acc)));
}
__device__ __forceinline__ float4 f4_mul2(float4 a, float4 b) { return cat4(__fmul2_rn(lo2(a), lo2(b)), __fmul2_rn(hi2(a), hi2(b))); }
__device__ __forceinline__ float4 f4_scale(float4 a, float2 s) { return cat4(__fmul2_rn(lo2(a), s), __fmul2_rn(hi2(a), s)); }
__device__ __forceinline__ void f2_dot_acc(float2& acc, float4 a, float4 b) {      // acc += (a.xy*b.xy) + (a.zw*b.zw), lane-wise
    acc = __ffma2_rn(lo2(a), lo2(b), acc);
    acc = __ffma2_rn(hi2(a), hi2(b), acc);
}
__device__ __forceinline__ bool f4_any(float4 a) { return a.x != 0.f || a.y != 0.f || a.z != 0.f || a.w != 0.f; }

// unclamped tap position on an axis of n texels (ATen grid_sampler, align_corners=True)
struct Pos { int i0; float f; float scale; };
__device__ __forceinline__ Pos axis_pos(float g, int n) {
    Pos p;
    p.scale = 0.5f * (float)(n - 1);
    const float x = (g + 1.0f) * p.scale;
    const float xf = floorf(x);
    p.f = x - xf;
    p.i0 = (int)fminf(fmaxf(xf, -2.0f), (float)n);       // NaN -> -2: both taps out of range
    return p;
}

struct ScatterArgs {
    Factors F;
    FactorGrads G;
    const float4* samp;     // [V] (u_x, u_y, u_z, t)
    const int* slot;        // element e -> sample slot (appearance list) or nullptr
    const int* sidx;        // [V] ray * S + k
    const int* n_dev;
    int n_fixed;
    const float* gin;       // APP: [n][ctot] (fp32, or bf16 when gin_bf16); density: [n]
    int gin_bf16;
    float* d_o;             // [N][3], accumulated
    float* d_d;             // [N][3], accumulated
    float inv[3];           // 2 / aabbSize (normalize_coord)
    int S;                  // samples per ray (sidx decoding)
    int seg;                // samples per walker segment (fixed), or
    int seg_target;         // > 0: persistent grid, segment length chosen in the kernel (see vm_scatter_walk_kernel)
    int plane_mask;         // bit i: walk plane / line pair i in this launch (7 = all three)
};

// One walker = LW lanes; lane `sub` owns the NQ channel quads sub, sub + LW, ... of a plane
// (C = 4 LW NQ), i.e. per tap the walker's lanes read LW x 16 contiguous bytes NQ times.
// Work unit = a segment of `seg` consecutive elements; the walker walks it once per plane
// (plane index is a compile-time constant of walk_plane). Walkers are laid out over the
// CTA's threads contiguously and use no warp-level collectives.
//
// Walking the three 16-channel density planes in ONE pass instead (per step: one record / sidx / gin load and one
// ray-change test; per plane only the cell state, 4 lanes x 1 quad per plane, 36 staging slots per lane) is slower:
// it needs 247 registers without spills (MINB 2; at MINB 3 it spills 420 B), so 8 warps per SM instead of 16, and
// the three planes' cell state costs more moves than the shared loads save (static loop body 1418 SASS instructions
// vs 3 x 486). Measured on one B200 at 1000 W (profiles/r03_density_onepass_ab.jsonl): density scatter
// 0.405 -> 0.563 ms on cfg2_sh, 0.555 -> 0.731 ms on cfg4; coordinate-only (134 registers, MINB 3) no faster either.
// The 2 lanes x 2 quads layout doubles the per-lane accumulators and cannot fit at all.
//
// Tap staging: the kernel is latency-bound, not RED-bound, once the REDs are merged, and the
// accumulators leave no registers to keep loads in flight. So each lane owns a private,
// double-buffered shared-memory slot set for the taps of its quads: when the look-ahead
// (one step) sees that the next sample enters another plane / line cell, the lane issues
// cp.async copies of the new cell's taps into the idle buffer while the current step
// computes out of the active one. A lane only ever reads what it copied itself, so no
// barrier is needed -- cp.async.wait_group orders it.
struct RaySums { float o[3], d[3]; };      // per axis: sum_j dL/du_j, sum_j dL/du_j * t_j (this lane's channels)

constexpr int SC_THREADS = 128;

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait0() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

struct StepPos {          // tap position of one sample on one plane/line pair
    int x0, y0, l0;       // unclamped cell indices (NaN -> -2: both taps out of range)
    float fx, fy, fl;     // fractions
    float t;              // depth along the ray
    int sid;              // ray * S + k
};

// B16: the factor taps are bf16 (8-byte quads: half the staging traffic), everything else is unchanged -- the
// gradients and the arithmetic stay fp32.
// FG = false: coordinate-only walk for a frozen field (test-time pose optimisation). The corner / line gradient
// accumulators, the cell bookkeeping of their flushes and every RED into the factor gradients are compiled out; the
// tap staging, the look-ahead and the per-ray sums (all the pose gradient needs) are the same code as with FG.
template <bool APP, int NQ, int I, bool GB16, bool B16, bool FG, int THR = SC_THREADS>
__device__ __forceinline__ void walk_plane(const ScatterArgs& A, const int e0, const int e1, const int q, const int qs,
                                           int& ray, int& ray_end, RaySums& rs,
                                           typename std::conditional<B16, uint2, float4>::type* __restrict__ sm) {
    using SlotT = typename std::conditional<B16, uint2, float4>::type;          // one staged channel quad
    using ElemT = typename std::conditional<B16, unsigned short, float>::type;  // one factor element
    const Factors& F = A.F;
    constexpr int ax = I == 2 ? 1 : 0, ay = I == 0 ? 1 : 2, al = 2 - I;      // matMode / vecMode (tensorBase.py:405-406)
    const int W = F.W[I], H = F.H[I], L = F.L[I], C = F.C[I];
    if (q >= C) return;
    const ElemT* __restrict__ P = reinterpret_cast<const ElemT*>(F.plane[I]) + q;
    const ElemT* __restrict__ Ln = reinterpret_cast<const ElemT*>(F.line[I]) + q;
    float* __restrict__ GP = FG ? A.G.plane[I] + q : nullptr;
    float* __restrict__ GL = FG ? A.G.line[I] + q : nullptr;
    const float sclx = 0.5f * (float)(W - 1), scly = 0.5f * (float)(H - 1), scll = 0.5f * (float)(L - 1);
    // this lane's staging slots (float4 index = slot * SC_THREADS): plane buffer b, tap c, quad k -> (b*4 + c)*NQ + k;
    // line buffer b, tap c, quad k -> 8 NQ + (b*2 + c)*NQ + k
    auto pslot = [&](int b, int c, int k) -> SlotT* { return sm + ((b * 4 + c) * NQ + k) * THR; };
    auto lslot = [&](int b, int c, int k) -> SlotT* { return sm + (8 * NQ + (b * 2 + c) * NQ + k) * THR; };
    auto rd = [&](const SlotT* p) -> float4 {
        if constexpr (B16) return bf16x4_to_f4(*p); else return *p;
    };
    auto cp = [&](SlotT* dst, const ElemT* src) { if constexpr (B16) cp_async8(dst, src); else cp_async16(dst, src); };

    auto make_pos = [&](const float4 u4, const int sid) {
        const float u[3] = {u4.x, u4.y, u4.z};
        StepPos p;
        const float fxp = (u[ax] + 1.0f) * sclx, fyp = (u[ay] + 1.0f) * scly, flp = (u[al] + 1.0f) * scll;
        const float xf = floorf(fxp), yf = floorf(fyp), lf = floorf(flp);
        p.x0 = (int)fminf(fmaxf(xf, -2.0f), (float)W); p.y0 = (int)fminf(fmaxf(yf, -2.0f), (float)H);
        p.l0 = (int)fminf(fmaxf(lf, -2.0f), (float)L);
        p.fx = fxp - xf; p.fy = fyp - yf; p.fl = flp - lf;
        p.t = u4.w; p.sid = sid;
        return p;
    };
    // clamped element offsets of the 4 plane corners / 2 line taps of a cell
    auto plane_offs = [&](int x0, int y0, unsigned o[4]) {
        const int xc0 = min(max(x0, 0), W - 1), xc1 = min(max(x0 + 1, 0), W - 1);
        const int yc0 = min(max(y0, 0), H - 1), yc1 = min(max(y0 + 1, 0), H - 1);
        o[0] = (unsigned)((yc0 * W + xc0) * C); o[1] = (unsigned)((yc0 * W + xc1) * C);
        o[2] = (unsigned)((yc1 * W + xc0) * C); o[3] = (unsigned)((yc1 * W + xc1) * C);
    };
    auto line_offs = [&](int l0, unsigned o[2]) {
        o[0] = (unsigned)(min(max(l0, 0), L - 1) * C); o[1] = (unsigned)(min(max(l0 + 1, 0), L - 1) * C);
    };
    auto fetch_plane = [&](int b, const unsigned o[4]) {
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int k = 0; k < NQ; ++k) cp(pslot(b, c, k), P + o[c] + k * qs);
    };
    auto fetch_line = [&](int b, const unsigned o[2]) {
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
            for (int k = 0; k < NQ; ++k) cp(lslot(b, c, k), Ln + o[c] + k * qs);
    };
    // upstream gradient of element e for this lane's quads: fetched raw one step ahead (the
    // conversion happens at use, so the load latency stays off the issue path)
    struct GinRaw { float4 f; uint2 h; float s; };
    auto load_gin = [&](int e, GinRaw g[NQ]) {
        if (APP && GB16) {                       // bf16 row of the tensor-core head's dcomps
            const unsigned short* row = reinterpret_cast<const unsigned short*>(A.gin) + (size_t)e * F.ctot + F.off[I] + q;
#pragma unroll
            for (int k = 0; k < NQ; ++k) g[k].h = __ldcs(reinterpret_cast<const uint2*>(row + k * qs));
        } else if (APP) {
            const float* row = A.gin + (size_t)e * F.ctot + F.off[I] + q;
#pragma unroll
            for (int k = 0; k < NQ; ++k) g[k].f = __ldcs(reinterpret_cast<const float4*>(row + k * qs));
        } else {
            g[0].s = A.gin[e];
        }
    };
    auto gin_value = [&](const GinRaw g[NQ], int k) -> float4 {
        if (APP && GB16)
            return make_float4(__uint_as_float(g[k].h.x << 16), __uint_as_float(g[k].h.x & 0xFFFF0000u),
                               __uint_as_float(g[k].h.y << 16), __uint_as_float(g[k].h.y & 0xFFFF0000u));
        if (APP) return g[k].f;
        return make_float4(g[0].s, g[0].s, g[0].s, g[0].s);
    };

    // accumulated cell: indices and clamped element offsets
    int cx = INT_MIN, cy = INT_MIN, cl = INT_MIN;
    unsigned s00 = 0, s10 = 0, s01 = 0, s11 = 0, sl0 = 0, sl1 = 0;
    float4 g00[NQ], g10[NQ], g01[NQ], g11[NQ], gl0[NQ], gl1[NQ];
#pragma unroll
    for (int k = 0; k < NQ; ++k) { g00[k] = g10[k] = g01[k] = g11[k] = gl0[k] = gl1[k] = f4z(); }

    auto flush_ray = [&]() {
        if (ray >= 0) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                if (rs.o[a] != 0.f) atomicAdd(A.d_o + 3 * ray + a, rs.o[a] * A.inv[a]);
                if (rs.d[a] != 0.f) atomicAdd(A.d_d + 3 * ray + a, rs.d[a] * A.inv[a]);
            }
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) rs.o[a] = rs.d[a] = 0.f;
    };

    // ---- prologue: position + taps of element e0, record of e0 + 1, upstream gradient of e0
    StepPos pn;
    unsigned on[4], oln[2];          // offsets of the cell whose taps sit in the "next" buffers
    int pbn = 0, lbn = 0;
    {
        const int j0 = A.slot ? A.slot[e0] : e0;
        pn = make_pos(A.samp[j0], A.sidx[j0]);
        plane_offs(pn.x0, pn.y0, on);
        line_offs(pn.l0, oln);
        fetch_plane(0, on);
        fetch_line(0, oln);
        cp_async_commit();
    }
    // sample records are fetched two steps ahead and their slot indices three steps ahead, so that no
    // load waits on the result of another load issued in the same step
    auto slot_of = [&](int e) -> int { return e < e1 ? (A.slot ? A.slot[e] : e) : 0; };
    float4 un = f4z();
    int sn = 0;
    if (e0 + 1 < e1) {
        const int j1 = slot_of(e0 + 1);
        un = A.samp[j1];
        sn = A.sidx[j1];
    }
    int jn2 = slot_of(e0 + 2);
    GinRaw gn[NQ];
    load_gin(e0, gn);

    for (int e = e0; e < e1; ++e) {
        const StepPos pc = pn;
        const int pb = pbn, lb = lbn;
        const unsigned o00 = on[0], o10 = on[1], o01 = on[2], o11 = on[3], ol0 = oln[0], ol1 = oln[1];
        GinRaw gc[NQ];
#pragma unroll
        for (int k = 0; k < NQ; ++k) gc[k] = gn[k];
        // ---- look-ahead: position of e+1; its taps are copied into the idle buffers if it enters a new cell
        if (e + 1 < e1) {
            pn = make_pos(un, sn);
            if (pn.x0 != pc.x0 || pn.y0 != pc.y0) {
                plane_offs(pn.x0, pn.y0, on);
                pbn = pb ^ 1;
                fetch_plane(pbn, on);
            }
            if (pn.l0 != pc.l0) {
                line_offs(pn.l0, oln);
                lbn = lb ^ 1;
                fetch_line(lbn, oln);
            }
            load_gin(e + 1, gn);
            if (e + 2 < e1) {
                un = A.samp[jn2];
                sn = A.sidx[jn2];
            }
            jn2 = slot_of(e + 3);
        }
        cp_async_commit();
        cp_async_wait1();                                    // everything but the look-ahead copies has landed

        if (pc.sid >= ray_end || pc.sid < ray_end - A.S) {   // another ray (lists are ray-major)
            flush_ray();
            ray = pc.sid / A.S;
            ray_end = (ray + 1) * A.S;
        }
        const int x0 = pc.x0, y0 = pc.y0, l0 = pc.l0;
        const float mx0 = (x0 >= 0 && x0 < W) ? 1.f : 0.f, mx1 = (x0 + 1 >= 0 && x0 + 1 < W) ? 1.f : 0.f;
        const float my0 = (y0 >= 0 && y0 < H) ? 1.f : 0.f, my1 = (y0 + 1 >= 0 && y0 + 1 < H) ? 1.f : 0.f;
        const float ml0 = (l0 >= 0 && l0 < L) ? 1.f : 0.f, ml1 = (l0 + 1 >= 0 && l0 + 1 < L) ? 1.f : 0.f;
        if (FG && (x0 != cx || y0 != cy)) {                  // plane cell changed: flush the 4 corners
            if (cx != INT_MIN) {
#pragma unroll
                for (int k = 0; k < NQ; ++k) {
                    red_add_v4(GP + s00 + k * qs, g00[k]); red_add_v4(GP + s10 + k * qs, g10[k]);
                    red_add_v4(GP + s01 + k * qs, g01[k]); red_add_v4(GP + s11 + k * qs, g11[k]);
                }
            }
#pragma unroll
            for (int k = 0; k < NQ; ++k) { g00[k] = f4z(); g10[k] = f4z(); g01[k] = f4z(); g11[k] = f4z(); }
            cx = x0; cy = y0; s00 = o00; s10 = o10; s01 = o01; s11 = o11;
        }
        if (FG && l0 != cl) {                                // line cell changed
            if (cl != INT_MIN) {
#pragma unroll
                for (int k = 0; k < NQ; ++k) { red_add_v4(GL + sl0 + k * qs, gl0[k]); red_add_v4(GL + sl1 + k * qs, gl1[k]); }
            }
#pragma unroll
            for (int k = 0; k < NQ; ++k) { gl0[k] = f4z(); gl1[k] = f4z(); }
            cl = l0; sl0 = ol0; sl1 = ol1;
        }
        const float fx = pc.fx, fy = pc.fy, fl = pc.fl;
        const float wx0 = (1.f - fx) * mx0, wx1 = fx * mx1, wy0 = (1.f - fy) * my0, wy1 = fy * my1;
        const float wl0 = (1.f - fl) * ml0, wl1 = fl * ml1;
        const float2 w00 = dup2(wx0 * wy0), w10 = dup2(wx1 * wy0), w01 = dup2(wx0 * wy1), w11 = dup2(wx1 * wy1);
        const float2 wl0p = dup2(wl0), wl1p = dup2(wl1);
        float2 dA2 = dup2(0.f), dB2 = dup2(0.f), dC2 = dup2(0.f), dD2 = dup2(0.f), dLa2 = dup2(0.f), dLb2 = dup2(0.f);
#pragma unroll
        for (int k = 0; k < NQ; ++k) {
            const float4 a = rd(pslot(pb, 0, k)), b = rd(pslot(pb, 1, k)), c = rd(pslot(pb, 2, k)), d = rd(pslot(pb, 3, k));
            const float4 la = rd(lslot(lb, 0, k)), lb4 = rd(lslot(lb, 1, k));
            float4 pv = f4_scale(a, w00), lv = f4_scale(la, wl0p);
            f4_fma(pv, b, w10); f4_fma(pv, c, w01); f4_fma(pv, d, w11);
            f4_fma(lv, lb4, wl1p);
            const float4 g4 = gin_value(gc, k);
            const float4 gl = f4_mul2(g4, lv);       // dL/dP (interpolated plane value)
            const float4 gp = f4_mul2(g4, pv);       // dL/dL (interpolated line value)
            if constexpr (FG) {
                f4_fma(g00[k], gl, w00); f4_fma(g10[k], gl, w10); f4_fma(g01[k], gl, w01); f4_fma(g11[k], gl, w11);
                f4_fma(gl0[k], gp, wl0p); f4_fma(gl1[k], gp, wl1p);
            }
            f2_dot_acc(dA2, gl, a); f2_dot_acc(dB2, gl, b); f2_dot_acc(dC2, gl, c); f2_dot_acc(dD2, gl, d);
            f2_dot_acc(dLa2, gp, la); f2_dot_acc(dLb2, gp, lb4);
        }
        const float dA = dA2.x + dA2.y, dB = dB2.x + dB2.y, dC = dC2.x + dC2.y, dD = dD2.x + dD2.y;   // sum_c gl*tap
        const float dLa = dLa2.x + dLa2.y, dLb = dLb2.x + dLb2.y;                                    // sum_c gp*tap
        // d/d index (ATen grid_sampler_2d_backward: out-of-range taps read as 0)
        const float dux = ((dB * mx1 - dA * mx0) * wy0 + (dD * mx1 - dC * mx0) * wy1) * sclx;
        const float duy = ((dC * my1 - dA * my0) * wx0 + (dD * my1 - dB * my0) * wx1) * scly;
        const float dul = (dLb * ml1 - dLa * ml0) * scll;
        const float t = pc.t;
        rs.o[ax] += dux; rs.d[ax] = fmaf(dux, t, rs.d[ax]);
        rs.o[ay] += duy; rs.d[ay] = fmaf(duy, t, rs.d[ay]);
        rs.o[al] += dul; rs.d[al] = fmaf(dul, t, rs.d[al]);
    }
    cp_async_wait0();
    if (FG && cx != INT_MIN) {
#pragma unroll
        for (int k = 0; k < NQ; ++k) {
            red_add_v4(GP + s00 + k * qs, g00[k]); red_add_v4(GP + s10 + k * qs, g10[k]);
            red_add_v4(GP + s01 + k * qs, g01[k]); red_add_v4(GP + s11 + k * qs, g11[k]);
        }
    }
    if (FG && cl != INT_MIN) {
#pragma unroll
        for (int k = 0; k < NQ; ++k) { red_add_v4(GL + sl0 + k * qs, gl0[k]); red_add_v4(GL + sl1 + k * qs, gl1[k]); }
    }
    flush_ray();
}

template <bool APP, int NQ, int MINB, bool GB16, int LWC, bool B16, bool FG>
__global__ void __launch_bounds__(SC_THREADS, MINB) vm_scatter_walk_kernel(const ScatterArgs A, int LW_rt, int walkers_per_cta) {
    extern __shared__ __align__(16) unsigned char sc_smem[];   // 12 NQ slots x SC_THREADS quads (16 B fp32 / 8 B bf16)
    using SlotT = typename std::conditional<B16, uint2, float4>::type;
    const int LW = LWC > 0 ? LWC : LW_rt;                // lanes per walker (compile-time strides when LWC > 0)
    const int n = A.n_dev ? *A.n_dev : A.n_fixed;
    const int wl = threadIdx.x / LW;                     // walker within the CTA
    const int q = (threadIdx.x - wl * LW) * 4;           // first channel of this lane's first quad
    const int qs = LW * 4;                               // channel stride between this lane's quads
    if (wl >= walkers_per_cta) return;
    SlotT* sm = reinterpret_cast<SlotT*>(sc_smem) + threadIdx.x;
    const int stride = gridDim.x * walkers_per_cta;      // walkers in the grid
    // Segment length. The grid is persistent (one wave of resident CTAs) and the units are dealt round-robin, so the
    // kernel takes ceil(units / walkers) rounds: a fixed length leaves up to a whole round idle at the end (measured
    // on cfg2, fixed 32/48/64/80 samples: 1.11 / 1.02 / 1.05 / 0.97 ms). The count n is only known on the device,
    // so every CTA derives the same length here: k = round(n / (walkers * target)) rounds of ceil(n / (k * walkers)).
    int seg = A.seg;
    if (A.seg_target > 0) {
        const long long wt = (long long)stride * A.seg_target;
        const long long k = max(1LL, ((long long)n + wt / 2) / wt);
        seg = (int)max(1LL, ((long long)n + k * stride - 1) / (k * stride));
    }
    const int n_units = (n + seg - 1) / seg;
    for (int unit = blockIdx.x * walkers_per_cta + wl; unit < n_units; unit += stride) {
        const int e0 = unit * seg;
        const int e1 = min(e0 + seg, n);
        int ray = -1, ray_end = INT_MIN;
        RaySums rs;
#pragma unroll
        for (int a = 0; a < 3; ++a) rs.o[a] = rs.d[a] = 0.f;
        if (A.plane_mask & 1) walk_plane<APP, NQ, 0, GB16, B16, FG>(A, e0, e1, q, qs, ray, ray_end, rs, sm);
        if (A.plane_mask & 2) walk_plane<APP, NQ, 1, GB16, B16, FG>(A, e0, e1, q, qs, ray, ray_end, rs, sm);
        if (A.plane_mask & 4) walk_plane<APP, NQ, 2, GB16, B16, FG>(A, e0, e1, q, qs, ray, ray_end, rs, sm);
    }
}

}  // namespace jt

using namespace jt;

extern "C" int jt_vm_scatter_rays(int app, const void* const* h_factors, void* const* h_factor_grads,
                                  const int* h_dims, const float* samp, const int* slot, const int* sidx,
                                  const int* n_dev, int n_max, const void* gin, int gin_bf16, int n_samples, const float* h_inv,
                                  float* d_o, float* d_d, int max_ctas, int plane_mask, cudaStream_t stream) {
    JT_CHECK_ARG(h_factors && h_dims && samp && sidx && gin && h_inv && d_o && d_d && n_samples > 0);
    JT_CHECK_ARG(plane_mask > 0 && plane_mask <= 7);
    if (n_max <= 0) return JT_OK;
    ScatterArgs A;
    if (int rc = fill_factors(A.F, h_factors, h_dims)) return rc;
    const bool fg = h_factor_grads != nullptr;              // NULL: coordinate-only walk (d_o / d_d alone)
    int cmax = 0;
    for (int i = 0; i < 3; ++i) {
        A.G.plane[i] = fg ? static_cast<float*>(h_factor_grads[i]) : nullptr;
        A.G.line[i] = fg ? static_cast<float*>(h_factor_grads[3 + i]) : nullptr;
        JT_CHECK_ARG(!fg || (A.G.plane[i] && A.G.line[i]));
        cmax = A.F.C[i] > cmax ? A.F.C[i] : cmax;
        JT_CHECK_ARG((long long)A.F.H[i] * A.F.W[i] * A.F.C[i] < 2147483647LL);
    }
    JT_CHECK_ARG((long long)n_max < 2147483647LL);
    A.samp = reinterpret_cast<const float4*>(samp);
    A.slot = slot; A.sidx = sidx; A.n_dev = n_dev; A.n_fixed = n_max; A.gin = static_cast<const float*>(gin); A.gin_bf16 = gin_bf16;
    JT_CHECK_ARG(!gin_bf16 || app);
    A.d_o = d_o; A.d_d = d_d;
    for (int a = 0; a < 3; ++a) A.inv[a] = h_inv[a];
    A.S = n_samples;
    A.plane_mask = plane_mask;
    // default: persistent grid, segment length derived in the kernel from the device-side count (target ~100
    // samples). JT_SCATTER_SEG=<n> (tuning) restores fixed n-sample segments on a non-persistent grid.
    static const int seg_env = getenv("JT_SCATTER_SEG") ? atoi(getenv("JT_SCATTER_SEG")) : 0;
    A.seg = seg_env > 0 ? seg_env : 32;
    A.seg_target = seg_env > 0 ? 0 : 100;
    // max_ctas < 0: fixed segments of -max_ctas samples on a non-persistent grid. The fused render op asks for this
    // for the density scatter of a data-parallel step: the NCCL all-reduce of the appearance gradients runs next to
    // it and its CTAs can only get onto an SM when scatter CTAs retire (a persistent wave would hold every SM's
    // registers until the end of the kernel and serialise the collective behind it).
    if (max_ctas < 0) { A.seg = -max_ctas; A.seg_target = 0; max_ctas = 0; }
    // lanes per walker / quads per lane: 48 or 32 uniform channels -> 4 lanes x C/16 quads, anything else -> one
    // quad per lane. (One lane owning all 4 quads of a 16-channel plane has 2.4x fewer instructions but
    // un-coalesced taps: measured 0.77 ms vs 0.49 ms for the cfg2 density planes.)
    int nq = 1, LW = cmax / 4;
    const bool uniform = A.F.C[0] == A.F.C[1] && A.F.C[1] == A.F.C[2];
    if (uniform && (cmax == 48 || cmax == 32)) { nq = cmax / 16; LW = 4; }
    JT_CHECK_ARG(LW >= 1 && LW <= 128);
    const int wpc = SC_THREADS / LW;                          // walkers per CTA
    const int threads = ((wpc * LW + 31) / 32) * 32;
    long long units = ((long long)n_max + A.seg - 1) / A.seg;
    long long want = (units + wpc - 1) / wpc;
    // CTAs per SM of the variant launched below (its MINB). Without the gradient accumulators the coordinate-only
    // variants fit more CTAs per SM; nq = 3 with fp32 taps is then bound by shared memory (3 x 72 KB).
    const int resident = fg ? (nq == 3 ? 2 : (nq == 2 || app) ? 3 : 4) : (nq == 3 ? 3 : nq == 2 ? 4 : 5);
    long long cap = max_ctas > 0 ? (long long)max_ctas
                                 : (A.seg_target > 0 ? (long long)kNumSMs * resident : (long long)kNumSMs * 32);
    if (A.seg_target > 0) want = cap;                         // one resident wave; the kernel sizes the segments to fit
    int grid = (int)(want < cap ? (want < 1 ? 1 : want) : cap);
    g_launches += 1;
    const int smem = 12 * nq * SC_THREADS * (A.F.bf16 ? 8 : 16);
#define JT_SCB(APPV, NQV, MB, GB, LWV, BV, FGV)                                                                     \
    {                                                                                                               \
        if (smem > 48 * 1024 &&                                                                                     \
            cudaFuncSetAttribute(vm_scatter_walk_kernel<APPV, NQV, MB, GB, LWV, BV, FGV>,                           \
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess)                 \
            return JT_ERR_LAUNCH;                                                                                   \
        vm_scatter_walk_kernel<APPV, NQV, MB, GB, LWV, BV, FGV><<<grid, threads, smem, stream>>>(A, LW, wpc);       \
    }
#define JT_SC(APPV, NQV, MB, GB, LWV) { if (A.F.bf16) JT_SCB(APPV, NQV, MB, GB, LWV, true, true) else JT_SCB(APPV, NQV, MB, GB, LWV, false, true) }
#define JT_SCC(APPV, NQV, MB, GB, LWV) { if (A.F.bf16) JT_SCB(APPV, NQV, MB, GB, LWV, true, false) else JT_SCB(APPV, NQV, MB, GB, LWV, false, false) }
    // (64-thread CTAs with a 200-register cap -- five CTAs per SM instead of two -- spill and lose: 1.55 vs 1.22 ms;
    // a minimum-blocks bound of 3 (168 registers) likewise: 2.28 ms.)
    if (!fg) {      // coordinate-only: MINB as `resident` above (no spills at these bounds, -Xptxas -v)
        if (app && gin_bf16) { if (nq == 3) JT_SCC(true, 3, 3, true, 4) else if (nq == 2) JT_SCC(true, 2, 4, true, 4) else JT_SCC(true, 1, 5, true, 0) }
        else if (app) { if (nq == 3) JT_SCC(true, 3, 3, false, 4) else if (nq == 2) JT_SCC(true, 2, 4, false, 4) else JT_SCC(true, 1, 5, false, 0) }
        else { if (nq == 3) JT_SCC(false, 3, 3, false, 4) else if (nq == 2) JT_SCC(false, 2, 4, false, 4) else JT_SCC(false, 1, 5, false, 0) }
    }
    else if (app && gin_bf16) { if (nq == 3) JT_SC(true, 3, 2, true, 4) else if (nq == 2) JT_SC(true, 2, 3, true, 4) else JT_SC(true, 1, 3, true, 0) }
    else if (app) { if (nq == 3) JT_SC(true, 3, 2, false, 4) else if (nq == 2) JT_SC(true, 2, 3, false, 4) else JT_SC(true, 1, 3, false, 0) }
    else { if (nq == 3) JT_SC(false, 3, 2, false, 4) else if (nq == 2) JT_SC(false, 2, 3, false, 4) else JT_SC(false, 1, 4, false, 0) }
#undef JT_SCC
#undef JT_SC
#undef JT_SCB
    JT_RETURN_LAUNCH();
}
