// Mesh export: marching cubes over a dense scalar volume [gz][gy][gx] (the dense alpha grid of jt_field_alpha),
// the step TensoRF-family exporters take after getDenseAlpha. The case table is generated (gen_mc_tables.py).
//
// Three launches, welded output in an order that does not depend on scheduling:
//   classify  one thread per lattice point, coalesced along x: the case of the cell the point anchors and the
//             3-bit mask of its owned crossing edges (x, y, z edge from the point). Per chunk of 32 points it
//             stores the ballots of those bits and the chunk's vertex / triangle offsets inside its tile of
//             2048 points; per tile the two counts.
//   scan      one block: exclusive scan of the tile counts in 64 bits, and the two totals.
//   emit      one warp per chunk, chunks without crossings skipped: vertex id = tile base + chunk offset + popc of
//             the chunk's bits below the lane; triangles of the non-empty cells look up the ids of edges owned by
//             neighbouring points the same way.
//   normals   (optional, after classify + scan) the same walk over chunks with crossings: per vertex the volume
//             gradient at both ends of its edge (central differences), blended with emit's t, negated, normalised.
// Scratch: 20 bytes per chunk of 32 points + 24 bytes per tile (jt_mc_scratch_bytes).
#include <climits>

#include "jt_common.cuh"
#include "mc_tables.cuh"
#include "../../include/jt_vm.h"

namespace jt {

constexpr int kMcThreads = 256;                  // 8 warps
constexpr int kMcTileChunks = 64;                // chunks of 32 points per classify block
constexpr int kMcTile = kMcTileChunks * 32;      // 2048 points
constexpr int kMcTriMax = 5;

struct McScratch {
    uint4* bits;          // [chunks] x, y, z crossing-edge ballots, w = ballot of non-empty cells
    uint32_t* loc;        // [chunks] vertex offset (low 16 bits) | triangle offset (high 16) inside the tile
    int2* tile_cnt;       // [tiles] vertices, triangles of the tile
    longlong2* tile_base; // [tiles] exclusive prefix of tile_cnt
};

__host__ __device__ inline long long mc_tiles(long long n) { return (n + kMcTile - 1) / kMcTile; }

inline McScratch mc_scratch(void* base, long long tiles) {
    char* p = static_cast<char*>(base);
    McScratch s;
    s.tile_base = reinterpret_cast<longlong2*>(p);
    p += tiles * sizeof(longlong2);
    s.bits = reinterpret_cast<uint4*>(p);
    p += tiles * kMcTileChunks * sizeof(uint4);
    s.tile_cnt = reinterpret_cast<int2*>(p);
    p += tiles * sizeof(int2);
    s.loc = reinterpret_cast<uint32_t*>(p);
    return s;
}

// case of the cell anchored at point p = (x, y, z): bit i set when corner (i&1, i>>1&1, i>>2&1) is > level
__device__ __forceinline__ int mc_case(const float* __restrict__ vol, int p, int sy, int sz, float level) {
    int c = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int q = p + (i & 1) + ((i >> 1) & 1) * sy + ((i >> 2) & 1) * sz;
        c |= (__ldg(vol + q) > level ? 1 : 0) << i;
    }
    return c;
}

__global__ void __launch_bounds__(kMcThreads) mc_classify_kernel(const float* __restrict__ vol, int gx, int gy, int gz,
                                                                 float level, McScratch S) {
    __shared__ unsigned char s_ntri[256];
    __shared__ int s_cnt[2][kMcTileChunks];
    s_ntri[threadIdx.x] = kMcNumTri[threadIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sy = gx, sz = gx * gy, n = sz * gz;
    for (int k = 0; k < kMcTileChunks / 8; ++k) {
        const int cl = k * 8 + warp;
        const long long chunk = (long long)blockIdx.x * kMcTileChunks + cl;
        const long long pl = chunk * 32 + lane;
        unsigned ex = 0, ey = 0, ez = 0;
        int nt = 0;
        if (pl < n) {
            const int p = (int)pl;
            const int x = p % gx, r = p / gx, y = r % gy, z = r / gy;
            const bool in0 = __ldg(vol + p) > level;
            if (x + 1 < gx) ex = in0 != (__ldg(vol + p + 1) > level);
            if (y + 1 < gy) ey = in0 != (__ldg(vol + p + sy) > level);
            if (z + 1 < gz) ez = in0 != (__ldg(vol + p + sz) > level);
            if (x + 1 < gx && y + 1 < gy && z + 1 < gz) nt = s_ntri[mc_case(vol, p, sy, sz, level)];
        }
        const unsigned bx = __ballot_sync(0xffffffffu, ex), by = __ballot_sync(0xffffffffu, ey);
        const unsigned bz = __ballot_sync(0xffffffffu, ez), bc = __ballot_sync(0xffffffffu, nt > 0);
        const int tri = __reduce_add_sync(0xffffffffu, nt);
        if (lane == 0) {
            S.bits[chunk] = make_uint4(bx, by, bz, bc);
            s_cnt[0][cl] = __popc(bx) + __popc(by) + __popc(bz);
            s_cnt[1][cl] = tri;
        }
    }
    __syncthreads();
    if (warp == 0) {                      // exclusive scan of the 64 chunk counts, two per lane
        const int v0 = s_cnt[0][2 * lane], v1 = s_cnt[0][2 * lane + 1];
        const int t0 = s_cnt[1][2 * lane], t1 = s_cnt[1][2 * lane + 1];
        int iv = v0 + v1, it = t0 + t1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int a = __shfl_up_sync(0xffffffffu, iv, o), b = __shfl_up_sync(0xffffffffu, it, o);
            if (lane >= o) { iv += a; it += b; }
        }
        const int ev = iv - v0 - v1, et = it - t0 - t1;     // <= 2048*3 and 2048*5: 16 bits each
        const long long c0 = (long long)blockIdx.x * kMcTileChunks + 2 * lane;
        S.loc[c0] = (uint32_t)ev | ((uint32_t)et << 16);
        S.loc[c0 + 1] = (uint32_t)(ev + v0) | ((uint32_t)(et + t0) << 16);
        if (lane == 31) S.tile_cnt[blockIdx.x] = make_int2(iv, it);
    }
}

// One block: each thread scans a contiguous run of tiles; 64-bit sums, so that a total past INT32_MAX is reported
// rather than wrapped.
__global__ void __launch_bounds__(1024) mc_scan_kernel(McScratch S, long long tiles, long long* __restrict__ totals) {
    __shared__ long long s_v[32], s_t[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long per = (tiles + blockDim.x - 1) / blockDim.x;
    const long long beg = min(tiles, tid * per), end = min(tiles, beg + per);
    long long sv = 0, st = 0;
    for (long long i = beg; i < end; ++i) {
        const int2 c = S.tile_cnt[i];
        sv += c.x;
        st += c.y;
    }
    long long iv = sv, it = st;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long a = __shfl_up_sync(0xffffffffu, iv, o), b = __shfl_up_sync(0xffffffffu, it, o);
        if (lane >= o) { iv += a; it += b; }
    }
    if (lane == 31) { s_v[warp] = iv; s_t[warp] = it; }
    __syncthreads();
    if (warp == 0) {
        long long wv = lane < (int)(blockDim.x >> 5) ? s_v[lane] : 0, wt = lane < (int)(blockDim.x >> 5) ? s_t[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long a = __shfl_up_sync(0xffffffffu, wv, o), b = __shfl_up_sync(0xffffffffu, wt, o);
            if (lane >= o) { wv += a; wt += b; }
        }
        s_v[lane] = wv;
        s_t[lane] = wt;
    }
    __syncthreads();
    long long ev = iv - sv + (warp ? s_v[warp - 1] : 0), et = it - st + (warp ? s_t[warp - 1] : 0);
    for (long long i = beg; i < end; ++i) {
        const int2 c = S.tile_cnt[i];
        S.tile_base[i] = make_longlong2(ev, et);
        ev += c.x;
        et += c.y;
    }
    if (tid == blockDim.x - 1) { totals[0] = ev; totals[1] = et; }
}

struct McEmitArgs {
    const float* lin[3];
    float a0[3], a1[3];
    int gx, gy, gz;
    float level;
};

// aabb0*(1-s) + aabb1*s, separately rounded: the points of getDenseAlpha's dense_xyz
__device__ __forceinline__ float mc_coord(const McEmitArgs& A, int a, int i) {
    const float s = __ldg(A.lin[a] + i);
    return __fadd_rn(__fmul_rn(A.a0[a], __fsub_rn(1.0f, s)), __fmul_rn(A.a1[a], s));
}

// id of the vertex on the edge along `axis` owned by point q
__device__ __forceinline__ int mc_vertex_id(const McScratch& S, int q, int axis) {
    const int chunk = q >> 5, l = q & 31;
    const uint4 b = S.bits[chunk];
    const unsigned below = (1u << l) - 1u;
    int id = (int)S.tile_base[chunk / kMcTileChunks].x + (int)(S.loc[chunk] & 0xFFFFu) +
             __popc(b.x & below) + __popc(b.y & below) + __popc(b.z & below);
    if (axis > 0) id += (b.x >> l) & 1;
    if (axis > 1) id += (b.y >> l) & 1;
    return id;
}

__global__ void __launch_bounds__(kMcThreads) mc_emit_kernel(const float* __restrict__ vol, McEmitArgs A, McScratch S,
                                                             const long long* __restrict__ totals,
                                                             float* __restrict__ verts, int* __restrict__ faces) {
    __shared__ unsigned char s_tri[256][3 * kMcTriMax];
    __shared__ unsigned char s_ntri[256];
    __shared__ unsigned char s_edge[12];
    for (int i = threadIdx.x; i < 256 * 3 * kMcTriMax; i += blockDim.x) (&s_tri[0][0])[i] = (&kMcTri[0][0])[i];
    s_ntri[threadIdx.x] = kMcNumTri[threadIdx.x];
    if (threadIdx.x < 12) s_edge[threadIdx.x] = kMcEdgeCorner[threadIdx.x];
    __syncthreads();
    if (totals[0] > INT_MAX || totals[1] > INT_MAX) return;      // the caller cannot have allocated the output
    const int lane = threadIdx.x & 31;
    const int sy = A.gx, sz = A.gx * A.gy, n = sz * A.gz;
    const int nchunks = (n + 31) >> 5;
    const unsigned below = (1u << lane) - 1u;
    for (int chunk = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; chunk < nchunks;
         chunk += (gridDim.x * blockDim.x) >> 5) {
        const uint4 b = S.bits[chunk];
        if ((b.x | b.y | b.z | b.w) == 0) continue;
        const int p = chunk * 32 + lane;
        const int x = p % A.gx, r = p / A.gx, y = r % A.gy, z = r / A.gy;
        const longlong2 base = S.tile_base[chunk / kMcTileChunks];
        const uint32_t loc = S.loc[chunk];
        // vertices of the edges this point owns
        const int own = ((b.x >> lane) & 1) | (((b.y >> lane) & 1) << 1) | (((b.z >> lane) & 1) << 2);
        if (own) {
            int id = (int)base.x + (int)(loc & 0xFFFFu) + __popc(b.x & below) + __popc(b.y & below) + __popc(b.z & below);
            const float v0 = __ldg(vol + p);
            const float p0[3] = {mc_coord(A, 0, x), mc_coord(A, 1, y), mc_coord(A, 2, z)};
            const int idx[3] = {x, y, z}, stride[3] = {1, sy, sz};
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                if (!((own >> a) & 1)) continue;
                const float v1 = __ldg(vol + p + stride[a]);
                const float t = __fdiv_rn(__fsub_rn(A.level, v0), __fsub_rn(v1, v0));
                const float pb = mc_coord(A, a, idx[a] + 1);
                float q[3] = {p0[0], p0[1], p0[2]};
                q[a] = __fadd_rn(p0[a], __fmul_rn(t, __fsub_rn(pb, p0[a])));
                verts[3LL * id] = q[0];
                verts[3LL * id + 1] = q[1];
                verts[3LL * id + 2] = q[2];
                ++id;
            }
        }
        // triangles of the cell this point anchors
        int cs = 0, nt = 0;
        if ((b.w >> lane) & 1) {
            cs = mc_case(vol, p, sy, sz, A.level);
            nt = s_ntri[cs];
        }
        int inc = nt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
        long long t = base.y + (loc >> 16) + inc - nt;
        for (int k = 0; k < 3 * nt; ++k) {
            const int e = s_tri[cs][k];
            const int c = s_edge[e];
            const int q = p + (c & 1) + ((c >> 1) & 1) * sy + ((c >> 2) & 1) * sz;
            faces[3 * t + k] = mc_vertex_id(S, q, e >> 2);
        }
    }
}

// Volume gradient at lattice point p = (x, y, z) in world units: central difference (v[i+1] - v[i-1]) /
// (c(i+1) - c(i-1)) per axis, one-sided at the grid's border. fp32, no contraction: the same value wherever it is
// evaluated.
__device__ __forceinline__ void mc_grad(const float* __restrict__ vol, const McEmitArgs& A, int p, const int idx[3],
                                        const int stride[3], float g[3]) {
    const int dims[3] = {A.gx, A.gy, A.gz};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int lo = idx[a] > 0 ? idx[a] - 1 : idx[a], hi = idx[a] + 1 < dims[a] ? idx[a] + 1 : idx[a];
        const float dv = __fsub_rn(__ldg(vol + p + (hi - idx[a]) * stride[a]), __ldg(vol + p + (lo - idx[a]) * stride[a]));
        g[a] = __fdiv_rn(dv, __fsub_rn(mc_coord(A, a, hi), mc_coord(A, a, lo)));
    }
}

// One warp per chunk with crossing edges, vertex ids as in mc_emit_kernel. Normal = -normalize((1-t) g(p0) + t g(p1))
// with emit's fp32 t; (0,0,0) when that vector is zero. Scaled by its largest component before the length, so small
// gradients neither underflow nor lose precision.
__global__ void __launch_bounds__(kMcThreads) mc_normals_kernel(const float* __restrict__ vol, McEmitArgs A, McScratch S,
                                                                const long long* __restrict__ totals,
                                                                float* __restrict__ normals) {
    if (totals[0] > INT_MAX || totals[1] > INT_MAX) return;      // the caller cannot have allocated the output
    const int lane = threadIdx.x & 31;
    const int sy = A.gx, sz = A.gx * A.gy, n = sz * A.gz;
    const int nchunks = (n + 31) >> 5;
    const unsigned below = (1u << lane) - 1u;
    for (int chunk = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; chunk < nchunks;
         chunk += (gridDim.x * blockDim.x) >> 5) {
        const uint4 b = S.bits[chunk];
        if ((b.x | b.y | b.z) == 0) continue;
        const int own = ((b.x >> lane) & 1) | (((b.y >> lane) & 1) << 1) | (((b.z >> lane) & 1) << 2);
        if (!own) continue;
        const int p = chunk * 32 + lane;
        const int x = p % A.gx, r = p / A.gx, y = r % A.gy, z = r / A.gy;
        int id = (int)S.tile_base[chunk / kMcTileChunks].x + (int)(S.loc[chunk] & 0xFFFFu) + __popc(b.x & below) +
                 __popc(b.y & below) + __popc(b.z & below);
        const float v0 = __ldg(vol + p);
        const int idx[3] = {x, y, z}, stride[3] = {1, sy, sz};
        float g0[3];
        mc_grad(vol, A, p, idx, stride, g0);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (!((own >> a) & 1)) continue;
            const float v1 = __ldg(vol + p + stride[a]);
            const float t = __fdiv_rn(__fsub_rn(A.level, v0), __fsub_rn(v1, v0));
            int idx1[3] = {x, y, z};
            ++idx1[a];
            float g1[3];
            mc_grad(vol, A, p + stride[a], idx1, stride, g1);
            const float s = __fsub_rn(1.0f, t);
            float q[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) q[c] = __fadd_rn(__fmul_rn(s, g0[c]), __fmul_rn(t, g1[c]));
            const float m = fmaxf(fabsf(q[0]), fmaxf(fabsf(q[1]), fabsf(q[2])));
            float nrm[3] = {0.0f, 0.0f, 0.0f};
            if (m > 0.0f) {
#pragma unroll
                for (int c = 0; c < 3; ++c) q[c] = __fdiv_rn(q[c], m);
                const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(q[0], q[0]), __fmul_rn(q[1], q[1])),
                                                       __fmul_rn(q[2], q[2])));
#pragma unroll
                for (int c = 0; c < 3; ++c) nrm[c] = -__fdiv_rn(q[c], len);
            }
            normals[3LL * id] = nrm[0];
            normals[3LL * id + 1] = nrm[1];
            normals[3LL * id + 2] = nrm[2];
            ++id;
        }
    }
}

}  // namespace jt

using namespace jt;

static bool mc_grid_ok(int gx, int gy, int gz) {
    return gx >= 2 && gy >= 2 && gz >= 2 && (long long)gx * gy * gz <= INT_MAX - 31;
}

extern "C" long long jt_mc_scratch_bytes(int gx, int gy, int gz) {
    if (!mc_grid_ok(gx, gy, gz)) return -1;
    const long long tiles = mc_tiles((long long)gx * gy * gz);
    return tiles * (long long)(sizeof(longlong2) + kMcTileChunks * (sizeof(uint4) + sizeof(uint32_t)) + sizeof(int2));
}

extern "C" int jt_mc_count(const float* vol, int gx, int gy, int gz, float level, void* scratch, long long* totals,
                           cudaStream_t stream) {
    JT_CHECK_ARG(vol && scratch && totals && mc_grid_ok(gx, gy, gz));
    JT_CHECK_ARG((reinterpret_cast<uintptr_t>(scratch) & 15) == 0);
    const long long tiles = mc_tiles((long long)gx * gy * gz);
    McScratch S = mc_scratch(scratch, tiles);
    mc_classify_kernel<<<(unsigned)tiles, kMcThreads, 0, stream>>>(vol, gx, gy, gz, level, S);
    mc_scan_kernel<<<1, 1024, 0, stream>>>(S, tiles, totals);
    g_launches += 2;
    JT_RETURN_LAUNCH();
}

// Launch set-up shared by the two per-vertex passes: lattice description and a persistent grid of warps over chunks.
static McEmitArgs mc_args(int gx, int gy, int gz, float level, const float* lin_x, const float* lin_y,
                          const float* lin_z, const float* h_aabb) {
    McEmitArgs A;
    A.lin[0] = lin_x; A.lin[1] = lin_y; A.lin[2] = lin_z;
    for (int a = 0; a < 3; ++a) { A.a0[a] = h_aabb[a]; A.a1[a] = h_aabb[3 + a]; }
    A.gx = gx; A.gy = gy; A.gz = gz; A.level = level;
    return A;
}

static int mc_chunk_grid(long long n) {
    const long long warps = (n + 31) / 32;
    const long long want = (warps + 7) / 8;
    return (int)(want < (long long)kNumSMs * 8 ? want : (long long)kNumSMs * 8);
}

extern "C" int jt_mc_emit(const float* vol, int gx, int gy, int gz, float level, const float* lin_x,
                          const float* lin_y, const float* lin_z, const float* h_aabb, const void* scratch,
                          const long long* totals, float* verts, int* faces, cudaStream_t stream) {
    JT_CHECK_ARG(vol && lin_x && lin_y && lin_z && h_aabb && scratch && totals && verts && faces);
    JT_CHECK_ARG(mc_grid_ok(gx, gy, gz) && (reinterpret_cast<uintptr_t>(scratch) & 15) == 0);
    const long long n = (long long)gx * gy * gz;
    McScratch S = mc_scratch(const_cast<void*>(scratch), mc_tiles(n));
    mc_emit_kernel<<<mc_chunk_grid(n), kMcThreads, 0, stream>>>(
        vol, mc_args(gx, gy, gz, level, lin_x, lin_y, lin_z, h_aabb), S, totals, verts, faces);
    ++g_launches;
    JT_RETURN_LAUNCH();
}

extern "C" int jt_mc_normals(const float* vol, int gx, int gy, int gz, float level, const float* lin_x,
                             const float* lin_y, const float* lin_z, const float* h_aabb, const void* scratch,
                             const long long* totals, float* normals, cudaStream_t stream) {
    JT_CHECK_ARG(vol && lin_x && lin_y && lin_z && h_aabb && scratch && totals && normals);
    JT_CHECK_ARG(mc_grid_ok(gx, gy, gz) && (reinterpret_cast<uintptr_t>(scratch) & 15) == 0);
    const long long n = (long long)gx * gy * gz;
    McScratch S = mc_scratch(const_cast<void*>(scratch), mc_tiles(n));
    mc_normals_kernel<<<mc_chunk_grid(n), kMcThreads, 0, stream>>>(
        vol, mc_args(gx, gy, gz, level, lin_x, lin_y, lin_z, h_aabb), S, totals, normals);
    ++g_launches;
    JT_RETURN_LAUNCH();
}
