// query.cuh — sm_100a kernels of the query side.
//
//   k_sat_nodes      a11-a12  batched separating-axis test: (location, node cube) -> Relation
//   k_propagate      a11      BFS semantics of NodeIdsIterator: a node is visited iff all ancestors passed
//   k_visible_eval   a17      per node: Relation vs the view frustum + relative_size_on_screen
//   k_cull_count / k_cull_write   a13-a15  decode + PointCulling::contains + interval filters +
//                                 order-preserving compaction (FilteredIterator, iterator.rs:96-119)
//   k_xray_accum / k_xray_resolve a19  discretise + per-pixel 1024-bit z-bucket set + grey mapping
//
// All arithmetic is binary64 in the reference's operation order (compiled with -fmad=false).
#pragma once
#include <cuda_runtime.h>

#include "chain.h"
#include "geometry_host.hpp"
#include "lod_order.h"

namespace pcv {

struct QNode {
    double m[3];
    double e;
    uint64_t point_off;
    uint64_t xyz_off;
    uint32_t n;
    int32_t enc;
    int32_t parent;
    int32_t level;
};

enum : uint8_t { REL_IN = 0, REL_CROSS = 1, REL_OUT = 2 };  // sat.rs:39-47

// Project the 8 corners of the cube (min m, edge e) on an axis: Aabb corners order x fastest (aabb.rs:114-125),
// max = min + edge (aabb.rs:175-181).
__device__ __forceinline__ void project_cube(const double m[3], double e, const double ax[3], double& lo, double& hi) {
    const double mx[3] = {m[0] + e, m[1] + e, m[2] + e};
    lo = 1.7976931348623157e308;
    hi = -1.7976931348623157e308;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const double cx = (i & 1) ? mx[0] : m[0], cy = (i & 2) ? mx[1] : m[1], cz = (i & 4) ? mx[2] : m[2];
        const double p = cx * ax[0] + cy * ax[1] + cz * ax[2];
        lo = fmin(lo, p);
        hi = fmax(hi, p);
    }
}

// sat() of sat.rs:174-194 with A = the location (projections precomputed in aproj) and B = the node cube.
__device__ __forceinline__ uint8_t sat_cube(const QueryGeom& g, const double (*aproj)[2], const double m[3], double e) {
    uint8_t rel = REL_IN;
    for (int k = 0; k < g.naxes; ++k) {
        double bmin, bmax;
        project_cube(m, e, g.axes[k], bmin, bmax);
        const double amin = aproj[k][0], amax = aproj[k][1];
        if (bmin > amax || bmax < amin) return REL_OUT;
        if (amin > bmin || bmax > amax) rel = REL_CROSS;
    }
    return rel;
}

__device__ __forceinline__ void project_location(const QueryGeom& g, double (*aproj)[2]) {
    for (int k = threadIdx.x; k < g.naxes; k += blockDim.x) {
        double lo = 1.7976931348623157e308, hi = -1.7976931348623157e308;
        for (int i = 0; i < 8; ++i) {
            const double p = g.corners[i][0] * g.axes[k][0] + g.corners[i][1] * g.axes[k][1] + g.corners[i][2] * g.axes[k][2];
            lo = fmin(lo, p);
            hi = fmax(hi, p);
        }
        aproj[k][0] = lo;
        aproj[k][1] = hi;
    }
}

// grid = (ceil(nnodes/256), nloc).  rel[loc * nnodes + node]
__global__ void __launch_bounds__(256) k_sat_nodes(const QueryGeom* __restrict__ geoms, const QNode* __restrict__ nodes, uint32_t nnodes,
                                                   uint8_t* __restrict__ rel) {
    __shared__ double aproj[26][2];
    const QueryGeom& g = geoms[blockIdx.y];
    project_location(g, aproj);
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nnodes) return;
    uint8_t r = REL_IN;
    if (g.kind != PCV_LOC_ALL) {
        const QNode nd = nodes[i];
        r = sat_cube(g, aproj, nd.m, nd.e);
    }
    rel[(size_t)blockIdx.y * nnodes + i] = r;
}

// One block per location; nodes are sorted by level so parents precede children.  pass = not Out && parent passed.
__global__ void __launch_bounds__(1024) k_propagate(const QNode* __restrict__ nodes, const uint32_t* __restrict__ level_start, int nlevels,
                                                    uint32_t nnodes, uint8_t* __restrict__ rel, uint8_t* __restrict__ pass) {
    uint8_t* r = rel + (size_t)blockIdx.x * nnodes;
    uint8_t* p = pass + (size_t)blockIdx.x * nnodes;
    for (int L = 0; L < nlevels; ++L) {
        for (uint32_t i = level_start[L] + threadIdx.x; i < level_start[L + 1]; i += blockDim.x) {
            const int par = nodes[i].parent;
            p[i] = (r[i] != REL_OUT && (par < 0 || p[par])) ? 1 : 0;
        }
        __syncthreads();
    }
}

// relative_size_on_screen (octree/mod.rs:103-139): project the 8 cube corners with the 4x4 (homogeneous divide),
// clamp to [-1,1]^2 x [0,1], grow an Aabb, return diag.x * diag.y.  bad[0] is set if any w == 0 (reference panics).
__device__ __forceinline__ double num_clamp_d(double x, double lo, double hi) { return x < lo ? lo : (x > hi ? hi : x); }
__global__ void __launch_bounds__(256) k_visible_eval(const QueryGeom* __restrict__ geom, const double* __restrict__ M,
                                                      const QNode* __restrict__ nodes, uint32_t nnodes, uint8_t* __restrict__ rel,
                                                      double* __restrict__ size) {
    __shared__ double aproj[26][2];
    const QueryGeom& g = geom[0];
    project_location(g, aproj);
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nnodes) return;
    const QNode nd = nodes[i];
    uint8_t relv = sat_cube(g, aproj, nd.m, nd.e);
    const double mn[3] = {nd.m[0], nd.m[1], nd.m[2]}, mx[3] = {nd.m[0] + nd.e, nd.m[1] + nd.e, nd.m[2] + nd.e};
    double lo[2] = {0, 0}, hi[2] = {0, 0};
    // corner order of mod.rs:122-137: min, max, then 6 mixed corners (order is irrelevant for min/max)
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const double px = (c & 1) ? mx[0] : mn[0], py = (c & 2) ? mx[1] : mn[1], pz = (c & 4) ? mx[2] : mn[2];
        double q[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            double a = M[r] * px;
            a = M[4 + r] * py + a;
            a = M[8 + r] * pz + a;
            a = M[12 + r] * 1.0 + a;
            q[r] = a;
        }
        if (q[3] == 0.0) relv |= 0x80;  // Point3::from_homogeneous(..).unwrap() panics for this node (mod.rs:103-106) - if it is ever pushed
        const double x = num_clamp_d(q[0] / q[3], -1., 1.), y = num_clamp_d(q[1] / q[3], -1., 1.);
        if (c == 0) {
            lo[0] = hi[0] = x;
            lo[1] = hi[1] = y;
        } else {
            lo[0] = fmin(lo[0], x);
            hi[0] = fmax(hi[0], x);
            lo[1] = fmin(lo[1], y);
            hi[1] = fmax(hi[1], y);
        }
    }
    size[i] = (hi[0] - lo[0]) * (hi[1] - lo[1]);
    rel[i] = relv;
}

// ---- per-point culling -----------------------------------------------------------------------------
__device__ __forceinline__ bool loc_contains(const QueryGeom& g, double x, double y, double z) {
    if (g.kind == PCV_LOC_AABB) {  // aabb.rs:46-48
        return g.aabb_min[0] <= x && g.aabb_min[1] <= y && g.aabb_min[2] <= z && x < g.aabb_max[0] && y < g.aabb_max[1] && z < g.aabb_max[2];
    }
    if (g.kind == PCV_LOC_FRUSTUM) {  // frustum.rs:120-125
        // q = clip_from_query.transform_point(p) divides by the homogeneous w, then every component must lie strictly inside
        // (-1, 1).  The three IEEE divisions dominate the point test, and they only matter within an ulp of the planes:
        // |fl(r / w)| < 1  <=>  |r / w| < 1 - 2^-54 (the midpoint below 1 rounds to 1), so with T = fl(|w| (1 - 2^-52)) <
        // |w| (1 - 2^-54):  |r| <= T is certainly inside,  |r| >= |w| certainly outside;  only the band in between (and
        // w == 0, tiny, huge or NaN) takes the divisions.  Same result as the reference's arithmetic for every input.
        const double* m = g.clip_from_query;
        double n = m[3] * x;
        n = n + m[7] * y;
        n = n + m[11] * z;
        n = n + m[15];
        double r[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            double a = m[i] * x;
            a = m[4 + i] * y + a;
            a = m[8 + i] * z + a;
            r[i] = a + m[12 + i];
        }
        const double an = fabs(n);
        if (an > 1e-290 && an < 1e300) {
            const double T = an * 0.99999999999999977795539507496869;  // 1 - 2^-52
            bool sure = true, inside = true;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const double ar = fabs(r[i]);
                if (ar >= an)
                    inside = false;
                else if (!(ar <= T))
                    sure = false;
            }
            if (!inside) return false;
            if (sure) return true;
        }
        double c[3] = {r[0], r[1], r[2]};
        if (n != 0.0) {
            c[0] = r[0] / n;
            c[1] = r[1] / n;
            c[2] = r[2] / n;
        }
        const double mn = fmin(fmin(c[0], c[1]), c[2]), mx = fmax(fmax(c[0], c[1]), c[2]);
        return mn > -1.0 && mx < 1.0;
    }
    if (g.kind == PCV_LOC_OBB) {  // obb.rs:83-90
        const V3 q = iso_apply(g.obb_from_query, V3{x, y, z});
        return fabs(q.x) <= g.half_extent[0] && fabs(q.y) <= g.half_extent[1] && fabs(q.z) <= g.half_extent[2];
    }
    return true;  // AllPoints, math/mod.rs:157-161
}

struct QTile {
    uint32_t loc;
    uint32_t node;
    uint32_t first;   // first point of the tile inside the node
    uint32_t count;
};
constexpr uint32_t kQueryTile = 2048;

struct CullArgs {
    const QueryGeom* geoms;
    const QNode* nodes;
    const QTile* tiles;
    const uint8_t* xyz;
    const uint8_t* rgb;
    const float* intensity;
    const uint32_t* src;
    const pcv_interval* filters;
    uint32_t nfilt;
    uint32_t* tile_keep;     // count pass output, then (after the scan) exclusive offsets
    double* out_xyz;         // write pass outputs (AoS)
    uint8_t* out_rgb;
    float* out_intensity;
    uint32_t* out_src;
    uint32_t* out_loc;       // k_cull_fused only (may be null): the location index of every survivor
};

__device__ __forceinline__ uint64_t load_code(const uint8_t* p, int enc) {
    if (enc == ENC_U8) return *p;
    if (enc == ENC_U16) return *reinterpret_cast<const uint16_t*>(p);
    if (enc == ENC_F32) return *reinterpret_cast<const uint32_t*>(p);
    return *reinterpret_cast<const uint64_t*>(p);
}

__device__ __forceinline__ bool eval_point(const CullArgs& a, const QueryGeom& g, const QNode& nd, uint32_t i, double p[3]) {
    const int bpc = enc_bytes(nd.enc);
    const uint8_t* s = a.xyz + nd.xyz_off + (uint64_t)i * 3 * bpc;
#pragma unroll
    for (int k = 0; k < 3; ++k) p[k] = decode1_fast(load_code(s + k * bpc, nd.enc), nd.m[k], nd.e, nd.enc);  // == decode1, integer-built unit fraction
    bool keep = loc_contains(g, p[0], p[1], p[2]);
    if (a.nfilt) {
        const double v = (double)a.intensity[nd.point_off + i];  // iterator.rs:82-91: attribute as f64, closed interval
        for (uint32_t f = 0; f < a.nfilt; ++f) keep = keep && (a.filters[f].lo <= v && v <= a.filters[f].hi);
    }
    return keep;
}

template <bool WRITE>
__global__ void __launch_bounds__(256) k_cull(const __grid_constant__ CullArgs a) {
    __shared__ uint32_t warp_cnt[8];
    __shared__ uint32_t running;
    const QTile t = a.tiles[blockIdx.x];
    const QueryGeom& g = a.geoms[t.loc];
    const QNode nd = a.nodes[t.node];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) running = WRITE ? a.tile_keep[blockIdx.x] : 0u;
    __syncthreads();
    for (uint32_t r0 = 0; r0 < t.count; r0 += 256) {
        const uint32_t i = r0 + threadIdx.x;
        double p[3] = {0, 0, 0};
        bool keep = false;
        if (i < t.count) keep = eval_point(a, g, nd, t.first + i, p);
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) warp_cnt[warp] = __popc(bal);
        __syncthreads();
        uint32_t before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const uint32_t c = warp_cnt[w];
            if (w < warp) before += c;
            total += c;
        }
        if (WRITE && keep) {
            const uint64_t dst = (uint64_t)running + before + __popc(bal & ((1u << lane) - 1u));
            const uint64_t sp = nd.point_off + t.first + i;
            a.out_xyz[3 * dst] = p[0];
            a.out_xyz[3 * dst + 1] = p[1];
            a.out_xyz[3 * dst + 2] = p[2];
            a.out_rgb[3 * dst] = a.rgb[3 * sp];
            a.out_rgb[3 * dst + 1] = a.rgb[3 * sp + 1];
            a.out_rgb[3 * dst + 2] = a.rgb[3 * sp + 2];
            if (a.out_intensity) a.out_intensity[dst] = a.intensity[sp];
            a.out_src[dst] = a.src[sp];
        }
        __syncthreads();
        if (threadIdx.x == 0) running += total;
        __syncthreads();
    }
    if (!WRITE && threadIdx.x == 0) a.tile_keep[blockIdx.x] = running;
}

// Exclusive scan of n u32 values in place; total (u64) to *total_out.  Single block; n is at most a few million tiles.
__global__ void __launch_bounds__(1024) k_scan_u32(uint32_t* v, uint32_t n, unsigned long long* total_out) {
    __shared__ uint32_t wsum[32];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t x = i < n ? v[i] : 0u;
        uint32_t incl = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += y;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            uint32_t s = wsum[lane], si = s;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, si, o);
                if (lane >= o) si += y;
            }
            wsum[lane] = si - s;  // exclusive over warps
        }
        __syncthreads();
        const unsigned long long c = carry;
        if (i < n) v[i] = (uint32_t)(c + wsum[warp] + (incl - x));
        __syncthreads();
        if (threadIdx.x == 1023) carry = c + wsum[warp] + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total_out = carry;
}

// Work list of the batched query: one QTile per kQueryTile points of every (location, node) pair that passed.
// The order of the list is irrelevant for the batched form (only per-location totals and the compacted survivors
// are produced), so tiles are appended with one atomic per pair.
__global__ void __launch_bounds__(256) k_count_tiles(const uint8_t* __restrict__ pass, const QNode* __restrict__ nodes, uint32_t nnodes,
                                                     uint64_t npairs, unsigned long long* __restrict__ total) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long c = 0;
    if (i < npairs && pass[i]) c = (nodes[i % nnodes].n + kQueryTile - 1) / kQueryTile;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(total, c);
}
__global__ void __launch_bounds__(256) k_fill_tiles(const uint8_t* __restrict__ pass, const QNode* __restrict__ nodes, uint32_t nnodes,
                                                    uint64_t npairs, unsigned long long* __restrict__ cursor, QTile* __restrict__ tiles) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npairs || !pass[i]) return;
    const uint32_t node = (uint32_t)(i % nnodes), loc = (uint32_t)(i / nnodes);
    const uint32_t n = nodes[node].n;
    if (n == 0) return;
    const uint32_t nt = (n + kQueryTile - 1) / kQueryTile;
    const unsigned long long base = atomicAdd(cursor, (unsigned long long)nt);
    for (uint32_t k = 0; k < nt; ++k) tiles[base + k] = QTile{loc, node, k * kQueryTile, min(kQueryTile, n - k * kQueryTile)};
}

// per-location totals: kept[loc] += keep counts, tested[loc] += tile counts
__global__ void k_tile_totals(const QTile* tiles, const uint32_t* keep_counts, uint32_t ntiles, unsigned long long* kept,
                              unsigned long long* tested) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ntiles) return;
    atomicAdd(&kept[tiles[i].loc], (unsigned long long)keep_counts[i]);
    atomicAdd(&tested[tiles[i].loc], (unsigned long long)tiles[i].count);
}

// ---- LOD draw order applied at build time (lod_order.h): gather every node's points into their shuffled order ------------------
struct LodArgs {
    const QNode* nodes;
    const QTile* tiles;  // (node, first, count) pieces of every node; loc unused
    const uint64_t* keys;  // [nnodes] permutation key of every node
    const uint8_t* xyz;
    const uint8_t* rgb;
    const float* intensity;
    const uint32_t* src;
    uint8_t* out_xyz;
    uint8_t* out_rgb;
    float* out_intensity;
    uint32_t* out_src;
};
__global__ void __launch_bounds__(256) k_lod_shuffle(const __grid_constant__ LodArgs a, uint32_t ntiles) {
    for (uint32_t ti = blockIdx.x; ti < ntiles; ti += gridDim.x) {
        const QTile t = a.tiles[ti];
        const QNode nd = a.nodes[t.node];
        const uint64_t key = a.keys[t.node];
        const int bpc = enc_bytes(nd.enc);
        for (uint32_t k = threadIdx.x; k < t.count; k += blockDim.x) {
            const uint32_t i = t.first + k, j = lod_order(key, nd.n, i);  // new[i] = old[j]
            const uint8_t* sx = a.xyz + nd.xyz_off + (uint64_t)j * 3 * bpc;
            uint8_t* dx = a.out_xyz + nd.xyz_off + (uint64_t)i * 3 * bpc;
            if (bpc == 1) {
                dx[0] = sx[0], dx[1] = sx[1], dx[2] = sx[2];
            } else if (bpc == 2) {
                const uint16_t* s16 = reinterpret_cast<const uint16_t*>(sx);
                uint16_t* d16 = reinterpret_cast<uint16_t*>(dx);
                d16[0] = s16[0], d16[1] = s16[1], d16[2] = s16[2];
            } else if (bpc == 4) {
                const uint32_t* s32 = reinterpret_cast<const uint32_t*>(sx);
                uint32_t* d32 = reinterpret_cast<uint32_t*>(dx);
                d32[0] = s32[0], d32[1] = s32[1], d32[2] = s32[2];
            } else {
                const uint64_t* s64 = reinterpret_cast<const uint64_t*>(sx);
                uint64_t* d64 = reinterpret_cast<uint64_t*>(dx);
                d64[0] = s64[0], d64[1] = s64[1], d64[2] = s64[2];
            }
            const uint64_t sp = nd.point_off + j, dp = nd.point_off + i;
            a.out_rgb[3 * dp] = a.rgb[3 * sp];
            a.out_rgb[3 * dp + 1] = a.rgb[3 * sp + 1];
            a.out_rgb[3 * dp + 2] = a.rgb[3 * sp + 2];
            a.out_src[dp] = a.src[sp];
            if (a.out_intensity) a.out_intensity[dp] = a.intensity[sp];
        }
    }
}

// ---- batched query: hierarchical node selection + single-pass culling ---------------------------------------------
// nodes_in_location for many locations at once, level by level like NodeIdsIterator (octree_iterator.rs:30-43): a frontier of
// (location, node) pairs; every pair is tested once (sat.rs:174-194), a pair that is not Out joins the work list (if the node
// holds points) and hands its existing children to the next level's frontier.  Only visited nodes are ever tested - the
// all-pairs kernel above (k_sat_nodes) stays for the single-location entry points that need the BFS order.
struct LocProj {
    double a[26][2];  // projections of the location's 8 corners on each of its cached axes
};
__global__ void __launch_bounds__(32) k_loc_proj(const QueryGeom* __restrict__ geoms, LocProj* __restrict__ out) {
    project_location(geoms[blockIdx.x], out[blockIdx.x].a);
}
struct BfsArgs {
    const QueryGeom* geoms;
    const LocProj* proj;
    const QNode* nodes;
    const int32_t* children;  // [nnodes][8]
    const uint2* fin;
    uint2* fout;
    const uint32_t* nin;   // size of the incoming frontier (device resident)
    uint32_t* nout;
    uint32_t cap;          // frontier / pair list capacity
    uint2* pairs;          // (location, node) pairs to cull
    uint32_t* npairs;
    unsigned long long* ntiles;
    unsigned long long* tested;  // [nloc] points of the nodes the location visits
    unsigned long long* bytes;   // sum of n * (3 bpc + 3) over the visited pairs
    int* overflow;
};
constexpr uint32_t kQueryTileBfs = 2048;
__global__ void __launch_bounds__(256) k_bfs_level(const __grid_constant__ BfsArgs a) {
    const uint32_t n = min(*a.nin, a.cap);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint2 pr = a.fin[i];
        const QueryGeom& g = a.geoms[pr.x];
        const QNode nd = a.nodes[pr.y];
        uint8_t rel = REL_IN;
        if (g.kind != PCV_LOC_ALL) rel = sat_cube(g, a.proj[pr.x].a, nd.m, nd.e);
        if (rel == REL_OUT) continue;
        if (nd.n) {
            const uint32_t k = atomicAdd(a.npairs, 1u);
            if (k < a.cap)
                a.pairs[k] = pr;
            else
                *a.overflow = 1;
            atomicAdd(a.ntiles, (unsigned long long)((nd.n + kQueryTileBfs - 1) / kQueryTileBfs));
            atomicAdd(&a.tested[pr.x], (unsigned long long)nd.n);
            atomicAdd(a.bytes, (unsigned long long)nd.n * (3ull * (unsigned long long)enc_bytes(nd.enc) + 3ull));
        }
        const int32_t* ch = a.children + (size_t)pr.y * 8;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int32_t cn = ch[c];
            if (cn < 0) continue;
            const uint32_t k = atomicAdd(a.nout, 1u);
            if (k < a.cap)
                a.fout[k] = make_uint2(pr.x, (uint32_t)cn);
            else
                *a.overflow = 1;
        }
    }
}
__global__ void __launch_bounds__(256) k_bfs_seed(uint2* f, uint32_t nloc, uint32_t root, uint32_t* n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nloc) f[i] = make_uint2(i, root);
    if (i == 0) *n = nloc;
}
__global__ void __launch_bounds__(256) k_pairs_to_tiles(const uint2* __restrict__ pairs, const uint32_t* __restrict__ npairs, uint32_t cap,
                                                        const QNode* __restrict__ nodes, unsigned long long* __restrict__ cursor, QTile* __restrict__ tiles) {
    const uint32_t n = min(*npairs, cap);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint2 pr = pairs[i];
        const uint32_t cnt = nodes[pr.y].n;
        const uint32_t nt = (cnt + kQueryTile - 1) / kQueryTile;
        const unsigned long long base = atomicAdd(cursor, (unsigned long long)nt);
        for (uint32_t k = 0; k < nt; ++k) tiles[base + k] = QTile{pr.x, pr.y, k * kQueryTile, min(kQueryTile, cnt - k * kQueryTile)};
    }
}

// FilteredIterator (iterator.rs:96-119) over one tile, in ONE pass: the tile's position bytes are staged in shared memory with
// 16-byte loads (node blocks and 2048-point tiles are 16-byte aligned), every point is decoded and tested once; per round of
// 256 points the block counts its survivors with ballots, reserves their output range with one atomic, stages them in shared
// memory and copies them out as contiguous words (the order inside a round is kept; rounds land in the order they finish -
// the batched form only promises per-location totals and the compacted set).  Survivors beyond `cap` are counted, not stored.
// With out_loc set, every stored survivor also gets the index of its location.
struct CullFusedArgs {
    CullArgs c;
    unsigned long long* cursor;  // output slots handed out so far
    unsigned long long cap;
    unsigned long long* kept;    // [nloc]
};
constexpr uint32_t kCullStage = kQueryTile * 12 + 32;  // F32 codes: the widest staged encoding
__device__ __forceinline__ void decode_staged(const uint8_t* s, uint32_t i, const QNode& nd, double p[3]) {
    if (nd.enc == ENC_U8) {
        const uint8_t* q = s + 3 * i;
#pragma unroll
        for (int k = 0; k < 3; ++k) p[k] = decode_axis<ENC_U8>(q[k], nd.m[k], nd.e);
    } else if (nd.enc == ENC_U16) {
        const uint16_t* q = reinterpret_cast<const uint16_t*>(s) + 3 * i;
#pragma unroll
        for (int k = 0; k < 3; ++k) p[k] = decode_axis<ENC_U16>(q[k], nd.m[k], nd.e);
    } else {
        const uint32_t* q = reinterpret_cast<const uint32_t*>(s) + 3 * i;
#pragma unroll
        for (int k = 0; k < 3; ++k) p[k] = decode_axis<ENC_F32>(q[k], nd.m[k], nd.e);
    }
}
__global__ void __launch_bounds__(256) k_cull_fused(const __grid_constant__ CullFusedArgs f, uint32_t ntiles) {
    __shared__ __align__(16) uint8_t sxyz[kCullStage];
    // survivors of one round of 256 points, staged so that the copy-out is contiguous 8 / 4 / 1-byte-per-lane stores
    __shared__ __align__(16) double st_xyz[256 * 3];
    __shared__ uint32_t st_src[256];
    __shared__ float st_int[256];
    __shared__ uint8_t st_rgb[256 * 3];
    __shared__ uint32_t wcnt[8];
    __shared__ unsigned long long sbase;
    const CullArgs& a = f.c;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t ti = blockIdx.x; ti < ntiles; ti += gridDim.x) {
        const QTile t = a.tiles[ti];
        const QueryGeom& g = a.geoms[t.loc];
        const QNode nd = a.nodes[t.node];
        const bool staged = nd.enc != ENC_F64;
        const int bpc = enc_bytes(nd.enc);
        const uint8_t* src = a.xyz + nd.xyz_off + (uint64_t)t.first * 3 * bpc;
        if (staged) {
            const uint32_t nvec = (t.count * 3u * (uint32_t)bpc + 15u) >> 4;
            for (uint32_t v = threadIdx.x; v < nvec; v += 256) reinterpret_cast<uint4*>(sxyz)[v] = __ldcg(reinterpret_cast<const uint4*>(src) + v);
        }
        __syncthreads();
        uint32_t kept_tile = 0;  // thread 0 only
        for (uint32_t r0 = 0; r0 < t.count; r0 += 256) {
            const uint32_t i = r0 + threadIdx.x;
            bool keep = false;
            double p[3] = {0, 0, 0};
            if (i < t.count) {
                if (staged) {
                    decode_staged(sxyz, i, nd, p);
                } else {
#pragma unroll
                    for (int k = 0; k < 3; ++k) p[k] = decode1_fast(load_code(src + ((size_t)i * 3 + k) * bpc, nd.enc), nd.m[k], nd.e, nd.enc);
                }
                keep = loc_contains(g, p[0], p[1], p[2]);
                if (a.nfilt) {
                    const double v = (double)a.intensity[nd.point_off + t.first + i];  // iterator.rs:82-91
                    for (uint32_t q = 0; q < a.nfilt; ++q) keep = keep && (a.filters[q].lo <= v && v <= a.filters[q].hi);
                }
            }
            const unsigned bal = __ballot_sync(0xffffffffu, keep);
            if (lane == 0) wcnt[warp] = __popc(bal);
            __syncthreads();
            uint32_t before = 0, total = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                const uint32_t c = wcnt[w];
                if (w < warp) before += c;
                total += c;
            }
            if (total == 0) {  // uniform: nothing survived this round
                __syncthreads();
                continue;
            }
            if (threadIdx.x == 0) {
                sbase = atomicAdd(f.cursor, (unsigned long long)total);  // one reservation per round: the round's survivors stay contiguous
                kept_tile += total;
            }
            if (keep) {
                const uint32_t li = before + __popc(bal & ((1u << lane) - 1u));
                const uint64_t sp = nd.point_off + t.first + i;
                st_xyz[3 * li] = p[0];
                st_xyz[3 * li + 1] = p[1];
                st_xyz[3 * li + 2] = p[2];
                st_rgb[3 * li] = a.rgb[3 * sp];
                st_rgb[3 * li + 1] = a.rgb[3 * sp + 1];
                st_rgb[3 * li + 2] = a.rgb[3 * sp + 2];
                st_src[li] = a.src[sp];
                if (a.out_intensity) st_int[li] = a.intensity[sp];
            }
            __syncthreads();
            const unsigned long long base = sbase;
            const uint32_t room = base >= f.cap ? 0u : (uint32_t)min((unsigned long long)total, f.cap - base);
            for (uint32_t k = threadIdx.x; k < 3 * room; k += 256) a.out_xyz[3 * base + k] = st_xyz[k];
            for (uint32_t k = threadIdx.x; k < 3 * room; k += 256) a.out_rgb[3 * base + k] = st_rgb[k];
            for (uint32_t k = threadIdx.x; k < room; k += 256) {
                a.out_src[base + k] = st_src[k];
                if (a.out_intensity) a.out_intensity[base + k] = st_int[k];
                if (a.out_loc) a.out_loc[base + k] = t.loc;  // tile-uniform: no staging
            }
            __syncthreads();  // the staging arrays and wcnt are reused by the next round
        }
        if (threadIdx.x == 0 && kept_tile) atomicAdd(&f.kept[t.loc], (unsigned long long)kept_tile);
        __syncthreads();  // sxyz is reused by the next tile
    }
}

// ---- X-ray -----------------------------------------------------------------------------------------
// Pixels no point falls into get TRANSPARENT.to_u8() = (255, 255, 255, 0) (src/color.rs:154-159, generation.rs:506-511).
constexpr uint32_t kXrayTransparent = 0x00FFFFFFu;  // r | g << 8 | b << 16 | a << 24
__global__ void __launch_bounds__(256) k_fill_u32(uint32_t* __restrict__ dst, uint32_t value, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = value;
}
struct XrayArgs {
    QueryGeom geom;
    const QNode* nodes;
    const QTile* tiles;
    const uint8_t* xyz;
    double tmin[3], tdiag[3];
    double rdiag[3];  // RN(1 / tdiag) for div_known (chain.h): the correctly rounded quotient without the division instruction
    int div_ok;       // every tdiag is admissible for div_known (host check), else the IEEE operator
    double query_from_global[7];
    int has_q;
    uint32_t w, h;
    uint32_t* zbits;   // w*h*32
    uint8_t* zover;    // w*h
    int* any;
};

// (p - tmin) / tdiag of one axis (process_point_data, generation.rs:108-127), bit-identical to the IEEE quotient
__device__ __forceinline__ double xray_unit(const XrayArgs& a, int k, double p) {
    const double d = p - a.tmin[k];
    return a.div_ok ? div_known(d, a.tdiag[k], a.rdiag[k]) : d / a.tdiag[k];
}

// Rust `f64 as u32`: truncating, saturating, NaN -> 0.  cvt.rzi.u32.f64 saturates but returns 0x80000000 for NaN (measured).
__device__ __forceinline__ uint32_t rust_as_u32_dev(double v) {
    const uint32_t u = __double2uint_rz(v);
    return v != v ? 0u : u;
}

__global__ void __launch_bounds__(256) k_xray_accum(const __grid_constant__ XrayArgs a) {
    const QTile t = a.tiles[blockIdx.x];
    const QNode nd = a.nodes[t.node];
    const int bpc = enc_bytes(nd.enc);
    bool seen = false;
    for (uint32_t i = threadIdx.x; i < t.count; i += blockDim.x) {
        const uint8_t* s = a.xyz + nd.xyz_off + (uint64_t)(t.first + i) * 3 * bpc;
        double p[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) p[k] = decode1_fast(load_code(s + k * bpc, nd.enc), nd.m[k], nd.e, nd.enc);  // == decode1, integer-built unit fraction
        if (!loc_contains(a.geom, p[0], p[1], p[2])) continue;
        seen = true;
        if (a.has_q) {  // generation.rs:493-497
            const V3 q = iso_apply(a.query_from_global, V3{p[0], p[1], p[2]});
            p[0] = q.x;
            p[1] = q.y;
            p[2] = q.z;
        }
        // process_point_data, generation.rs:108-127 (`as u32` saturates, NaN -> 0)
        const uint32_t x = rust_as_u32_dev(xray_unit(a, 0, p[0]) * (double)a.w);
        const uint32_t y = rust_as_u32_dev((1. - xray_unit(a, 1, p[1])) * (double)a.h);
        const uint32_t z = rust_as_u32_dev(xray_unit(a, 2, p[2]) * 1024.);
        if (x < a.w && y < a.h) {
            const size_t px = (size_t)y * a.w + x;
            if (z < 1024)
                atomicOr(&a.zbits[px * 32 + (z >> 5)], 1u << (z & 31));
            else
                a.zover[px] = 1;
        }
    }
    if (__syncthreads_or(seen) && threadIdx.x == 0) atomicExch(a.any, 1);
}

// The same accumulation with the z-bucket sets in SHARED memory (the global-memory form above needs 128 B per pixel: 2 GiB for
// a 4096 x 4096 tile, written and read once more than it is used).  The points are first binned by 32 x 32 pixel sub-tile of
// the image with a counting sort of 4-byte keys (k_xray_bin<0>: count, k_xray_bin<1>: place; octree nodes are spatially
// coherent, so the lanes of a warp mostly share their sub-tile and the atomics are issued once per warp and sub-tile), then
// one block per non-empty sub-tile ORs its keys into 1024 pixels x 1024 bits of shared memory (128 KB) and resolves them to
// RGBA itself.  Per-point arithmetic and the pixel / bucket indices are exactly those of k_xray_accum.
constexpr uint32_t kXraySub = 32;  // sub-tile edge in pixels
struct XrayBinArgs {
    XrayArgs x;               // geom, nodes, tiles, xyz, tile box, transform, w, h, any
    uint32_t ntiles;
    uint32_t sub_w;           // sub-tiles per row
    uint32_t* sub_count;      // [nsub] points per sub-tile; after the scan: exclusive offsets
    uint32_t* sub_cursor;     // [nsub] place pass: keys written so far
    uint32_t* keys;           // ly << 16 | lx << 11 | min(z, 1024)
};
template <int PLACE>
__global__ void __launch_bounds__(256) k_xray_bin(const __grid_constant__ XrayBinArgs b) {
    const XrayArgs& a = b.x;
    const int lane = threadIdx.x & 31;
    for (uint32_t ti = blockIdx.x; ti < b.ntiles; ti += gridDim.x) {
        const QTile t = a.tiles[ti];
        const QNode nd = a.nodes[t.node];
        const int bpc = enc_bytes(nd.enc);
        for (uint32_t i0 = 0; i0 < t.count; i0 += blockDim.x) {
            const uint32_t i = i0 + threadIdx.x;
            uint32_t sub = 0xFFFFFFFFu, key = 0;
            if (i < t.count) {
                const uint8_t* s = a.xyz + nd.xyz_off + (uint64_t)(t.first + i) * 3 * bpc;
                double p[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) p[k] = decode1_fast(load_code(s + k * bpc, nd.enc), nd.m[k], nd.e, nd.enc);
                if (loc_contains(a.geom, p[0], p[1], p[2])) {
                    if (a.has_q) {  // generation.rs:493-497
                        const V3 q = iso_apply(a.query_from_global, V3{p[0], p[1], p[2]});
                        p[0] = q.x, p[1] = q.y, p[2] = q.z;
                    }
                    // process_point_data, generation.rs:108-127 (`as u32` saturates, NaN -> 0)
                    const uint32_t x = rust_as_u32_dev(xray_unit(a, 0, p[0]) * (double)a.w);
                    const uint32_t y = rust_as_u32_dev((1. - xray_unit(a, 1, p[1])) * (double)a.h);
                    const uint32_t z = rust_as_u32_dev(xray_unit(a, 2, p[2]) * 1024.);
                    if (x < a.w && y < a.h) {
                        sub = (y / kXraySub) * b.sub_w + (x / kXraySub);
                        key = ((y % kXraySub) << 16) | ((x % kXraySub) << 11) | min(z, 1024u);
                    }
                }
            }
            // one atomic per warp and distinct sub-tile
            const unsigned mask = __match_any_sync(0xffffffffu, sub);
            if (sub != 0xFFFFFFFFu) {
                const int leader = __ffs(mask) - 1;
                const uint32_t rank = __popc(mask & ((1u << lane) - 1u));
                if (PLACE) {
                    uint32_t base = 0;
                    if (lane == leader) base = atomicAdd(&b.sub_cursor[sub], (uint32_t)__popc(mask));
                    base = __shfl_sync(mask, base, leader);
                    b.keys[b.sub_count[sub] + base + rank] = key;
                } else if (lane == leader) {
                    atomicAdd(&b.sub_count[sub], (uint32_t)__popc(mask));
                }
            }
        }
    }
}
struct XraySubArgs {
    const uint32_t* sub_id;     // unused (every sub-tile has a block; empty ones leave at once)
    const uint32_t* sub_off;    // [nsub + 1] exclusive offsets into keys
    const uint32_t* keys;
    const uint8_t* grey;        // [1026]
    uint8_t* rgba;              // w * h * 4, zero-initialised
    uint32_t* zbits_out;        // optional: w * h * 32, zero-initialised
    uint32_t sub_w, w, h;
};
__global__ void __launch_bounds__(512, 1) k_xray_subtile(const __grid_constant__ XraySubArgs b) {
    extern __shared__ __align__(16) uint32_t sbits[];  // [1024 pixels][32 words]
    __shared__ uint8_t sover[kXraySub * kXraySub];
    const uint32_t sid = blockIdx.x;
    const uint32_t k0 = b.sub_off[sid], k1 = b.sub_off[sid + 1];
    if (k1 == k0) return;  // no point falls into this sub-tile: its pixels stay transparent (the image is pre-filled with TRANSPARENT)
    const uint32_t px0 = (sid % b.sub_w) * kXraySub, py0 = (sid / b.sub_w) * kXraySub;
    {
        uint4* z4 = reinterpret_cast<uint4*>(sbits);
        for (uint32_t i = threadIdx.x; i < kXraySub * kXraySub * 8; i += blockDim.x) z4[i] = make_uint4(0, 0, 0, 0);
    }
    for (uint32_t i = threadIdx.x; i < kXraySub * kXraySub; i += blockDim.x) sover[i] = 0;
    __syncthreads();
    auto put = [&](uint32_t key) {
        const uint32_t lp = (key >> 16) * kXraySub + ((key >> 11) & 31u), z = key & 2047u;
        if (z < 1024)
            atomicOr(&sbits[lp * 32 + (z >> 5)], 1u << (z & 31));
        else
            sover[lp] = 1;
    };
    uint32_t k = k0 + threadIdx.x;
    for (; k + 3 * blockDim.x < k1; k += 4 * blockDim.x) {  // four independent loads in flight per thread
        const uint32_t q0 = __ldcs(b.keys + k), q1 = __ldcs(b.keys + k + blockDim.x), q2 = __ldcs(b.keys + k + 2 * blockDim.x), q3 = __ldcs(b.keys + k + 3 * blockDim.x);
        put(q0), put(q1), put(q2), put(q3);
    }
    for (; k < k1; k += blockDim.x) put(__ldcs(b.keys + k));
    __syncthreads();
    // resolve: popcount of the pixel's bucket set -> grey (generation.rs:186-197)
    for (uint32_t lp = threadIdx.x; lp < kXraySub * kXraySub; lp += blockDim.x) {
        const uint32_t x = px0 + (lp % kXraySub), y = py0 + (lp / kXraySub);
        if (x >= b.w || y >= b.h) continue;
        uint32_t cnt = sover[lp];
#pragma unroll
        for (int k = 0; k < 32; ++k) cnt += __popc(sbits[lp * 32 + ((k + lp) & 31)]);  // rotated start: no 32-way bank conflict
        if (cnt) {
            const uint8_t gv = b.grey[cnt];
            reinterpret_cast<uchar4*>(b.rgba)[(size_t)y * b.w + x] = make_uchar4(gv, gv, gv, 255);
        }
        if (b.zbits_out) {
            uint32_t* o = b.zbits_out + ((size_t)y * b.w + x) * 32;
            for (int k = 0; k < 32; ++k) o[k] = sbits[lp * 32 + k];
        }
    }
}

// grey[count] LUT is computed on the host with libm log (generation.rs:186-197) so the cast boundary matches.
__global__ void __launch_bounds__(256) k_xray_resolve(const uint32_t* __restrict__ zbits, const uint8_t* __restrict__ zover,
                                                      const uint8_t* __restrict__ grey, uint32_t npix, uint8_t* __restrict__ rgba) {
    const uint32_t px = blockIdx.x * blockDim.x + threadIdx.x;
    if (px >= npix) return;
    uint32_t cnt = zover[px];
    const uint4* b = reinterpret_cast<const uint4*>(zbits + (size_t)px * 32);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const uint4 v = b[k];
        cnt += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
    }
    uchar4 o = make_uchar4(255, 255, 255, 0);  // TRANSPARENT.to_u8() (color.rs:154-159; generation.rs:506-511)
    if (cnt) {
        const uint8_t gval = grey[cnt];
        o = make_uchar4(gval, gval, gval, 255);
    }
    reinterpret_cast<uchar4*>(rgba)[px] = o;
}

// ------------------------------------------------------------------------------------------------
// The other colouring strategies of the X-ray tiles (xray/src/generation.rs:200-405), Binning = None:
//   1 point colour mean, 2 intensity mean (log-brightened), 3 height standard deviation through a colormap.
// The reference accumulates per column in arrival order (f32 sums, Welford in f64) and its batches arrive from several
// threads in unspecified order; here the columns are accumulated with atomics (f32 sums like the reference; for the
// variance, f64 sums of (z - z0) and (z - z0)^2 around the tile's mid height), so results agree up to rounding.
// ------------------------------------------------------------------------------------------------
struct XrayAttrArgs {
    XrayArgs x;
    const uint8_t* rgb;      // node-contiguous colours
    const float* intensity;  // node-contiguous intensities (mode 2)
    float* sum;              // mode 1: npix * 4; mode 2: npix
    double* dsum;            // mode 3: npix * 2
    uint32_t* count;
    double z0;
};

template <int MODE>
__global__ void __launch_bounds__(256) k_xray_accum_attr(const __grid_constant__ XrayAttrArgs b) {
    const XrayArgs& a = b.x;
    const QTile t = a.tiles[blockIdx.x];
    const QNode nd = a.nodes[t.node];
    const int bpc = enc_bytes(nd.enc);
    bool seen = false;
    for (uint32_t i = threadIdx.x; i < t.count; i += blockDim.x) {
        const uint8_t* s = a.xyz + nd.xyz_off + (uint64_t)(t.first + i) * 3 * bpc;
        double p[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) p[k] = decode1_fast(load_code(s + k * bpc, nd.enc), nd.m[k], nd.e, nd.enc);
        if (!loc_contains(a.geom, p[0], p[1], p[2])) continue;
        seen = true;
        if (a.has_q) {
            const V3 q = iso_apply(a.query_from_global, V3{p[0], p[1], p[2]});
            p[0] = q.x, p[1] = q.y, p[2] = q.z;
        }
        const uint32_t x = rust_as_u32_dev(xray_unit(a, 0, p[0]) * (double)a.w);
        const uint32_t y = rust_as_u32_dev((1. - xray_unit(a, 1, p[1])) * (double)a.h);
        if (!(x < a.w && y < a.h)) continue;
        const size_t px = (size_t)y * a.w + x;
        const uint64_t slot = nd.point_off + t.first + i;
        if (MODE == 1) {  // Color<u8>::to_f32: f32::from(c) / 255.
            const uint8_t* c = b.rgb + 3 * slot;
            atomicAdd(&b.sum[px * 4 + 0], (float)c[0] / 255.f);
            atomicAdd(&b.sum[px * 4 + 1], (float)c[1] / 255.f);
            atomicAdd(&b.sum[px * 4 + 2], (float)c[2] / 255.f);
            atomicAdd(&b.count[px], 1u);
        } else if (MODE == 2) {
            const float v = b.intensity[slot];
            if (v < 0.f) continue;
            atomicAdd(&b.sum[px], v);
            atomicAdd(&b.count[px], 1u);
        } else {
            const double d = p[2] - b.z0;
            atomicAdd(&b.dsum[px * 2], d);
            atomicAdd(&b.dsum[px * 2 + 1], d * d);
            atomicAdd(&b.count[px], 1u);
        }
    }
    if (__syncthreads_or(seen) && threadIdx.x == 0) atomicExch(a.any, 1);
}

__device__ __forceinline__ uint8_t f32_to_u8_dev(float v) {  // Color<f32>::to_u8: (v * 255.) as u8 (saturating, NaN -> 0)
    const float s = v * 255.f;
    if (!(s == s) || s <= 0.f) return 0;
    return s >= 255.f ? (uint8_t)255 : (uint8_t)s;
}
__device__ __forceinline__ float jet_base_dev(float val) {  // xray/src/colormap.rs:30-46
    if (val <= -0.75f) return 0.f;
    if (val <= -0.25f) return (val - -0.75f) * (1.0f - 0.0f) / (-0.25f - -0.75f) + 0.0f;
    if (val <= 0.25f) return 1.0f;
    if (val <= 0.75f) return (val - 0.25f) * (0.0f - 1.0f) / (0.75f - 0.25f) + 1.0f;
    return 0.0f;
}

__global__ void __launch_bounds__(256) k_xray_resolve_attr(int mode, float p0, float p1, int colormap, const float* __restrict__ sum,
                                                           const double* __restrict__ dsum, const uint32_t* __restrict__ count, uint32_t npix,
                                                           uint8_t* __restrict__ rgba) {
    const uint32_t px = blockIdx.x * blockDim.x + threadIdx.x;
    if (px >= npix) return;
    uchar4 o = make_uchar4(255, 255, 255, 0);  // TRANSPARENT.to_u8() (color.rs:154-159; generation.rs:506-511)
    const uint32_t n = count[px];
    if (n) {
        if (mode == 1) {
            o = make_uchar4(f32_to_u8_dev(sum[px * 4] / (float)n), f32_to_u8_dev(sum[px * 4 + 1] / (float)n), f32_to_u8_dev(sum[px * 4 + 2] / (float)n), 255);
        } else if (mode == 2) {
            float m = sum[px] / (float)n;
            m = fminf(fmaxf(m, p0), p1);
            const uint8_t g = f32_to_u8_dev(logf(m - p0) / logf(p1 - p0));
            o = make_uchar4(g, g, g, 255);
        } else {
            const double mean = dsum[px * 2] / (double)n;
            double var = dsum[px * 2 + 1] / (double)n - mean * mean;
            var = var > 0.0 ? var : 0.0;
            float sd = (float)sqrt(var);
            sd = sd < 0.f ? 0.f : (sd > p0 ? p0 : sd);
            const float val = sd / p0;
            if (colormap == 0)
                o = make_uchar4(f32_to_u8_dev(jet_base_dev(val - 0.5f)), f32_to_u8_dev(jet_base_dev(val)), f32_to_u8_dev(jet_base_dev(val + 0.5f)), 255);
            else
                o = make_uchar4(f32_to_u8_dev((1.0f - val) * 0.8f), f32_to_u8_dev((1.0f - val) * 0.8f), f32_to_u8_dev((1.0f - val) * 1.0f), 255);
        }
    }
    reinterpret_cast<uchar4*>(rgba)[px] = o;
}

// ------------------------------------------------------------------------------------------------
// /nodes_data blob (octree_web_viewer/src/backend.rs:92-165): gather the position and colour bytes of the requested
// nodes from their places in the octree arrays into one contiguous, 8-byte-padded reply buffer.
// ------------------------------------------------------------------------------------------------
// One work item = up to kBlobSeg destination bytes of one node part.  Destination offsets are multiples of 8 (the
// blob's padding rule); sources start at arbitrary byte offsets (a Uint8 node has 3 n bytes), so every destination word
// is assembled from two aligned source words with a funnel shift.  HBM-bound byte copy: 2 bytes moved per byte of reply.
struct BlobItem {
    uint64_t src;   // byte offset into the source array
    uint64_t dst;   // byte offset into the blob (multiple of 8)
    uint32_t bytes;
    uint32_t from_rgb;  // 0: position bytes, 1: colour bytes
};
constexpr uint32_t kBlobSeg = 32768;

__global__ void __launch_bounds__(256) k_blob_gather(const BlobItem* __restrict__ items, const uint8_t* __restrict__ xyz, const uint8_t* __restrict__ rgb,
                                                     uint8_t* __restrict__ blob) {
    const BlobItem it = items[blockIdx.x];
    const uint8_t* src = (it.from_rgb ? rgb : xyz) + it.src;
    uint32_t* dst = reinterpret_cast<uint32_t*>(blob + it.dst);
    const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(src) & 3), sh = mis * 8;
    const uint32_t* w = reinterpret_cast<const uint32_t*>(src - mis);
    const uint32_t nwords = it.bytes / 4;
    for (uint32_t i = threadIdx.x; i < nwords; i += blockDim.x) {
        const uint32_t lo = __ldg(w + i);
        const uint32_t hi = mis ? __ldg(w + i + 1) : 0u;  // never read a word the source range does not touch
        dst[i] = __funnelshift_r(lo, hi, sh);
    }
    // the last 0..3 bytes; the blob's zero padding is written by the host-side memset of the reply buffer
    if (threadIdx.x < (it.bytes & 3u)) blob[it.dst + 4ull * nwords + threadIdx.x] = src[4ull * nwords + threadIdx.x];
}

}  // namespace pcv
