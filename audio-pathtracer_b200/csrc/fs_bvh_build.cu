// fs_bvh_build.cu -- LBVH build on the device (one-time per fs_scene_commit).
//
// Pipeline (all kernels hand-written, no CUB/thrust):
//   k_tri_bounds   per-triangle AABB + centroid-bounds reduction (ordered-uint atomics)
//   k_morton       63-bit Morton code of the normalised AABB centre (21 bits per axis)
//   radix sort     8 LSD passes of 8 bits over (u64 key, u32 triangle id): k_sort_hist,
//                  k_sort_scan, k_sort_scatter (stable: warp match + ordered warp hand-over)
//   k_pack         64 B triangle records (v0,e1,e2,n,orig id,material) in sorted order,
//                  leaf boxes
//   k_karras       binary radix tree topology (Karras 2012), ties broken by sorted index
//   k_refit        bottom-up box fit with one atomic arrival counter per inner node
//   k_emit         64 B traversal nodes holding both children's padded boxes; subtrees of
//                  <= FS_LEAF_MAX triangles collapse into one leaf (ranges are contiguous)
//   k_top_treelet  BFS copy of the top levels for shared-memory staging
//
// Replaces UAudioRayTracingSubsystem::RegisterGeometry (SUB.h:99-100) + the Chaos scene query
// acceleration behind UWorld::LineTraceSingleByObjectType (SUB.cpp:252, 340).
#include "fs_internal.h"
#include <vector>
#include <utility>
#include <stdlib.h>

namespace {

__device__ __forceinline__ uint32_t f2ord(float f)
{
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float ord2f(uint32_t u)
{
    u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f; memcpy(&f, &u, 4); return f;
#endif
}

// bounds[0..2] = min (ordered uint), bounds[3..5] = max of AABB centres
__global__ void k_init_bounds(uint32_t* bounds)
{
    if (threadIdx.x < 3) bounds[threadIdx.x] = 0xffffffffu;
    else if (threadIdx.x < 6) bounds[threadIdx.x] = 0u;
    if (threadIdx.x >= 9 && threadIdx.x < 12) bounds[threadIdx.x] = 0xffffffffu;   // scene box min
    else if (threadIdx.x >= 12 && threadIdx.x < 15) bounds[threadIdx.x] = 0u;      // scene box max
}

// raw-vertex box of one triangle: the leaf boxes of the build and of fs_bvh_refit
__device__ __forceinline__ void tri_box(const float* __restrict__ p, float4& lo, float4& hi)
{
    float x0 = p[0], y0 = p[1], z0 = p[2], x1 = p[3], y1 = p[4], z1 = p[5], x2 = p[6], y2 = p[7], z2 = p[8];
    lo = make_float4(fminf(x0, fminf(x1, x2)), fminf(y0, fminf(y1, y2)), fminf(z0, fminf(z1, z2)), 0.f);
    hi = make_float4(fmaxf(x0, fmaxf(x1, x2)), fmaxf(y0, fmaxf(y1, y2)), fmaxf(z0, fmaxf(z1, z2)), 0.f);
}

__global__ void k_tri_bounds(const float* __restrict__ verts, uint32_t n, float4* __restrict__ tlo,
                             float4* __restrict__ thi, uint32_t* __restrict__ bounds,
                             uint32_t* __restrict__ extent_ord)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    float cx = 0, cy = 0, cz = 0, ext = 0;
    float blx = INFINITY, bly = INFINITY, blz = INFINITY, bhx = -INFINITY, bhy = -INFINITY, bhz = -INFINITY;
    bool valid = i < n;
    if (valid) {
        float4 lo, hi;
        tri_box(verts + (size_t)i * 9, lo, hi);
        const float lx = lo.x, ly = lo.y, lz = lo.z, hx = hi.x, hy = hi.y, hz = hi.z;
        tlo[i] = lo;
        thi[i] = hi;
        blx = lx; bly = ly; blz = lz; bhx = hx; bhy = hy; bhz = hz;
        cx = 0.5f * lx + 0.5f * hx; cy = 0.5f * ly + 0.5f * hy; cz = 0.5f * lz + 0.5f * hz;
        ext = fmaxf(fmaxf(fmaxf(fabsf(lx), fabsf(hx)), fmaxf(fabsf(ly), fabsf(hy))), fmaxf(fabsf(lz), fabsf(hz)));
    }
    // warp reduce then one atomic per warp
    uint32_t m = __ballot_sync(0xffffffffu, valid);
    if (!m) return;
    float mnx = valid ? cx : INFINITY, mny = valid ? cy : INFINITY, mnz = valid ? cz : INFINITY;
    float mxx = valid ? cx : -INFINITY, mxy = valid ? cy : -INFINITY, mxz = valid ? cz : -INFINITY;
    for (int o = 16; o; o >>= 1) {
        mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o));
        mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o));
        mnz = fminf(mnz, __shfl_xor_sync(0xffffffffu, mnz, o));
        mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
        mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
        mxz = fmaxf(mxz, __shfl_xor_sync(0xffffffffu, mxz, o));
        ext = fmaxf(ext, __shfl_xor_sync(0xffffffffu, ext, o));
        blx = fminf(blx, __shfl_xor_sync(0xffffffffu, blx, o)); bly = fminf(bly, __shfl_xor_sync(0xffffffffu, bly, o));
        blz = fminf(blz, __shfl_xor_sync(0xffffffffu, blz, o)); bhx = fmaxf(bhx, __shfl_xor_sync(0xffffffffu, bhx, o));
        bhy = fmaxf(bhy, __shfl_xor_sync(0xffffffffu, bhy, o)); bhz = fmaxf(bhz, __shfl_xor_sync(0xffffffffu, bhz, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(bounds + 0, f2ord(mnx)); atomicMin(bounds + 1, f2ord(mny)); atomicMin(bounds + 2, f2ord(mnz));
        atomicMax(bounds + 3, f2ord(mxx)); atomicMax(bounds + 4, f2ord(mxy)); atomicMax(bounds + 5, f2ord(mxz));
        atomicMax(extent_ord, f2ord(ext));
        atomicMin(bounds + 9, f2ord(blx)); atomicMin(bounds + 10, f2ord(bly)); atomicMin(bounds + 11, f2ord(blz));
        atomicMax(bounds + 12, f2ord(bhx)); atomicMax(bounds + 13, f2ord(bhy)); atomicMax(bounds + 14, f2ord(bhz));
    }
}

__device__ __forceinline__ uint64_t expand21(uint32_t v)
{
    uint64_t x = v & 0x1fffffu;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

__global__ void k_morton(const float4* __restrict__ tlo, const float4* __restrict__ thi, uint32_t n,
                         const uint32_t* __restrict__ bounds, uint64_t* __restrict__ keys,
                         uint32_t* __restrict__ vals)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float bx = ord2f(bounds[0]), by = ord2f(bounds[1]), bz = ord2f(bounds[2]);
    float ex = ord2f(bounds[3]) - bx, ey = ord2f(bounds[4]) - by, ez = ord2f(bounds[5]) - bz;
    float4 lo = tlo[i], hi = thi[i];
    float cx = 0.5f * lo.x + 0.5f * hi.x, cy = 0.5f * lo.y + 0.5f * hi.y, cz = 0.5f * lo.z + 0.5f * hi.z;
    const float S = 2097151.0f;   // 2^21 - 1
    float fx = ex > 0.f ? (cx - bx) / ex : 0.f, fy = ey > 0.f ? (cy - by) / ey : 0.f, fz = ez > 0.f ? (cz - bz) / ez : 0.f;
    uint32_t qx = (uint32_t)fminf(fmaxf(fx * S, 0.f), S);
    uint32_t qy = (uint32_t)fminf(fmaxf(fy * S, 0.f), S);
    uint32_t qz = (uint32_t)fminf(fmaxf(fz * S, 0.f), S);
    keys[i] = (expand21(qx) << 2) | (expand21(qy) << 1) | expand21(qz);
    vals[i] = i;
}

// ---------------------------------------------------------------------------------------------
// LSD radix sort, 8 bits per pass
// ---------------------------------------------------------------------------------------------
constexpr int SORT_THREADS = 256;
constexpr int SORT_ITEMS = 8;
constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS;

__global__ void __launch_bounds__(SORT_THREADS)
k_sort_hist(const uint64_t* __restrict__ keys, uint32_t n, int shift, uint32_t* __restrict__ block_hist,
            uint32_t n_blocks)
{
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    uint32_t base = blockIdx.x * SORT_TILE;
#pragma unroll
    for (int r = 0; r < SORT_ITEMS; ++r) {
        uint32_t i = base + r * SORT_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&h[(uint32_t)(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    block_hist[(size_t)threadIdx.x * n_blocks + blockIdx.x] = h[threadIdx.x];
}

// exclusive scan of `total` counters, one CTA, chunked with a running carry
__global__ void __launch_bounds__(1024) k_sort_scan(uint32_t* __restrict__ data, uint32_t total)
{
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t base = 0; base < total; base += 1024) {
        uint32_t i = base + threadIdx.x;
        uint32_t v = (i < total) ? data[i] : 0u;
        uint32_t x = v;
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if ((int)lane >= o) x += y;
        }
        if (lane == 31) warp_sums[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = warp_sums[lane];
            for (int o = 1; o < 32; o <<= 1) {
                uint32_t y = __shfl_up_sync(0xffffffffu, w, o);
                if ((int)lane >= o) w += y;
            }
            warp_sums[lane] = w;
        }
        __syncthreads();
        uint32_t carry = carry_s;
        uint32_t incl = x + (warp ? warp_sums[warp - 1] : 0u) + carry;
        if (i < total) data[i] = incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = incl;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(SORT_THREADS)
k_sort_scatter(const uint64_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
               uint64_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out, uint32_t n, int shift,
               const uint32_t* __restrict__ block_hist, uint32_t n_blocks)
{
    __shared__ uint32_t base_s[256];
    base_s[threadIdx.x] = block_hist[(size_t)threadIdx.x * n_blocks + blockIdx.x];
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    uint32_t tile = blockIdx.x * SORT_TILE;
    for (int r = 0; r < SORT_ITEMS; ++r) {
        uint32_t i = tile + r * SORT_THREADS + threadIdx.x;
        bool valid = i < n;
        uint64_t k = valid ? keys_in[i] : 0ull;
        uint32_t v = valid ? vals_in[i] : 0u;
        uint32_t digit = valid ? ((uint32_t)(k >> shift) & 255u) : 256u;
        uint32_t peers = __match_any_sync(0xffffffffu, digit);
        uint32_t rank = __popc(peers & lt);
        // warps take turns in index order so that equal digits keep their input order (stable)
        for (uint32_t w = 0; w < SORT_THREADS / 32; ++w) {
            if (warp == w) {
                uint32_t pos = 0;
                if (valid) pos = base_s[digit] + rank;
                __syncwarp();
                if (valid && rank == 0) base_s[digit] += __popc(peers);
                if (valid) { keys_out[pos] = k; vals_out[pos] = v; }
            }
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------------------------
// tree
// ---------------------------------------------------------------------------------------------
// the 64 B triangle record of sorted position j and its (normal, material) record: the build (k_pack) and the refit
// (k_refit_tris) share this arithmetic, so a refitted record is bit-identical to a freshly built one
__device__ __forceinline__ void pack_tri(const float* __restrict__ verts, uint32_t id, uint32_t mat, uint32_t j,
                                         float4* __restrict__ tris, float4* __restrict__ tri_nm)
{
    const float* p = verts + (size_t)id * 9;
    fs_vec3 v0 = fs_mk(p[0], p[1], p[2]);
    fs_vec3 e1 = fs_mk(p[3] - p[0], p[4] - p[1], p[5] - p[2]);
    fs_vec3 e2 = fs_mk(p[6] - p[0], p[7] - p[1], p[8] - p[2]);
    fs_vec3 nn = fs_tri_normal(e1, e2);
    tris[(size_t)j * 4 + 0] = make_float4(v0.x, v0.y, v0.z, nn.x);
    tris[(size_t)j * 4 + 1] = make_float4(e1.x, e1.y, e1.z, nn.y);
    tris[(size_t)j * 4 + 2] = make_float4(e2.x, e2.y, e2.z, nn.z);
    tris[(size_t)j * 4 + 3] = make_float4(__uint_as_float(id), __uint_as_float(mat), 0.f, 0.f);
    tri_nm[j] = make_float4(nn.x, nn.y, nn.z, __uint_as_float(mat));
}

__global__ void k_pack(const float* __restrict__ verts, const uint32_t* __restrict__ mats,
                       const uint32_t* __restrict__ sorted_ids, uint32_t n,
                       const float4* __restrict__ tlo, const float4* __restrict__ thi,
                       float4* __restrict__ tris, uint32_t* __restrict__ tri_orig,
                       uint32_t* __restrict__ tri_mat, float4* __restrict__ tri_nm, float4* __restrict__ bb_lo,
                       float4* __restrict__ bb_hi)
{
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    uint32_t id = sorted_ids[j];
    const uint32_t mat = mats[id];
    pack_tri(verts, id, mat, j, tris, tri_nm);
    tri_orig[j] = id;
    tri_mat[j] = mat;
    bb_lo[(n - 1) + j] = tlo[id];
    bb_hi[(n - 1) + j] = thi[id];
}

__device__ __forceinline__ int delta(const uint64_t* __restrict__ keys, int n, int i, int j)
{
    if (j < 0 || j >= n) return -1;
    uint64_t a = keys[i], b = keys[j];
    if (a != b) return __clzll((long long)(a ^ b));
    return 64 + __clz(i ^ j);
}

// node ids: inner i in [0, n-1), leaf j -> (n-1)+j
__global__ void k_karras(const uint64_t* __restrict__ keys, int n, int2* __restrict__ children,
                         int2* __restrict__ ranges, int* __restrict__ parent)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    int dmin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = delta(keys, n, i, j);
    int s = 0;
    int t = l;
    do {
        t = (t + 1) >> 1;
        if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    int gamma = i + s * d + min(d, 0);
    int lo = min(i, j), hi = max(i, j);
    int left = (lo == gamma) ? (n - 1) + gamma : gamma;
    int right = (hi == gamma + 1) ? (n - 1) + gamma + 1 : gamma + 1;
    children[i] = make_int2(left, right);
    ranges[i] = make_int2(lo, hi);
    parent[left] = i;
    parent[right] = i;
    if (i == 0) parent[0] = -1;
}

__global__ void k_refit(int n, const int2* __restrict__ children, const int* __restrict__ parent,
                        float4* bb_lo, float4* bb_hi, uint32_t* __restrict__ arrive)
{
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    int cur = parent[(n - 1) + j];
    for (int guard = 0; cur >= 0 && guard < 4096; ++guard) {     // bounded: a tree is never this deep
        __threadfence();
        if (atomicAdd(&arrive[cur], 1u) == 0u) return;      // first arrival stops
        __threadfence();
        int2 c = children[cur];
        float4 l0 = __ldcg(bb_lo + c.x), h0 = __ldcg(bb_hi + c.x);
        float4 l1 = __ldcg(bb_lo + c.y), h1 = __ldcg(bb_hi + c.y);
        __stcg(bb_lo + cur, make_float4(fminf(l0.x, l1.x), fminf(l0.y, l1.y), fminf(l0.z, l1.z), 0.f));
        __stcg(bb_hi + cur, make_float4(fmaxf(h0.x, h1.x), fmaxf(h0.y, h1.y), fmaxf(h0.z, h1.z), 0.f));
        cur = parent[cur];
    }
}

__device__ __forceinline__ int encode_child(int c, int n, const int2* __restrict__ ranges, int leaf_max)
{
    if (c >= n - 1) {                       // leaf j, one triangle
        uint32_t j = (uint32_t)(c - (n - 1));
        return ~(int)((j << 3) | 0u);
    }
    int2 r = ranges[c];
    int cnt = r.y - r.x + 1;
    if (cnt <= leaf_max) return ~(int)(((uint32_t)r.x << 3) | (uint32_t)(cnt - 1));
    return c;
}

// Conservative padding of a child box: 2^-17 of its largest |coordinate| (~128 float ulps at that magnitude) + 1e-5 m.
// It must cover (a) the rounding of the FMA slab test (~3 ulps of max(|o|, |plane|), as a displacement of the plane),
// (b) v0+e1 / v0+e2 differing from v1 / v2 by an ulp, (c) the rounding of fs_intersect_tri's barycentrics (tvec = o - v0
// carries 2^-24 of max(|o|, |v0|): a hit can be accepted ~1e-5 m outside the triangle at 50 m coordinates), so that every
// triangle the exact-sequence test accepts is reached: together ~2e-5 m at 50 m, i.e. 2^-21 relative; 2^-17 leaves a factor
// of 16.  The first version used 2^-15: at the concert hall's coordinates that is 1.5 mm on every side of 6 cm triangles,
// and the looser leaf boxes cost 3.4 % of the update (hall 10.29 -> 9.94 ms; room unchanged).  The quantised 4-wide boxes add
// their own outward rounding + one spare quantum on top.  tests/test_gpu_intersect.py checks BVH == brute force on the
// device, the full-size parity tests compare 16 M + 4.5 M rays with the CPU oracle.
#ifndef FS_BOX_PAD_REL
#define FS_BOX_PAD_REL (1.0f / 131072.0f)
#endif
__device__ __forceinline__ float box_pad(float4 lo, float4 hi)
{
    float m = fmaxf(fmaxf(fmaxf(fabsf(lo.x), fabsf(hi.x)), fmaxf(fabsf(lo.y), fabsf(hi.y))),
                    fmaxf(fabsf(lo.z), fabsf(hi.z)));
    return fmaf(m, FS_BOX_PAD_REL, 1e-5f);
}

__global__ void k_emit(int n, const int2* __restrict__ children, const int2* __restrict__ ranges,
                       const float4* __restrict__ bb_lo, const float4* __restrict__ bb_hi,
                       float4* __restrict__ nodes, int leaf_max)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int2 c = children[i];
    float4 l0 = bb_lo[c.x], h0 = bb_hi[c.x], l1 = bb_lo[c.y], h1 = bb_hi[c.y];
    float p0 = box_pad(l0, h0), p1 = box_pad(l1, h1);
    int e0 = encode_child(c.x, n, ranges, leaf_max), e1 = encode_child(c.y, n, ranges, leaf_max);
    nodes[(size_t)i * 4 + 0] = make_float4(l0.x - p0, h0.x + p0, l0.y - p0, h0.y + p0);
    nodes[(size_t)i * 4 + 1] = make_float4(l1.x - p1, h1.x + p1, l1.y - p1, h1.y + p1);
    nodes[(size_t)i * 4 + 2] = make_float4(l0.z - p0, h0.z + p0, l1.z - p1, h1.z + p1);
    nodes[(size_t)i * 4 + 3] = make_float4(__int_as_float(e0), __int_as_float(e1), 0.f, 0.f);
}


// ---------------------------------------------------------------------------------------------
// PLOC: parallel locally-ordered clustering (Meister & Bittner 2018) over the Morton-sorted
// triangles.  Every round each cluster looks R neighbours to the left and right in the cluster
// array for the partner minimising the surface area of the merged box; mutual nearest neighbours
// merge into one inner node.  Bottom-up agglomeration by surface area gives near-SAH trees
// (the LBVH topology splits on Morton bits only).  One triangle per leaf; inner node ids are
// handed out from the back so the root ends up at index 0 and the top of the tree is contiguous.
// ---------------------------------------------------------------------------------------------
// search radius: FS_TUNE_PLOC_R (default 10)

__device__ __forceinline__ float box_area(float4 lo, float4 hi)
{
    float dx = hi.x - lo.x, dy = hi.y - lo.y, dz = hi.z - lo.z;
    return dx * dy + dy * dz + dz * dx;
}

__global__ void k_ploc_init(uint32_t n, const float4* __restrict__ bb_lo, const float4* __restrict__ bb_hi,
                            float4* __restrict__ clo, float4* __restrict__ chi, int* __restrict__ cref)
{
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    clo[j] = bb_lo[(n - 1) + j];
    chi[j] = bb_hi[(n - 1) + j];
    cref[j] = ~(int)(j << 3);                       // leaf: triangle j, count 1
}

__global__ void k_ploc_nn(uint32_t n, const float4* __restrict__ clo, const float4* __restrict__ chi,
                          uint32_t* __restrict__ nn, const int PLOC_R)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 lo = clo[i], hi = chi[i];
    float best = INFINITY; uint32_t bj = i;
    const uint32_t j0 = i > (uint32_t)PLOC_R ? i - PLOC_R : 0u;
    const uint32_t j1 = min(n - 1u, i + (uint32_t)PLOC_R);
    for (uint32_t j = j0; j <= j1; ++j) {
        if (j == i) continue;
        const float4 l = clo[j], h = chi[j];
        const float4 ul = make_float4(fminf(lo.x, l.x), fminf(lo.y, l.y), fminf(lo.z, l.z), 0.f);
        const float4 uh = make_float4(fmaxf(hi.x, h.x), fmaxf(hi.y, h.y), fmaxf(hi.z, h.z), 0.f);
        const float a = box_area(ul, uh);
        if (a < best) { best = a; bj = j; }          // ties keep the lower index: deterministic
    }
    nn[i] = bj;
}

// flags[i] = 1 if cluster i survives this round (it is not the right half of a merging pair);
// mflag[i] = 1 if cluster i is the left half of a merging pair (creates one inner node)
__global__ void k_ploc_flags(uint32_t n, const uint32_t* __restrict__ nn, uint32_t* __restrict__ keep,
                             uint32_t* __restrict__ mflag)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t j = nn[i];
    const bool mutual = (j != i) && (nn[j] == i);
    keep[i] = (mutual && j < i) ? 0u : 1u;
    mflag[i] = (mutual && i < j) ? 1u : 0u;
}

__global__ void k_ploc_merge(uint32_t n, const uint32_t* __restrict__ nn, const uint32_t* __restrict__ keep_scan,
                             const uint32_t* __restrict__ merge_scan, const uint32_t* __restrict__ keep,
                             const uint32_t* __restrict__ mflag, uint32_t nodes_made, uint32_t n_inner,
                             const float4* __restrict__ clo, const float4* __restrict__ chi, const int* __restrict__ cref,
                             float4* __restrict__ nlo, float4* __restrict__ nhi, int* __restrict__ nref,
                             float4* __restrict__ nodes)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !keep[i]) return;
    const uint32_t pos = keep_scan[i];
    if (mflag[i]) {
        const uint32_t j = nn[i];
        const float4 l0 = clo[i], h0 = chi[i], l1 = clo[j], h1 = chi[j];
        const uint32_t id = n_inner - 1u - (nodes_made + merge_scan[i]);      // root (made last) gets id 0
        const float p0 = box_pad(l0, h0), p1 = box_pad(l1, h1);
        nodes[(size_t)id * 4 + 0] = make_float4(l0.x - p0, h0.x + p0, l0.y - p0, h0.y + p0);
        nodes[(size_t)id * 4 + 1] = make_float4(l1.x - p1, h1.x + p1, l1.y - p1, h1.y + p1);
        nodes[(size_t)id * 4 + 2] = make_float4(l0.z - p0, h0.z + p0, l1.z - p1, h1.z + p1);
        nodes[(size_t)id * 4 + 3] = make_float4(__int_as_float(cref[i]), __int_as_float(cref[j]), 0.f, 0.f);
        nlo[pos] = make_float4(fminf(l0.x, l1.x), fminf(l0.y, l1.y), fminf(l0.z, l1.z), 0.f);
        nhi[pos] = make_float4(fmaxf(h0.x, h1.x), fmaxf(h0.y, h1.y), fmaxf(h0.z, h1.z), 0.f);
        nref[pos] = (int)id;
    } else {
        nlo[pos] = clo[i]; nhi[pos] = chi[i]; nref[pos] = cref[i];
    }
}

// three-phase exclusive scan of n u32 (tile sums -> scan of tile sums by one CTA -> add)
constexpr int SCAN_TILE = 1024;
__global__ void __launch_bounds__(SCAN_TILE) k_scan_tiles(const uint32_t* __restrict__ in, uint32_t* __restrict__ out,
                                                           uint32_t n, uint32_t* __restrict__ tile_sums)
{
    __shared__ uint32_t ws[32];
    const uint32_t i = blockIdx.x * SCAN_TILE + threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t v = i < n ? in[i] : 0u;
    uint32_t x = v;
    for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if ((int)lane >= o) x += y; }
    if (lane == 31) ws[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = ws[lane];
        for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, w, o); if ((int)lane >= o) w += y; }
        ws[lane] = w;
    }
    __syncthreads();
    const uint32_t incl = x + (warp ? ws[warp - 1] : 0u);
    if (i < n) out[i] = incl - v;
    if (threadIdx.x == SCAN_TILE - 1) tile_sums[blockIdx.x] = incl;
}
__global__ void k_scan_add(uint32_t* __restrict__ out, uint32_t n, const uint32_t* __restrict__ tile_offs)
{
    const uint32_t i = blockIdx.x * SCAN_TILE + threadIdx.x;
    if (i < n) out[i] += tile_offs[blockIdx.x];
}
// total[0] = last exclusive value + last input (after the add phase)
__global__ void k_scan_total(const uint32_t* __restrict__ in, const uint32_t* __restrict__ out, uint32_t n, uint32_t* total)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) *total = n ? out[n - 1] + in[n - 1] : 0u;
}


// ---------------------------------------------------------------------------------------------
// 4-wide quantised nodes from the finished BVH2 (see fs_bvh.cuh).  One thread per BVH2 node.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t quant_lo(float v, float base, float inv_scale)
{
    float q = floorf((v - base) * inv_scale) - 1.0f;          // outward + one spare quantum
    return (uint32_t)fminf(fmaxf(q, 0.0f), 65535.0f);
}
__device__ __forceinline__ uint32_t quant_hi(float v, float base, float inv_scale)
{
    float q = ceilf((v - base) * inv_scale) + 1.0f;
    return (uint32_t)fminf(fmaxf(q, 0.0f), 65535.0f);
}

// grid[0..2] = qbase, grid[3..5] = qscale from the root's two (padded) child boxes
__global__ void k_quant_grid(const float4* __restrict__ nodes, float* __restrict__ grid)
{
    const int a = threadIdx.x;
    if (a >= 3) return;
    const float4 n0 = nodes[0], n1 = nodes[1], n2 = nodes[2];
    float lo, hi;
    if (a == 0) { lo = fminf(n0.x, n1.x); hi = fmaxf(n0.y, n1.y); }
    else if (a == 1) { lo = fminf(n0.z, n1.z); hi = fmaxf(n0.w, n1.w); }
    else { lo = fminf(n2.x, n2.z); hi = fmaxf(n2.y, n2.w); }
    if (!(hi < 1e29f)) hi = (a == 0) ? n0.y : (a == 1 ? n0.w : n2.y);     // single-triangle root: ignore the dummy child
    if (!(lo < 1e29f)) lo = (a == 0) ? n0.x : (a == 1 ? n0.z : n2.x);
    float scale = (hi - lo) / 65500.0f;
    if (!(scale > 1e-12f)) scale = 1e-12f;
    grid[a] = lo - 16.0f * scale;
    grid[3 + a] = scale;
}

__device__ __forceinline__ uint4 quant_box(float lox, float hix, float loy, float hiy, float loz, float hiz, int ref,
                                           const float* __restrict__ g)
{
    const float ix = 1.0f / g[3], iy = 1.0f / g[4], iz = 1.0f / g[5];
    uint4 u;
    u.x = quant_lo(lox, g[0], ix) | (quant_hi(hix, g[0], ix) << 16);
    u.y = quant_lo(loy, g[1], iy) | (quant_hi(hiy, g[1], iy) << 16);
    u.z = quant_lo(loz, g[2], iz) | (quant_hi(hiz, g[2], iz) << 16);
    u.w = (uint32_t)ref;
    return u;
}

// Wide node i = BVH2 node i with up to two of its descendants opened.  collapse = 1 (default): greedy by
// surface area -- repeatedly replace the inner child with the largest box by its two children until there are
// four slots (Wald et al. 2008 / Ylitie et al. 2017 collapse, restricted to width 4): every slot is used and the
// big, often-hit boxes are the ones that get resolved one level further.  collapse = 0: the four grandchildren
// (a leaf child leaves a slot empty).  Child references stay BVH2 node indices, so every BVH2 node can be emitted
// independently; the ones no wide node refers to are simply never visited.
// src: where the box was loaded from, BVH2 node * 2 + side (the provenance of a wide-node slot, see fs_bvh_refit)
struct cbox { float lx, hx, ly, hy, lz, hz; int ref, src; };
__device__ __forceinline__ void load_children(const float4* __restrict__ nodes, int i, cbox& a, cbox& b)
{
    const float4 n0 = nodes[(size_t)i * 4], n1 = nodes[(size_t)i * 4 + 1], n2 = nodes[(size_t)i * 4 + 2], n3 = nodes[(size_t)i * 4 + 3];
    a.lx = n0.x; a.hx = n0.y; a.ly = n0.z; a.hy = n0.w; a.lz = n2.x; a.hz = n2.y; a.ref = __float_as_int(n3.x); a.src = 2 * i;
    b.lx = n1.x; b.hx = n1.y; b.ly = n1.z; b.hy = n1.w; b.lz = n2.z; b.hz = n2.w; b.ref = __float_as_int(n3.y); b.src = 2 * i + 1;
}
__device__ __forceinline__ float cbox_area(const cbox& c)
{
    const float dx = c.hx - c.lx, dy = c.hy - c.ly, dz = c.hz - c.lz;
    return dx * dy + dy * dz + dz * dx;
}

__global__ void k_emit4(uint32_t n_inner, const float4* __restrict__ nodes, const float* __restrict__ grid,
                        uint4* __restrict__ wnodes, int* __restrict__ wsrc, int collapse)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_inner) return;
    const uint4 EMPTY = make_uint4(0x0000ffffu, 0x0000ffffu, 0x0000ffffu, 0x7fffffffu);   // lo = 65535 > hi = 0
    cbox c[4];
    int k = 2;
    load_children(nodes, (int)i, c[0], c[1]);
    if (collapse) {
        while (k < 4) {
            int pick = -1; float best = -1.0f;
            for (int j = 0; j < k; ++j)
                if (c[j].ref >= 0) { const float a = cbox_area(c[j]); if (a > best) { best = a; pick = j; } }
            if (pick < 0) break;
            const int r = c[pick].ref;
            load_children(nodes, r, c[pick], c[k]);
            ++k;
        }
    } else {
        const int r0 = c[0].ref, r1 = c[1].ref;
        if (r1 >= 0) { load_children(nodes, r1, c[1], c[k]); ++k; }
        if (r0 >= 0) { load_children(nodes, r0, c[0], c[k]); ++k; }
    }
    for (int j = 0; j < 4; ++j) {
        wnodes[(size_t)i * 4 + j] = (j < k) ? quant_box(c[j].lx, c[j].hx, c[j].ly, c[j].hy, c[j].lz, c[j].hz, c[j].ref, grid) : EMPTY;
        wsrc[(size_t)i * 4 + j] = (j < k) ? c[j].src : -1;
    }
}

// ---------------------------------------------------------------------------------------------
// Dense breadth-first relayout of the REACHABLE wide nodes.  k_emit4 makes a wide node for every BVH2
// node, but a traversal that starts at the root only ever visits the ones other wide nodes refer to
// (about half with the grandchild collapse, fewer with the greedy one); left interleaved in memory the
// unreachable ones halve the useful part of every 128 B line and of the L1/L2 capacity.  Level by
// level: count the inner children of the frontier, exclusive scan, copy each frontier node to its
// dense slot with its inner-child references rewritten.  The children of a node get consecutive
// slots (one or two lines), the top of the tree is a contiguous prefix.  Deterministic.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ bool wide_is_inner(uint32_t ref) { return (int)ref >= 0 && ref != 0x7fffffffu; }

__global__ void k_wide_count(const uint4* __restrict__ src, const int* __restrict__ frontier, uint32_t nf, uint32_t* __restrict__ cnt)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nf) return;
    const uint4* p = src + (size_t)frontier[t] * 4;
    uint32_t c = 0;
    for (int j = 0; j < 4; ++j) c += wide_is_inner(p[j].w) ? 1u : 0u;
    cnt[t] = c;
}

__global__ void k_wide_place(const uint4* __restrict__ src, uint4* __restrict__ dst, const int* __restrict__ src_prov,
                             int* __restrict__ dst_prov, const int* __restrict__ frontier, uint32_t nf,
                             const uint32_t* __restrict__ off, uint32_t level_base, int* __restrict__ next_frontier)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nf) return;
    const uint4* p = src + (size_t)frontier[t] * 4;
    uint4* q = dst + (size_t)(level_base + t) * 4;
    uint32_t o = off[t];
    for (int j = 0; j < 4; ++j) {
        uint4 u = p[j];
        if (wide_is_inner(u.w)) { next_frontier[o] = (int)u.w; u.w = level_base + nf + o; ++o; }
        q[j] = u;
        dst_prov[(size_t)(level_base + t) * 4 + j] = src_prov[(size_t)frontier[t] * 4 + j];
    }
}

// ---------------------------------------------------------------------------------------------
// 8-wide compressed nodes (fs_bvh.cuh: w8nodes) from the finished BVH2.
//
// k_emit8 (one thread per BVH2 node): open the inner child with the largest box until there are eight slots (greedy by
// surface area, as for the 4-wide nodes), quantise the child boxes to 8 bits on a grid LOCAL to the node (origin = the
// node's low corner, a power-of-two quantum per axis, outward rounding), and place the children in the slots so that
// slot s holds the child lying farthest in the direction (s&1 ? +x : -x, s&2 ? +y : -y, s&4 ? +z : -z): the traversal
// then visits the hit children in the order of (slot XOR ray octant), near to far, without sorting by distance
// (Ylitie, Karras, Laine 2017).  Greedy assignment on cost(c, s) = <centre(c) - centre(node), sigma_s>.
// k_w8_count / k_w8_place: dense breadth-first relayout of the reachable nodes, as for the 4-wide nodes.  The inner
// children of a node get CONSECUTIVE node slots in slot order and its leaf children consecutive slots of a triangle
// array in W8 order (tris8), so a child is addressed by base + popc(mask below its slot): no per-child reference.
// ---------------------------------------------------------------------------------------------
#define W8_EMPTY 0x7fffffff
__device__ __forceinline__ uint32_t q8_lo(float v, float p, float inv)
{
    const float q = floorf((v - p) * inv - 0.001953125f);
    return (uint32_t)fminf(fmaxf(q, 0.0f), 255.0f);
}
__device__ __forceinline__ uint32_t q8_hi(float v, float p, float inv)
{
    const float q = ceilf((v - p) * inv + 0.001953125f);
    return (uint32_t)fminf(fmaxf(q, 0.0f), 255.0f);
}
// biased exponent eb of the quantum 2^(eb-127) for an axis of extent ext: 254 quanta cover the extent
__device__ __forceinline__ int q8_exponent(float ext)
{
    int k = -60;
    if (ext > 1e-18f) { (void)frexpf(ext / 254.0f, &k); }      // ext / 254 = m 2^k, m in [0.5, 1): 2^k > ext / 254
    k = k < -60 ? -60 : (k > 60 ? 60 : k);
    return k + 127;
}

// Which BVH2 nodes become 8-wide nodes: minimise the summed surface area of the 8-wide nodes (= the expected number of
// node steps of a random line) under the eight-slot limit, by dynamic programming over the BVH2 (the optimal collapse of
// Ylitie et al. 2017, with unit node cost).  T[n][j-1] = least cost of the subtree of n when it may occupy at most j slots
// of its parent's node: T[n][1] = area(n) + min_a T[l][a] + T[r][8-a] (n is a node of its own), T[n][j] = min(T[n][j-1],
// min_a T[l][a] + T[r][j-a]) (n is dissolved into the parent); leaves cost nothing.  Bottom-up with one arrival counter
// per node (as k_refit); k_emit8 then walks the choices down from each node.
__global__ void k_w8_parents(uint32_t n_inner, const float4* __restrict__ nodes, int* __restrict__ parent, uint32_t* __restrict__ need)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_inner) return;
    const float4 n3 = nodes[(size_t)i * 4 + 3];
    const int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
    need[i] = (c0 >= 0 ? 1u : 0u) + (c1 >= 0 ? 1u : 0u);
    if (c0 >= 0) parent[c0] = (int)i;
    if (c1 >= 0) parent[c1] = (int)i;
    if (i == 0) parent[0] = -1;
}
template <int W>
__device__ __forceinline__ float wide_t(const float* T, int ref, int j) { return ref >= 0 ? __ldcg(T + (size_t)ref * W + (j - 1)) : 0.0f; }
__device__ __forceinline__ float w8_t(const float* T, int ref, int j) { return wide_t<8>(T, ref, j); }
// W = node width (8: compressed nodes, 4: the quantised 4-wide nodes)
template <int W>
__global__ void k_wide_dp(uint32_t n_inner, const float4* __restrict__ nodes, const int* __restrict__ parent,
                        const uint32_t* __restrict__ need, uint32_t* __restrict__ arrive, float* T)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_inner || need[i] != 0u) return;
    int n = (int)i;
    for (;;) {
        cbox a, b;
        load_children(nodes, n, a, b);
        float ta[W], tb[W], t[W];
        for (int j = 1; j <= W; ++j) { ta[j - 1] = wide_t<W>(T, a.ref, j); tb[j - 1] = wide_t<W>(T, b.ref, j); }
        cbox u;
        u.lx = fminf(a.lx, b.lx); u.hx = fmaxf(a.hx, b.hx); u.ly = fminf(a.ly, b.ly); u.hy = fmaxf(a.hy, b.hy);
        u.lz = fminf(a.lz, b.lz); u.hz = fmaxf(a.hz, b.hz);
        float best = 3.0e38f;
        for (int x = 1; x <= W - 1; ++x) best = fminf(best, ta[x - 1] + tb[W - 1 - x]);
        t[0] = cbox_area(u) + best;
        for (int j = 2; j <= W; ++j) {
            float m = t[j - 2];
            for (int x = 1; x < j; ++x) m = fminf(m, ta[x - 1] + tb[j - x - 1]);
            t[j - 1] = m;
        }
        for (int j = 0; j < W; ++j) T[(size_t)n * W + j] = t[j];
        __threadfence();
        const int p = parent[n];
        if (p < 0) break;
        if (atomicAdd(arrive + p, 1u) + 1u < need[p]) break;
        n = p;
    }
}

// the children of wide node i chosen by the table: walks the choices of k_wide_dp down from BVH2 node i; returns their number
template <int W>
__device__ __forceinline__ int dp_cut(const float4* __restrict__ nodes, const float* __restrict__ T, int i, cbox* c)
{
    cbox st[W]; int sb[W]; int sp = 0, k = 0;
    {
        cbox l, r;
        load_children(nodes, i, l, r);
        float best = 3.0e38f; int ba = 1;
        for (int x = 1; x <= W - 1; ++x) { const float v = wide_t<W>(T, l.ref, x) + wide_t<W>(T, r.ref, W - x); if (v < best) { best = v; ba = x; } }
        st[0] = l; sb[0] = ba; st[1] = r; sb[1] = W - ba; sp = 2;
    }
    while (sp) {
        --sp;
        const cbox m = st[sp]; const int j = sb[sp];
        if (m.ref < 0 || j == 1) { c[k++] = m; continue; }
        cbox x, y;
        load_children(nodes, m.ref, x, y);
        float best = wide_t<W>(T, m.ref, 1); int ba = 0;                     // stay a node of its own ...
        for (int q = 1; q < j; ++q) { const float v = wide_t<W>(T, x.ref, q) + wide_t<W>(T, y.ref, j - q); if (v < best) { best = v; ba = q; } }
        if (!ba) { c[k++] = m; continue; }
        st[sp] = x; sb[sp] = ba; st[sp + 1] = y; sb[sp + 1] = j - ba; sp += 2;      // ... or dissolve into this one
    }
    return k;
}

// the 4-wide nodes with the children chosen by the table instead of greedily (FS_TUNE_COLLAPSE bit 4)
__global__ void k_emit4_dp(uint32_t n_inner, const float4* __restrict__ nodes, const float* __restrict__ T, const float* __restrict__ grid,
                           uint4* __restrict__ wnodes, int* __restrict__ wsrc)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_inner) return;
    const uint4 EMPTY = make_uint4(0x0000ffffu, 0x0000ffffu, 0x0000ffffu, 0x7fffffffu);
    cbox c[4];
    const int k = dp_cut<4>(nodes, T, (int)i, c);
    for (int j = 0; j < 4; ++j) {
        wnodes[(size_t)i * 4 + j] = (j < k) ? quant_box(c[j].lx, c[j].hx, c[j].ly, c[j].hy, c[j].lz, c[j].hz, c[j].ref, grid) : EMPTY;
        wsrc[(size_t)i * 4 + j] = (j < k) ? c[j].src : -1;
    }
}

// T = null: greedy collapse (open the inner child with the largest box until there are eight slots)
__global__ void k_emit8(uint32_t n_inner, const float4* __restrict__ nodes, const float* __restrict__ T, uint4* __restrict__ w8tmp,
                        int* __restrict__ w8ref)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_inner) return;
    cbox c[8];
    int k = 2;
    if (T) {
        k = dp_cut<8>(nodes, T, (int)i, c);
    } else {
        load_children(nodes, (int)i, c[0], c[1]);
        while (k < 8) {
            int pick = -1; float best = -1.0f;
            for (int j = 0; j < k; ++j)
                if (c[j].ref >= 0) { const float a = cbox_area(c[j]); if (a > best) { best = a; pick = j; } }
            if (pick < 0) break;
            const int r = c[pick].ref;
            load_children(nodes, r, c[pick], c[k]);
            ++k;
        }
    }
    float lx = c[0].lx, hx = c[0].hx, ly = c[0].ly, hy = c[0].hy, lz = c[0].lz, hz = c[0].hz;
    for (int j = 1; j < k; ++j) {
        lx = fminf(lx, c[j].lx); hx = fmaxf(hx, c[j].hx); ly = fminf(ly, c[j].ly); hy = fmaxf(hy, c[j].hy);
        lz = fminf(lz, c[j].lz); hz = fmaxf(hz, c[j].hz);
    }
    if (!(hx < 1e29f) || !(lx > -1e29f) || !(hy < 1e29f) || !(hz < 1e29f)) {       // single-triangle dummy child: never here (n >= 3)
        hx = fminf(hx, 1e29f); hy = fminf(hy, 1e29f); hz = fminf(hz, 1e29f);
    }
    // slot assignment: greedy on <centre(c) - centre(node), sigma_s>
    const float mx = 0.5f * (lx + hx), my = 0.5f * (ly + hy), mz = 0.5f * (lz + hz);
    int slot_of[8], child_in[8];
    for (int j = 0; j < 8; ++j) { slot_of[j] = -1; child_in[j] = -1; }
    for (int it = 0; it < k; ++it) {
        float best = -3.0e38f; int bc = -1, bs = -1;
        for (int j = 0; j < k; ++j) {
            if (slot_of[j] >= 0) continue;
            const float dx = 0.5f * (c[j].lx + c[j].hx) - mx, dy = 0.5f * (c[j].ly + c[j].hy) - my, dz = 0.5f * (c[j].lz + c[j].hz) - mz;
            for (int s = 0; s < 8; ++s) {
                if (child_in[s] >= 0) continue;
                const float cost = ((s & 1) ? dx : -dx) + ((s & 2) ? dy : -dy) + ((s & 4) ? dz : -dz);
                if (cost > best) { best = cost; bc = j; bs = s; }
            }
        }
        slot_of[bc] = bs; child_in[bs] = bc;
    }
    const int ebx = q8_exponent(hx - lx), eby = q8_exponent(hy - ly), ebz = q8_exponent(hz - lz);
    const float ix = __uint_as_float((uint32_t)(254 - ebx) << 23), iy = __uint_as_float((uint32_t)(254 - eby) << 23),
                iz = __uint_as_float((uint32_t)(254 - ebz) << 23);            // 2^-(eb-127)
    uint32_t q[12];                                 // lox[2] loy[2] loz[2] hix[2] hiy[2] hiz[2], one byte per slot
    for (int w = 0; w < 12; ++w) q[w] = 0u;
    uint32_t imask = 0, lmask = 0;
    int refs[8];
    for (int s = 0; s < 8; ++s) {
        const int j = child_in[s];
        uint32_t b[6];
        if (j < 0) { b[0] = b[1] = b[2] = 255u; b[3] = b[4] = b[5] = 0u; refs[s] = W8_EMPTY; }      // inverted box: never entered
        else {
            b[0] = q8_lo(c[j].lx, lx, ix); b[1] = q8_lo(c[j].ly, ly, iy); b[2] = q8_lo(c[j].lz, lz, iz);
            b[3] = q8_hi(c[j].hx, lx, ix); b[4] = q8_hi(c[j].hy, ly, iy); b[5] = q8_hi(c[j].hz, lz, iz);
            refs[s] = c[j].ref;
            if (c[j].ref >= 0) imask |= 1u << s; else lmask |= 1u << s;
        }
        for (int a = 0; a < 6; ++a) q[a * 2 + (s >> 2)] |= b[a] << (8 * (s & 3));
    }
    uint4* o = w8tmp + (size_t)i * 5;
    o[0] = make_uint4(__float_as_uint(lx), __float_as_uint(ly), __float_as_uint(lz), ((uint32_t)ebx << 23) | imask | (lmask << 8));
    o[1] = make_uint4((uint32_t)eby << 23, (uint32_t)ebz << 23, 0u, 0u);
    o[2] = make_uint4(q[0], q[1], q[2], q[3]);
    o[3] = make_uint4(q[4], q[5], q[6], q[7]);
    o[4] = make_uint4(q[8], q[9], q[10], q[11]);
    for (int s = 0; s < 8; ++s) w8ref[(size_t)i * 8 + s] = refs[s];
}

__global__ void k_w8_count(const uint4* __restrict__ w8tmp, const int* __restrict__ frontier, uint32_t nf,
                           uint32_t* __restrict__ cnt_in, uint32_t* __restrict__ cnt_leaf)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nf) return;
    const uint32_t w = w8tmp[(size_t)frontier[t] * 5].w;
    cnt_in[t] = (uint32_t)__popc(w & 0xffu);
    cnt_leaf[t] = (uint32_t)__popc((w >> 8) & 0xffu);
}

__global__ void k_w8_place(const uint4* __restrict__ w8tmp, const int* __restrict__ w8ref, uint4* __restrict__ dst,
                           const int* __restrict__ frontier, uint32_t nf, const uint32_t* __restrict__ off_in,
                           const uint32_t* __restrict__ off_leaf, uint32_t level_base, uint32_t tri_level_base,
                           int* __restrict__ next_frontier, const float4* __restrict__ tris, float4* __restrict__ tris8,
                           uint32_t* __restrict__ tri8_map)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nf) return;
    const int src = frontier[t];
    const uint4* p = w8tmp + (size_t)src * 5;
    uint4* q = dst + (size_t)(level_base + t) * 5;
    uint4 u1 = p[1];
    uint32_t oi = off_in[t], ol = tri_level_base + off_leaf[t];
    u1.z = level_base + nf + oi;
    u1.w = ol;
    q[0] = p[0]; q[1] = u1; q[2] = p[2]; q[3] = p[3]; q[4] = p[4];
    for (int s = 0; s < 8; ++s) {
        const int r = w8ref[(size_t)src * 8 + s];
        if (r == W8_EMPTY) continue;
        if (r >= 0) next_frontier[oi++] = r;
        else {
            const uint32_t first = (uint32_t)(~r) >> 3;          // single-triangle leaves (PLOC)
            for (int a = 0; a < 4; ++a) tris8[(size_t)ol * 4 + a] = tris[(size_t)first * 4 + a];
            tri8_map[ol] = first;
            ++ol;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Tree rotations (Kensler 2008) on the finished BVH2: for a node N with children L, R, swapping L with a child of
// R (or R with a child of L) changes only the box of R (or L); take the swap that shrinks it most.  Nodes of one
// depth own disjoint subtrees, so a whole level is processed in parallel, levels bottom-up (a rotation only changes
// depths below it).  The level lists come from a breadth-first expansion (k_bvh2_count / k_bvh2_place).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void store_children(float4* __restrict__ nodes, int i, const cbox& a, const cbox& b)
{
    nodes[(size_t)i * 4] = make_float4(a.lx, a.hx, a.ly, a.hy);
    nodes[(size_t)i * 4 + 1] = make_float4(b.lx, b.hx, b.ly, b.hy);
    nodes[(size_t)i * 4 + 2] = make_float4(a.lz, a.hz, b.lz, b.hz);
    nodes[(size_t)i * 4 + 3] = make_float4(__int_as_float(a.ref), __int_as_float(b.ref), 0.f, 0.f);
}
__device__ __forceinline__ cbox cbox_union(const cbox& a, const cbox& b, int ref)
{
    cbox u;
    u.lx = fminf(a.lx, b.lx); u.hx = fmaxf(a.hx, b.hx); u.ly = fminf(a.ly, b.ly); u.hy = fmaxf(a.hy, b.hy);
    u.lz = fminf(a.lz, b.lz); u.hz = fmaxf(a.hz, b.hz); u.ref = ref; u.src = -1;
    return u;
}

__global__ void k_bvh2_count(const float4* __restrict__ nodes, const int* __restrict__ frontier, uint32_t nf, uint32_t* __restrict__ cnt)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nf) return;
    const float4 n3 = nodes[(size_t)frontier[t] * 4 + 3];
    cnt[t] = (__float_as_int(n3.x) >= 0 ? 1u : 0u) + (__float_as_int(n3.y) >= 0 ? 1u : 0u);
}
__global__ void k_bvh2_place(const float4* __restrict__ nodes, const int* __restrict__ frontier, uint32_t nf,
                             const uint32_t* __restrict__ off, int* __restrict__ next)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nf) return;
    const float4 n3 = nodes[(size_t)frontier[t] * 4 + 3];
    uint32_t o = off[t];
    const int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
    if (c0 >= 0) next[o++] = c0;
    if (c1 >= 0) next[o] = c1;
}

__global__ void k_rotate(float4* __restrict__ nodes, const int* __restrict__ level, uint32_t nl, uint32_t* __restrict__ n_done)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nl) return;
    const int N = level[t];
    cbox L, R;
    load_children(nodes, N, L, R);
    float best = 0.0f; int op = 0;
    cbox LL, LR, RL, RR;
    if (R.ref >= 0) {
        load_children(nodes, R.ref, RL, RR);
        const float aR = cbox_area(R);
        const float d1 = cbox_area(cbox_union(L, RR, 0)) - aR;        // L <-> RL
        const float d2 = cbox_area(cbox_union(RL, L, 0)) - aR;        // L <-> RR
        if (d1 < best) { best = d1; op = 1; }
        if (d2 < best) { best = d2; op = 2; }
    }
    if (L.ref >= 0) {
        load_children(nodes, L.ref, LL, LR);
        const float aL = cbox_area(L);
        const float d3 = cbox_area(cbox_union(R, LR, 0)) - aL;        // R <-> LL
        const float d4 = cbox_area(cbox_union(LL, R, 0)) - aL;        // R <-> LR
        if (d3 < best) { best = d3; op = 3; }
        if (d4 < best) { best = d4; op = 4; }
    }
    if (op == 0) return;
    if (op == 1) {            // N = (RL, R'), R' = (L, RR)
        const cbox Rn = cbox_union(L, RR, R.ref);
        store_children(nodes, R.ref, L, RR);
        store_children(nodes, N, RL, Rn);
    } else if (op == 2) {     // N = (RR, R'), R' = (RL, L)
        const cbox Rn = cbox_union(RL, L, R.ref);
        store_children(nodes, R.ref, RL, L);
        store_children(nodes, N, RR, Rn);
    } else if (op == 3) {     // N = (L', LL), L' = (R, LR)
        const cbox Ln = cbox_union(R, LR, L.ref);
        store_children(nodes, L.ref, R, LR);
        store_children(nodes, N, Ln, LL);
    } else {                  // N = (L', LR), L' = (LL, R)
        const cbox Ln = cbox_union(LL, R, L.ref);
        store_children(nodes, L.ref, LL, R);
        store_children(nodes, N, Ln, LR);
    }
    atomicAdd(n_done, 1u);
}

// surface-area cost of the BVH2: sum of the areas of all child boxes (the expected number of boxes a random line crosses,
// up to the root's area); used to compare candidate trees
__global__ void k_sah_cost(uint32_t n_inner, const float4* __restrict__ nodes, double* __restrict__ out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    double a = 0.0;
    if (i < n_inner) {
        cbox c0, c1;
        load_children(nodes, (int)i, c0, c1);
        a = (double)cbox_area(c0) + (double)cbox_area(c1);
    }
    for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if ((threadIdx.x & 31) == 0 && a != 0.0) atomicAdd(out, a);
}

// single-triangle scene: root whose second child is a far-away point box (never entered in practice)
__device__ __forceinline__ void emit_single(float4 l0, float4 h0, float4* __restrict__ nodes)
{
    float pad = box_pad(l0, h0);
    const float F = 1e30f;
    nodes[0] = make_float4(l0.x - pad, h0.x + pad, l0.y - pad, h0.y + pad);
    nodes[1] = make_float4(F, F, F, F);
    nodes[2] = make_float4(l0.z - pad, h0.z + pad, F, F);
    nodes[3] = make_float4(__int_as_float(~0), __int_as_float(~0), 0.f, 0.f);
}
__global__ void k_emit_single(const float4* __restrict__ bb_lo, const float4* __restrict__ bb_hi,
                              float4* __restrict__ nodes)
{
    emit_single(bb_lo[0], bb_hi[0], nodes);
}

// BFS copy of the top of the tree; children inside the copy get FS_TOP_FLAG | local index.
// One thread: the order of local-index assignment is sequential by construction (<= 2048 nodes).
__global__ void k_top_treelet(const float4* __restrict__ nodes, uint32_t n_inner, uint32_t cap,
                              float4* __restrict__ top, uint32_t* __restrict__ n_top_out, int* __restrict__ queue)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint32_t qn = 0;
    queue[qn++] = 0;
    for (uint32_t p = 0; p < qn; ++p) {
        const float4* src = nodes + (size_t)queue[p] * 4;
        float4 n3 = src[3];
        int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
        if (c0 >= 0 && qn < cap) { queue[qn] = c0; c0 = FS_TOP_FLAG | (int)qn; ++qn; }
        if (c1 >= 0 && qn < cap) { queue[qn] = c1; c1 = FS_TOP_FLAG | (int)qn; ++qn; }
        top[(size_t)p * 4 + 0] = src[0];
        top[(size_t)p * 4 + 1] = src[1];
        top[(size_t)p * 4 + 2] = src[2];
        top[(size_t)p * 4 + 3] = make_float4(__int_as_float(c0), __int_as_float(c1), 0.f, 0.f);
    }
    *n_top_out = qn;
    (void)n_inner;
}

// largest leaf / reachable inner-node statistics are cheap enough on one pass over ranges
__global__ void k_leaf_stats(int n, const int2* __restrict__ ranges, uint32_t* __restrict__ max_leaf, int leaf_max)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int cnt = ranges[i].y - ranges[i].x + 1;
    if (cnt <= leaf_max) atomicMax(max_leaf, (uint32_t)cnt);
}

// ---------------------------------------------------------------------------------------------
// Refit (fs_bvh_refit): the committed topology with boxes recomputed from moved triangles.  Every box of the build is
// box_pad(unpadded box) and every unpadded box a fminf / fmaxf union of raw triangle bounds: exact and independent of
// the order of the union, so refitting unchanged triangles reproduces the committed arrays bit for bit.
// ---------------------------------------------------------------------------------------------
__global__ void k_refit_tris(uint32_t n, const float* __restrict__ verts, const uint32_t* __restrict__ tri_orig,
                             const uint32_t* __restrict__ tri_mat, float4* __restrict__ tris, float4* __restrict__ tri_nm)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    pack_tri(verts, tri_orig[j], tri_mat[j], j, tris, tri_nm);
}

// unpadded box of child reference r: a leaf ~(j << 3 | cnt - 1) is the union of the raw bounds of sorted triangles
// j .. j + cnt - 1, an inner child the box its own thread stored before it released this node
__device__ __forceinline__ void refit_child(int r, const float* __restrict__ verts, const uint32_t* __restrict__ tri_orig,
                                            const float4* ubox, float4& lo, float4& hi)
{
    if (r >= 0) { lo = __ldcg(ubox + 2 * (size_t)r); hi = __ldcg(ubox + 2 * (size_t)r + 1); return; }
    const uint32_t e = (uint32_t)~r, first = e >> 3, cnt = (e & 7u) + 1u;
    tri_box(verts + (size_t)tri_orig[first] * 9, lo, hi);
    for (uint32_t k = 1; k < cnt; ++k) {
        float4 l, h;
        tri_box(verts + (size_t)tri_orig[first + k] * 9, l, h);
        lo = make_float4(fminf(lo.x, l.x), fminf(lo.y, l.y), fminf(lo.z, l.z), 0.f);
        hi = make_float4(fmaxf(hi.x, h.x), fmaxf(hi.y, h.y), fmaxf(hi.z, h.z), 0.f);
    }
}

// bottom-up over the BVH2 with one arrival counter per node (as k_wide_dp): a thread starts at every node without inner
// children; the last of a node's inner children to finish carries on with the parent.  Child entries are written in the
// float form of k_ploc_merge / k_emit; the child references (node word 3) are left alone.
__global__ void k_refit_nodes(uint32_t n_inner, const float* __restrict__ verts, const uint32_t* __restrict__ tri_orig,
                              const int* __restrict__ parent, const uint32_t* __restrict__ need, uint32_t* __restrict__ arrive,
                              float4* __restrict__ nodes, float4* ubox)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_inner || need[i] != 0u) return;
    int n = (int)i;
    for (;;) {
        const float4 n3 = nodes[(size_t)n * 4 + 3];
        float4 l0, h0, l1, h1;
        refit_child(__float_as_int(n3.x), verts, tri_orig, ubox, l0, h0);
        refit_child(__float_as_int(n3.y), verts, tri_orig, ubox, l1, h1);
        const float p0 = box_pad(l0, h0), p1 = box_pad(l1, h1);
        nodes[(size_t)n * 4 + 0] = make_float4(l0.x - p0, h0.x + p0, l0.y - p0, h0.y + p0);
        nodes[(size_t)n * 4 + 1] = make_float4(l1.x - p1, h1.x + p1, l1.y - p1, h1.y + p1);
        nodes[(size_t)n * 4 + 2] = make_float4(l0.z - p0, h0.z + p0, l1.z - p1, h1.z + p1);
        __stcg(ubox + 2 * (size_t)n, make_float4(fminf(l0.x, l1.x), fminf(l0.y, l1.y), fminf(l0.z, l1.z), 0.f));
        __stcg(ubox + 2 * (size_t)n + 1, make_float4(fmaxf(h0.x, h1.x), fmaxf(h0.y, h1.y), fmaxf(h0.z, h1.z), 0.f));
        __threadfence();
        const int p = parent[n];
        if (p < 0) break;
        if (atomicAdd(arrive + p, 1u) + 1u < need[p]) break;
        __threadfence();
        n = p;
    }
}

// single-triangle scene: the root of k_emit_single, from the moved triangle
__global__ void k_refit_single(const float* __restrict__ verts, const uint32_t* __restrict__ tri_orig, float4* __restrict__ nodes)
{
    float4 lo, hi;
    tri_box(verts + (size_t)tri_orig[0] * 9, lo, hi);
    emit_single(lo, hi, nodes);
}

// every slot of the wide nodes re-quantised from the BVH2 child entry it was made from (wsrc = node * 2 + side); the
// child reference (u.w) and the empty slots stay as they are
__global__ void k_requant4(uint32_t n_slots, const float4* __restrict__ nodes, const int* __restrict__ wsrc,
                           const float* __restrict__ grid, uint4* __restrict__ wnodes)
{
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_slots) return;
    const int src = wsrc[s];
    if (src < 0) return;
    cbox a, b;
    load_children(nodes, src >> 1, a, b);
    const cbox& c = (src & 1) ? b : a;
    const uint4 q = quant_box(c.lx, c.hx, c.ly, c.hy, c.lz, c.hz, 0, grid);
    uint4 u = wnodes[s];
    u.x = q.x; u.y = q.y; u.z = q.z;
    wnodes[s] = u;
}

// ---------------------------------------------------------------------------------------------
// Parallel reinsertion on the BVH2 (Bittner et al. 2013; on the GPU: Meister & Bittner 2018).  A move takes the subtree
// N out of its parent P (the sibling S takes P's place under the grandparent G) and puts it back as the sibling of some
// other subtree X, reusing P as their new parent.  Unlike a rotation it can move N anywhere in the tree.  Slots are
// child entries, slot = 2 * node + side.  One iteration:
//   k_ri_search  one thread per candidate slot (N's box at least `thr`): the best X by the change of the surface-area
//                cost (sum of all non-root boxes).  The removal saves area(P) plus the shrinkage of P's ancestors below
//                the lowest common ancestor of P and X; the insertion adds area(X u N) plus the growth of X's ancestors
//                below it.  Depth-first from the ancestors' off-path children with the branch-and-bound of Bittner et al.
//                (whatever lies below X pays at least area(N) on top of the growth down to X).
//   k_ri_lock    a move locks the nodes on the paths from P and from X's parent up to their common ancestor, and G:
//                u64 atomicMax of (saving, slot), so the winner of every node is independent of the thread order
//   k_ri_apply   moves that hold all their locks rewrite the child references of G, X's parent and P.  Disjoint lock
//                paths keep the moves independent (no cycles: a move into N's subtree crosses P).
// then the boxes are refitted bottom-up (k_refit_nodes: exact unions, padded as PLOC pads them).  The root stays node 0.
// ---------------------------------------------------------------------------------------------
#ifndef FS_REINSERT_ITERS
#define FS_REINSERT_ITERS 32        // default iteration cap (FS_TUNE_REINSERT overrides)
#endif
constexpr int RI_MAXD = 64;         // ancestors of P a search may use; deeper candidates are skipped
constexpr int RI_STACK = 128;       // search stack; a full stack drops branches (the search stays a valid heuristic)

__device__ __forceinline__ cbox slot_box(const float4* __restrict__ nodes, int slot)
{
    cbox a, b;
    load_children(nodes, slot >> 1, a, b);
    return (slot & 1) ? b : a;
}
__device__ __forceinline__ int slot_ref(const float4* nodes, int slot)
{
    return ((const int*)(nodes + (size_t)(slot >> 1) * 4 + 3))[slot & 1];
}

// area histogram of the candidate slots (12 high bits of the ordered float): picks the size threshold of the candidates
__global__ void k_ri_hist(uint32_t n_inner, const float4* __restrict__ nodes, uint32_t* __restrict__ hist)
{
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x + 2u;
    if (s >= 2u * n_inner) return;
    atomicAdd(hist + (f2ord(cbox_area(slot_box(nodes, (int)s))) >> 20), 1u);
}

__global__ void k_ri_search(uint32_t n_inner, const float4* __restrict__ nodes, const int* __restrict__ parent, float thr,
                            float min_gain, float* __restrict__ mv_gain, int* __restrict__ mv_dst)
{
    const int s = (int)(blockIdx.x * blockDim.x + threadIdx.x) + 2;       // the root's slots never move (P = root has no G)
    if (s >= 2 * (int)n_inner) return;
    mv_dst[s] = -1;
    const int P = s >> 1;
    cbox a, b;
    load_children(nodes, P, a, b);
    const cbox N = (s & 1) ? b : a, S = (s & 1) ? a : b;
    const float aN = cbox_area(N);
    if (!(aN >= thr)) return;
    struct ent { int slot; float c, g; };
    ent st[RI_STACK];
    int sp = 0;
    // up from P: the off-path child of every ancestor, with the saving of the removal when that ancestor is the common one
    cbox cur = S;                   // the box of the current ancestor once N has left it
    float g = 0.0f;
    for (int c = P, d = 0;; ++d) {
        const int u = parent[c];
        if (u < 0) break;
        if (d == RI_MAXD) return;
        cbox l, r;
        load_children(nodes, u, l, r);
        const int cs = (l.ref == c) ? 0 : 1;
        const cbox& cb = cs ? r : l;
        const cbox& ob = cs ? l : r;
        g += (c == P) ? cbox_area(cb) : cbox_area(cb) - cbox_area(cur);
        cur = cbox_union(cur, ob, 0);
        st[sp++] = ent{2 * u + (cs ^ 1), 0.0f, g};
        c = u;
    }
    for (int i = 0, j = sp - 1; i < j; ++i, --j) { const ent t = st[i]; st[i] = st[j]; st[j] = t; }   // nearest first off the stack
    if (S.ref >= 0) {               // inside S (S itself is where N is now): S grows by N
        const float c0 = cbox_area(cbox_union(S, N, 0)) - cbox_area(S), aP = st[sp - 1].g;
        st[sp++] = ent{2 * S.ref, c0, aP};
        st[sp++] = ent{2 * S.ref + 1, c0, aP};
    }
    float best = -min_gain * aN; int bdst = -1;       // a move must save a little more than float noise
    while (sp) {
        const ent e = st[--sp];
        if (e.c + aN - e.g >= best) continue;
        const cbox X = slot_box(nodes, e.slot);
        const float u = cbox_area(cbox_union(X, N, 0));
        const float tot = e.c + u - e.g;
        if (tot < best) { best = tot; bdst = e.slot; }
        if (X.ref >= 0) {
            const float c2 = e.c + u - cbox_area(X);
            if (c2 + aN - e.g < best && sp + 2 <= RI_STACK) {
                st[sp++] = ent{2 * X.ref + 1, c2, e.g};
                st[sp++] = ent{2 * X.ref, c2, e.g};
            }
        }
    }
    mv_gain[s] = -best;
    mv_dst[s] = bdst;
}

// the lock set of move (slot s -> slot dst): P .. common ancestor, X's parent .. below it, and G; visits each node with f
template <typename F>
__device__ __forceinline__ void ri_lockset(const int* __restrict__ parent, int s, int dst, F f)
{
    int up[RI_MAXD + 2]; int d = 0;
    for (int c = s >> 1; c >= 0 && d < RI_MAXD + 2; c = parent[c]) up[d++] = c;      // P, G, ..., root (the search bounded it)
    int lca = 0;
    for (int v = dst >> 1; v >= 0; v = parent[v]) {
        bool on = false;
        for (int k = 0; k < d; ++k) if (up[k] == v) { on = true; break; }
        if (on) { lca = v; break; }
        f(v);
    }
    for (int k = 0; k < d; ++k) { f(up[k]); if (up[k] == lca) break; }
    if (d > 1) f(up[1]);
}

__device__ __forceinline__ unsigned long long ri_key(float gain, int s)
{
    return ((unsigned long long)__float_as_uint(gain) << 32) | (unsigned long long)(uint32_t)s;     // gain > 0: ordered as uint
}

__global__ void k_ri_lock(uint32_t n_inner, const int* __restrict__ parent, const float* __restrict__ mv_gain,
                          const int* __restrict__ mv_dst, unsigned long long* __restrict__ lock)
{
    const int s = (int)(blockIdx.x * blockDim.x + threadIdx.x) + 2;
    if (s >= 2 * (int)n_inner || mv_dst[s] < 0) return;
    const unsigned long long key = ri_key(mv_gain[s], s);
    ri_lockset(parent, s, mv_dst[s], [&](int v) { atomicMax(lock + v, key); });
}

__device__ __forceinline__ void set_ref(float4* nodes, int slot, int ref)
{
    ((int*)(nodes + (size_t)(slot >> 1) * 4 + 3))[slot & 1] = ref;
}

__global__ void k_ri_apply(uint32_t n_inner, const int* __restrict__ parent, const float* __restrict__ mv_gain,
                           const int* __restrict__ mv_dst, const unsigned long long* __restrict__ lock, float4* nodes,
                           uint32_t* __restrict__ n_moved)
{
    const int s = (int)(blockIdx.x * blockDim.x + threadIdx.x) + 2;
    if (s >= 2 * (int)n_inner) return;
    const int dst = mv_dst[s];
    if (dst < 0) return;
    const unsigned long long key = ri_key(mv_gain[s], s);
    bool own = true;
    ri_lockset(parent, s, dst, [&](int v) { own = own && (lock[v] == key); });
    if (!own) return;
    const int P = s >> 1, G = parent[P];
    const int Nr = slot_ref(nodes, s), Sr = slot_ref(nodes, s ^ 1), Xr = slot_ref(nodes, dst);
    set_ref(nodes, 2 * G + (slot_ref(nodes, 2 * G) == P ? 0 : 1), Sr);
    set_ref(nodes, dst, P);
    set_ref(nodes, 2 * P, Nr);
    set_ref(nodes, 2 * P + 1, Xr);
    atomicAdd(n_moved, 1u);
}

}  // namespace

uint32_t fs_radix_sort_blocks(uint32_t n) { return (n + SORT_TILE - 1) / SORT_TILE; }

void fs_radix_sort_u64(cudaStream_t st, uint64_t* keys, uint32_t* vals, uint64_t* keys_tmp, uint32_t* vals_tmp, uint32_t n,
                       uint32_t* block_hist, uint64_t* launches)
{
    const uint32_t n_blocks = fs_radix_sort_blocks(n);
    uint64_t *ki = keys, *ko = keys_tmp;
    uint32_t *vi = vals, *vo = vals_tmp;
    for (int pass = 0; pass < 8; ++pass) {
        int shift = pass * 8;
        k_sort_hist<<<n_blocks, SORT_THREADS, 0, st>>>(ki, n, shift, block_hist, n_blocks);
        k_sort_scan<<<1, 1024, 0, st>>>(block_hist, 256u * n_blocks);
        k_sort_scatter<<<n_blocks, SORT_THREADS, 0, st>>>(ki, vi, ko, vo, n, shift, block_hist, n_blocks);
        *launches += 3;
        uint64_t* tk = ki; ki = ko; ko = tk;
        uint32_t* tv = vi; vi = vo; vo = tv;
    }
    // 8 passes: the result is back in keys / vals
}

#define BCHECK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { err = e_; goto fail; } } while (0)

// exclusive scan helper (device arrays); tile_sums must hold ceil(n/1024) + 1 entries
void fs_scan_u32(cudaStream_t st, const uint32_t* in, uint32_t* out, uint32_t n, uint32_t* tile_sums,
                 uint32_t* total, uint64_t* launches)
{
    const uint32_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    k_scan_tiles<<<tiles, SCAN_TILE, 0, st>>>(in, out, n, tile_sums);
    k_sort_scan<<<1, 1024, 0, st>>>(tile_sums, tiles);
    k_scan_add<<<tiles, SCAN_TILE, 0, st>>>(out, n, tile_sums);
    k_scan_total<<<1, 32, 0, st>>>(in, out, n, total);
    *launches += 4;
}

static cudaError_t ploc_build(cudaStream_t st, uint32_t n, const float4* bb_lo, const float4* bb_hi, float4* nodes,
                              uint64_t* launches, int radius)
{
    cudaError_t err = cudaSuccess;
    float4 *lo[2] = {nullptr, nullptr}, *hi[2] = {nullptr, nullptr};
    int* ref[2] = {nullptr, nullptr};
    uint32_t *nn = nullptr, *keep = nullptr, *mflag = nullptr, *keep_scan = nullptr, *merge_scan = nullptr,
             *tile_sums = nullptr, *totals = nullptr;
    const uint32_t n_inner = n - 1;
    const int TPB = 256;
    uint32_t cur = n, made = 0;
    int pp = 0;
    for (int k = 0; k < 2; ++k) {
        BCHECK(cudaMalloc(&lo[k], sizeof(float4) * n));
        BCHECK(cudaMalloc(&hi[k], sizeof(float4) * n));
        BCHECK(cudaMalloc(&ref[k], sizeof(int) * n));
    }
    BCHECK(cudaMalloc(&nn, 4ull * n)); BCHECK(cudaMalloc(&keep, 4ull * n)); BCHECK(cudaMalloc(&mflag, 4ull * n));
    BCHECK(cudaMalloc(&keep_scan, 4ull * n)); BCHECK(cudaMalloc(&merge_scan, 4ull * n));
    BCHECK(cudaMalloc(&tile_sums, 4ull * ((n + SCAN_TILE - 1) / SCAN_TILE + 2)));
    BCHECK(cudaMalloc(&totals, 4 * 2));
    k_ploc_init<<<(n + TPB - 1) / TPB, TPB, 0, st>>>(n, bb_lo, bb_hi, lo[0], hi[0], ref[0]); ++*launches;
    for (int round = 0; cur > 1 && round < 4096; ++round) {
        const uint32_t g = (cur + TPB - 1) / TPB;
        k_ploc_nn<<<g, TPB, 0, st>>>(cur, lo[pp], hi[pp], nn, radius);
        k_ploc_flags<<<g, TPB, 0, st>>>(cur, nn, keep, mflag);
        *launches += 2;
        fs_scan_u32(st, keep, keep_scan, cur, tile_sums, totals, launches);
        fs_scan_u32(st, mflag, merge_scan, cur, tile_sums, totals + 1, launches);
        k_ploc_merge<<<g, TPB, 0, st>>>(cur, nn, keep_scan, merge_scan, keep, mflag, made, n_inner, lo[pp], hi[pp], ref[pp],
                                        lo[pp ^ 1], hi[pp ^ 1], ref[pp ^ 1], nodes);
        ++*launches;
        uint32_t h[2];
        BCHECK(cudaMemcpyAsync(h, totals, sizeof(h), cudaMemcpyDeviceToHost, st));
        BCHECK(cudaStreamSynchronize(st));
        if (h[1] == 0 || h[0] >= cur) { err = cudaErrorUnknown; goto fail; }      // no progress: cannot happen (the global minimum pair is mutual)
        made += h[1];
        cur = h[0];
        pp ^= 1;
    }
    if (cur != 1 || made != n_inner) err = cudaErrorUnknown;
fail:
    for (int k = 0; k < 2; ++k) { cudaFree(lo[k]); cudaFree(hi[k]); cudaFree(ref[k]); }
    cudaFree(nn); cudaFree(keep); cudaFree(mflag); cudaFree(keep_scan); cudaFree(merge_scan); cudaFree(tile_sums); cudaFree(totals);
    return err;
}

// `sweeps` bottom-up rotation sweeps over the BVH2 in `nodes`; *n_rot = rotations applied
static cudaError_t bvh2_rotate(cudaStream_t st, uint32_t n_inner, float4* nodes, int sweeps, uint64_t* launches, uint32_t* n_rot)
{
    cudaError_t err = cudaSuccess;
    int* order = nullptr;                 // breadth-first list of the inner nodes, level after level
    uint32_t *cnt = nullptr, *off = nullptr, *tile_sums = nullptr, *total = nullptr, *d_done = nullptr;
    const int TPB = 256;
    std::vector<std::pair<uint32_t, uint32_t>> levels;
    const int zero = 0;
    *n_rot = 0;
    BCHECK(cudaMalloc(&order, 4ull * n_inner));
    BCHECK(cudaMalloc(&cnt, 4ull * n_inner)); BCHECK(cudaMalloc(&off, 4ull * n_inner));
    BCHECK(cudaMalloc(&tile_sums, 4ull * ((n_inner + SCAN_TILE - 1) / SCAN_TILE + 2)));
    BCHECK(cudaMalloc(&total, 4)); BCHECK(cudaMalloc(&d_done, 4));
    BCHECK(cudaMemsetAsync(d_done, 0, 4, st));
    for (int sw = 0; sw < sweeps; ++sw) {
        levels.clear();
        BCHECK(cudaMemcpyAsync(order, &zero, 4, cudaMemcpyHostToDevice, st));
        uint32_t base = 0, nf = 1;
        while (nf) {
            levels.push_back(std::make_pair(base, nf));
            const uint32_t g = (nf + TPB - 1) / TPB;
            uint32_t next = 0;
            k_bvh2_count<<<g, TPB, 0, st>>>(nodes, order + base, nf, cnt); ++*launches;
            fs_scan_u32(st, cnt, off, nf, tile_sums, total, launches);
            BCHECK(cudaMemcpyAsync(&next, total, 4, cudaMemcpyDeviceToHost, st));
            BCHECK(cudaStreamSynchronize(st));
            if (base + nf + next > n_inner) { err = cudaErrorUnknown; goto fail; }
            if (next) { k_bvh2_place<<<g, TPB, 0, st>>>(nodes, order + base, nf, off, order + base + nf); ++*launches; }
            base += nf; nf = next;
        }
        for (size_t l = levels.size(); l-- > 0;) {
            const uint32_t nl = levels[l].second;
            k_rotate<<<(nl + TPB - 1) / TPB, TPB, 0, st>>>(nodes, order + levels[l].first, nl, d_done); ++*launches;
        }
    }
    BCHECK(cudaMemcpyAsync(n_rot, d_done, 4, cudaMemcpyDeviceToHost, st));
    BCHECK(cudaStreamSynchronize(st));
    BCHECK(cudaGetLastError());
fail:
    cudaFree(order); cudaFree(cnt); cudaFree(off); cudaFree(tile_sums); cudaFree(total); cudaFree(d_done);
    return err;
}

// Up to `iters` reinsertion iterations over the BVH2 in `nodes` (see k_ri_search).  The candidates are the largest 10 %
// of the child boxes of the tree as it comes in.  The loop stops early when an iteration moves nothing or saves less
// than 0.01 % of the surface-area cost (on the room an iteration saves < 0.1 % from the 9th on, because few moves win all
// their locks, yet iterations 9-32 still take another 3 % off the 4-wide nodes' summed area); an iteration that raised
// the cost (its moves were judged on the boxes before the others moved) is undone, so the result never costs more than
// the input.
static cudaError_t bvh2_reinsert(cudaStream_t st, uint32_t n_inner, const float* d_verts, const uint32_t* tri_orig,
                                 float4* nodes, int iters, uint64_t* launches)
{
    cudaError_t err = cudaSuccess;
    int *parent = nullptr, *mv_dst = nullptr;
    uint32_t *need = nullptr, *arrive = nullptr, *hist = nullptr;
    float4 *ubox = nullptr, *backup = nullptr;
    float* mv_gain = nullptr;
    unsigned long long* lock = nullptr;
    char* misc = nullptr;                         // [0] cost (double), [8] moves (u32)
    const int TPB = 256;
    const uint32_t n_slots = 2u * n_inner - 2u, gs = (n_slots + TPB - 1) / TPB, gi = (n_inner + TPB - 1) / TPB;
    std::vector<uint32_t> h_hist(4096);
    double cost0 = 0.0, prev = 0.0;
    int it = 0;
    uint32_t total_moves = 0;
    float thr = 0.0f;
    BCHECK(cudaMalloc(&parent, 4ull * n_inner)); BCHECK(cudaMalloc(&need, 4ull * n_inner)); BCHECK(cudaMalloc(&arrive, 4ull * n_inner));
    BCHECK(cudaMalloc(&ubox, sizeof(float4) * 2ull * n_inner)); BCHECK(cudaMalloc(&backup, sizeof(float4) * 4ull * n_inner));
    BCHECK(cudaMalloc(&lock, 8ull * n_inner));
    BCHECK(cudaMalloc(&mv_gain, 4ull * 2 * n_inner)); BCHECK(cudaMalloc(&mv_dst, 4ull * 2 * n_inner));
    BCHECK(cudaMalloc(&hist, 4ull * 4096)); BCHECK(cudaMalloc(&misc, 16));
    BCHECK(cudaMemsetAsync(hist, 0, 4ull * 4096, st));
    BCHECK(cudaMemsetAsync(misc, 0, 16, st));
    k_ri_hist<<<gs, TPB, 0, st>>>(n_inner, nodes, hist);
    k_sah_cost<<<gi, TPB, 0, st>>>(n_inner, nodes, (double*)misc);
    *launches += 2;
    BCHECK(cudaMemcpyAsync(h_hist.data(), hist, 4ull * 4096, cudaMemcpyDeviceToHost, st));
    BCHECK(cudaMemcpyAsync(&cost0, misc, 8, cudaMemcpyDeviceToHost, st));
    BCHECK(cudaStreamSynchronize(st));
    {
        uint64_t acc = 0;
        for (int bin = 4095; bin >= 0; --bin) {
            acc += h_hist[bin];
            if (acc * 10 >= n_slots) { thr = ord2f((uint32_t)bin << 20); break; }
        }
    }
    prev = cost0;
    for (it = 0; it < iters; ++it) {
        struct { double cost; uint32_t moved; } h;
        BCHECK(cudaMemsetAsync(lock, 0, 8ull * n_inner, st));
        BCHECK(cudaMemsetAsync(misc, 0, 16, st));
        k_w8_parents<<<gi, TPB, 0, st>>>(n_inner, nodes, parent, need);
        k_ri_search<<<gs, TPB, 0, st>>>(n_inner, nodes, parent, thr, 1e-5f, mv_gain, mv_dst);
        k_ri_lock<<<gs, TPB, 0, st>>>(n_inner, parent, mv_gain, mv_dst, lock);
        BCHECK(cudaMemcpyAsync(backup, nodes, sizeof(float4) * 4ull * n_inner, cudaMemcpyDeviceToDevice, st));
        k_ri_apply<<<gs, TPB, 0, st>>>(n_inner, parent, mv_gain, mv_dst, lock, nodes, (uint32_t*)(misc + 8));
        BCHECK(cudaMemsetAsync(arrive, 0, 4ull * n_inner, st));
        k_w8_parents<<<gi, TPB, 0, st>>>(n_inner, nodes, parent, need);
        k_refit_nodes<<<gi, TPB, 0, st>>>(n_inner, d_verts, tri_orig, parent, need, arrive, nodes, ubox);
        k_sah_cost<<<gi, TPB, 0, st>>>(n_inner, nodes, (double*)misc);
        *launches += 7;
        BCHECK(cudaMemcpyAsync(&h, misc, sizeof(h), cudaMemcpyDeviceToHost, st));
        BCHECK(cudaStreamSynchronize(st));
        BCHECK(cudaGetLastError());
        if (h.moved == 0) break;
        if (h.cost > prev) {
            BCHECK(cudaMemcpyAsync(nodes, backup, sizeof(float4) * 4ull * n_inner, cudaMemcpyDeviceToDevice, st));
            BCHECK(cudaStreamSynchronize(st));
            break;
        }
        total_moves += h.moved;
        const bool small = prev - h.cost < 1e-4 * prev;
        prev = h.cost;
        if (small) { ++it; break; }
    }
    if (getenv("FS_VERBOSE"))
        fprintf(stderr, "[frequensee] reinsertion: %d iterations, %u moves, surface-area cost %.6g -> %.6g (%.2f %%)\n", it,
                total_moves, cost0, prev, cost0 > 0.0 ? 100.0 * (prev - cost0) / cost0 : 0.0);
fail:
    cudaFree(parent); cudaFree(need); cudaFree(arrive); cudaFree(ubox); cudaFree(backup); cudaFree(lock);
    cudaFree(mv_gain); cudaFree(mv_dst); cudaFree(hist); cudaFree(misc);
    return err;
}

// sparse (one wide node per BVH2 node) -> dense breadth-first array; *dense_out is allocated here
// (the slot provenance sparse_prov is carried along into *dense_prov_out, also allocated here)
static cudaError_t wide_compact(cudaStream_t st, uint32_t n_inner, const uint4* sparse, const int* sparse_prov, uint4** dense_out,
                                int** dense_prov_out, uint32_t* n_wide_out, uint64_t* launches)
{
    cudaError_t err = cudaSuccess;
    int* fr[2] = {nullptr, nullptr};
    uint32_t *cnt = nullptr, *off = nullptr, *tile_sums = nullptr, *total = nullptr;
    uint4* dense = nullptr;
    int* dense_prov = nullptr;
    const int TPB = 256;
    uint32_t nf = 1, base = 0;
    int pp = 0;
    const int zero = 0;
    BCHECK(cudaMalloc(&fr[0], 4ull * n_inner)); BCHECK(cudaMalloc(&fr[1], 4ull * n_inner));
    BCHECK(cudaMalloc(&cnt, 4ull * n_inner)); BCHECK(cudaMalloc(&off, 4ull * n_inner));
    BCHECK(cudaMalloc(&tile_sums, 4ull * ((n_inner + SCAN_TILE - 1) / SCAN_TILE + 2)));
    BCHECK(cudaMalloc(&total, 4));
    BCHECK(cudaMalloc(&dense, sizeof(uint4) * 4ull * n_inner));
    BCHECK(cudaMalloc(&dense_prov, sizeof(int) * 4ull * n_inner));
    BCHECK(cudaMemcpyAsync(fr[0], &zero, 4, cudaMemcpyHostToDevice, st));
    while (nf) {
        const uint32_t g = (nf + TPB - 1) / TPB;
        uint32_t next = 0;
        k_wide_count<<<g, TPB, 0, st>>>(sparse, fr[pp], nf, cnt); ++*launches;
        fs_scan_u32(st, cnt, off, nf, tile_sums, total, launches);
        k_wide_place<<<g, TPB, 0, st>>>(sparse, dense, sparse_prov, dense_prov, fr[pp], nf, off, base, fr[pp ^ 1]); ++*launches;
        BCHECK(cudaMemcpyAsync(&next, total, 4, cudaMemcpyDeviceToHost, st));
        BCHECK(cudaStreamSynchronize(st));
        base += nf; nf = next; pp ^= 1;
        if (base + nf > n_inner) { err = cudaErrorUnknown; goto fail; }     // cannot happen for a tree
    }
    BCHECK(cudaGetLastError());
    *dense_out = dense; dense = nullptr; *dense_prov_out = dense_prov; dense_prov = nullptr; *n_wide_out = base;
fail:
    cudaFree(fr[0]); cudaFree(fr[1]); cudaFree(cnt); cudaFree(off); cudaFree(tile_sums); cudaFree(total); cudaFree(dense); cudaFree(dense_prov);
    return err;
}

// 8-wide compressed nodes + the triangle array in their order; single-triangle leaves only (PLOC trees)
static cudaError_t w8_build(cudaStream_t st, uint32_t n, uint32_t n_inner, const float4* nodes, const float4* tris,
                            fs_bvh_device* out, uint64_t* launches, bool dp)
{
    cudaError_t err = cudaSuccess;
    float* T = nullptr; int* parent = nullptr; uint32_t *need = nullptr, *arrive = nullptr;
    uint4 *tmp = nullptr, *dense = nullptr, *fit = nullptr;
    int *ref = nullptr, *fr[2] = {nullptr, nullptr};
    uint32_t *cnt_in = nullptr, *cnt_leaf = nullptr, *off_in = nullptr, *off_leaf = nullptr, *tile_sums = nullptr, *total = nullptr;
    float4* tris8 = nullptr; uint32_t* map = nullptr;
    const int TPB = 256;
    uint32_t nf = 1, base = 0, tri_base = 0;
    int pp = 0;
    const int zero = 0;
    BCHECK(cudaMalloc(&tmp, sizeof(uint4) * 5ull * n_inner));
    BCHECK(cudaMalloc(&ref, 4ull * 8 * n_inner));
    BCHECK(cudaMalloc(&dense, sizeof(uint4) * 5ull * n_inner));
    BCHECK(cudaMalloc(&fr[0], 4ull * n_inner)); BCHECK(cudaMalloc(&fr[1], 4ull * n_inner));
    BCHECK(cudaMalloc(&cnt_in, 4ull * n_inner)); BCHECK(cudaMalloc(&cnt_leaf, 4ull * n_inner));
    BCHECK(cudaMalloc(&off_in, 4ull * n_inner)); BCHECK(cudaMalloc(&off_leaf, 4ull * n_inner));
    BCHECK(cudaMalloc(&tile_sums, 4ull * ((n_inner + SCAN_TILE - 1) / SCAN_TILE + 2)));
    BCHECK(cudaMalloc(&total, 8));
    BCHECK(cudaMalloc(&tris8, sizeof(float4) * 4ull * n));
    BCHECK(cudaMalloc(&map, 4ull * n));
    if (dp) {
        BCHECK(cudaMalloc(&T, sizeof(float) * 8ull * n_inner));
        BCHECK(cudaMalloc(&parent, 4ull * n_inner)); BCHECK(cudaMalloc(&need, 4ull * n_inner)); BCHECK(cudaMalloc(&arrive, 4ull * n_inner));
        BCHECK(cudaMemsetAsync(arrive, 0, 4ull * n_inner, st));
        k_w8_parents<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, nodes, parent, need);
        k_wide_dp<8><<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, nodes, parent, need, arrive, T);
        *launches += 2;
    }
    k_emit8<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, nodes, T, tmp, ref); ++*launches;
    BCHECK(cudaMemcpyAsync(fr[0], &zero, 4, cudaMemcpyHostToDevice, st));
    while (nf) {
        const uint32_t g = (nf + TPB - 1) / TPB;
        uint32_t next[2] = {0, 0};
        k_w8_count<<<g, TPB, 0, st>>>(tmp, fr[pp], nf, cnt_in, cnt_leaf); ++*launches;
        fs_scan_u32(st, cnt_in, off_in, nf, tile_sums, total, launches);
        fs_scan_u32(st, cnt_leaf, off_leaf, nf, tile_sums, total + 1, launches);
        k_w8_place<<<g, TPB, 0, st>>>(tmp, ref, dense, fr[pp], nf, off_in, off_leaf, base, tri_base, fr[pp ^ 1], tris, tris8, map);
        ++*launches;
        BCHECK(cudaMemcpyAsync(next, total, 8, cudaMemcpyDeviceToHost, st));
        BCHECK(cudaStreamSynchronize(st));
        base += nf; nf = next[0]; tri_base += next[1]; pp ^= 1;
        if ((uint64_t)base + nf > n_inner || tri_base > n) { err = cudaErrorUnknown; goto fail; }     // cannot happen for a tree
    }
    BCHECK(cudaGetLastError());
    if (tri_base != n) { err = cudaErrorUnknown; goto fail; }
    BCHECK(cudaMalloc(&fit, sizeof(uint4) * 5ull * base));                  // right-sized copy (the bound was one node per BVH2 node)
    BCHECK(cudaMemcpyAsync(fit, dense, sizeof(uint4) * 5ull * base, cudaMemcpyDeviceToDevice, st));
    BCHECK(cudaStreamSynchronize(st));
    out->w8nodes = fit; fit = nullptr; out->n_w8 = base;
    out->tris8 = tris8; tris8 = nullptr; out->tri8_map = map; map = nullptr;
fail:
    cudaFree(T); cudaFree(parent); cudaFree(need); cudaFree(arrive);
    cudaFree(tmp); cudaFree(ref); cudaFree(dense); cudaFree(fit); cudaFree(fr[0]); cudaFree(fr[1]); cudaFree(cnt_in); cudaFree(cnt_leaf);
    cudaFree(off_in); cudaFree(off_leaf); cudaFree(tile_sums); cudaFree(total); cudaFree(tris8); cudaFree(map);
    return err;
}

cudaError_t fs_bvh_build(cudaStream_t st, const float* d_verts, const uint32_t* d_mats, uint64_t T64,
                         fs_bvh_device* out, uint64_t* launches, uint32_t leaf_max_u, uint32_t builder, uint32_t collapse_u)
{
    const int leaf_max = (int)(leaf_max_u < 1 ? 1 : (leaf_max_u > 8 ? 8 : leaf_max_u));
    const int collapse = (int)collapse_u;     // bit 0: greedy surface-area collapse, bit 1: skip the dense relayout
    cudaError_t err = cudaSuccess;
    const uint32_t n = (uint32_t)T64;
    fs_bvh_free(out);
    out->n_tris = n;
    if (n == 0) return cudaSuccess;
    const uint32_t n_inner = n > 1 ? n - 1 : 1;
    const uint32_t n_blocks_sort = fs_radix_sort_blocks(n);
    float4 *tlo = nullptr, *thi = nullptr, *bb_lo = nullptr, *bb_hi = nullptr;
    uint64_t *keys0 = nullptr, *keys1 = nullptr;
    uint32_t *vals0 = nullptr, *vals1 = nullptr, *block_hist = nullptr, *misc = nullptr, *arrive = nullptr;
    float* grid = nullptr;
    int2 *children = nullptr, *ranges = nullptr;
    int *parent = nullptr, *queue = nullptr;
    const int TPB = 256;
    const uint32_t gb = (n + TPB - 1) / TPB;

    BCHECK(cudaMalloc(&tlo, sizeof(float4) * n));
    BCHECK(cudaMalloc(&thi, sizeof(float4) * n));
    BCHECK(cudaMalloc(&bb_lo, sizeof(float4) * (2ull * n)));
    BCHECK(cudaMalloc(&bb_hi, sizeof(float4) * (2ull * n)));
    BCHECK(cudaMalloc(&keys0, 8ull * n));
    BCHECK(cudaMalloc(&keys1, 8ull * n));
    BCHECK(cudaMalloc(&vals0, 4ull * n));
    BCHECK(cudaMalloc(&vals1, 4ull * n));
    BCHECK(cudaMalloc(&block_hist, 4ull * 256 * n_blocks_sort));
    BCHECK(cudaMalloc(&misc, 4 * 16));   // [0..5] centre bounds [6] extent [7] n_top [8] max_leaf [9..14] scene box
    BCHECK(cudaMalloc(&arrive, 4ull * n_inner));
    BCHECK(cudaMalloc(&children, sizeof(int2) * n_inner));
    BCHECK(cudaMalloc(&ranges, sizeof(int2) * n_inner));
    BCHECK(cudaMalloc(&parent, 4ull * 2 * n));
    BCHECK(cudaMalloc(&queue, 4ull * FS_TOP_CAP));
    BCHECK(cudaMalloc(&out->nodes, sizeof(float4) * 4ull * n_inner));
    BCHECK(cudaMalloc(&out->wnodes, sizeof(uint4) * 4ull * n_inner));
    BCHECK(cudaMalloc(&out->wsrc, sizeof(int) * 4ull * n_inner));
    BCHECK(cudaMalloc(&grid, sizeof(float) * 8));
    BCHECK(cudaMalloc(&out->tris, sizeof(float4) * 4ull * n));
    BCHECK(cudaMalloc(&out->tri_orig, 4ull * n));
    BCHECK(cudaMalloc(&out->tri_mat, 4ull * n));
    BCHECK(cudaMalloc(&out->tri_nm, sizeof(float4) * (size_t)n));
    BCHECK(cudaMalloc(&out->top_nodes, sizeof(float4) * 4ull * FS_TOP_CAP));
    out->n_inner = n_inner;

    BCHECK(cudaMemsetAsync(misc, 0, 4 * 16, st));
    BCHECK(cudaMemsetAsync(arrive, 0, 4ull * n_inner, st));
    // misc[0..5] centre bounds, misc[6] extent (ordered), misc[7] n_top, misc[8] max_leaf
    k_init_bounds<<<1, 32, 0, st>>>(misc); ++*launches;
    k_tri_bounds<<<gb, TPB, 0, st>>>(d_verts, n, tlo, thi, misc, misc + 6); ++*launches;
    k_morton<<<gb, TPB, 0, st>>>(tlo, thi, n, misc, keys0, vals0); ++*launches;
    fs_radix_sort_u64(st, keys0, vals0, keys1, vals1, n, block_hist, launches);
    k_pack<<<gb, TPB, 0, st>>>(d_verts, d_mats, vals0, n, tlo, thi, out->tris, out->tri_orig, out->tri_mat, out->tri_nm, bb_lo, bb_hi);
    ++*launches;
    if (n == 1) {
        k_emit_single<<<1, 1, 0, st>>>(bb_lo, bb_hi, out->nodes); ++*launches;
        out->max_leaf = 1;
    } else if (builder == 1 && n >= 3) {
        // PLOC over the Morton-sorted leaves; nodes are emitted as clusters merge
        // The search radius that gives the best tree depends on the scene (hall: 5 beats 24 by 8 % in node visits, mine
        // tunnels: 96 beats 5 by 22 %, room: 10), and the surface-area cost of the BVH2 ranks the candidates the same way
        // as the measured node visits: build the candidates, keep the cheapest (commit time only).
        // FS_TUNE_PLOC_R pins one radius.
        int cand[4] = {5, 10, 24, 64}, n_cand = 4;
        if (const char* e = getenv("FS_TUNE_PLOC_R")) { int v = atoi(e); if (v >= 1 && v <= 256) { cand[0] = v; n_cand = 1; } }
        if (n < 4096) n_cand = 1;                         // tiny scenes: nothing to gain
        double best_cost = 0.0; int best = -1;
        float4* alt = nullptr; double* d_cost = nullptr;
        float* cT4 = nullptr; int* cpar = nullptr; uint32_t *cneed = nullptr, *carr = nullptr;
        if (n_cand > 1) { BCHECK(cudaMalloc(&alt, sizeof(float4) * 4ull * n_inner)); BCHECK(cudaMalloc(&d_cost, 8)); }
        for (int ci = 0; ci < n_cand; ++ci) {
            float4* dst = (n_cand > 1) ? alt : out->nodes;
            BCHECK(ploc_build(st, n, bb_lo, bb_hi, dst, launches, cand[ci]));
            if (n_cand == 1) break;
            double h_cost = 0.0;
            BCHECK(cudaMemsetAsync(d_cost, 0, 8, st));
            k_sah_cost<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, dst, d_cost); ++*launches;
            BCHECK(cudaMemcpyAsync(&h_cost, d_cost, 8, cudaMemcpyDeviceToHost, st));
            BCHECK(cudaStreamSynchronize(st));
            if (getenv("FS_VERBOSE")) fprintf(stderr, "[frequensee] PLOC radius %d: surface-area cost %.6g\n", cand[ci], h_cost);
            if (collapse & 16) {
                // rank the candidates by what the traversal will walk: the summed area of the 4-wide nodes after the optimal
                // collapse (= the root's entry of the dynamic programme's table; the leaf boxes are the same in every tree)
                if (!cT4) {
                    BCHECK(cudaMalloc(&cT4, sizeof(float) * 4ull * n_inner)); BCHECK(cudaMalloc(&cpar, 4ull * n_inner));
                    BCHECK(cudaMalloc(&cneed, 4ull * n_inner)); BCHECK(cudaMalloc(&carr, 4ull * n_inner));
                }
                float root_cost = 0.f;
                BCHECK(cudaMemsetAsync(carr, 0, 4ull * n_inner, st));
                k_w8_parents<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, dst, cpar, cneed);
                k_wide_dp<4><<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, dst, cpar, cneed, carr, cT4);
                *launches += 2;
                BCHECK(cudaMemcpyAsync(&root_cost, cT4, 4, cudaMemcpyDeviceToHost, st));
                BCHECK(cudaStreamSynchronize(st));
                if (getenv("FS_VERBOSE")) fprintf(stderr, "[frequensee] PLOC radius %d: summed area of the 4-wide nodes %.6g\n", cand[ci], (double)root_cost);
                h_cost = (double)root_cost;
            }
            if (best < 0 || h_cost < best_cost) {
                best = ci; best_cost = h_cost;
                BCHECK(cudaMemcpyAsync(out->nodes, alt, sizeof(float4) * 4ull * n_inner, cudaMemcpyDeviceToDevice, st));
            }
        }
        if (alt) { cudaStreamSynchronize(st); cudaFree(alt); cudaFree(d_cost); }
        cudaFree(cT4); cudaFree(cpar); cudaFree(cneed); cudaFree(carr);
        out->max_leaf = 1;
        {
            int sweeps = 0;      // measured: PLOC trees gain 0.3-0.5 % of surface-area cost and < 1 % of node visits; off by default
            if (const char* e = getenv("FS_TUNE_ROTATE")) { int v = atoi(e); if (v >= 0 && v <= 64) sweeps = v; }
            if (sweeps && n >= 4096) {
                uint32_t n_rot = 0;
                BCHECK(bvh2_rotate(st, n_inner, out->nodes, sweeps, launches, &n_rot));
                if (getenv("FS_VERBOSE")) {
                    double* d_c = nullptr; double h_c = 0.0;
                    if (cudaMalloc(&d_c, 8) == cudaSuccess) {
                        cudaMemsetAsync(d_c, 0, 8, st);
                        k_sah_cost<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, out->nodes, d_c);
                        cudaMemcpyAsync(&h_c, d_c, 8, cudaMemcpyDeviceToHost, st); cudaStreamSynchronize(st); cudaFree(d_c);
                    }
                    fprintf(stderr, "[frequensee] %d rotation sweeps: %u rotations, surface-area cost %.6g\n", sweeps, n_rot, h_c);
                }
            }
        }
        {
            // FS_TUNE_REINSERT = most reinsertion iterations (0: off)
            int iters = FS_REINSERT_ITERS;
            if (const char* e = getenv("FS_TUNE_REINSERT")) { int v = atoi(e); if (v >= 0 && v <= 256) iters = v; }
            if (iters && n >= 4096) BCHECK(bvh2_reinsert(st, n_inner, d_verts, out->tri_orig, out->nodes, iters, launches));
        }
    } else {
        k_karras<<<gb, TPB, 0, st>>>(keys0, (int)n, children, ranges, parent); ++*launches;
        k_refit<<<gb, TPB, 0, st>>>((int)n, children, parent, bb_lo, bb_hi, arrive); ++*launches;
        k_emit<<<gb, TPB, 0, st>>>((int)n, children, ranges, bb_lo, bb_hi, out->nodes, leaf_max); ++*launches;
        k_leaf_stats<<<gb, TPB, 0, st>>>((int)n, ranges, misc + 8, leaf_max); ++*launches;
    }
    k_quant_grid<<<1, 32, 0, st>>>(out->nodes, grid); ++*launches;
    if ((collapse & 16) && n >= 3) {
        // optimal collapse (dynamic programme over the BVH2, as for the 8-wide nodes) instead of the greedy one
        float* T4 = nullptr; int* par = nullptr; uint32_t *need = nullptr, *arr = nullptr;
        cudaError_t e4 = cudaSuccess;
        if ((e4 = cudaMalloc(&T4, sizeof(float) * 4ull * n_inner)) == cudaSuccess && (e4 = cudaMalloc(&par, 4ull * n_inner)) == cudaSuccess &&
            (e4 = cudaMalloc(&need, 4ull * n_inner)) == cudaSuccess && (e4 = cudaMalloc(&arr, 4ull * n_inner)) == cudaSuccess &&
            (e4 = cudaMemsetAsync(arr, 0, 4ull * n_inner, st)) == cudaSuccess) {
            k_w8_parents<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, out->nodes, par, need);
            k_wide_dp<4><<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, out->nodes, par, need, arr, T4);
            k_emit4_dp<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, out->nodes, T4, grid, out->wnodes, out->wsrc);
            *launches += 3;
            e4 = cudaStreamSynchronize(st);
        }
        cudaFree(T4); cudaFree(par); cudaFree(need); cudaFree(arr);
        BCHECK(e4);
    } else {
        k_emit4<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, out->nodes, grid, out->wnodes, out->wsrc, collapse & 1); ++*launches;
    }
    out->n_wide = n_inner;
    if (!(collapse & 2)) {                          // FS_TUNE_COLLAPSE bit 1 keeps the sparse layout (A/B)
        uint4* dense = nullptr; int* dense_prov = nullptr; uint32_t n_wide = 0;
        BCHECK(wide_compact(st, n_inner, out->wnodes, out->wsrc, &dense, &dense_prov, &n_wide, launches));
        cudaFree(out->wnodes); out->wnodes = dense; out->n_wide = n_wide;
        cudaFree(out->wsrc); out->wsrc = dense_prov;
    }
    {
        cudaResourceDesc rd; memset(&rd, 0, sizeof(rd));
        rd.resType = cudaResourceTypeLinear;
        rd.res.linear.devPtr = out->nodes;
        rd.res.linear.desc = cudaCreateChannelDesc<float4>();
        rd.res.linear.sizeInBytes = sizeof(float4) * 4ull * n_inner;
        cudaTextureDesc td; memset(&td, 0, sizeof(td));
        td.readMode = cudaReadModeElementType;
        if (cudaCreateTextureObject(&out->nodes_tex, &rd, &td, nullptr) != cudaSuccess) { out->nodes_tex = 0; (void)cudaGetLastError(); }
        rd.res.linear.devPtr = out->tris;
        rd.res.linear.sizeInBytes = sizeof(float4) * 4ull * n;
        if (cudaCreateTextureObject(&out->tris_tex, &rd, &td, nullptr) != cudaSuccess) { out->tris_tex = 0; (void)cudaGetLastError(); }
        rd.res.linear.devPtr = out->wnodes;
        rd.res.linear.desc = cudaCreateChannelDesc<uint4>();
        rd.res.linear.sizeInBytes = sizeof(uint4) * 4ull * out->n_wide;
        if (cudaCreateTextureObject(&out->wnodes_tex, &rd, &td, nullptr) != cudaSuccess) { out->wnodes_tex = 0; (void)cudaGetLastError(); }
    }
    k_top_treelet<<<1, 32, 0, st>>>(out->nodes, n_inner, FS_TOP_CAP, out->top_nodes, misc + 7, queue); ++*launches;
    BCHECK(cudaGetLastError());
    // 8-wide compressed nodes (FS_TUNE_W8=1 -> collapse bit 2): optional traversal format, see profiles/r2_experiments.md
    if (builder == 1 && n >= 3 && out->max_leaf == 1 && (collapse & 4)) BCHECK(w8_build(st, n, n_inner, out->nodes, out->tris, out, launches, !(collapse & 8)));   // bit 3: greedy instead of the optimal collapse
    {
        uint32_t h[16];   // misc[0..15]
        BCHECK(cudaMemcpyAsync(h, misc, sizeof(h), cudaMemcpyDeviceToHost, st));
        BCHECK(cudaStreamSynchronize(st));
        out->n_top = h[7];
        if (n > 1 && !(builder == 1 && n >= 3)) out->max_leaf = h[8] ? h[8] : 1;
        out->extent = ord2f(h[6]);
        float hg[6];
        BCHECK(cudaMemcpy(hg, grid, sizeof(hg), cudaMemcpyDeviceToHost));
        for (int a = 0; a < 3; ++a) { out->qbase[a] = hg[a]; out->qscale[a] = hg[3 + a]; }
    }
fail:
    cudaFree(tlo); cudaFree(thi); cudaFree(bb_lo); cudaFree(bb_hi); cudaFree(keys0); cudaFree(keys1);
    cudaFree(vals0); cudaFree(vals1); cudaFree(block_hist); cudaFree(misc); cudaFree(arrive);
    cudaFree(children); cudaFree(ranges); cudaFree(parent); cudaFree(queue); cudaFree(grid);
    if (err != cudaSuccess) fs_bvh_free(out);
    return err;
}

void fs_bvh_free(fs_bvh_device* b)
{
    if (b->nodes_tex) cudaDestroyTextureObject(b->nodes_tex);
    if (b->tris_tex) cudaDestroyTextureObject(b->tris_tex);
    if (b->wnodes_tex) cudaDestroyTextureObject(b->wnodes_tex);
    cudaFree(b->w8nodes); cudaFree(b->tris8); cudaFree(b->tri8_map);
    cudaFree(b->nodes); cudaFree(b->wnodes); cudaFree(b->tris); cudaFree(b->tri_orig); cudaFree(b->tri_mat); cudaFree(b->tri_nm); cudaFree(b->top_nodes);
    cudaFree(b->wsrc);
    cudaFree(b->rf.parent); cudaFree(b->rf.need); cudaFree(b->rf.arrive); cudaFree(b->rf.ubox); cudaFree(b->rf.queue); cudaFree(b->rf.misc);
    memset(b, 0, sizeof(*b));
}

// Refit of a committed tree (see fs_internal.h).  Stream-ordered on `st`; the one synchronisation is the read-back of the
// quantisation grid and the two costs.  The 8-wide nodes (FS_TUNE_W8) are not refitted: the caller rebuilds them.
cudaError_t fs_bvh_refit(cudaStream_t st, const float* d_verts, fs_bvh_device* b, uint64_t* launches, float* cost_ratio)
{
    cudaError_t err = cudaSuccess;
    const uint32_t n = b->n_tris, n_inner = b->n_inner;
    const int TPB = 256;
    fs_bvh_device::refit_scratch& r = b->rf;
    struct { double cost[2]; float grid[8]; uint32_t n_top; } h;
    if (cost_ratio) *cost_ratio = 1.0f;
    if (n == 0) return cudaSuccess;
    if (!r.misc) {
        // first refit: the topology tables, and the cost of the tree as committed before anything overwrites it
        BCHECK(cudaMalloc(&r.parent, 4ull * n_inner));
        BCHECK(cudaMalloc(&r.need, 4ull * n_inner));
        BCHECK(cudaMalloc(&r.arrive, 4ull * n_inner));
        BCHECK(cudaMalloc(&r.ubox, sizeof(float4) * 2ull * n_inner));
        BCHECK(cudaMalloc(&r.queue, 4ull * FS_TOP_CAP));
        BCHECK(cudaMalloc(&r.misc, sizeof(h)));
        // -1 everywhere first: the inner nodes inside a multi-triangle leaf (LBVH) have no parent; their subtrees are
        // refitted as trees of their own, which keeps the whole node array equal to a fresh build's
        BCHECK(cudaMemsetAsync(r.parent, 0xff, 4ull * n_inner, st));
        BCHECK(cudaMemsetAsync(r.misc, 0, sizeof(h), st));
        k_w8_parents<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, b->nodes, r.parent, r.need);
        k_sah_cost<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, b->nodes, (double*)r.misc);
        *launches += 2;
        BCHECK(cudaMemcpyAsync(&r.cost0, r.misc, sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    BCHECK(cudaMemsetAsync(r.arrive, 0, 4ull * n_inner, st));
    BCHECK(cudaMemsetAsync((double*)r.misc + 1, 0, sizeof(double), st));
    k_refit_tris<<<(n + TPB - 1) / TPB, TPB, 0, st>>>(n, d_verts, b->tri_orig, b->tri_mat, b->tris, b->tri_nm);
    if (n == 1) k_refit_single<<<1, 1, 0, st>>>(d_verts, b->tri_orig, b->nodes);
    else k_refit_nodes<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, d_verts, b->tri_orig, r.parent, r.need, r.arrive, b->nodes, r.ubox);
    k_sah_cost<<<(n_inner + TPB - 1) / TPB, TPB, 0, st>>>(n_inner, b->nodes, (double*)r.misc + 1);
    {
        float* d_grid = (float*)((char*)r.misc + offsetof(decltype(h), grid));
        k_quant_grid<<<1, 32, 0, st>>>(b->nodes, d_grid);
        const uint32_t n_slots = 4u * b->n_wide;
        k_requant4<<<(n_slots + TPB - 1) / TPB, TPB, 0, st>>>(n_slots, b->nodes, b->wsrc, d_grid, b->wnodes);
        k_top_treelet<<<1, 32, 0, st>>>(b->nodes, n_inner, FS_TOP_CAP, b->top_nodes,
                                        (uint32_t*)((char*)r.misc + offsetof(decltype(h), n_top)), r.queue);
    }
    *launches += 6;
    BCHECK(cudaGetLastError());
    BCHECK(cudaMemcpyAsync(&h, r.misc, sizeof(h), cudaMemcpyDeviceToHost, st));
    BCHECK(cudaStreamSynchronize(st));
    for (int a = 0; a < 3; ++a) { b->qbase[a] = h.grid[a]; b->qscale[a] = h.grid[3 + a]; }
    b->n_top = h.n_top;
    if (cost_ratio) *cost_ratio = r.cost0 > 0.0 ? (float)(h.cost[1] / r.cost0) : 1.0f;
fail:
    return err;
}
