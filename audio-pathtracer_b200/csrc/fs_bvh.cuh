// fs_bvh.cuh -- device BVH layout and stack-based traversal (closest hit / any hit).
//
// Layout in HBM (all 16-byte aligned, fetched as float4 through the read-only path):
//   nodes : float4[n_inner][4]   64 B per BVH2 inner node, holding BOTH children's boxes:
//             n0 = (c0.lo.x, c0.hi.x, c0.lo.y, c0.hi.y)
//             n1 = (c1.lo.x, c1.hi.x, c1.lo.y, c1.hi.y)
//             n2 = (c0.lo.z, c0.hi.z, c1.lo.z, c1.hi.z)
//             n3 = (child0, child1, -, -) as int bits.  child >= 0: inner node index;
//                  child < 0: leaf, payload = ~child = (first_tri << 3) | (count - 1)
//   tris  : float4[T][4]         64 B per triangle in leaf (Morton) order, fetched as two 256-bit
//             loads: (v0.xyz, n.x) (e1.xyz, n.y) | (e2.xyz, n.z) (bits(orig id), bits(material), -, -)
//             n = unit geometric normal; orig id = tie-break key (closest hit = min (t, orig id))
//   tri_orig : uint32[T]  original triangle id (copy, for the debug entry points)
//   tri_mat  : uint32[T]  material id (copy)
// Fetches are 128-bit ld.global.nc.  ncu shows the traversal bound by the L1TEX LSU data pipe
// (l1tex__data_pipe_lsu_wavefronts ~ 88 %): a divergent warp load costs one wavefront per lane,
// whatever its width -- 256-bit loads (LDG.E.ENL2.256) were measured and are not cheaper.
// A 32 B node format (16-bit quantised boxes, octant plane selection by PRMT) halves those
// wavefronts (48 %) but was measured no faster: the kernel then waits on load latency with the
// ALU pipe as the busiest unit (profiles/r1_experiments.md); it is not kept in the tree.
//   wnodes : uint4[n_wide][4]    64 B per 4-WIDE node (production traversal format).  A wide node is a BVH2
//             node with up to two of its descendants opened (greedy by surface area), so a ray takes about
//             half as many dependent steps; only the nodes reachable from the root are kept, in a dense
//             breadth-first array (children of a node adjacent).  Boxes are quantised to 16 bits per coordinate
//             on a scene-wide grid, rounded outward plus one spare quantum:
//               u_k = (lo.x | hi.x << 16, lo.y | hi.y << 16, lo.z | hi.z << 16, child_k), k = 0..3
//             empty slot: inverted box (lo = 65535, hi = 0).  Dequantisation is folded into the slab FMA:
//             t = fma(2^23 + q, s, b'), s = qscale * idir, b' = (qbase - o) * idir - 2^23 s (one PRMT per
//             plane, chosen by the ray octant so there is no per-axis min/max).
//   w8nodes : uint4[n_w8][5]     80 B per 8-WIDE compressed node (production traversal format, after Ylitie, Karras,
//             Laine 2017).  Child boxes are quantised to 8 bits on a grid local to the node: origin p (the node's low
//             corner, float3), one power-of-two quantum per axis, outward rounding.
//               u0 = (p.x, p.y, p.z, 2^ex as float bits | imask | lmask << 8)   (masks in the mantissa bits)
//               u1 = (2^ey, 2^ez, child_base, tri_base)
//               u2 = (lo.x[0..3], lo.x[4..7], lo.y[0..3], lo.y[4..7])           one byte per child slot
//               u3 = (lo.z[0..3], lo.z[4..7], hi.x[0..3], hi.x[4..7])
//               u4 = (hi.y[0..3], hi.y[4..7], hi.z[0..3], hi.z[4..7])
//             imask / lmask: slots holding an inner node / a leaf (one triangle); empty slot: inverted box (lo 255, hi 0).
//             Inner child in slot s = node child_base + popc(imask below s); leaf child = triangle tri_base + popc(lmask
//             below s) of tris8 (the triangle records in W8 order; tri8_map gives the index into tris / tri_nm that hit
//             records carry).  Children sit in the slots by direction from the node centre, so visiting the hit slots in
//             the order of (slot XOR ray octant), highest first, is near-to-far without a sort.  Slab test:
//             t = fma(2^15 + q, A, B), A = 2^e / d, B = (p - o) / d - 2^15 A; the byte goes into bits 8..15 of a float
//             with exponent 2^15 by one PRMT, so the cancellation error is 2^-9 of a quantum (no spare quantum needed).
// Boxes are padded at build time so that the slab test (FMA form, not bit-reproducible against
// the oracle and not required to be) is conservative: any triangle whose exact-arithmetic
// fs_intersect_tri() succeeds is reached.  The hit itself comes from fs_intersect_tri() only.
#pragma once

#include "fs_math.cuh"

#define FS_STACK_SIZE 64
#define FS_LEAF_MAX 4
#define FS_TOP_FLAG 0x40000000     // node index refers to the shared-memory treelet copy

// Optional bring-up guard: bounds the number of inner-node visits per ray so that a malformed
// tree can never hang the GPU (sets the overflow flag instead).  Off in release builds.
#if defined(FS_TRAVERSAL_GUARD)
#define FS_GUARD_DECL uint32_t guard_ = 0;
#define FS_GUARD_STEP if (++guard_ > 4000000u) { *overflow = 2u; node = SENTINEL; sp = 0; break; }
#else
#define FS_GUARD_DECL
#define FS_GUARD_STEP
#endif

struct fs_bvh_view {
    unsigned long long nodes_tex;   // cudaTextureObject_t over `nodes` (float4 texels), 0 if absent
    unsigned long long tris_tex;    // same over `tris`
    unsigned long long wnodes_tex;  // cudaTextureObject_t over `wnodes` (uint4 texels)
    const uint4* wnodes;            // 4-wide quantised nodes (below), indexed like `nodes`
    const uint4* w8nodes;           // 8-wide compressed nodes, 5 x uint4 each; null = not built / switched off
    const float4* tris8;            // triangle records in W8 order
    const uint32_t* tri8_map;       // W8 triangle position -> index into tris / tri_nm
    uint32_t w8_magic;              // 0x47000000 (2^15 as float bits), kept out of the compiler's sight as a kernel parameter: a literal
                                    // takes PRMT's only immediate slot and pushes the byte selector into a register (+1 MOV per plane)
    float qbase[3], qscale[3];      // world = qbase + q * qscale, q in [0, 65535]
    const float4* nodes;
    const float4* tris;
    const uint32_t* tri_orig;
    const uint32_t* tri_mat;
    const float4* tri_nm;           // [T] (unit normal.xyz, bits(material)) in leaf order: one 16 B fetch per hit when shading
    uint32_t n_tris;
    uint32_t n_inner;
};

struct fs_visit_counters { uint32_t nodes, tris; };

#if defined(__CUDACC__)

__device__ __forceinline__ float4 fs_ldg4(const float4* p)
{
    float4 r;
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

// 256-bit read-only load (LDG.E.256 on sm_100a); p must be 32-byte aligned
__device__ __forceinline__ void fs_ldg8(const float4* p, float4& a, float4& b)
{
    asm volatile("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p));
}

struct fs_ray_prep {
    fs_vec3 o, d;
    float idx, idy, idz, oodx, oody, oodz;
};

__device__ __forceinline__ fs_ray_prep fs_prep_ray(fs_vec3 o, fs_vec3 d)
{
    fs_ray_prep r;
    r.o = o; r.d = d;
    float dx = (fabsf(d.x) > 1e-30f) ? d.x : ((d.x < 0.0f) ? -1e-30f : 1e-30f);
    float dy = (fabsf(d.y) > 1e-30f) ? d.y : ((d.y < 0.0f) ? -1e-30f : 1e-30f);
    float dz = (fabsf(d.z) > 1e-30f) ? d.z : ((d.z < 0.0f) ? -1e-30f : 1e-30f);
    r.idx = 1.0f / dx; r.idy = 1.0f / dy; r.idz = 1.0f / dz;
    r.oodx = o.x * r.idx; r.oody = o.y * r.idy; r.oodz = o.z * r.idz;
    return r;
}

// Both children of one node against the ray interval [0, tmax].
__device__ __forceinline__ void fs_slab2(const fs_ray_prep& r, float4 n0, float4 n1, float4 n2,
                                         float tmax, bool& h0, bool& h1, float& t0n, float& t1n)
{
    float c0lox = fmaf(n0.x, r.idx, -r.oodx), c0hix = fmaf(n0.y, r.idx, -r.oodx);
    float c0loy = fmaf(n0.z, r.idy, -r.oody), c0hiy = fmaf(n0.w, r.idy, -r.oody);
    float c0loz = fmaf(n2.x, r.idz, -r.oodz), c0hiz = fmaf(n2.y, r.idz, -r.oodz);
    float c1lox = fmaf(n1.x, r.idx, -r.oodx), c1hix = fmaf(n1.y, r.idx, -r.oodx);
    float c1loy = fmaf(n1.z, r.idy, -r.oody), c1hiy = fmaf(n1.w, r.idy, -r.oody);
    float c1loz = fmaf(n2.z, r.idz, -r.oodz), c1hiz = fmaf(n2.w, r.idz, -r.oodz);
    float c0min = fmaxf(fmaxf(fminf(c0lox, c0hix), fminf(c0loy, c0hiy)), fmaxf(fminf(c0loz, c0hiz), 0.0f));
    float c0max = fminf(fminf(fmaxf(c0lox, c0hix), fmaxf(c0loy, c0hiy)), fminf(fmaxf(c0loz, c0hiz), tmax));
    float c1min = fmaxf(fmaxf(fminf(c1lox, c1hix), fminf(c1loy, c1hiy)), fmaxf(fminf(c1loz, c1hiz), 0.0f));
    float c1max = fminf(fminf(fmaxf(c1lox, c1hix), fmaxf(c1loy, c1hiy)), fminf(fmaxf(c1loz, c1hiz), tmax));
    h0 = c0min <= c0max;
    h1 = c1min <= c1max;
    t0n = c0min; t1n = c1min;
}

// Closest hit.  Returns sorted triangle index (>= 0) or -1; best_t receives t.
// `top`/`n_top`: optional shared-memory copy of the top treelet (node indices with FS_TOP_FLAG).
template <bool COUNT, bool USE_TOP>
__device__ __forceinline__ int fs_closest_hit(const fs_bvh_view& bv, const float4* __restrict__ top,
                                              fs_vec3 o, fs_vec3 d, float& best_t,
                                              fs_visit_counters* cnt, uint32_t* overflow)
{
    int best = -1;
    uint32_t best_orig = 0xffffffffu;
    float bt = __int_as_float(0x7f800000);
    if (bv.n_tris == 0) { best_t = bt; return -1; }
    const fs_ray_prep r = fs_prep_ray(o, d);
    int stack[FS_STACK_SIZE];
    int sp = 0;
    const int SENTINEL = 0x7fffffff;
    int node = USE_TOP ? FS_TOP_FLAG : 0;
    FS_GUARD_DECL
    while (node != SENTINEL) {
        while (node >= 0 && node != SENTINEL) {
            FS_GUARD_STEP
            float4 n0, n1, n2, n3;
            if (USE_TOP && (node & FS_TOP_FLAG)) {
                const float4* p = top + (size_t)(node & ~FS_TOP_FLAG) * 4;
                n0 = p[0]; n1 = p[1]; n2 = p[2]; n3 = p[3];
            } else {
                const float4* p = bv.nodes + (size_t)node * 4;
                n0 = fs_ldg4(p); n1 = fs_ldg4(p + 1); n2 = fs_ldg4(p + 2); n3 = fs_ldg4(p + 3);
            }
            if (COUNT) cnt->nodes++;
            bool h0, h1; float t0, t1;
            fs_slab2(r, n0, n1, n2, bt, h0, h1, t0, t1);
            int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
            if (!h0 && !h1) {
                node = sp ? stack[--sp] : SENTINEL;
            } else {
                node = h0 ? c0 : c1;
                if (h0 && h1) {
                    int far_ = c1;
                    if (t1 < t0) { far_ = c0; node = c1; }
                    if (sp < FS_STACK_SIZE) stack[sp++] = far_; else *overflow = 1u;
                }
            }
        }
        while (node < 0) {
            uint32_t payload = (uint32_t)(~node);
            uint32_t first = payload >> 3, count = (payload & 7u) + 1u;
            for (uint32_t i = 0; i < count; ++i) {
                const float4* tp = bv.tris + (size_t)(first + i) * 4;
                const float4 a = fs_ldg4(tp), b = fs_ldg4(tp + 1), c = fs_ldg4(tp + 2);
                if (COUNT) cnt->tris++;
                float t;
                if (fs_intersect_tri(o, d, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z), fs_mk(c.x, c.y, c.z), t) && t <= bt) {
                    // tie: lower ORIGINAL id wins (acceleration-structure independent)
                    const uint32_t oi = __float_as_uint(fs_ldg4(tp + 3).x);
                    if (t < bt || (t == bt && oi < best_orig)) { bt = t; best = (int)(first + i); best_orig = oi; }
                }
            }
            node = sp ? stack[--sp] : SENTINEL;
        }
    }
    best_t = bt;
    return best;
}

// Any hit with 0 < t < tmax.
template <bool COUNT, bool USE_TOP>
__device__ __forceinline__ bool fs_any_hit(const fs_bvh_view& bv, const float4* __restrict__ top,
                                           fs_vec3 o, fs_vec3 d, float tmax,
                                           fs_visit_counters* cnt, uint32_t* overflow)
{
    if (bv.n_tris == 0) return false;
    const fs_ray_prep r = fs_prep_ray(o, d);
    int stack[FS_STACK_SIZE];
    int sp = 0;
    const int SENTINEL = 0x7fffffff;
    int node = USE_TOP ? FS_TOP_FLAG : 0;
    FS_GUARD_DECL
    while (node != SENTINEL) {
        while (node >= 0 && node != SENTINEL) {
            FS_GUARD_STEP
            float4 n0, n1, n2, n3;
            if (USE_TOP && (node & FS_TOP_FLAG)) {
                const float4* p = top + (size_t)(node & ~FS_TOP_FLAG) * 4;
                n0 = p[0]; n1 = p[1]; n2 = p[2]; n3 = p[3];
            } else {
                const float4* p = bv.nodes + (size_t)node * 4;
                n0 = fs_ldg4(p); n1 = fs_ldg4(p + 1); n2 = fs_ldg4(p + 2); n3 = fs_ldg4(p + 3);
            }
            if (COUNT) cnt->nodes++;
            bool h0, h1; float t0, t1;
            fs_slab2(r, n0, n1, n2, tmax, h0, h1, t0, t1);
            int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
            if (!h0 && !h1) {
                node = sp ? stack[--sp] : SENTINEL;
            } else {
                node = h0 ? c0 : c1;
                if (h0 && h1) {
                    if (sp < FS_STACK_SIZE) stack[sp++] = c1; else *overflow = 1u;
                }
            }
        }
        while (node < 0) {
            uint32_t payload = (uint32_t)(~node);
            uint32_t first = payload >> 3, count = (payload & 7u) + 1u;
            for (uint32_t i = 0; i < count; ++i) {
                const float4* tp = bv.tris + (size_t)(first + i) * 4;
                const float4 a = fs_ldg4(tp), b = fs_ldg4(tp + 1), c = fs_ldg4(tp + 2);
                if (COUNT) cnt->tris++;
                float t;
                if (fs_intersect_tri(o, d, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z), fs_mk(c.x, c.y, c.z), t)
                    && t < tmax)
                    return true;
            }
            node = sp ? stack[--sp] : SENTINEL;
        }
    }
    return false;
}

// Every hit with 0 < t < tmax (fs_occlusion): the walk of fs_any_hit without the early exit, over the BVH2 `nodes`, which
// every node format keeps and whose leaves address `tris` (the 8-wide format copies the records into tris8).
// on_hit(t, original id, material) is called once per hit in traversal order; the walk stops when it returns false.
template <class F>
__device__ __forceinline__ void fs_all_hits(const fs_bvh_view& bv, fs_vec3 o, fs_vec3 d, float tmax, F&& on_hit,
                                            uint32_t* overflow)
{
    if (bv.n_tris == 0) return;
    const fs_ray_prep r = fs_prep_ray(o, d);
    int stack[FS_STACK_SIZE];
    int sp = 0;
    const int SENTINEL = 0x7fffffff;
    int node = 0;
    FS_GUARD_DECL
    while (node != SENTINEL) {
        while (node >= 0 && node != SENTINEL) {
            FS_GUARD_STEP
            const float4* p = bv.nodes + (size_t)node * 4;
            const float4 n0 = fs_ldg4(p), n1 = fs_ldg4(p + 1), n2 = fs_ldg4(p + 2), n3 = fs_ldg4(p + 3);
            bool h0, h1; float t0, t1;
            fs_slab2(r, n0, n1, n2, tmax, h0, h1, t0, t1);
            int c0 = __float_as_int(n3.x), c1 = __float_as_int(n3.y);
            if (!h0 && !h1) {
                node = sp ? stack[--sp] : SENTINEL;
            } else {
                node = h0 ? c0 : c1;
                if (h0 && h1) {
                    if (sp < FS_STACK_SIZE) stack[sp++] = c1; else *overflow = 1u;
                }
            }
        }
        while (node < 0) {
            uint32_t payload = (uint32_t)(~node);
            uint32_t first = payload >> 3, count = (payload & 7u) + 1u;
            for (uint32_t i = 0; i < count; ++i) {
                const float4* tp = bv.tris + (size_t)(first + i) * 4;
                const float4 a = fs_ldg4(tp), b = fs_ldg4(tp + 1), c = fs_ldg4(tp + 2);
                float t;
                if (fs_intersect_tri(o, d, fs_mk(a.x, a.y, a.z), fs_mk(b.x, b.y, b.z), fs_mk(c.x, c.y, c.z), t) && t < tmax) {
                    const float4 e = fs_ldg4(tp + 3);
                    if (!on_hit(t, __float_as_uint(e.x), __float_as_uint(e.y))) return;
                }
            }
            node = sp ? stack[--sp] : SENTINEL;
        }
    }
}

#endif  // __CUDACC__
