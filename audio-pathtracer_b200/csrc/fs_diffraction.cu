// fs_diffraction.cu -- first-order edge diffraction of the direct path (fs_diffraction).
//
// Edge extraction (once per commit, refit or threshold, cached by fs_api.cu):
//   k_diff_keys   one thread per triangle edge e = 3 tri + k: 63-bit hash of its canonical endpoint pair, value e
//   radix sort    the LSD sort of the BVH build (fs_radix_sort_u64), stable: equal hashes stay in ascending e
//   k_diff_group  one thread per sorted entry: the first entry of a group of equal endpoints (exact compare, which also
//                 separates hash collisions) is its lowest (tri, k); it classifies the group (1, 2, >= 3 triangles),
//                 applies the fold test and marks keep[e]
//   scan          keep -> output slots (fs_scan_u32), so the edges come out in ascending (tri, k)
//   k_diff_emit   one thread per kept e: its 64-byte fs_diff_edge record
// Query:
//   k_diff_cand   edge-major: each thread holds one edge and tests it against the sources staged in shared memory;
//                 surviving (source, edge) pairs are appended with one atomic per warp and source
//   k_diff_legs   one thread per candidate: the two legs through fs_any_hit, then atomicMin on (bits(length) << 32 | edge
//                 rank) and a path count per source
//   k_diff_final  one thread per source: the winner re-evaluated through fs_diffraction.h into fs_diffraction_result
#include <algorithm>

#include "fs_internal.h"
#include "fs_diffraction.h"

#define DIFF_TPB 256

__global__ void __launch_bounds__(DIFF_TPB) k_diff_keys(const float* __restrict__ verts, uint32_t n_edges, uint64_t* __restrict__ keys,
                                                        uint32_t* __restrict__ vals, uint32_t* __restrict__ keep)
{
    const uint32_t e = blockIdx.x * DIFF_TPB + threadIdx.x;
    if (e >= n_edges) return;
    const float* v = verts + (size_t)(e / 3u) * 9u;
    float a[3], b[3];
    const bool ok = !fs_diff_degenerate(v) && fs_diff_endpoints(v, e % 3u, a, b);
    keys[e] = ok ? fs_diff_hash(a, b) : FS_DIFF_NO_KEY;
    vals[e] = e;
    keep[e] = 0u;
}

// part[e]: the second triangle edge of a wedge, or 0xffffffff for a screen (read by k_diff_emit for kept e only)
__global__ void __launch_bounds__(DIFF_TPB) k_diff_group(const float* __restrict__ verts, const uint64_t* __restrict__ keys,
                                                         const uint32_t* __restrict__ vals, uint32_t n, float c_min,
                                                         uint32_t* __restrict__ keep, uint32_t* __restrict__ part)
{
    const uint32_t i = blockIdx.x * DIFF_TPB + threadIdx.x;
    if (i >= n) return;
    const uint64_t key = keys[i];
    if (key == FS_DIFF_NO_KEY) return;
    const uint32_t e = vals[i];
    const float* v = verts + (size_t)(e / 3u) * 9u;
    float a[3], b[3], c[3], d[3];
    fs_diff_endpoints(v, e % 3u, a, b);
    uint32_t r0 = i;
    while (r0 > 0u && keys[r0 - 1u] == key) --r0;
    for (uint32_t j = r0; j < i; ++j) {                      // an earlier entry with the same endpoints names the group
        const uint32_t f = vals[j];
        fs_diff_endpoints(verts + (size_t)(f / 3u) * 9u, f % 3u, c, d);
        if (fs_diff_same(a, b, c, d)) return;
    }
    uint32_t count = 1u, other = 0xffffffffu;
    for (uint32_t j = i + 1u; j < n && keys[j] == key && count < 3u; ++j) {
        const uint32_t f = vals[j];
        fs_diff_endpoints(verts + (size_t)(f / 3u) * 9u, f % 3u, c, d);
        if (fs_diff_same(a, b, c, d)) { if (count == 1u) other = f; ++count; }
    }
    if (count >= 3u) return;                                 // non-manifold: never diffracts
    if (count == 2u && !fs_diff_fold_ok(a, b, v, e % 3u, verts + (size_t)(other / 3u) * 9u, other % 3u, c_min)) return;
    keep[e] = 1u;
    part[e] = other;
}

__global__ void __launch_bounds__(DIFF_TPB) k_diff_emit(const float* __restrict__ verts, uint32_t n_edges, const uint32_t* __restrict__ keep,
                                                        const uint32_t* __restrict__ part, const uint32_t* __restrict__ slot,
                                                        fs_diff_edge* __restrict__ out)
{
    const uint32_t e = blockIdx.x * DIFF_TPB + threadIdx.x;
    if (e >= n_edges || !keep[e]) return;
    const float* v = verts + (size_t)(e / 3u) * 9u;
    float a[3], b[3];
    fs_diff_endpoints(v, e % 3u, a, b);
    const uint32_t f = part[e];
    fs_diff_edge r;
    fs_diff_make_edge(a, b, v, e / 3u, e % 3u, f == 0xffffffffu ? nullptr : verts + (size_t)(f / 3u) * 9u, f % 3u, &r);
    out[slot[e]] = r;
}

cudaError_t fs_diffraction_edges(cudaStream_t st, const float* d_verts, uint32_t n_tris, float c_min, fs_diff_edge** d_edges,
                                 uint32_t* n_out, uint64_t* launches)
{
    *n_out = 0;
    const uint32_t n = 3u * n_tris;
    if (!n) return cudaSuccess;
    const uint32_t tiles = (n + 1023u) / 1024u;
    uint64_t *keys = nullptr, *keys_tmp = nullptr;
    uint32_t *vals = nullptr, *vals_tmp = nullptr, *keep = nullptr, *part = nullptr, *slot = nullptr, *hist = nullptr,
             *tile_sums = nullptr, *total = nullptr;
    uint32_t h_total = 0;
    cudaError_t err = cudaSuccess;
    const uint32_t g = (n + DIFF_TPB - 1u) / DIFF_TPB;
#define DCHECK(x) do { if ((err = (x)) != cudaSuccess) goto done; } while (0)
    DCHECK(cudaMalloc(&keys, 8ull * n));
    DCHECK(cudaMalloc(&keys_tmp, 8ull * n));
    DCHECK(cudaMalloc(&vals, 4ull * n));
    DCHECK(cudaMalloc(&vals_tmp, 4ull * n));
    DCHECK(cudaMalloc(&keep, 4ull * n));
    DCHECK(cudaMalloc(&part, 4ull * n));
    DCHECK(cudaMalloc(&slot, 4ull * n));
    DCHECK(cudaMalloc(&hist, 4ull * 256u * fs_radix_sort_blocks(n)));
    DCHECK(cudaMalloc(&tile_sums, 4ull * (tiles + 2u)));
    DCHECK(cudaMalloc(&total, 4));
    k_diff_keys<<<g, DIFF_TPB, 0, st>>>(d_verts, n, keys, vals, keep);
    ++*launches;
    fs_radix_sort_u64(st, keys, vals, keys_tmp, vals_tmp, n, hist, launches);
    k_diff_group<<<g, DIFF_TPB, 0, st>>>(d_verts, keys, vals, n, c_min, keep, part);
    ++*launches;
    fs_scan_u32(st, keep, slot, n, tile_sums, total, launches);
    DCHECK(cudaGetLastError());
    DCHECK(cudaMemcpyAsync(&h_total, total, 4, cudaMemcpyDeviceToHost, st));
    DCHECK(cudaStreamSynchronize(st));
    if (h_total) {
        DCHECK(cudaMalloc(d_edges, sizeof(fs_diff_edge) * (size_t)h_total));
        k_diff_emit<<<g, DIFF_TPB, 0, st>>>(d_verts, n, keep, part, slot, *d_edges);
        ++*launches;
        DCHECK(cudaGetLastError());
        DCHECK(cudaStreamSynchronize(st));
    }
    *n_out = h_total;
#undef DCHECK
done:
    cudaFree(keys); cudaFree(keys_tmp); cudaFree(vals); cudaFree(vals_tmp); cudaFree(keep); cudaFree(part); cudaFree(slot);
    cudaFree(hist); cudaFree(tile_sums); cudaFree(total);
    return err;
}

// (source, edge) pairs that pass the geometric tests, appended to cand[0 .. cap); *count counts every pair, also those
// beyond cap (the caller then grows the buffer and repeats the edge range)
__global__ void __launch_bounds__(DIFF_TPB) k_diff_cand(const fs_diff_edge* __restrict__ edges, uint32_t e0, uint32_t e1,
                                                        const float4* __restrict__ src, uint32_t n_src, float lx, float ly, float lz,
                                                        float eps_offset, uint2* __restrict__ cand, unsigned long long cap,
                                                        unsigned long long* __restrict__ count)
{
    __shared__ float4 ss[DIFF_TPB];
    const uint32_t e = e0 + blockIdx.x * DIFF_TPB + threadIdx.x;
    const bool live = e < e1;
    fs_diff_edge E;
    if (live) E = edges[e];
    const float l[3] = {lx, ly, lz};
    const uint32_t lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
    for (uint32_t s0 = 0; s0 < n_src; s0 += DIFF_TPB) {
        const uint32_t m = min(n_src - s0, (uint32_t)DIFF_TPB);
        __syncthreads();
        if (threadIdx.x < m) ss[threadIdx.x] = src[s0 + threadIdx.x];
        __syncthreads();
        for (uint32_t j = 0; j < m; ++j) {
            const float4 q = ss[j];
            const float s[3] = {q.x, q.y, q.z};
            float p[3];
            const bool pass = live && fs_diff_apex(&E, s, l, eps_offset, p);
            const uint32_t mask = __ballot_sync(0xffffffffu, pass);
            if (!mask) continue;
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(count, (unsigned long long)__popc(mask));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (pass) {
                const unsigned long long idx = base + __popc(mask & lt);
                if (idx < cap) cand[idx] = make_uint2(s0 + j, e);
            }
        }
    }
}

__global__ void __launch_bounds__(DIFF_TPB) k_diff_legs(fs_bvh_view bv, const fs_diff_edge* __restrict__ edges,
                                                        const uint2* __restrict__ cand, uint32_t n_cand, const float4* __restrict__ src,
                                                        float lx, float ly, float lz, float eps_offset, float eps_connect,
                                                        unsigned long long* __restrict__ best, uint32_t* __restrict__ n_paths,
                                                        unsigned long long* __restrict__ rays, uint32_t* overflow)
{
    const uint32_t i = blockIdx.x * DIFF_TPB + threadIdx.x;
    uint32_t traced = 0;
    if (i < n_cand) {
        const uint2 c = cand[i];
        const fs_diff_edge E = edges[c.y];
        const float4 q = __ldg(src + c.x);
        const float s[3] = {q.x, q.y, q.z}, l[3] = {lx, ly, lz};
        float p[3], ds[3], dl[3], ts, tl;
        fs_diff_apex(&E, s, l, eps_offset, p);
        const float ls = fs_diff_leg(s, p, eps_connect, ds, &ts);
        const float ll = fs_diff_leg(l, p, eps_connect, dl, &tl);
        bool clear = true;
        if (ts > 0.0f) {
            ++traced;
            clear = !fs_any_hit<false, false>(bv, nullptr, fs_mk(s[0], s[1], s[2]), fs_mk(ds[0], ds[1], ds[2]), ts, nullptr, overflow);
        }
        if (clear && tl > 0.0f) {
            ++traced;
            clear = !fs_any_hit<false, false>(bv, nullptr, fs_mk(l[0], l[1], l[2]), fs_mk(dl[0], dl[1], dl[2]), tl, nullptr, overflow);
        }
        if (clear) {
            const float length = ls + ll;
            atomicMin(best + c.x, ((unsigned long long)__float_as_uint(length) << 32) | c.y);
            atomicAdd(n_paths + c.x, 1u);
        }
    }
    for (int o = 16; o; o >>= 1) traced += __shfl_xor_sync(0xffffffffu, traced, o);
    if ((threadIdx.x & 31u) == 0 && traced) atomicAdd(rays, (unsigned long long)traced);
}

struct fs_diff_bands { float hz[FS_MAX_BANDS]; };

__global__ void k_diff_final(const fs_diff_edge* __restrict__ edges, const float4* __restrict__ src, uint32_t n_src, float lx, float ly,
                             float lz, float eps_offset, float eps_connect, float sound_speed, fs_diff_bands bands, uint32_t n_bands,
                             const unsigned long long* __restrict__ best, const uint32_t* __restrict__ n_paths,
                             fs_diffraction_result* __restrict__ out)
{
    const uint32_t s_i = blockIdx.x * blockDim.x + threadIdx.x;
    if (s_i >= n_src) return;
    fs_diffraction_result r;
    memset(&r, 0, sizeof(r));
    const unsigned long long w = best[s_i];
    if (w != ~0ull) {
        const fs_diff_edge E = edges[(uint32_t)w];
        const float4 q = src[s_i];
        const float s[3] = {q.x, q.y, q.z}, l[3] = {lx, ly, lz};
        float p[3], d[3], t;
        fs_diff_apex(&E, s, l, eps_offset, p);
        const float length = fs_diff_leg(s, p, eps_connect, d, &t) + fs_diff_leg(l, p, eps_connect, d, &t);
        const float z = fs_diff_z(s, l, length);
        r.found = 1u;
        r.n_paths = n_paths[s_i];
        r.edge_tri = E.tri;
        r.edge_k = E.k & 3u;
        r.apex[0] = p[0]; r.apex[1] = p[1]; r.apex[2] = p[2];
        r.length = length;
        r.path_difference = z;
        for (uint32_t b = 0; b < n_bands; ++b) r.gain[b] = fs_diff_gain(z, bands.hz[b], sound_speed);
    }
    out[s_i] = r;
}

cudaError_t fs_diffraction_run(const fs_diff_run& a, cudaStream_t st, uint64_t* launches, uint64_t* n_cand_out)
{
    cudaError_t err;
    uint64_t total = 0;
    uint32_t e0 = 0;
    uint32_t step = a.n_edges;
    while (e0 < a.n_edges) {
        const uint32_t e1 = (uint32_t)std::min<uint64_t>((uint64_t)e0 + step, a.n_edges);
        if ((err = cudaMemsetAsync(a.d_count, 0, 8, st)) != cudaSuccess) return err;
        k_diff_cand<<<(e1 - e0 + DIFF_TPB - 1u) / DIFF_TPB, DIFF_TPB, 0, st>>>(a.edges, e0, e1, a.src, a.n_src, a.lis[0], a.lis[1],
                                                                             a.lis[2], a.eps_offset, *a.cand, *a.cand_cap, a.d_count);
        ++*launches;
        unsigned long long n = 0;
        if ((err = cudaMemcpyAsync(&n, a.d_count, 8, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return err;
        if ((err = cudaStreamSynchronize(st)) != cudaSuccess) return err;
        if (n > *a.cand_cap) {
            // grow up to FS_DIFF_CAND_MAX pairs and repeat the range; beyond that, halve the range
            if (n <= FS_DIFF_CAND_MAX) {
                cudaFree(*a.cand); *a.cand = nullptr; *a.cand_cap = 0;
                if ((err = cudaMalloc(a.cand, sizeof(uint2) * n)) != cudaSuccess) return err;
                *a.cand_cap = n;
            } else {
                step = std::max<uint32_t>((e1 - e0) / 2u, 1u);
                if (e1 - e0 == 1u) return cudaErrorMemoryAllocation;    // one edge cannot exceed 4096 pairs
            }
            continue;
        }
        if (n) {
            k_diff_legs<<<(uint32_t)((n + DIFF_TPB - 1u) / DIFF_TPB), DIFF_TPB, 0, st>>>(a.bv, a.edges, *a.cand, (uint32_t)n, a.src,
                                                                                      a.lis[0], a.lis[1], a.lis[2], a.eps_offset,
                                                                                      a.eps_connect, a.best, a.n_paths, a.rays,
                                                                                      a.overflow);
            ++*launches;
        }
        total += n;
        e0 = e1;
    }
    fs_diff_bands bands;
    for (int b = 0; b < FS_MAX_BANDS; ++b) bands.hz[b] = a.band_hz[b];
    k_diff_final<<<(a.n_src + 127u) / 128u, 128, 0, st>>>(a.edges, a.src, a.n_src, a.lis[0], a.lis[1], a.lis[2], a.eps_offset,
                                                         a.eps_connect, a.sound_speed, bands, a.n_bands, a.best, a.n_paths, a.out);
    ++*launches;
    if (n_cand_out) *n_cand_out = total;
    return cudaGetLastError();
}
