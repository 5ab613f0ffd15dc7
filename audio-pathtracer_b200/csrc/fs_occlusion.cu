// fs_occlusion.cu -- direct-path occlusion and transmission (fs_occlusion): one thread per (source, sample ray), every
// surface the ray crosses on its way to the listener, per-band transmitted gains summed exactly in Q32.32.
#include "fs_internal.h"
#include "fs_occlusion.h"

#define OCC_TPB 256

// source of flat ray index i: the last s with off[s] <= i (off strictly increasing, off[0] = 0)
__device__ __forceinline__ uint32_t occl_source(const uint32_t* __restrict__ off, uint32_t n_src, uint32_t i)
{
    uint32_t lo = 0, hi = n_src - 1u;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1u) >> 1;
        if (__ldg(off + mid) <= i) lo = mid; else hi = mid - 1u;
    }
    return lo;
}

// acc [S][B+1]: per band the sum of trunc(gain 2^32), slot B the visible rays.  The rays of a source are contiguous, so a CTA
// sums into shared memory first (it spans at most OCC_TPB sources) and adds each non-zero (source, slot) to global memory once.
__global__ void __launch_bounds__(OCC_TPB) k_occlusion(fs_bvh_view bv, const float4* __restrict__ src, const uint32_t* __restrict__ off,
                                                       uint32_t n_src, uint32_t n_rays, float lx, float ly, float lz,
                                                       const float* __restrict__ tau, uint32_t n_bands, uint32_t max_crossings,
                                                       float eps_connect, float eps_offset, uint64_t seed,
                                                       unsigned long long* __restrict__ acc, uint32_t* overflow)
{
    __shared__ unsigned long long sacc[OCC_TPB * (FS_MAX_BANDS + 1)];
    const uint32_t W = n_bands + 1u;
    const uint32_t i0 = blockIdx.x * OCC_TPB;
    const uint32_t s0 = occl_source(off, n_src, i0);
    const uint32_t span = occl_source(off, n_src, min(i0 + OCC_TPB, n_rays) - 1u) - s0 + 1u;
    for (uint32_t k = threadIdx.x; k < span * W; k += OCC_TPB) sacc[k] = 0ull;
    __syncthreads();
    const uint32_t i = i0 + threadIdx.x;
    if (i < n_rays) {
        const uint32_t s = occl_source(off, n_src, i);
        const float4 c4 = __ldg(src + s);
        const float c[3] = {c4.x, c4.y, c4.z};
        float q[3];
        fs_occl_point(c, c4.w, i - __ldg(off + s), s, seed, q);
        const fs_vec3 dl = fs_mk(lx - q[0], ly - q[1], lz - q[2]);
        const float len = sqrtf(fs_dot(dl, dl));
        const float tmax = len - eps_connect;
        float g[FS_OCCL_BANDS];
        int visible = 1;
#pragma unroll
        for (int b = 0; b < FS_OCCL_BANDS; ++b) g[b] = 1.0f;
        if (tmax > 0.0f) {
            const float inv = 1.0f / len;
            fs_occl_hit h[FS_OCCL_MAX_HITS];
            uint32_t n = 0;
            fs_all_hits(bv, fs_mk(q[0], q[1], q[2]), fs_mk(dl.x * inv, dl.y * inv, dl.z * inv), tmax,
                        [&](float t, uint32_t id, uint32_t mat) {
                            if (n < FS_OCCL_MAX_HITS) { h[n].t = t; h[n].id = id; h[n].mat = mat; }
                            return ++n <= FS_OCCL_MAX_HITS;        // one hit over the cap blocks the ray: stop there
                        }, overflow);
            visible = fs_occl_ray(h, n, eps_offset, max_crossings, tau, n_bands, g);
        }
        unsigned long long* row = sacc + (size_t)(s - s0) * W;
#pragma unroll
        for (int b = 0; b < FS_OCCL_BANDS; ++b) {
            const unsigned long long v = (unsigned long long)(g[b] * 4294967296.0f);
            if ((uint32_t)b < n_bands && v) atomicAdd(row + b, v);
        }
        if (visible) atomicAdd(row + n_bands, 1ull);
    }
    __syncthreads();
    for (uint32_t k = threadIdx.x; k < span * W; k += OCC_TPB)
        if (sacc[k]) atomicAdd(acc + (size_t)s0 * W + k, sacc[k]);
}

cudaError_t fs_occlusion_run(const fs_bvh_view& bv, const float4* d_src, const uint32_t* d_off, uint32_t n_src, uint32_t n_rays,
                             const float lis[3], const float* d_tau, uint32_t n_bands, uint32_t max_crossings, float eps_connect,
                             float eps_offset, uint64_t seed, unsigned long long* d_acc, uint32_t* d_overflow, cudaStream_t st)
{
    const uint32_t grid = (n_rays + OCC_TPB - 1u) / OCC_TPB;
    k_occlusion<<<grid, OCC_TPB, 0, st>>>(bv, d_src, d_off, n_src, n_rays, lis[0], lis[1], lis[2], d_tau, n_bands, max_crossings,
                                          eps_connect, eps_offset, seed, d_acc, d_overflow);
    return cudaGetLastError();
}
