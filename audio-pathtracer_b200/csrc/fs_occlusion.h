/* fs_occlusion.h -- the per-ray arithmetic of fs_occlusion, written once for k_occlusion and the CPU reference
 * (tests/oracle_ext/fso_occlusion.c), which include this file as C.  The CUDA side takes Philox, fs_u01, fs_pow and
 * fs_sample_sphere from fs_math.cuh; the C side takes their fso_* twins, which the reference defines before it includes this
 * file and the trace parity tests already hold bit-identical.
 *
 * Bit-exactness: binary32 * + / sqrt and explicit fmaf only, in a fixed order (the CUDA translation units are compiled with
 * --fmad=false, the reference with -ffp-contract=off).
 *   sample point j >= 1 of source s:  Philox4x32-10 block, key = seed, counter = (j, s, 0, FS_OCCL_TAG);
 *     u1, u2, u3 = u01 of its first three words, rho = radius u3^(1/3) (fs_pow; 0 when u3 = 0),
 *     q = centre + rho sample_sphere(u1, u2), one fmaf per component.  q_0 = centre.
 *   hits: sorted by (t, original triangle id); a hit of the same material as the last COUNTED crossing and less than
 *     eps_offset further along is that crossing again (a shared edge or vertex of a tessellated wall counts once).
 *   gain_b = prod over the k counted crossings, in order, starting at 1.0f, of tau[mat][b]; 0 when k > max_crossings or
 *     when the ray had more than FS_OCCL_MAX_HITS raw hits.  Visible = no counted crossing (and not over the cap). */
#ifndef FS_OCCLUSION_H
#define FS_OCCLUSION_H

#include <math.h>
#include <stdint.h>

#define FS_OCCL_MAX_HITS 32u
#define FS_OCCL_TAG 0x4F43434Cu        /* 'OCCL': trace blocks carry the side (0, 1) in this word, the IR noise carriers a band < 8 */
#define FS_OCCL_BANDS 8

#if defined(__CUDACC__)
#define FS_OCCL_HD __host__ __device__ __forceinline__
#else
#define FS_OCCL_HD static inline
#endif

typedef struct fs_occl_hit { float t; uint32_t id, mat; } fs_occl_hit;

/* sample point j of source s: centre c, radius r */
FS_OCCL_HD void fs_occl_point(const float c[3], float r, uint32_t j, uint32_t s, uint64_t seed, float q[3])
{
    if (j == 0u) { q[0] = c[0]; q[1] = c[1]; q[2] = c[2]; return; }
    uint32_t w[4];
    float d[3];
#if defined(__CUDACC__)
    fs_philox4x32_10(j, s, 0u, FS_OCCL_TAG, (uint32_t)seed, (uint32_t)(seed >> 32), w);
    const float u1 = fs_u01(w[0]), u2 = fs_u01(w[1]), u3 = fs_u01(w[2]);
    const fs_vec3 dv = fs_sample_sphere(u1, u2);
    d[0] = dv.x; d[1] = dv.y; d[2] = dv.z;
    const float rho = (u3 > 0.0f) ? r * fs_pow(u3, 1.0f / 3.0f) : 0.0f;
#else
    const uint32_t ctr[4] = {j, s, 0u, FS_OCCL_TAG}, key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    fso_philox4x32_10(ctr, key, w);
    const float u1 = fso_u01(w[0]), u2 = fso_u01(w[1]), u3 = fso_u01(w[2]);
    fso_sample_sphere(u1, u2, d);
    const float rho = (u3 > 0.0f) ? r * fso_powf(u3, 1.0f / 3.0f) : 0.0f;
#endif
    q[0] = fmaf(rho, d[0], c[0]);
    q[1] = fmaf(rho, d[1], c[1]);
    q[2] = fmaf(rho, d[2], c[2]);
}

/* one ray from its raw hits h[0 .. min(n_raw, FS_OCCL_MAX_HITS)) (any order; sorted and compacted in place): per-band gains
 * g[0 .. FS_OCCL_BANDS) (bands >= n_bands: 0) from tau [M][n_bands]; returns 1 when the ray crosses no surface */
FS_OCCL_HD int fs_occl_ray(fs_occl_hit* h, uint32_t n_raw, float eps_offset, uint32_t max_crossings, const float* tau,
                           uint32_t n_bands, float* g)
{
    if (n_raw > FS_OCCL_MAX_HITS) {
        for (int b = 0; b < FS_OCCL_BANDS; ++b) g[b] = 0.0f;
        return 0;
    }
    for (uint32_t i = 1; i < n_raw; ++i) {                 /* insertion sort by (t, id) */
        const fs_occl_hit x = h[i];
        uint32_t k = i;
        while (k > 0u && (h[k - 1u].t > x.t || (h[k - 1u].t == x.t && h[k - 1u].id > x.id))) { h[k] = h[k - 1u]; --k; }
        h[k] = x;
    }
    uint32_t n = 0;                                        /* counted crossings, compacted to h[0 .. n) */
    for (uint32_t i = 0; i < n_raw; ++i) {
        if (n > 0u && h[i].mat == h[n - 1u].mat && h[i].t - h[n - 1u].t < eps_offset) continue;
        h[n++] = h[i];
    }
    for (int b = 0; b < FS_OCCL_BANDS; ++b) g[b] = ((uint32_t)b < n_bands && n <= max_crossings) ? 1.0f : 0.0f;
    if (n <= max_crossings)
        for (uint32_t i = 0; i < n; ++i) {
            const float* row = tau + (size_t)h[i].mat * n_bands;
            for (int b = 0; b < FS_OCCL_BANDS; ++b)
                if ((uint32_t)b < n_bands) g[b] = g[b] * row[b];
        }
    return n == 0u;
}

#endif
