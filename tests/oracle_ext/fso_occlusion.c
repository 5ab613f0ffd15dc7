/* CPU reference of fs_occlusion (direct-path occlusion and transmission): for every source and sample ray, the sample point
 * and the per-ray gains come from audio-pathtracer_b200/csrc/fs_occlusion.h, the code k_occlusion runs; the hits are found
 * by brute force over all triangles or through the oracle's own BVH (fso_scene_create's use_bvh), walked without an early exit.
 * The ray is the endpoint connection ray of the oracle (fs_oracle.c, trace_one): from the sample point to the listener,
 * tmax = |dl| - eps_connect.  tau_eff is slot 2 of fso_scene_set_material_model's table, or 0 for every material of a scene
 * without the model (surfaces block).  Single thread; the sums are exact 64-bit integers as on the device. */
#include "../../oracle/fs_oracle.c"
#include "../../audio-pathtracer_b200/csrc/fs_occlusion.h"

typedef struct { fs_occl_hit h[FS_OCCL_MAX_HITS]; uint32_t n; } hitlist;

static void add_hit(hitlist* L, float t, uint32_t id, uint32_t mat)
{
    if (L->n < FS_OCCL_MAX_HITS) { L->h[L->n].t = t; L->h[L->n].id = id; L->h[L->n].mat = mat; }
    L->n++;
}

static void all_hits(const fso_scene* sc, const float o[3], const float d[3], float tmax, hitlist* L)
{
    L->n = 0;
    if (!sc->use_bvh || sc->n_tris == 0) {
        for (uint64_t t = 0; t < sc->n_tris; ++t) {
            float tt;
            if (fso_intersect_tri(o, d, sc->v0 + 3 * t, sc->e1 + 3 * t, sc->e2 + 3 * t, &tt) && tt < tmax)
                add_hit(L, tt, (uint32_t)t, sc->mat[t]);
        }
        return;
    }
    float inv[3];
    safe_inv(d, inv);
    int32_t stack[128];
    int sp = 0;
    stack[sp++] = 0;
    while (sp) {
        const onode* n = &sc->nodes[stack[--sp]];
        float tn;
        if (!slab(n, o, inv, tmax, &tn)) continue;
        if (n->left < 0) {
            for (uint32_t i = 0; i < n->count; ++i) {
                uint32_t t = sc->order[n->first + i];
                float tt;
                if (fso_intersect_tri(o, d, sc->v0 + 3 * (uint64_t)t, sc->e1 + 3 * (uint64_t)t, sc->e2 + 3 * (uint64_t)t, &tt)
                    && tt < tmax)
                    add_hit(L, tt, t, sc->mat[t]);
            }
        } else {
            stack[sp++] = n->left;
            stack[sp++] = n->right;
        }
    }
}

/* tau_eff [M][B] the reference uses */
void fso_occlusion_tau(const fso_scene* sc, float* out)
{
    const size_t n = (size_t)sc->n_mats * sc->n_bands;
    for (size_t i = 0; i < n; ++i) out[i] = sc->bsdf_tab ? sc->bsdf_tab[2 * n + i] : 0.0f;
}

/* pos [S][3], radius [S], n_rays [S] (ignored for radius 0); visible [S], trans [S][8] (bands >= n_bands: 0), used [S].
 * Returns 0, or -1 for an argument fs_occlusion rejects. */
int fso_occlusion(const fso_scene* sc, const float* pos, const float* radius, const uint32_t* n_rays, uint32_t n_src,
                  const float lis[3], uint32_t max_crossings, uint64_t seed, float eps_connect, float eps_offset, float* visible,
                  float* trans, uint32_t* used)
{
    if (n_src == 0 || max_crossings > 16) return -1;
    const uint32_t B = sc->n_bands;
    const size_t MB = (size_t)(sc->n_mats ? sc->n_mats : 1) * B;
    float* tau = (float*)malloc(sizeof(float) * MB);
    fso_occlusion_tau(sc, tau);
    hitlist L;
    for (uint32_t s = 0; s < n_src; ++s) {
        if (!(radius[s] >= 0.0f) || (radius[s] > 0.0f && (n_rays[s] == 0 || n_rays[s] > 65536u))) { free(tau); return -1; }
        const uint32_t n = radius[s] > 0.0f ? n_rays[s] : 1u;
        uint64_t acc[FS_OCCL_BANDS] = {0}, vis = 0;
        for (uint32_t j = 0; j < n; ++j) {
            float q[3], g[FS_OCCL_BANDS];
            fs_occl_point(pos + 3ull * s, radius[s], j, s, seed, q);
            const float dl[3] = {lis[0] - q[0], lis[1] - q[1], lis[2] - q[2]};
            const float len = sqrtf(dot3(dl, dl));
            const float tmax = len - eps_connect;
            int v = 1;
            for (int b = 0; b < FS_OCCL_BANDS; ++b) g[b] = 1.0f;
            if (tmax > 0.0f) {
                const float inv = 1.0f / len;
                const float dir[3] = {dl[0] * inv, dl[1] * inv, dl[2] * inv};
                all_hits(sc, q, dir, tmax, &L);
                v = fs_occl_ray(L.h, L.n, eps_offset, max_crossings, tau, B, g);
            }
            for (uint32_t b = 0; b < B; ++b) acc[b] += (uint64_t)(g[b] * 4294967296.0f);
            vis += (uint64_t)v;
        }
        visible[s] = (float)((double)vis / (double)n);
        for (uint32_t b = 0; b < FS_OCCL_BANDS; ++b)
            trans[(size_t)s * FS_OCCL_BANDS + b] = b < B ? (float)((double)acc[b] * 0x1p-32 / (double)n) : 0.0f;
        used[s] = n;
    }
    free(tau);
    return 0;
}
