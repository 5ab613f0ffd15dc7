/* CPU reference of fs_diffraction (first-order edge diffraction of the direct path).  The per-edge arithmetic comes from
 * audio-pathtracer_b200/csrc/fs_diffraction.h, the code the kernels run; everything around it is independent of them:
 *   edges: every triangle edge with its canonical endpoints, sorted with qsort by the endpoint bits and then by 3 tri + k
 *     (no hash), grouped by equal endpoints, classified (1, 2, >= 3 triangles) and fold-tested;
 *   query: every (source, edge) pair in turn, the two legs through fso_any_hit (brute force over all triangles, or the
 *     oracle's own BVH when the scene was created with use_bvh), the shortest path kept by (length, edge rank).
 * Single thread. */
#include "../../oracle/fs_oracle.c"
#include "../../audio-pathtracer_b200/csrc/fs_diffraction.h"

typedef struct { uint32_t found, n_paths, edge_tri, edge_k; float apex[3], length, path_difference, gain[8]; } fso_diff_result;

typedef struct { uint32_t key[6]; uint32_t e; } tedge;

static int tedge_cmp(const void* x, const void* y)
{
    const tedge *a = (const tedge*)x, *b = (const tedge*)y;
    for (int i = 0; i < 6; ++i)
        if (a->key[i] != b->key[i]) return a->key[i] < b->key[i] ? -1 : 1;
    return a->e < b->e ? -1 : (a->e > b->e);
}

static int u32_cmp(const void* x, const void* y)
{
    const uint32_t a = *(const uint32_t*)x, b = *(const uint32_t*)y;
    return a < b ? -1 : (a > b);
}

static float c_min_of(float min_fold_deg) { return (float)(-cos((double)min_fold_deg * (M_PI / 180.0))); }

/* the edge set of verts [T][3][3] for min_fold_deg: records in ascending (tri, k) into *out (malloc'ed); returns the count */
static uint32_t build_edges(const float* verts, uint64_t n_tris, float min_fold_deg, fs_diff_edge** out)
{
    const float c_min = c_min_of(min_fold_deg);
    tedge* t = (tedge*)malloc(sizeof(tedge) * (3 * n_tris + 1));
    uint64_t n = 0;
    for (uint64_t tri = 0; tri < n_tris; ++tri) {
        const float* v = verts + 9 * tri;
        if (fs_diff_degenerate(v)) continue;
        for (uint32_t k = 0; k < 3; ++k) {
            float a[3], b[3];
            if (!fs_diff_endpoints(v, k, a, b)) continue;
            for (int i = 0; i < 3; ++i) { t[n].key[i] = fs_diff_bits(a[i]); t[n].key[3 + i] = fs_diff_bits(b[i]); }
            t[n].e = (uint32_t)(3 * tri + k);
            ++n;
        }
    }
    qsort(t, n, sizeof(tedge), tedge_cmp);
    uint32_t* kept = (uint32_t*)malloc(sizeof(uint32_t) * 2 * (n + 1));   /* (e, other) */
    uint32_t m = 0;
    for (uint64_t i = 0; i < n;) {
        uint64_t j = i + 1;
        while (j < n && !memcmp(t[j].key, t[i].key, sizeof(t[i].key))) ++j;
        const uint32_t e = t[i].e;
        int keep = 0;
        uint32_t other = 0xffffffffu;
        if (j - i == 1) keep = 1;
        else if (j - i == 2) {
            float a[3], b[3];
            fs_diff_endpoints(verts + 9ull * (e / 3), e % 3, a, b);
            other = t[i + 1].e;
            keep = fs_diff_fold_ok(a, b, verts + 9ull * (e / 3), e % 3, verts + 9ull * (other / 3), other % 3, c_min);
        }
        if (keep) { kept[2 * m] = e; kept[2 * m + 1] = other; ++m; }
        i = j;
    }
    qsort(kept, m, 2 * sizeof(uint32_t), u32_cmp);
    fs_diff_edge* E = (fs_diff_edge*)malloc(sizeof(fs_diff_edge) * (m + 1));
    for (uint32_t i = 0; i < m; ++i) {
        const uint32_t e = kept[2 * i], f = kept[2 * i + 1];
        float a[3], b[3];
        fs_diff_endpoints(verts + 9ull * (e / 3), e % 3, a, b);
        fs_diff_make_edge(a, b, verts + 9ull * (e / 3), e / 3, e % 3, f == 0xffffffffu ? NULL : verts + 9ull * (f / 3), f % 3, &E[i]);
    }
    free(t);
    free(kept);
    *out = E;
    return m;
}

/* (tri, k) pairs of the edge set, the first min(n, cap) into out [cap][2]; returns n */
uint64_t fso_diffraction_edges(const float* verts, uint64_t n_tris, float min_fold_deg, uint32_t* out, uint64_t cap)
{
    fs_diff_edge* E;
    const uint32_t n = build_edges(verts, n_tris, min_fold_deg, &E);
    for (uint32_t i = 0; i < n && i < cap; ++i) { out[2 * i] = E[i].tri; out[2 * i + 1] = E[i].k & 3u; }
    free(E);
    return n;
}

/* src [S][3], lis [3], band_hz [n_bands] (NULL: 62.5 2^b); out [S]; stats [3] = edges, candidates (pairs passing the
 * geometric tests), leg rays traced */
void fso_diffraction(const fso_scene* sc, const float* verts, float min_fold_deg, const float* src, uint32_t n_src,
                     const float lis[3], const float* band_hz, uint32_t n_bands, float eps_offset, float eps_connect,
                     float sound_speed, fso_diff_result* out, uint64_t* stats)
{
    fs_diff_edge* E;
    const uint32_t n = build_edges(verts, sc->n_tris, min_fold_deg, &E);
    float hz[8];
    for (uint32_t b = 0; b < n_bands; ++b) hz[b] = band_hz ? band_hz[b] : fs_diff_default_hz(b);
    uint64_t cand = 0, rays = 0;
    for (uint32_t s_i = 0; s_i < n_src; ++s_i) {
        const float* s = src + 3ull * s_i;
        uint32_t paths = 0, best = 0xffffffffu;
        float best_len = 0.0f;
        for (uint32_t e = 0; e < n; ++e) {
            float p[3], ds[3], dl[3], ts, tl;
            if (!fs_diff_apex(&E[e], s, lis, eps_offset, p)) continue;
            ++cand;
            const float ls = fs_diff_leg(s, p, eps_connect, ds, &ts);
            const float ll = fs_diff_leg(lis, p, eps_connect, dl, &tl);
            int clear = 1;
            if (ts > 0.0f) { ++rays; clear = !fso_any_hit(sc, s, ds, ts); }
            if (clear && tl > 0.0f) { ++rays; clear = !fso_any_hit(sc, lis, dl, tl); }
            if (!clear) continue;
            ++paths;
            const float length = ls + ll;
            if (best == 0xffffffffu || length < best_len) { best = e; best_len = length; }   /* e ascends: ties keep the lower */
        }
        fso_diff_result* r = out + s_i;
        memset(r, 0, sizeof(*r));
        if (best == 0xffffffffu) continue;
        float p[3], d[3], t;
        fs_diff_apex(&E[best], s, lis, eps_offset, p);
        const float length = fs_diff_leg(s, p, eps_connect, d, &t) + fs_diff_leg(lis, p, eps_connect, d, &t);
        const float z = fs_diff_z(s, lis, length);
        r->found = 1;
        r->n_paths = paths;
        r->edge_tri = E[best].tri;
        r->edge_k = E[best].k & 3u;
        for (int i = 0; i < 3; ++i) r->apex[i] = p[i];
        r->length = length;
        r->path_difference = z;
        for (uint32_t b = 0; b < n_bands; ++b) r->gain[b] = fs_diff_gain(z, hz[b], sound_speed);
    }
    if (stats) { stats[0] = n; stats[1] = cand; stats[2] = rays; }
    free(E);
}

/* the shared gain formula, for the known-answer tests */
float fso_diffraction_gain(float z, float f, float c) { return fs_diff_gain(z, f, c); }
