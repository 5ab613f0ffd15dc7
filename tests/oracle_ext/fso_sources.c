/* CPU reference for per-source path budgets and depths (fs_trace_sources): the oracle's own path code, compiled together
 * with it, over the flat work range of the per-source form.
 *
 * Source s owns g in [o_s, o_s + n_s) with o_s = sum_{s' < s} n_s'; both subpaths of its pairs stop at depth_s; Philox is
 * keyed by (seed, g) for both subpaths, except that with FSO_FLAG_SHARE_LISTENER the listener subpath is keyed by
 * i = g - o_s.  hist: [S][B][K] Q32.32, ACCUMULATED into (the caller zeroes).  Single thread, in g order. */
#include "../../oracle/fs_oracle.c"

static void trace_pair(const fso_scene* sc, const fso_config* cfg, const float* src, const float* lis, uint64_t g,
                       uint64_t g_lis, uint32_t max_depth, uint64_t seed, pnode* fn, pnode* bn, uint64_t* hist_src,
                       fso_stats* st, ocount* cnt)
{
    uint64_t rays = 0;
    uint32_t nf = gen_subpath(sc, cfg, src, g, 0u, max_depth, seed, fn, &rays, cnt);
    uint32_t nb = gen_subpath(sc, cfg, lis, g_lis, 1u, max_depth, seed, bn, &rays, cnt);
    st->ext_rays += rays;
    st->paths++;
    if (cfg->reserved[1] & (FSO_FLAG_CONNECT_ALL | FSO_FLAG_MIS)) {
        connect_all(sc, cfg, fn, nf, bn, nb, max_depth, hist_src, st, cnt);
        return;
    }
    const pnode* F = &fn[nf - 1];
    const pnode* Bn = &bn[nb - 1];
    float dl[3] = {Bn->p[0] - F->p[0], Bn->p[1] - F->p[1], Bn->p[2] - F->p[2]};
    float len = sqrtf(dot3(dl, dl));
    float tmax = len - cfg->eps_connect;
    int occluded = 0;
    if (tmax > 0.0f) {
        float inv = 1.0f / len;
        float dir[3] = {dl[0] * inv, dl[1] * inv, dl[2] * inv};
        st->shadow_rays++;
        occluded = any_hit_cnt(sc, F->p, dir, tmax, cnt);
    }
    if (occluded) return;
    st->connected++;
    splat_path(sc, cfg, fn, nf, bn, nb, len, 1.0f, hist_src, NULL);
}

int fso_trace_sources(const fso_scene* sc, const fso_config* cfg, const float* src_pos, const uint64_t* n_paths,
                      const uint32_t* depths, uint32_t n_src, const float lis_pos[3], uint64_t g_first, uint64_t g_count,
                      uint64_t seed, uint64_t* hist, fso_stats* stats)
{
    if (!sc || !cfg || !hist || n_src == 0) return -1;
    if (cfg->n_bands != sc->n_bands || cfg->n_bands > FSO_MAX_BANDS) return -2;
    uint64_t G = 0;
    uint32_t d_max = 0;
    for (uint32_t s = 0; s < n_src; ++s) {
        if (n_paths[s] == 0) return -3;
        G += n_paths[s];
        if (depths[s] > d_max) d_max = depths[s];
    }
    if (g_first + g_count > G) return -3;
    pnode* fn = (pnode*)malloc(sizeof(pnode) * (d_max + 2));
    pnode* bn = (pnode*)malloc(sizeof(pnode) * (d_max + 2));
    fso_stats st;
    ocount cnt;
    memset(&st, 0, sizeof(st));
    memset(&cnt, 0, sizeof(cnt));
    const int share = (cfg->reserved[1] & FSO_FLAG_SHARE_LISTENER) != 0;
    uint64_t o = 0;
    for (uint32_t s = 0; s < n_src; ++s) {
        const uint64_t lo = o > g_first ? o : g_first;
        const uint64_t hi = (o + n_paths[s] < g_first + g_count) ? o + n_paths[s] : g_first + g_count;
        for (uint64_t g = lo; g < hi; ++g)
            trace_pair(sc, cfg, src_pos + 3ull * s, lis_pos, g, share ? g - o : g, depths[s], seed, fn, bn,
                       hist + (uint64_t)s * cfg->n_bands * cfg->n_bins, &st, &cnt);
        o += n_paths[s];
    }
    free(fn); free(bn);
    st.node_visits = cnt.node_visits; st.tri_tests = cnt.tri_tests;
    if (stats) *stats = st;
    return 0;
}
