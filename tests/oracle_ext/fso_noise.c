/* CPU reference for FS_FLAG_NOISE_STATS: the pair loop of fso_trace_sources (fso_sources.c) over the oracle's own path code,
 * with the exact second moment of every pair's contribution.
 *
 * In the endpoint-connection mode a pair adds at most one connected path, i.e. one Q32.32 value q_b to one bin of every band.
 * hist: [S][B][K] (S1, as fso_trace_sources), m2: [S][B+1][K][2] (lo, hi) = sum of q_b^2 per band and of (sum_b q_b)^2 in
 * slot B, both ACCUMULATED into (the caller zeroes).  Sums mod 2^128 in unsigned __int128.  Single thread, in g order. */
#include "../../oracle/fs_oracle.c"

static void m2_add(uint64_t* m2, unsigned __int128 v)
{
    unsigned __int128 s = ((unsigned __int128)m2[1] << 64) | m2[0];
    s += v;
    m2[0] = (uint64_t)s; m2[1] = (uint64_t)(s >> 64);
}

static void trace_pair_m2(const fso_scene* sc, const fso_config* cfg, const float* src, const float* lis, uint64_t g,
                          uint64_t g_lis, uint32_t max_depth, uint64_t seed, pnode* fn, pnode* bn, uint64_t* hist_src,
                          uint64_t* m2_src, fso_stats* st, ocount* cnt)
{
    uint64_t rays = 0;
    uint32_t nf = gen_subpath(sc, cfg, src, g, 0u, max_depth, seed, fn, &rays, cnt);
    uint32_t nb = gen_subpath(sc, cfg, lis, g_lis, 1u, max_depth, seed, bn, &rays, cnt);
    st->ext_rays += rays;
    st->paths++;
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
    fso_path_dbg dbg;
    memset(&dbg, 0, sizeof(dbg));
    splat_path(sc, cfg, fn, nf, bn, nb, len, 1.0f, hist_src, &dbg);
    /* the splat's own Q32.32 values: the same float expression on the recorded clamped, gained energy */
    const uint32_t B = cfg->n_bands, K = cfg->n_bins;
    uint64_t qs = 0;
    for (uint32_t b = 0; b < B; ++b) {
        const uint64_t q = (uint64_t)(dbg.energy[b] * 4294967296.0f);
        qs += q;
        m2_add(m2_src + 2ull * ((uint64_t)b * K + (uint32_t)dbg.bin), (unsigned __int128)q * q);
    }
    m2_add(m2_src + 2ull * ((uint64_t)B * K + (uint32_t)dbg.bin), (unsigned __int128)qs * qs);
}

int fso_trace_sources_m2(const fso_scene* sc, const fso_config* cfg, const float* src_pos, const uint64_t* n_paths,
                         const uint32_t* depths, uint32_t n_src, const float lis_pos[3], uint64_t seed, uint64_t* hist,
                         uint64_t* m2, fso_stats* stats)
{
    if (!sc || !cfg || !hist || !m2 || n_src == 0) return -1;
    if (cfg->n_bands != sc->n_bands || cfg->n_bands > FSO_MAX_BANDS) return -2;
    if (cfg->reserved[1] & (FSO_FLAG_CONNECT_ALL | FSO_FLAG_MIS)) return -4;
    uint32_t d_max = 0;
    for (uint32_t s = 0; s < n_src; ++s) {
        if (n_paths[s] == 0) return -3;
        if (depths[s] > d_max) d_max = depths[s];
    }
    pnode* fn = (pnode*)malloc(sizeof(pnode) * (d_max + 2));
    pnode* bn = (pnode*)malloc(sizeof(pnode) * (d_max + 2));
    fso_stats st;
    ocount cnt;
    memset(&st, 0, sizeof(st));
    memset(&cnt, 0, sizeof(cnt));
    const int share = (cfg->reserved[1] & FSO_FLAG_SHARE_LISTENER) != 0;
    const uint64_t B = cfg->n_bands, K = cfg->n_bins;
    uint64_t o = 0;
    for (uint32_t s = 0; s < n_src; ++s) {
        for (uint64_t g = o; g < o + n_paths[s]; ++g)
            trace_pair_m2(sc, cfg, src_pos + 3ull * s, lis_pos, g, share ? g - o : g, depths[s], seed, fn, bn,
                          hist + (uint64_t)s * B * K, m2 + 2ull * (uint64_t)s * (B + 1) * K, &st, &cnt);
        o += n_paths[s];
    }
    free(fn); free(bn);
    st.node_visits = cnt.node_visits; st.tri_tests = cnt.tri_tests;
    if (stats) *stats = st;
    return 0;
}
