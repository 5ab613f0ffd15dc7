/* CPU reference for directional sources (fs_set_directivity_patterns / fs_set_source_directivity): the pair loop of
 * fso_trace_sources (fso_sources.c) over the oracle's own walk, with the splat restated so that every band's energy product
 * starts at the source pattern's gain at the path's emission direction instead of 1.
 *
 *   endpoint mode and FSO_FLAG_CONNECT_ALL: source prefix of >= 2 nodes -> the bounce-0 direction of the source subpath
 *     (fso_sample_sphere of Philox block (g, 0, 0), what gen_subpath drew); 1 node -> connection vector * (1 / length);
 *   FSO_FLAG_MIS: the direction of the path's first edge, normalize(x1 - x0), and the product that forms f starts at the gain.
 * The gain itself comes from audio-pathtracer_b200/csrc/fs_directivity.h, the code k_eval runs.  A source with pattern
 * 0xffffffff (FS_OMNI) is not multiplied.  With every gain 1 the result is fso_trace_sources' bit for bit.
 * hist: [S][B][K] Q32.32, ACCUMULATED into (the caller zeroes); dbg: [G] or NULL, endpoint mode only (one record per pair as
 * fso_trace writes them).  Single thread, in g order. */
#include "../../oracle/fs_oracle.c"
#include "../../audio-pathtracer_b200/csrc/fs_directivity.h"

#define DIR_OMNI 0xffffffffu

typedef struct {
    const float* gain;    /* [8][33] of this source's pattern; NULL = omni */
    float f[3];           /* unit forward axis */
} dsrc;

static void dir_factor(const dsrc* ds, uint32_t n_bands, const float d[3], float* g)
{
    for (uint32_t b = 0; b < n_bands; ++b) g[b] = 1.0f;
    if (!ds->gain) return;
    float t;
    const uint32_t i = fs_dir_index(fs_dir_cos(d[0], d[1], d[2], ds->f[0], ds->f[1], ds->f[2]), &t);
    for (uint32_t b = 0; b < n_bands; ++b) {
        const float* T = ds->gain + (size_t)b * 33u + i;
        g[b] = fs_dir_lerp(T[0], T[1], t);
    }
}

/* emission direction of a connected prefix path of the endpoint / all-prefix modes */
static void emission_dir(uint64_t g, uint32_t nf, const float* F, const float* Bp, float len, uint64_t seed, float d[3])
{
    if (nf >= 2u) {
        const uint32_t ctr[4] = {(uint32_t)g, (uint32_t)(g >> 32), 0u, 0u}, key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
        uint32_t r[4];
        fso_philox4x32_10(ctr, key, r);
        fso_sample_sphere(fso_u01(r[1]), fso_u01(r[2]), d);
        return;
    }
    const float inv = 1.0f / len;
    for (int a = 0; a < 3; ++a) d[a] = (Bp[a] - F[a]) * inv;
}

/* splat_path with E[b] starting at g[b] */
static void splat_path_dir(const fso_scene* sc, const fso_config* cfg, const pnode* fn, uint32_t nf, const pnode* bn, uint32_t nb,
                           float len, float weight, const float* gdir, uint64_t* hist_src, fso_path_dbg* dbg)
{
    float E[FSO_MAX_BANDS];
    for (uint32_t b = 0; b < cfg->n_bands; ++b) E[b] = gdir[b];
    float total = 0.0f;
    for (uint32_t i = 0; i + 1 < nf; ++i)
        eval_segment_ev(sc, cfg, fn[i].mat, fn[i].ev, fn[i].prob, dist3(fn[i].ro, fn[i + 1].p), &total, E);
    eval_segment_ev(sc, cfg, fn[nf - 1].mat, FSO_EV_DIFFUSE, fn[nf - 1].prob, len, &total, E);
    for (uint32_t j = nb - 1; j >= 1; --j)
        eval_segment_ev(sc, cfg, bn[j].mat, (j == nb - 1) ? FSO_EV_DIFFUSE : bn[j].ev, bn[j].prob, dist3(bn[j - 1].ro, bn[j].p), &total, E);
    float delay = total / cfg->sound_speed;
    const int32_t bin = fso_bin_index(cfg, delay);
    for (uint32_t b = 0; b < cfg->n_bands; ++b) {
        float e = E[b];
        e = (e < cfg->energy_clamp) ? e : cfg->energy_clamp;
        e = e * cfg->energy_gain;
        if (weight != 1.0f) e = e * weight;
        uint64_t q = (uint64_t)(e * 4294967296.0f);
        hist_src[(uint64_t)b * cfg->n_bins + (uint32_t)bin] += q;
        if (dbg) dbg->energy[b] = e;
    }
    if (dbg) { dbg->connected = 1; dbg->bin = bin; dbg->delay_s = delay; dbg->total_dist = total; }
}

/* mis_splat with val starting at g[b] * 1/(4 pi), g taken at the first edge's direction */
static void mis_splat_dir(const fso_scene* sc, const fso_config* cfg, const pnode* fn, uint32_t s, const pnode* bn, uint32_t t,
                          uint32_t max_depth, const dsrc* ds, uint64_t* hist_src)
{
    const uint32_t k = s + t;
    if (k > FSO_MIS_MAXV) return;
    float pf[FSO_MIS_MAXV], pb[FSO_MIS_MAXV], gg[FSO_MIS_MAXV], dlen[FSO_MIS_MAXV], gdir[FSO_MAX_BANDS];
    float total = 0.0f;
    for (uint32_t i = 0; i + 1 < k; ++i) {
        const pnode* a = (i < s) ? &fn[i] : &bn[k - 1u - i];
        const pnode* b = (i + 1u < s) ? &fn[i + 1u] : &bn[k - 2u - i];
        const float dl[3] = {b->p[0] - a->p[0], b->p[1] - a->p[1], b->p[2] - a->p[2]};
        const float d2 = dot3(dl, dl);
        const float d = sqrtf(d2);
        total += d;
        if (d < cfg->min_seg) return;
        const float inv = 1.0f / d;
        const float dir[3] = {dl[0] * inv, dl[1] * inv, dl[2] * inv};
        if (i == 0u) dir_factor(ds, cfg->n_bands, dir, gdir);
        const float cp = (i == 0u) ? 1.0f : fabsf(dot3(a->n, dir));
        const float cm = (i + 2u == k) ? 1.0f : fabsf(dot3(b->n, dir));
        const float rd2 = 1.0f / d2;
        gg[i] = (cp * cm) * rd2;
        if (!(gg[i] > 0.0f)) return;
        pf[i] = (cfg->rr_prob * ((i == 0u) ? FSO_INV_4PI : cp * FSO_INV_PI)) * (cm * rd2);
        pb[i] = (cfg->rr_prob * ((i + 2u == k) ? FSO_INV_4PI : cm * FSO_INV_PI)) * (cp * rd2);
        dlen[i] = d;
    }
    float sum = 1.0f, r = 1.0f;
    for (uint32_t sp = s; sp + 1u < k && sp <= max_depth; ++sp) { r = r * (pf[sp - 1u] / pb[sp]); sum += r; }
    r = 1.0f;
    for (uint32_t sp = s; sp > 1u && k - sp <= max_depth; --sp) { r = r * (pb[sp - 1u] / pf[sp - 2u]); sum += r; }
    const float delay = total / cfg->sound_speed;
    const int32_t bin = fso_bin_index(cfg, delay);
    for (uint32_t b = 0; b < cfg->n_bands; ++b) {
        float val = ds->gain ? gdir[b] * FSO_INV_4PI : FSO_INV_4PI;
        for (uint32_t i = 0; i + 1 < k; ++i) {
            val = val * gg[i];
            val = val * fso_expf(-cfg->air_absorption[b] * dlen[i]);
            const uint32_t j = i + 1u;
            if (j + 1u < k) {
                const pnode* v = (j < s) ? &fn[j] : &bn[k - 1u - j];
                val = val * sc->refl_over_pi[(uint32_t)v->mat * sc->n_bands + b];
                val = val / ((j < s) ? pf[j - 1u] : pb[j]);
            }
        }
        float e = val / sum;
        e = (e < cfg->energy_clamp) ? e : cfg->energy_clamp;
        e = e * cfg->energy_gain;
        hist_src[(uint64_t)b * cfg->n_bins + (uint32_t)bin] += (uint64_t)(e * 4294967296.0f);
    }
}

static void connect_all_dir(const fso_scene* sc, const fso_config* cfg, const pnode* fn, uint32_t nf, const pnode* bn, uint32_t nb,
                            uint32_t max_depth, uint64_t g, uint64_t seed, const dsrc* ds, uint64_t* hist_src, fso_stats* st,
                            ocount* cnt)
{
    const int mis = (cfg->reserved[1] & FSO_FLAG_MIS) != 0;
    for (uint32_t s = 1; s <= nf; ++s)
        for (uint32_t t = 1; t <= nb; ++t) {
            const pnode* F = &fn[s - 1];
            const pnode* Bn = &bn[t - 1];
            float dl[3] = {Bn->p[0] - F->p[0], Bn->p[1] - F->p[1], Bn->p[2] - F->p[2]};
            float len = sqrtf(dot3(dl, dl));
            float tmax = len - cfg->eps_connect;
            if (tmax > 0.0f) {
                float inv = 1.0f / len;
                float dir[3] = {dl[0] * inv, dl[1] * inv, dl[2] * inv};
                st->shadow_rays++;
                if (any_hit_cnt(sc, F->p, dir, tmax, cnt)) continue;
            }
            st->connected++;
            if (mis) { mis_splat_dir(sc, cfg, fn, s, bn, t, max_depth, ds, hist_src); continue; }
            float d[3], gdir[FSO_MAX_BANDS];
            emission_dir(g, s, F->p, Bn->p, len, seed, d);
            dir_factor(ds, cfg->n_bands, d, gdir);
            splat_path_dir(sc, cfg, fn, s, bn, t, len, 1.0f / (float)(s + t - 1u), gdir, hist_src, NULL);
        }
}

static void trace_pair_dir(const fso_scene* sc, const fso_config* cfg, const float* src, const float* lis, uint64_t g,
                           uint64_t g_lis, uint32_t max_depth, uint64_t seed, const dsrc* ds, pnode* fn, pnode* bn,
                           uint64_t* hist_src, fso_path_dbg* dbg, fso_stats* st, ocount* cnt)
{
    uint64_t rays = 0;
    uint32_t nf = gen_subpath(sc, cfg, src, g, 0u, max_depth, seed, fn, &rays, cnt);
    uint32_t nb = gen_subpath(sc, cfg, lis, g_lis, 1u, max_depth, seed, bn, &rays, cnt);
    st->ext_rays += rays;
    st->paths++;
    if (cfg->reserved[1] & (FSO_FLAG_CONNECT_ALL | FSO_FLAG_MIS)) {
        connect_all_dir(sc, cfg, fn, nf, bn, nb, max_depth, g, seed, ds, hist_src, st, cnt);
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
    if (dbg) {
        memset(dbg, 0, sizeof(*dbg));
        dbg->n_src_nodes = nf; dbg->n_lis_nodes = nb; dbg->bin = -1;
        for (int a = 0; a < 3; ++a) { dbg->src_end[a] = F->p[a]; dbg->lis_end[a] = Bn->p[a]; }
    }
    if (occluded) return;
    st->connected++;
    float d[3], gdir[FSO_MAX_BANDS];
    emission_dir(g, nf, F->p, Bn->p, len, seed, d);
    dir_factor(ds, cfg->n_bands, d, gdir);
    splat_path_dir(sc, cfg, fn, nf, bn, nb, len, 1.0f, gdir, hist_src, dbg);
}

/* gains: [P][8][33]; forward: [S][3] (any non-zero vector, normalised here as the library does: double, rounded to float);
 * pattern: [S] (index < n_patterns or 0xffffffff) */
int fso_trace_sources_dir(const fso_scene* sc, const fso_config* cfg, const float* src_pos, const uint64_t* n_paths,
                          const uint32_t* depths, uint32_t n_src, const float lis_pos[3], uint64_t seed, const float* gains,
                          uint32_t n_patterns, const float* forward, const uint32_t* pattern, uint64_t* hist, fso_path_dbg* dbg,
                          fso_stats* stats)
{
    if (!sc || !cfg || !hist || n_src == 0) return -1;
    if (cfg->n_bands != sc->n_bands || cfg->n_bands > FSO_MAX_BANDS) return -2;
    if (dbg && (cfg->reserved[1] & (FSO_FLAG_CONNECT_ALL | FSO_FLAG_MIS))) return -4;
    uint32_t d_max = 0;
    dsrc* ds = (dsrc*)calloc(n_src, sizeof(dsrc));
    for (uint32_t s = 0; s < n_src; ++s) {
        if (n_paths[s] == 0) { free(ds); return -3; }
        if (depths[s] > d_max) d_max = depths[s];
        if (pattern[s] == DIR_OMNI) continue;
        if (pattern[s] >= n_patterns) { free(ds); return -5; }
        const double x = forward[3 * s], y = forward[3 * s + 1], z = forward[3 * s + 2];
        const double len = sqrt(x * x + y * y + z * z);
        if (!(len > 0.0)) { free(ds); return -5; }
        ds[s].gain = gains + (size_t)pattern[s] * 8u * 33u;
        ds[s].f[0] = (float)(x / len); ds[s].f[1] = (float)(y / len); ds[s].f[2] = (float)(z / len);
    }
    pnode* fn = (pnode*)malloc(sizeof(pnode) * (d_max + 2));
    pnode* bn = (pnode*)malloc(sizeof(pnode) * (d_max + 2));
    fso_stats st;
    ocount cnt;
    memset(&st, 0, sizeof(st));
    memset(&cnt, 0, sizeof(cnt));
    const int share = (cfg->reserved[1] & FSO_FLAG_SHARE_LISTENER) != 0;
    uint64_t o = 0;
    for (uint32_t s = 0; s < n_src; ++s) {
        for (uint64_t g = o; g < o + n_paths[s]; ++g)
            trace_pair_dir(sc, cfg, src_pos + 3ull * s, lis_pos, g, share ? g - o : g, depths[s], seed, &ds[s], fn, bn,
                           hist + (uint64_t)s * cfg->n_bands * cfg->n_bins, dbg ? dbg + g : NULL, &st, &cnt);
        o += n_paths[s];
    }
    free(fn); free(bn); free(ds);
    st.node_visits = cnt.node_visits; st.tri_tests = cnt.tri_tests;
    if (stats) *stats = st;
    return 0;
}
