/* fs_diffraction.h -- the per-edge arithmetic of fs_diffraction, written once for the kernels of fs_diffraction.cu and the
 * CPU reference (tests/oracle_ext/fso_diffraction.c), which includes this file as C.
 *
 * Bit-exactness: binary32 * + / sqrt and explicit fmaf only, in a fixed order (the CUDA translation units are compiled with
 * --fmad=false, the reference with -ffp-contract=off).  dot(a, b) = fmaf(a.z, b.z, fmaf(a.y, b.y, a.x b.x)), the order of
 * fs_dot, so a leg ray built here is the ray fs_debug_any_hits is given for the same two points.
 *   edge endpoints: each coordinate with -0.0 replaced by +0.0; A = the lexicographically smaller endpoint (x, then y, then
 *     z), B the other.  Two triangle edges are one scene edge iff their (A, B) are equal bit for bit.
 *   e = B - A, len = sqrt(dot(e, e)), u_hat = e (1 / len).
 *   face direction of a triangle with third vertex C: w = C - A, u = w - (dot(w, e) / dot(e, e)) e, u1 = u (1 / |u|).
 *   fold test of a wedge: dot(u1, u2) >= c_min.
 *   per source S and listener L: ps = (S - A) - dot(S - A, u_hat) u_hat, r_S = |ps| (likewise pl, r_L); both > eps_offset;
 *     x = s_a + ((l_a - s_a) r_S) / (r_S + r_L), valid for 0 <= x <= len; P = A + x u_hat;
 *     shadow: with c(a, b) = dot(u_hat, a x b), for every face half-line u: c(ps, u), c(u, pl) and c(ps, pl) all > 0 or all
 *     < 0 (the segment ps -> pl strictly crosses the half-line).
 *   legs: d = P - Q, |d| = sqrt(dot(d, d)), tmax = |d| - eps_connect (<= 0: clear, nothing traced), direction d (1 / |d|).
 *   length = |SP| + |PL|, z = max(length - |SL|, 0), gain_b = max(1 / (3 + ((40 z) f_b) / c), 0.01). */
#ifndef FS_DIFFRACTION_H
#define FS_DIFFRACTION_H

#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define FS_DIFF_HD __host__ __device__ __forceinline__
#else
#define FS_DIFF_HD static inline
#endif

#define FS_DIFF_NO_KEY 0xffffffffffffffffull   /* sort key of a skipped triangle edge: after every real key */
#define FS_DIFF_SCREEN 4u                       /* flag bit of fs_diff_edge::k: one face (u2 unused) */

/* one scene edge, as the query reads it (64 bytes) */
typedef struct fs_diff_edge {
    float a[3]; uint32_t tri;                   /* A, the naming triangle */
    float d[3]; float len;                      /* u_hat, |B - A| */
    float u1[3]; uint32_t k;                    /* face direction 1; edge slot k | FS_DIFF_SCREEN */
    float u2[3]; uint32_t pad;                  /* face direction 2 (wedges) */
} fs_diff_edge;

FS_DIFF_HD float fs_diff_dot(const float a[3], const float b[3]) { return fmaf(a[2], b[2], fmaf(a[1], b[1], a[0] * b[0])); }
FS_DIFF_HD void fs_diff_cross(const float a[3], const float b[3], float o[3])
{
    o[0] = fmaf(a[1], b[2], -(a[2] * b[1]));
    o[1] = fmaf(a[2], b[0], -(a[0] * b[2]));
    o[2] = fmaf(a[0], b[1], -(a[1] * b[0]));
}

FS_DIFF_HD uint32_t fs_diff_bits(float f)
{
    uint32_t u;
    memcpy(&u, &f, 4);
    return u == 0x80000000u ? 0u : u;
}
FS_DIFF_HD float fs_diff_canon(float f) { return f == 0.0f ? 0.0f : f; }

/* triangle with zero cross product (a degenerate triangle holds no edge) */
FS_DIFF_HD int fs_diff_degenerate(const float* v /* [3][3] */)
{
    const float e1[3] = {v[3] - v[0], v[4] - v[1], v[5] - v[2]}, e2[3] = {v[6] - v[0], v[7] - v[1], v[8] - v[2]};
    float c[3];
    fs_diff_cross(e1, e2, c);
    return c[0] == 0.0f && c[1] == 0.0f && c[2] == 0.0f;
}

/* canonical endpoints of triangle edge k of the triangle v [3][3]: a = the smaller; returns 0 for a zero-length edge */
FS_DIFF_HD int fs_diff_endpoints(const float* v, uint32_t k, float a[3], float b[3])
{
    const float* p = v + 3u * k;
    const float* q = v + 3u * (k == 2u ? 0u : k + 1u);
    float x[3], y[3];
    for (int i = 0; i < 3; ++i) { x[i] = fs_diff_canon(p[i]); y[i] = fs_diff_canon(q[i]); }
    int lt = 0, eq = 1;
    for (int i = 0; i < 3 && eq; ++i) {
        if (x[i] != y[i]) { eq = 0; lt = x[i] < y[i]; }
    }
    if (eq) return 0;
    for (int i = 0; i < 3; ++i) { a[i] = lt ? x[i] : y[i]; b[i] = lt ? y[i] : x[i]; }
    return 1;
}

/* 63-bit hash of the canonical endpoint pair (top bit clear, so FS_DIFF_NO_KEY sorts after every real key) */
FS_DIFF_HD uint64_t fs_diff_hash(const float a[3], const float b[3])
{
    uint64_t h = 0x9E3779B97F4A7C15ull;
    for (int i = 0; i < 6; ++i) {
        h ^= (uint64_t)fs_diff_bits(i < 3 ? a[i] : b[i - 3]);
        h *= 0xFF51AFD7ED558CCDull;
        h ^= h >> 33;
    }
    return h >> 1;
}

FS_DIFF_HD int fs_diff_same(const float a[3], const float b[3], const float c[3], const float d[3])
{
    for (int i = 0; i < 3; ++i)
        if (fs_diff_bits(a[i]) != fs_diff_bits(c[i]) || fs_diff_bits(b[i]) != fs_diff_bits(d[i])) return 0;
    return 1;
}

/* unit vector from the edge (a, b) into the face whose third vertex is c, perpendicular to the edge */
FS_DIFF_HD void fs_diff_face_dir(const float a[3], const float b[3], const float c[3], float u[3])
{
    const float e[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, w[3] = {c[0] - a[0], c[1] - a[1], c[2] - a[2]};
    const float s = fs_diff_dot(w, e) / fs_diff_dot(e, e);
    float t[3];
    for (int i = 0; i < 3; ++i) t[i] = w[i] - s * e[i];
    const float inv = 1.0f / sqrtf(fs_diff_dot(t, t));
    for (int i = 0; i < 3; ++i) u[i] = t[i] * inv;
}

/* the third vertex of triangle edge k */
FS_DIFF_HD const float* fs_diff_opposite(const float* v, uint32_t k) { return v + 3u * (k == 0u ? 2u : k - 1u); }

/* fold test of a wedge with faces from triangles v and w (their edges ka, kb are the same scene edge (a, b)) */
FS_DIFF_HD int fs_diff_fold_ok(const float a[3], const float b[3], const float* v, uint32_t kv, const float* w, uint32_t kw,
                               float c_min)
{
    float u1[3], u2[3];
    fs_diff_face_dir(a, b, fs_diff_opposite(v, kv), u1);
    fs_diff_face_dir(a, b, fs_diff_opposite(w, kw), u2);
    return fs_diff_dot(u1, u2) >= c_min;
}

/* the edge record of (tri, k) with canonical endpoints (a, b); w = the second triangle (and kw its slot), or null: a screen */
FS_DIFF_HD void fs_diff_make_edge(const float a[3], const float b[3], const float* v, uint32_t tri, uint32_t k, const float* w,
                                  uint32_t kw, fs_diff_edge* out)
{
    const float e[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]};
    const float len = sqrtf(fs_diff_dot(e, e));
    const float inv = 1.0f / len;
    for (int i = 0; i < 3; ++i) { out->a[i] = a[i]; out->d[i] = e[i] * inv; }
    out->len = len;
    out->tri = tri;
    fs_diff_face_dir(a, b, fs_diff_opposite(v, k), out->u1);
    if (w) {
        fs_diff_face_dir(a, b, fs_diff_opposite(w, kw), out->u2);
        out->k = k;
    } else {
        out->u2[0] = out->u2[1] = out->u2[2] = 0.0f;
        out->k = k | FS_DIFF_SCREEN;
    }
    out->pad = 0u;
}

/* c(a, b) = dot(u_hat, a x b) */
FS_DIFF_HD float fs_diff_side(const float d[3], const float a[3], const float b[3])
{
    float c[3];
    fs_diff_cross(a, b, c);
    return fs_diff_dot(d, c);
}

FS_DIFF_HD int fs_diff_crosses(const float d[3], const float ps[3], const float pl[3], const float u[3], float c3)
{
    const float c1 = fs_diff_side(d, ps, u), c2 = fs_diff_side(d, u, pl);
    return (c1 > 0.0f && c2 > 0.0f && c3 > 0.0f) || (c1 < 0.0f && c2 < 0.0f && c3 < 0.0f);
}

/* the geometric tests of one (source, listener, edge): returns 1 and the apex p when the edge line's closest path is on the
 * segment and in the shadow of every face */
FS_DIFF_HD int fs_diff_apex(const fs_diff_edge* E, const float s[3], const float l[3], float eps_offset, float p[3])
{
    const float ds[3] = {s[0] - E->a[0], s[1] - E->a[1], s[2] - E->a[2]};
    const float dl[3] = {l[0] - E->a[0], l[1] - E->a[1], l[2] - E->a[2]};
    const float sa = fs_diff_dot(ds, E->d), la = fs_diff_dot(dl, E->d);
    float ps[3], pl[3];
    for (int i = 0; i < 3; ++i) { ps[i] = ds[i] - sa * E->d[i]; pl[i] = dl[i] - la * E->d[i]; }
    const float rs = sqrtf(fs_diff_dot(ps, ps)), rl = sqrtf(fs_diff_dot(pl, pl));
    if (!(rs > eps_offset && rl > eps_offset)) return 0;
    const float x = sa + ((la - sa) * rs) / (rs + rl);
    if (!(x >= 0.0f && x <= E->len)) return 0;
    const float c3 = fs_diff_side(E->d, ps, pl);
    if (!fs_diff_crosses(E->d, ps, pl, E->u1, c3)) return 0;
    if (!(E->k & FS_DIFF_SCREEN) && !fs_diff_crosses(E->d, ps, pl, E->u2, c3)) return 0;
    for (int i = 0; i < 3; ++i) p[i] = E->a[i] + x * E->d[i];
    return 1;
}

/* the leg from q to the apex p: unit direction, tmax (<= 0: nothing to trace); returns |p - q| */
FS_DIFF_HD float fs_diff_leg(const float q[3], const float p[3], float eps_connect, float dir[3], float* tmax)
{
    const float d[3] = {p[0] - q[0], p[1] - q[1], p[2] - q[2]};
    const float len = sqrtf(fs_diff_dot(d, d));
    const float inv = 1.0f / len;
    for (int i = 0; i < 3; ++i) dir[i] = d[i] * inv;
    *tmax = len - eps_connect;
    return len;
}

/* path difference z of a path of this length */
FS_DIFF_HD float fs_diff_z(const float s[3], const float l[3], float length)
{
    const float d[3] = {l[0] - s[0], l[1] - s[1], l[2] - s[2]};
    const float z = length - sqrtf(fs_diff_dot(d, d));
    return z > 0.0f ? z : 0.0f;
}

/* Maekawa's energy attenuation 1 / (3 + 20 N), N = 2 z f / c, limited to 20 dB */
FS_DIFF_HD float fs_diff_gain(float z, float f, float c)
{
    const float g = 1.0f / (3.0f + ((40.0f * z) * f) / c);
    return g > 0.01f ? g : 0.01f;
}

/* centre frequency of band b when the caller gives none: 62.5 2^b Hz (the convention of fs_build_ir_bands) */
FS_DIFF_HD float fs_diff_default_hz(uint32_t b) { return 62.5f * (float)(1u << b); }

#endif
