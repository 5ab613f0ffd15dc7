/* fs_acoustics.h -- the per-slot finishing arithmetic of fs_get_acoustic_params, written once for k_acoustics (fs_acoustics.cu).
 * tests/acoustics_oracle.py reads the FS_AP_C_* constants from this file and repeats the formulas below in the same order.
 *
 * A slot is one band of one source, or its broadband sum.  The kernel hands over exact integer sums (128 bits, as (hi, lo))
 * and the fixed-order double sums of the three decay fits; everything after that is here.  Thresholds are compared
 * without a logarithm: point k is at or below x dB iff (double)R_k <= (double)S0 * C_x, with C_x the double nearest
 * 10^(x / 10). */
#ifndef FS_ACOUSTICS_H
#define FS_ACOUSTICS_H

#include <math.h>
#include <stdint.h>

#include "../../include/frequensee.h"

#define FS_AP_C_0DB   0x1.0000000000000p+0     /* 10^(0/10) */
#define FS_AP_C_M5DB  0x1.43d136248490fp-2     /* 10^(-5/10) */
#define FS_AP_C_M10DB 0x1.999999999999ap-4     /* 10^(-10/10) */
#define FS_AP_C_M25DB 0x1.9e7c6e43390b7p-9     /* 10^(-25/10) */
#define FS_AP_C_M35DB 0x1.4b96be9c2da2cp-12    /* 10^(-35/10) */
#define FS_AP_DB_PER_NEPER 0x1.15f2ced384f29p+2   /* 10 / ln 10 */
#define FS_AP_NO_ONSET 0xffffffffu
#define FS_AP_FITS 3                            /* EDT, T20, T30 */

#if defined(__CUDACC__)
#define FS_AP_HD __host__ __device__ __forceinline__
#else
#define FS_AP_HD static inline
#endif

/* the [hi, lo] range of fit i as (C_hi, C_lo) */
FS_AP_HD double fs_ap_c_hi(int i) { return i == 0 ? FS_AP_C_0DB : FS_AP_C_M5DB; }
FS_AP_HD double fs_ap_c_lo(int i) { return i == 0 ? FS_AP_C_M10DB : i == 1 ? FS_AP_C_M25DB : FS_AP_C_M35DB; }

/* an exact 128-bit sum as a double, the conversion of fs_noise.cu */
FS_AP_HD double fs_ap_u128(uint64_t hi, uint64_t lo) { return (double)hi * 0x1p64 + (double)lo; }

/* bins of a 50 / 80 ms window: nearest to ms / bin_ms */
FS_AP_HD uint32_t fs_ap_window(double ms, float bin_ms) { return (uint32_t)(ms / (double)bin_ms + 0.5); }

/* decay-curve level of a bin in dB: 10 log10(R / S0), -inf for R = 0 (S0 > 0) */
FS_AP_HD double fs_ap_level_db(double r, double s0) { return r > 0.0 ? 10.0 * log10(r / s0) : -INFINITY; }

/* level of fit point k relative to the fit's first point ka: L_k - L_ka = 10 log10(R_k / R_ka), evaluated as
 * 10 / ln 10 log1p(-(R_ka - R_k) / R_ka) from the exact integer drop.  The fits are taken on these values: the same points
 * shifted by a constant, so slope and r are those of L_k, but a nearly flat stretch of the curve keeps its digits (and
 * sum L^2 - (sum L)^2 / n does not cancel them away). */
FS_AP_HD double fs_ap_fit_level(double drop, double r_first) { return FS_AP_DB_PER_NEPER * log1p(-drop / r_first); }

/* one fit over points ka .. ka + n - 1: sw = sum w_k L_k with w_k = 2k - ka - kb, sl = sum L_k, sll = sum L_k^2 (L_k from
 * fs_ap_fit_level).
 * reached: the curve fell below the range's lower end before the overflow bin.  Returns 1 when the fit is valid. */
FS_AP_HD int fs_ap_fit(uint32_t ka, uint32_t n, int reached, double sw, double sl, double sll, double delta, fs_decay_fit* f)
{
    f->first_bin = ka;
    f->n_points = n;
    f->time_s = NAN;
    f->r = NAN;
    if (!reached || n < 3u) return 0;
    const double dn = (double)n, q = dn * (dn * dn - 1.0);
    const double m = 6.0 * sw / (delta * q);                 /* dB/s */
    if (!(m < 0.0)) return 0;
    const double sll_c = sll - sl * sl / dn;                  /* sum (L - mean L)^2 */
    f->time_s = -60.0 / m;
    f->r = sw / sqrt(q / 3.0 * sll_c);                         /* S_tL / sqrt(S_tt S_LL); delta cancels */
    return 1;
}

/* the integer inputs of one slot (128-bit values as hi, lo) */
typedef struct fs_ap_sums {
    uint32_t k0, n_bins;                       /* onset (FS_AP_NO_ONSET: no energy), K */
    uint32_t ka[FS_AP_FITS];                   /* first fit point (n_bins: none) */
    int32_t  kb[FS_AP_FITS];                   /* last fit point (-1: none) */
    uint32_t n50, n80;
    uint64_t s0_hi, s0_lo;                     /* sum of all bins */
    uint64_t last_hi, last_lo;                 /* the overflow bin K-1 */
    uint64_t e50_hi, e50_lo, e80_hi, e80_lo;   /* sum of bins k0 .. k0 + nX - 1 */
    uint64_t ts_hi, ts_lo;                     /* sum of (k - k0) E_k */
    double   fit[FS_AP_FITS][3];               /* sw, sl, sll of each fit */
} fs_ap_sums;

/* the record of one slot */
FS_AP_HD void fs_ap_finish(const fs_ap_sums* a, double delta, fs_acoustic_slot* o)
{
    uint32_t valid = 0u;
    const int energy = a->k0 != FS_AP_NO_ONSET;
    const uint32_t K = a->n_bins;
    const double s0 = fs_ap_u128(a->s0_hi, a->s0_lo), last = fs_ap_u128(a->last_hi, a->last_lo);
    fs_decay_fit* fits[FS_AP_FITS] = {&o->edt, &o->t20, &o->t30};
    for (int i = 0; i < FS_AP_FITS; ++i) {
        const uint32_t n = (energy && a->kb[i] >= 0 && (uint32_t)a->kb[i] >= a->ka[i]) ? (uint32_t)a->kb[i] - a->ka[i] + 1u : 0u;
        const int reached = energy && last < s0 * fs_ap_c_lo(i);
        if (fs_ap_fit(energy ? a->ka[i] : 0u, n, reached, a->fit[i][0], a->fit[i][1], a->fit[i][2], delta, fits[i])) valid |= FS_AP_EDT << i;
    }
    o->c50_db = o->c80_db = o->d50 = o->ts_s = NAN;
    if (energy) {
        const uint32_t nw[2] = {a->n50, a->n80};
        const uint64_t ehi[2] = {a->e50_hi, a->e80_hi}, elo[2] = {a->e50_lo, a->e80_lo};
        for (int w = 0; w < 2; ++w) {
            if (nw[w] < 1u || (uint64_t)a->k0 + nw[w] > (uint64_t)K - 1u) continue;
            const uint64_t lhi = a->s0_hi - ehi[w] - (a->s0_lo < elo[w] ? 1u : 0u), llo = a->s0_lo - elo[w];
            const double early = fs_ap_u128(ehi[w], elo[w]), late = fs_ap_u128(lhi, llo);
            const double c = late > 0.0 ? 10.0 * log10(early / late) : INFINITY;
            if (w == 0) { o->c50_db = c; o->d50 = early / s0; valid |= FS_AP_C50; }
            else        { o->c80_db = c; valid |= FS_AP_C80; }
        }
        if (!(a->last_hi | a->last_lo)) { o->ts_s = delta * (fs_ap_u128(a->ts_hi, a->ts_lo) / s0); valid |= FS_AP_TS; }
    }
    o->onset_bin = a->k0;
    o->valid = valid;
}

#endif
