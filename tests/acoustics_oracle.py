"""float64 / Python-int reference of fs_get_acoustic_params (include/frequensee.h): the Schroeder decay curve of every
(source, band or broadband) slot of an energy histogram, its EDT / T20 / T30 fits, C50 / C80 / D50 and the centre time.

Energies are Python ints, so every sum is exact.  The thresholds C_x are read from csrc/fs_acoustics.h, and the finishing
formulas repeat that header's operations in the same order (fit levels relative to the first fit point, from the exact
integer drop, as fs_ap_fit_level); the fit sums are taken with math.fsum (correctly rounded),
the device reduces them in a fixed tree, so the two agree to a few ulps."""
import math
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "audio-pathtracer_b200", "csrc", "fs_acoustics.h")
EDT, T20, T30, C50, C80, TS = 1, 2, 4, 8, 16, 32
NO_ONSET = 0xFFFFFFFF
FITS = ("edt", "t20", "t30")
MASK64 = (1 << 64) - 1


def constants():
    """{'0': C_0dB, '-5': ..., '-10': ..., '-25': ..., '-35': ...} from the FS_AP_C_* hex-float literals of the header"""
    src = open(HEADER).read()
    out = {}
    for name, lit in re.findall(r"#define\s+FS_AP_C_(M?\d+)DB\s+(0x[0-9a-fA-Fp.+-]+)", src):
        out[name.replace("M", "-")] = float.fromhex(lit)
    return out


_C = constants()
DB_PER_NEPER = float.fromhex(re.search(r"#define\s+FS_AP_DB_PER_NEPER\s+(0x[0-9a-fA-Fp.+-]+)", open(HEADER).read()).group(1))
RANGES = ((_C["0"], _C["-10"]), (_C["-5"], _C["-25"]), (_C["-5"], _C["-35"]))   # (C_hi, C_lo) of EDT, T20, T30


def to_double(x):
    """an exact non-negative integer below 2^128 as (double)hi 2^64 + (double)lo"""
    x = int(x)
    return float(x >> 64) * 18446744073709551616.0 + float(x & MASK64)


def window(ms, bin_ms):
    return int(ms / float(np.float32(bin_ms)) + 0.5)


def _fit(ka, n, reached, sw, sl, sll, delta):
    f = {"time_s": math.nan, "r": math.nan, "first_bin": ka, "n_points": n}
    if not reached or n < 3:
        return f, False
    dn = float(n)
    q = dn * (dn * dn - 1.0)
    m = 6.0 * sw / (delta * q)
    if not (m < 0.0):
        return f, False
    sll_c = sll - sl * sl / dn
    f["time_s"] = -60.0 / m
    f["r"] = sw / math.sqrt(q / 3.0 * sll_c)
    return f, True


def slot(E, bin_ms):
    """the record of one slot from its bin energies E (K non-negative ints) and the EDC (float32 [K])"""
    E = np.asarray([int(v) for v in E], dtype=object)
    K = len(E)
    delta = float(np.float32(bin_ms)) * 1e-3
    n50, n80 = window(50.0, bin_ms), window(80.0, bin_ms)
    rec = {"onset_bin": NO_ONSET, "valid": 0, "c50_db": math.nan, "c80_db": math.nan, "d50": math.nan, "ts_s": math.nan}
    nz = np.flatnonzero(E != 0)
    if len(nz) == 0:
        for name in FITS:
            rec[name] = {"time_s": math.nan, "r": math.nan, "first_bin": 0, "n_points": 0}
        return rec, np.full(K, np.nan, np.float32)
    k0 = int(nz[0])
    R = np.cumsum(E[::-1])[::-1]
    S0 = int(R[0])
    Rd = (R >> 64).astype(np.float64) * 18446744073709551616.0 + (R & MASK64).astype(np.float64)
    s0d = to_double(S0)
    with np.errstate(divide="ignore"):
        L = np.where(Rd > 0.0, 10.0 * np.log10(Rd / s0d), -np.inf)
    last = to_double(E[K - 1])
    for i, (chi, clo) in enumerate(RANGES):
        a = np.flatnonzero(Rd[k0:] <= s0d * chi)
        ka = k0 + int(a[0]) if len(a) else K
        b = np.flatnonzero(Rd[:K - 1] >= s0d * clo)
        kb = int(b[-1]) if len(b) else -1
        n = kb - ka + 1 if kb >= ka else 0
        k = np.arange(ka, ka + n)
        # levels relative to the first point from the exact drop, as fs_ap_fit_level: L_k - L_ka
        drop = int(R[ka]) - R[ka:ka + n] if n else np.zeros(0, dtype=object)
        dd = (drop >> 64).astype(np.float64) * 18446744073709551616.0 + (drop & MASK64).astype(np.float64)
        Lk = DB_PER_NEPER * np.log1p(-dd / to_double(R[ka])) if n else np.zeros(0)
        w = (2 * k - ka - kb).astype(np.float64)
        f, ok = _fit(ka, n, last < s0d * clo, math.fsum(w * Lk), math.fsum(Lk), math.fsum(Lk * Lk), delta)
        rec[FITS[i]] = f
        rec["valid"] |= (1 << i) if ok else 0
    for nw, key, bit in ((n50, "c50_db", C50), (n80, "c80_db", C80)):
        if nw < 1 or k0 + nw > K - 1:
            continue
        early = int(sum(E[k0:k0 + nw]))
        e, late = to_double(early), to_double(S0 - early)
        rec[key] = 10.0 * math.log10(e / late) if late > 0.0 else math.inf
        if bit == C50:
            rec["d50"] = e / s0d
        rec["valid"] |= bit
    if int(E[K - 1]) == 0:
        num = sum((int(k) - k0) * int(E[k]) for k in nz)
        rec["ts_s"] = delta * (to_double(num) / s0d)
        rec["valid"] |= TS
    rec["onset_bin"] = k0
    edc = L.astype(np.float32)
    edc[:k0] = 0.0
    return rec, edc


def acoustic_params(hist, bin_ms):
    """hist uint64 [S][B][K] -> (list of S dicts {no_energy, broadband, band: [B]}, EDC float32 [S][B+1][K])"""
    hist = np.asarray(hist, dtype=np.uint64)
    S, B, K = hist.shape
    out, edc = [], np.zeros((S, B + 1, K), np.float32)
    for s in range(S):
        rows = [[int(v) for v in hist[s, b]] for b in range(B)]
        bands = []
        for b in range(B):
            r, edc[s, b] = slot(rows[b], bin_ms)
            bands.append(r)
        bb, edc[s, B] = slot([sum(col) for col in zip(*rows)], bin_ms)
        out.append({"no_energy": int(bb["onset_bin"] == NO_ONSET), "broadband": bb, "band": bands})
    return out, edc


def from_ctypes(arr, n_bands):
    """the same dict layout from fs.capi.AcousticParams[S]"""
    def sl(a):
        d = {"onset_bin": a.onset_bin, "valid": a.valid, "c50_db": a.c50_db, "c80_db": a.c80_db, "d50": a.d50, "ts_s": a.ts_s}
        for name in FITS:
            f = getattr(a, name)
            d[name] = {"time_s": f.time_s, "r": f.r, "first_bin": f.first_bin, "n_points": f.n_points}
        return d
    return [{"no_energy": p.no_energy, "broadband": sl(p.broadband), "band": [sl(p.band[b]) for b in range(n_bands)]}
            for p in arr]


def _close(a, b, rtol=1e-12, atol=1e-9):
    if math.isnan(a) or math.isnan(b):
        return math.isnan(a) and math.isnan(b)
    if math.isinf(a) or math.isinf(b):
        return a == b
    return abs(a - b) <= max(atol, rtol * max(abs(a), abs(b)))


def compare(got, ref):
    """[] when every integer field is equal and every double within 1e-12 relative or 1e-9 absolute; else the differences"""
    bad = []

    def cmp_slot(g, r, where):
        for k in ("onset_bin", "valid"):
            if g[k] != r[k]:
                bad.append((where, k, g[k], r[k]))
        for k in ("c50_db", "c80_db", "d50", "ts_s"):
            if not _close(g[k], r[k]):
                bad.append((where, k, g[k], r[k]))
        for name in FITS:
            for k in ("first_bin", "n_points"):
                if g[name][k] != r[name][k]:
                    bad.append((where, name + "." + k, g[name][k], r[name][k]))
            for k in ("time_s", "r"):
                if not _close(g[name][k], r[name][k]):
                    bad.append((where, name + "." + k, g[name][k], r[name][k]))

    if len(got) != len(ref):
        return [("sources", len(got), len(ref))]
    for s, (g, r) in enumerate(zip(got, ref)):
        if g["no_energy"] != r["no_energy"]:
            bad.append((s, "no_energy", g["no_energy"], r["no_energy"]))
        cmp_slot(g["broadband"], r["broadband"], (s, "bb"))
        for b, (gb, rb) in enumerate(zip(g["band"], r["band"])):
            cmp_slot(gb, rb, (s, b))
    return bad


def edc_ulps(a, b):
    """largest distance in float32 ulps between two EDC arrays (NaN == NaN, inf == inf; 0 when identical)"""
    a = np.ascontiguousarray(a, np.float32).ravel()
    b = np.ascontiguousarray(b, np.float32).ravel()
    same = (a == b) | (np.isnan(a) & np.isnan(b))
    if same.all():
        return 0
    ia, ib = a.view(np.int32).astype(np.int64), b.view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    d = np.abs(ia - ib)
    d[same] = 0
    fin = np.isfinite(a) & np.isfinite(b)
    if not fin[~same].all():
        return 1 << 40
    return int(d.max())
