"""CPU reference of FS_FLAG_NOISE_STATS: fso_trace_sources_m2 (tests/oracle_ext/fso_noise.c, the pair loop of
fso_trace_sources with the exact second moment of every pair's contribution), compiled together with the oracle into a
temporary directory on first use, and the float64 statistics fs_get_noise computes from (S1, S2, n)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import pyoracle
import sources_oracle

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="fso_noise_"), "libfso_noise.so")
        cmd = ["gcc", "-O2", "-std=gnu99", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-fPIC", "-w", "-shared",
               "-o", out, os.path.join(HERE, "oracle_ext", "fso_noise.c"), "-lm"]
        if pyoracle._has_fma():
            cmd.insert(1, "-mfma")
        subprocess.check_call(cmd)
        L = C.CDLL(out)
        L.fso_trace_sources_m2.restype = C.c_int
        L.fso_trace_sources_m2.argtypes = [C.c_void_p, C.POINTER(pyoracle.Config), C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                           C.POINTER(pyoracle.Stats)]
        _lib = L
    return _lib


def trace_sources_m2(scene, cfg, src_pos, n_paths, depths, lis_pos, seed):
    """scene: a sources_oracle.Scene (its handle is an fso_scene of the same oracle source).  Returns (hist [S][B][K],
    m2 [S][B+1][K][2] (lo, hi), stats)"""
    src = np.ascontiguousarray(src_pos, dtype=np.float32).reshape(-1, 3)
    S = len(src)
    n = np.ascontiguousarray(np.broadcast_to(np.asarray(n_paths, np.uint64), (S,)))
    d = np.ascontiguousarray(np.broadcast_to(np.asarray(depths, np.uint32), (S,)))
    lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
    hist = np.zeros((S, cfg.n_bands, cfg.n_bins), dtype=np.uint64)
    m2 = np.zeros((S, cfg.n_bands + 1, cfg.n_bins, 2), dtype=np.uint64)
    st = pyoracle.Stats()
    rc = lib().fso_trace_sources_m2(scene.h, C.byref(cfg), src.ctypes.data, n.ctypes.data, d.ctypes.data, S,
                                    lis.ctypes.data, seed, hist.ctypes.data, m2.ctypes.data, C.byref(st))
    if rc != 0:
        raise RuntimeError("fso_trace_sources_m2 failed: %d" % rc)
    return hist, m2, st.as_dict()


def bin_stats(s1, s2_lo, s2_hi, n):
    """per-bin (mu, Var(mu_hat)) in energy units, float64, from S1 (Q32.32 sums), S2 (lo, hi) and the pair count n; the
    numerator n S2 - S1^2 is formed exactly (Python integers)"""
    s1 = [int(v) for v in np.asarray(s1).ravel()]
    s2 = [int(lo) | (int(hi) << 64) for lo, hi in zip(np.asarray(s2_lo).ravel(), np.asarray(s2_hi).ravel())]
    den = float(n) * float(n) * float(max(n - 1, 1))
    mu = np.array([v * 2.0 ** -32 / float(n) for v in s1])
    var = np.array([max(n * b - a * a, 0) * 2.0 ** -64 / den for a, b in zip(s1, s2)])
    return mu, var


def _snr_db(sig, var):
    if not sig > 0:
        return -np.inf
    if not var > 0:
        return np.inf
    return 10.0 * np.log10(sig / var)


def noise_stats(hist, m2, n_paths):
    """the float64 statistics of fs_get_noise: dict of arrays like frequensee.Context.noise_stats()"""
    S, B, K = hist.shape
    n = np.broadcast_to(np.asarray(n_paths, np.uint64), (S,))
    out = {k: [] for k in ("signal", "variance", "snr_db", "band_signal", "band_variance", "band_snr_db", "no_energy")}
    for s in range(S):
        bs, bv = [], []
        for b in range(B + 1):
            s1 = hist[s, b] if b < B else np.sum(hist[s].astype(object), axis=0)
            mu, var = bin_stats(s1, m2[s, b, :, 0], m2[s, b, :, 1], int(n[s]))
            bs.append(float(np.sum(mu * mu))); bv.append(float(np.sum(var)))
        out["band_signal"].append(bs[:B]); out["band_variance"].append(bv[:B])
        out["band_snr_db"].append([_snr_db(a, v) for a, v in zip(bs[:B], bv[:B])])
        out["signal"].append(bs[B]); out["variance"].append(bv[B]); out["snr_db"].append(_snr_db(bs[B], bv[B]))
        out["no_energy"].append(not bs[B] > 0)
    r = {k: np.array(v) for k, v in out.items()}
    r["n_paths"] = np.array(n, np.uint64)
    return r


Scene = sources_oracle.Scene
