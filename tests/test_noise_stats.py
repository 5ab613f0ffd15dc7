"""FS_FLAG_NOISE_STATS, host side: the CPU reference of the second moments (fso_trace_sources_m2) keeps the histogram of
fso_trace_sources bit for bit, its per-bin variance predicts the spread of the histogram across seeds, the float64
statistics the GPU is compared against, and the budget allocation fs_allocate_paths (host only, no GPU)."""
import os
import subprocess

import numpy as np
import pytest

import noise_oracle
import sources_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
POS5 = np.array([[1.0, 1.0, 1.0], [6.0, 4.0, 2.0], [3.5, 2.5, 1.5], [0.5, 4.5, 2.5], [5.0, 1.0, 0.5]], np.float32)
N5 = [1, 700, 4096, 33, 2000]
D5 = [0, 1, 8, 3, 16]


def _shoebox(model=False):
    from frequensee import scenes
    sc = scenes.shoebox()
    R = sources_oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=True)
    if model:
        rng = np.random.default_rng(3)
        M, B = sc.absorption.shape
        R.set_material_model(rng.uniform(0, 0.5, (M, B)).astype(np.float32), rng.uniform(0, 1, (M, B)).astype(np.float32),
                             rng.uniform(0.5, 10, M).astype(np.float32))
    return sc, R


def _m2_direct(hist, m2):
    """S2 is 0 exactly where S1 is 0, per band and broadband"""
    s1_bb = hist.astype(object).sum(axis=1)
    for s in range(hist.shape[0]):
        assert ((m2[s, :-1, :, 0] == 0) & (m2[s, :-1, :, 1] == 0) == (hist[s] == 0)).all()
        assert ((m2[s, -1, :, 0] == 0) & (m2[s, -1, :, 1] == 0) == (s1_bb[s] == 0)).all()


@pytest.mark.parametrize("mode", ["uniform", "uniform_share", "sources", "sources_share", "sources_model"])
def test_m2_reference_keeps_the_histogram(oracle, mode):
    flags = oracle.FLAG_SHARE_LISTENER if mode.endswith("share") else oracle.FLAG_MATERIAL_MODEL if mode.endswith("model") else 0
    sc, R = _shoebox(model=mode.endswith("model"))
    cfg = oracle.default_config(flags=flags)
    if mode.startswith("uniform"):
        pos, n, d = POS5[:3], 900, 6
    else:
        pos, n, d = POS5, N5, ([5] * 5 if mode.endswith("share") else D5)
    h0, s0 = R.trace_sources(cfg, pos, n, d, sc.listener, 0x5EED)
    h1, m2, s1 = noise_oracle.trace_sources_m2(R, cfg, pos, n, d, sc.listener, 0x5EED)
    assert np.array_equal(h0, h1)
    assert s0["connected"] == s1["connected"] > 0
    _m2_direct(h1, m2)


def test_m2_of_a_deterministic_path(oracle):
    """depth 0: every pair is the direct path, the same q in one bin: S2 = n q^2 exactly and the variance is 0"""
    sc, R = _shoebox()
    cfg = oracle.default_config()
    h, m2, _ = noise_oracle.trace_sources_m2(R, cfg, POS5[:1], 1000, 0, sc.listener, 1)
    k = int(np.flatnonzero(h[0, 0])[0])
    q = [int(h[0, b, k]) // 1000 for b in range(cfg.n_bands)]
    assert all(int(h[0, b, k]) == 1000 * q[b] for b in range(cfg.n_bands))
    for b in range(cfg.n_bands):
        assert int(m2[0, b, k, 0]) | (int(m2[0, b, k, 1]) << 64) == 1000 * q[b] ** 2
    assert int(m2[0, -1, k, 0]) | (int(m2[0, -1, k, 1]) << 64) == 1000 * sum(q) ** 2
    st = noise_oracle.noise_stats(h, m2, 1000)
    assert st["variance"][0] == 0.0 and st["snr_db"][0] == np.inf and (st["band_variance"][0] == 0).all()


def test_predicted_variance_matches_the_spread_over_seeds(oracle):
    """shoebox, 2^12 pairs, depth 8, 64 seeds.  Per seed r: mu_r[k] and the predicted Var_r[k] of fs_get_noise.  With
    mu_bar the mean over seeds, d_r = R / (R - 1) sum_k (mu_r[k] - mu_bar[k])^2 - sum_k Var_r[k] has mean
    (empirical variance of mu_hat summed over bins) - (mean predicted variance), which is 0 when the prediction is unbiased.
    Bound: |mean d| <= 5 std(d) / sqrt(R), five standard errors of that mean for R = 64 seeds."""
    sc, Rs = _shoebox()
    cfg = oracle.default_config()
    n, R = 1 << 12, 64
    runs = [noise_oracle.trace_sources_m2(Rs, cfg, sc.sources, n, 8, sc.listener, 1000 + seed)[:2] for seed in range(R)]
    for b in (cfg.n_bands, 0):                          # broadband, band 0
        mus, preds = [], []
        for h, m2 in runs:
            s1 = h[0].astype(object).sum(axis=0) if b == cfg.n_bands else h[0, b]
            mu, var = noise_oracle.bin_stats(s1, m2[0, b, :, 0], m2[0, b, :, 1], n)
            mus.append(mu); preds.append(var.sum())
        mus = np.array(mus); preds = np.array(preds)
        d = ((mus - mus.mean(axis=0)) ** 2).sum(axis=1) * R / (R - 1) - preds
        se = d.std(ddof=1) / np.sqrt(R)
        assert preds.mean() > 0
        assert abs(d.mean()) <= 5 * se, (b, d.mean(), se, preds.mean())


def test_float64_statistics_conventions():
    """+inf for variance 0 with signal, -inf and no_energy without signal; broadband is the band sum"""
    S, B, K = 2, 2, 3
    hist = np.zeros((S, B, K), np.uint64)
    m2 = np.zeros((S, B + 1, K, 2), np.uint64)
    # source 0: 4 pairs, band 0 values (1, 1, 3, 0) in bin 1 -> S1 = 5, S2 = 11 (Q32.32 units)
    hist[0, 0, 1] = 5 << 32
    m2[0, 0, 1, 1] = 11            # (11 * 2^64): q in 2^32 units -> q^2 in 2^64 units: hi word
    m2[0, 2, 1, 1] = 11
    st = noise_oracle.noise_stats(hist, m2, [4, 4])
    mu, var = 5 / 4, (11 / 4 - (5 / 4) ** 2) / 3
    assert np.isclose(st["band_signal"][0, 0], mu * mu, rtol=1e-15)
    assert np.isclose(st["band_variance"][0, 0], var, rtol=1e-15)
    assert np.isclose(st["snr_db"][0], 10 * np.log10(mu * mu / var), rtol=1e-15)
    assert st["band_snr_db"][0, 1] == -np.inf and not st["no_energy"][0]
    assert st["no_energy"][1] and st["snr_db"][1] == -np.inf


# ---- fs_allocate_paths ---------------------------------------------------------------------------------------------------
def _stats(n, sig, var, no_energy=None):
    S = len(n)
    return {"n_paths": np.asarray(n, np.uint64), "signal": np.asarray(sig, float), "variance": np.asarray(var, float),
            "no_energy": np.zeros(S, bool) if no_energy is None else np.asarray(no_energy, bool)}


def test_allocate_sum_and_clamps(fs):
    rng = np.random.default_rng(5)
    for trial in range(50):
        S = int(rng.integers(1, 40))
        st = _stats(rng.integers(1, 1 << 16, S), rng.uniform(0.1, 10, S), rng.uniform(1e-6, 1.0, S) ** 3)
        lo, hi = int(rng.integers(1, 1000)), 0
        hi = lo + int(rng.integers(0, 1 << 16))
        total = int(rng.integers(S * lo, S * hi + 1))
        w = rng.uniform(0, 3, S) if trial % 2 else None
        n = fs.allocate_paths(st, total, lo, hi, w)
        assert n.dtype == np.uint64 and int(n.sum()) == total
        assert (n >= lo).all() and (n <= hi).all()


def test_allocate_equal_demand_is_an_equal_split(fs):
    st = _stats([1000] * 8, [2.0] * 8, [0.5] * 8)
    assert (fs.allocate_paths(st, 8000, 1, 10 ** 6) == 1000).all()
    n = fs.allocate_paths(st, 8003, 1, 10 ** 6, [1.5] * 8)
    assert int(n.sum()) == 8003 and n.max() - n.min() <= 1


def test_allocate_equalises_predicted_noise(fs):
    """n_s ~ w_s a_s: unclamped sources end with equal w_s a_s / n_s, the predicted variance-to-signal ratio after the
    update scaled by the weight (a source of weight 2 is given twice its share of the SNR)"""
    rng = np.random.default_rng(9)
    S = 16
    n0 = rng.integers(1 << 10, 1 << 14, S)
    sig = rng.uniform(0.5, 2, S)
    var = rng.uniform(1e-4, 1e-2, S)
    w = rng.uniform(0.5, 2, S)
    lo, hi, total = 256, 1 << 16, int(n0.sum())
    n = fs.allocate_paths(_stats(n0, sig, var), total, lo, hi, w)
    a = n0 * var / sig
    free = (n > lo) & (n < hi)
    assert free.sum() >= S // 2
    r = w[free] * a[free] / n[free]
    # rounding moves n_s by < 1 path: relative spread <= 1 / min n_s (x2 for both ends)
    assert (r.max() - r.min()) / r.mean() <= 2.0 / n[free].min() + 1e-12


def test_allocate_clamped_sources(fs):
    st = _stats([1000, 1000, 1000], [1.0, 1.0, 1.0], [1.0, 1e-6, 1e-6])
    n = fs.allocate_paths(st, 3000, 100, 2000)
    assert list(n) == [2000, 500, 500]
    st = _stats([1000, 1000, 1000], [1.0, 1.0, 1.0], [0.0, 1e-6, 1e-6])      # noise-free source: min
    assert fs.allocate_paths(st, 3000, 100, 2000)[0] == 100


def test_allocate_no_energy_keeps_its_budget(fs):
    st = _stats([700, 1000, 1000, 1000], [0.0, 1.0, 1.0, 2.0], [0.0, 0.1, 0.2, 0.1], no_energy=[1, 0, 0, 0])
    n = fs.allocate_paths(st, 4000, 100, 5000)
    assert n[0] == 700 and int(n.sum()) == 4000
    assert fs.allocate_paths(st, 4000, 800, 5000)[0] == 800                    # kept count clamped
    # only no-energy sources: every one keeps its count when that is feasible; otherwise all split equally
    st2 = _stats([1000, 3000], [0, 0], [0, 0], no_energy=[1, 1])
    assert list(fs.allocate_paths(st2, 4000, 1, 10 ** 6)) == [1000, 3000]
    assert list(fs.allocate_paths(st2, 5000, 1, 10 ** 6)) == [2500, 2500]


def test_allocate_invalid_arguments(fs):
    st = _stats([1000, 1000], [1.0, 1.0], [0.1, 0.1])
    for args, w in [((2000, 0, 1000), None),           # min == 0
                    ((2000, 1001, 1000), None),        # min > max
                    ((100, 51, 1000), None),           # S min > total
                    ((3000, 1, 1000), None),           # S max < total
                    ((2000, 1, 1000), [1.0, -1.0]),    # negative weight
                    ((2000, 1, 1000), [1.0, np.nan]),
                    ((2000, 1, 1000), [np.inf, 1.0])]:
        with pytest.raises(fs.FrequenSeeError) as ei:
            fs.allocate_paths(st, *args, weight=w)
        assert ei.value.code == fs.capi.FS_ERR_INVALID
    L = fs.capi.load()
    out = np.zeros(1, np.uint64)
    assert L.fs_allocate_paths(fs.capi.noise_stats_array(st), 0, 10, 1, 100, None, out.ctypes.data) == fs.capi.FS_ERR_INVALID
    assert L.fs_allocate_paths(None, 2, 10, 1, 100, None, out.ctypes.data) == fs.capi.FS_ERR_INVALID


def test_noise_stats_struct_layout(fs):
    import ctypes as C
    assert C.sizeof(fs.capi.NoiseStats) == 232 and fs.capi.NoiseStats.signal.offset == 16


def build_noise_smoke(out_dir):
    exe = os.path.join(str(out_dir), "noise_smoke")
    libdir = os.path.join(ROOT, "audio-pathtracer_b200", "lib")
    env = dict(os.environ); env.pop("CC", None); env.pop("CXX", None)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "noise_smoke.cpp"), "-o", exe,
                           "-L", libdir, "-lfrequensee", "-Wl,-rpath," + libdir], env=env)
    return exe


def test_noise_smoke_compiles_and_fails_loudly_without_gpu(fs, tmp_path):
    """the mirror's automatic budgets (TotalRaysPerTick, NoiseWeight, LastNoise) build from plain C++"""
    import torch
    exe = build_noise_smoke(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([exe, "nogpu"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CPU fallback" in r.stdout


def test_allocate_extreme_demands(fs):
    """a source whose a_s overflows (signal far below its variance) is the noisiest there is: it is served first, up to
    max; a denormal weight is a tiny but positive demand and does not break the split"""
    st = _stats([1000, 1000, 1000], [1e-320, 1.0, 1.0], [1.0, 0.1, 0.1])
    n = fs.allocate_paths(st, 3000, 100, 2000)
    assert list(n) == [2000, 500, 500]
    st = _stats([1000, 1000, 1000], [1.0, 1.0, 1.0], [0.1, 0.1, 0.1])
    n = fs.allocate_paths(st, 3000, 100, 2000, [1e-40, 1.0, 1.0])
    assert int(n.sum()) == 3000 and n[0] == 100 and list(n[1:]) == [1450, 1450]
    n = fs.allocate_paths(st, 3000, 100, 2000, [1e-40, 1e-40, 1e-45])
    assert int(n.sum()) == 3000 and n[2] == 100 and n[0] == n[1] == 1450
