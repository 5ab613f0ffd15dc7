"""Directional sources, host side: the CPU reference (tests/oracle_ext/fso_directivity.c) reproduces fso_trace /
fso_trace_sources bit for bit with constant-1 patterns in every connection mode; a depth-0 known answer at three facings;
a pattern that is zero behind the source leaves no backwards emission; fs_directivity_polar against float64; the struct
layouts; the C++ mirror's smoke program compiles and fails loudly without a GPU."""
import ctypes as C
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import directivity_oracle
import sources_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
POS3 = np.array([[1.0, 1.0, 1.0], [6.0, 4.0, 2.0], [3.5, 2.5, 1.5]], np.float32)
MODES = {"default": 0, "share_listener": 128, "connect_all": 64, "mis": 512, "material_model": 256}


def _scene(oracle, model=False):
    from frequensee import scenes
    sc = scenes.shoebox()
    S = oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=True)
    R = sources_oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=True)
    D = directivity_oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=True)
    if model:
        rng = np.random.default_rng(3)
        M, B = sc.absorption.shape
        mm = (rng.uniform(0, 0.5, (M, B)).astype(np.float32), rng.uniform(0, 1, (M, B)).astype(np.float32),
              rng.uniform(0.5, 10, M).astype(np.float32))
        for x in (S, R, D):
            x.set_material_model(*mm)
    return sc, S, R, D


def _f32(fr):
    """the binary32 nearest to the exact rational fr (ties to even): what one fmaf rounds to"""
    f = np.float32(float(fr))
    best = f
    for c in (np.nextafter(f, np.float32(-np.inf)), np.nextafter(f, np.float32(np.inf))):
        dc, db = abs(Fraction(float(c)) - fr), abs(Fraction(float(best)) - fr)
        if dc < db or (dc == db and (int(c.view(np.uint32)) & 1) == 0):
            best = c
    return best


def gain_by_hand(table, c):
    """g = T[i] + t (T[i+1] - T[i]) for the float32 cosine c, formed as fs_directivity.h does (one fmaf)"""
    x = (np.float32(c) + np.float32(1.0)) * np.float32(16.0)
    i = min(int(np.floor(x)), 31)
    t = np.float32(x - np.float32(i))
    t0, t1 = np.float32(table[i]), np.float32(table[i + 1])
    return _f32(Fraction(float(t)) * Fraction(float(np.float32(t1 - t0))) + Fraction(float(t0)))


@pytest.mark.parametrize("mode", list(MODES))
def test_constant_one_patterns_reproduce_fso_trace(oracle, mode):
    """uniform budgets: the same bytes as fso_trace; per-source budgets (mixed depths, a depth-0 source): as
    fso_trace_sources -- with a constant-1 pattern on some sources and FS_OMNI on the others"""
    sc, S, R, D = _scene(oracle, model=(mode == "material_model"))
    cfg = oracle.default_config(flags=MODES[mode])
    ones = np.ones((2, 8, 33), np.float32)
    fwd = [[1, 0, 0], [0, -3, 1], [0.2, 0.1, -5]]
    h0, s0 = S.trace(cfg, POS3, sc.listener, 700, 6, 0x5EED)
    h1, s1 = D.trace_sources_dir(cfg, POS3, 700, 6, sc.listener, 0x5EED, ones, fwd, [0, 1, directivity_oracle.OMNI])
    assert np.array_equal(h0, h1) and h0.any()
    assert s0["connected"] == s1["connected"] and s0["shadow_rays"] == s1["shadow_rays"]
    if mode == "share_listener":
        depths = [6, 6, 6]
    else:
        depths = [0, 3, 8]
    n = [1, 500, 900]
    h2, _ = R.trace_sources(cfg, POS3, n, depths, sc.listener, 77)
    h3, _ = D.trace_sources_dir(cfg, POS3, n, depths, sc.listener, 77, ones, fwd, [1, 0, 0])
    assert np.array_equal(h2, h3) and h2[2].any()


@pytest.mark.parametrize("facing,forward", [("towards", [1, 0, 0]), ("away", [-1, 0, 0]), ("sideways", [0, 1, 0]),
                                            ("oblique", [1, 1, 0])])
def test_depth0_known_answer(oracle, facing, forward):
    """max_depth = 0: every pair is the direct pair along +x, so each bin holds n q with
    q = trunc(min(E, clamp) gain 2^32) and E = g 1/(4 pi d^2) exp(-air_b d) / 1^pdf_exponent, g interpolated by hand"""
    sc, S, R, D = _scene(oracle)
    L = oracle.lib()
    cfg = oracle.default_config()
    src = np.array([[1.0, 2.5, 1.5]], np.float32)
    lis = np.array([6.0, 2.5, 1.5], np.float32)
    rng = np.random.default_rng(11)
    table = rng.uniform(0.0, 3.0, (8, 33)).astype(np.float32)
    n = 37
    h, st = D.trace_sources_dir(cfg, src, n, 0, lis, 5, table, [forward], [0])
    assert st["connected"] == n
    f = np.array(forward, np.float64)
    f = (f / np.sqrt(f[0] * f[0] + f[1] * f[1] + f[2] * f[2])).astype(np.float32)
    dl = lis - src[0]
    d = np.float32(5.0)
    dirv = dl * (np.float32(1.0) / d)
    assert np.array_equal(dirv, np.array([1, 0, 0], np.float32))
    c = np.float32(min(max(float(f[0]), -1.0), 1.0))          # the dot with (1, 0, 0) is exact: f.x
    G = np.float32(1.0) / (np.float32(12.5663709640502930) * (d * d))
    P = np.float32(L.fso_powf(1.0, cfg.pdf_exponent))
    b_idx = oracle.bin_index(cfg, np.float32(d / np.float32(cfg.sound_speed)))
    for b in range(cfg.n_bands):
        g = gain_by_hand(table[b], c)
        e = np.float32(g * np.float32(1.0))
        e = np.float32(e * G)
        e = np.float32(e * np.float32(L.fso_expf(np.float32(-np.float32(cfg.air_absorption[b]) * d))))
        e = np.float32(e / P)
        e = np.float32(min(e, np.float32(cfg.energy_clamp)) * np.float32(cfg.energy_gain))
        q = int(np.float32(e * np.float32(4294967296.0)))
        expect = np.zeros(cfg.n_bins, np.uint64)
        expect[b_idx] = n * q
        assert np.array_equal(h[0, b], expect), (facing, b)
    if facing == "away":
        assert all(gain_by_hand(table[b], -1.0) == table[b][0] for b in range(8))


def test_backward_zero_pattern_leaves_no_backward_path(oracle):
    """a pattern that is 0 for c <= 0: no connected path of the source leaves it backwards.  The emission direction of
    each pair is taken from the oracle's own node lists (first segment of the source subpath, or the connection)"""
    sc, S, R, D = _scene(oracle)
    cfg = oracle.default_config()
    table = np.zeros((8, 33), np.float32)
    table[:, 17:] = np.linspace(0.2, 2.0, 16, dtype=np.float32)
    fwd = np.array([0.3, -1.0, 0.2], np.float64)
    fhat = fwd / np.linalg.norm(fwd)
    src, n, depth = POS3[2], 1500, 5
    h, st, dbg = D.trace_sources_dir(cfg, src[None], n, depth, sc.listener, 9, table, [fwd], [0], want_dbg=True)
    h_omni, _, dbg_omni = D.trace_sources_dir(cfg, src[None], n, depth, sc.listener, 9, table, [fwd],
                                              [directivity_oracle.OMNI], want_dbg=True)
    back = front = 0
    for g in range(n):
        if not dbg_omni[g]["connected"]:
            assert not dbg[g]["connected"]
            continue
        F, B = S.debug_path(cfg, src, sc.listener, g, n, depth, 9)
        d = (F["p"][1] - F["p"][0]) if len(F["p"]) >= 2 else (B["p"][-1] - F["p"][0])
        c = float(np.dot(d, fhat) / np.linalg.norm(d))
        if c < -1e-3:
            back += 1
            assert not np.any(dbg[g]["energy"]), g
        elif c > 0.1:
            front += 1
            assert np.all(dbg[g]["energy"][:cfg.n_bands] > 0), g
    assert back > 100 and front > 100
    assert h.sum() < h_omni.sum()


def test_directivity_polar_matches_float64(fs):
    w = np.array([0.0, 0.5, 1.0, 0.25, 0.75, 0.5, 0.1, 1.0], np.float32)
    p = np.array([1.0, 1.0, 2.0, 0.0, 3.5, 64.0, 0.5, 1.0], np.float32)
    out = fs.directivity_polar(w, p)
    assert out.shape == (8, 33) and out.dtype == np.float32
    c = -1.0 + np.arange(33) / 16.0
    for b in range(8):
        ref = np.abs((1.0 - float(w[b])) + float(w[b]) * c) ** float(p[b])
        assert np.array_equal(out[b], ref.astype(np.float32)), b
    assert np.all(out[0] == 1.0) and out[1][0] == 0.0 and out[1][32] == 1.0 and out[2][16] == 0.0
    assert fs.directivity_polar([0.5, 0.5], 1.0).shape == (2, 33)


@pytest.mark.parametrize("w,p", [(-0.1, 1.0), (1.5, 1.0), (0.5, -1.0), (0.5, 65.0), (float("nan"), 1.0),
                                 (0.5, float("inf")), (0.5, float("nan"))])
def test_directivity_polar_rejects(fs, w, p):
    with pytest.raises(fs.FrequenSeeError):
        fs.directivity_polar([w], [p])


def test_directivity_polar_band_count(fs):
    L = fs.capi.load()
    w = np.zeros(9, np.float32)
    out = np.zeros((8, 33), np.float32)
    assert L.fs_directivity_polar(w.ctypes.data, w.ctypes.data, 0, out.ctypes.data) == fs.capi.FS_ERR_INVALID
    assert L.fs_directivity_polar(w.ctypes.data, w.ctypes.data, 9, out.ctypes.data) == fs.capi.FS_ERR_INVALID
    assert L.fs_directivity_polar(None, w.ctypes.data, 1, out.ctypes.data) == fs.capi.FS_ERR_INVALID


def test_struct_layouts(fs):
    assert C.sizeof(fs.capi.SourceOrient) == 16 and fs.capi.SourceOrient.pattern.offset == 12
    assert fs.capi.DIR_POINTS == 33 and fs.OMNI == 0xFFFFFFFF
    assert fs.capi._patterns(np.ones((3, 2, 33))).shape == (3, 8, 33)
    with pytest.raises(ValueError):
        fs.capi._patterns(np.ones((1, 9, 33)))


def build_directivity_smoke(out_dir):
    exe = os.path.join(str(out_dir), "directivity_smoke")
    libdir = os.path.join(ROOT, "audio-pathtracer_b200", "lib")
    env = dict(os.environ); env.pop("CC", None); env.pop("CXX", None)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "directivity_smoke.cpp"), "-o", exe,
                           "-L", libdir, "-lfrequensee", "-Wl,-rpath," + libdir], env=env)
    return exe


def test_directivity_smoke_compiles_and_fails_loudly_without_gpu(fs, tmp_path):
    """the mirror's Forward / DirectivityPattern / SetDirectivityPatterns build from plain C++"""
    import torch
    exe = build_directivity_smoke(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([exe, "nogpu"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CPU fallback" in r.stdout
