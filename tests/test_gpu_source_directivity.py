"""Directional sources on the GPU: histograms bit-identical to the CPU reference (fso_trace_sources_dir) in every
connection mode, with per-source budgets, a mix of omni and directional sources, small batches and both settings of the
persistent per-batch kernel; constant-1 patterns, FS_OMNI everywhere and no call at all give the same bytes; the noise
moments are those of the weighted values; fs_multi equals the single context; the error and state rules; the C++ mirror."""
import re
import subprocess

import numpy as np
import pytest

import directivity_oracle
import sources_oracle
from test_gpu_source_budgets import _ctx, _mm
from test_source_budgets import POS5, N5, D5

pytestmark = pytest.mark.gpu

OMNI = directivity_oracle.OMNI
MODES = {"default": 0, "share_listener": 128, "material_model": 256, "connect_all": 64, "mis": 512}


@pytest.fixture(scope="module")
def shoebox():
    from frequensee import scenes
    return scenes.shoebox()


@pytest.fixture(scope="module")
def room():
    from frequensee import scenes
    return scenes.furnished_room()


def _patterns(seed=5):
    """two patterns: a rough cardioid per band and a random positive table"""
    rng = np.random.default_rng(seed)
    c = -1.0 + np.arange(33) / 16.0
    card = np.stack([(0.5 + 0.5 * c) ** (1 + b / 4.0) for b in range(8)]).astype(np.float32)
    return np.stack([card, rng.uniform(0.0, 2.5, (8, 33)).astype(np.float32)])


def _orient(S, seed=7, omni_every=3):
    rng = np.random.default_rng(seed)
    fwd = rng.normal(size=(S, 3)).astype(np.float32)
    pat = np.array([OMNI if s % omni_every == omni_every - 1 else s % 2 for s in range(S)], np.uint64)
    return fwd, pat


def _ref(sc, mm=None):
    D = directivity_oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=True)
    if mm is not None:
        D.set_material_model(*mm)
    return D


def _configs():
    """(name, FS_TUNE_* knobs, config overrides)"""
    return [("default", {}, {}), ("small_batches", {}, {"max_batch_paths": 1100}), ("mega_on", {"FS_TUNE_MEGA": 1}, {}),
            ("mega_off", {"FS_TUNE_MEGA": 0}, {})]


@pytest.mark.parametrize("mode", list(MODES))
def test_bit_exact_vs_cpu_reference_shoebox(fs, oracle, shoebox, mode):
    sc = shoebox
    mm = _mm(sc) if mode == "material_model" else None
    flags = MODES[mode]
    D = _ref(sc, mm)
    cfg = oracle.default_config(flags=flags)
    pats = _patterns()
    pos3 = np.concatenate([np.asarray(sc.sources[:1], np.float32).reshape(-1, 3), POS5[1:3]])
    fwd3, pat3 = _orient(3)
    n_uni, d_uni = 3000, 6
    h_u, _ = D.trace_sources_dir(cfg, pos3, n_uni, d_uni, sc.listener, 0x5EED, pats, fwd3, pat3)
    share = mode == "share_listener"
    depths = [6] * 5 if share else D5
    if mode in ("connect_all", "mis"):
        depths = [0, 1, 6, 3, 5]
    n5 = [1, 700, 2000, 33, 900] if mode in ("connect_all", "mis") else N5
    fwd5, pat5 = _orient(5, seed=8)
    h_s, _ = D.trace_sources_dir(cfg, POS5, n5, depths, sc.listener, 77, pats, fwd5, pat5)
    h_omni, _ = D.trace_sources_dir(cfg, pos3, n_uni, d_uni, sc.listener, 0x5EED, pats, fwd3, [OMNI] * 3)
    assert not np.array_equal(h_u, h_omni)                 # the patterns do something
    for name, env, over in _configs():
        ctx = _ctx(fs, sc, env=env, mm=mm, flags=flags, **over)
        try:
            ctx.set_directivity_patterns(pats)
            ctx.set_source_directivity(fwd3, pat3)
            assert np.array_equal(ctx.trace(pos3, sc.listener, n_uni, d_uni, 0x5EED), h_u), name
            ctx.set_source_directivity(fwd5, pat5)
            assert np.array_equal(ctx.trace_sources(POS5, n5, depths, sc.listener, 77), h_s), name
        finally:
            ctx.close()


@pytest.mark.parametrize("mode", ["default", "material_model"])
def test_bit_exact_vs_cpu_reference_room(fs, oracle, room, mode):
    """the furnished room (>= 4096 triangles: the persistent per-batch kernel is chosen on its own for large batches)"""
    sc = room
    mm = _mm(sc) if mode == "material_model" else None
    D = _ref(sc, mm)
    cfg = oracle.default_config(flags=MODES[mode])
    pats = _patterns(9)
    pos = POS5[:4] * np.float32(1.2)
    fwd, pat = _orient(4, seed=10)
    h_u, _ = D.trace_sources_dir(cfg, pos, 1 << 13, 8, sc.listener, 0x5EED, pats, fwd, pat)
    n4, d4 = [1, 3000, 5000, 64], [0, 3, 8, 16]
    h_s, _ = D.trace_sources_dir(cfg, pos, n4, d4, sc.listener, 12, pats, fwd, pat)
    for name, env, over in _configs():
        ctx = _ctx(fs, sc, env=env, mm=mm, flags=MODES[mode], **over)
        try:
            ctx.set_directivity_patterns(pats)
            ctx.set_source_directivity(fwd, pat)
            assert np.array_equal(ctx.trace(pos, sc.listener, 1 << 13, 8, 0x5EED), h_u), name
            assert np.array_equal(ctx.trace_sources(pos, n4, d4, sc.listener, 12), h_s), name
        finally:
            ctx.close()


@pytest.mark.parametrize("mode", ["default", "share_listener", "connect_all", "mis"])
def test_unit_patterns_omni_and_no_call_agree(fs, room, shoebox, mode):
    sc = room if mode in ("default", "share_listener") else shoebox
    pos = POS5[:3] * np.float32(1.2 if sc is room else 1.0)
    n, d = (1 << 15, 8) if sc is room else (4000, 6)
    ctx = _ctx(fs, sc, flags=MODES[mode])
    try:
        h0 = ctx.trace(pos, sc.listener, n, d, 3)
        ctx.set_directivity_patterns(np.ones((2, 8, 33), np.float32))
        ctx.set_source_directivity([[0, 0, 1], [1, 2, 3], [-1, 0, 0]], [0, 1, 0])
        h1 = ctx.trace(pos, sc.listener, n, d, 3)
        ctx.set_source_directivity([[0, 0, 1]] * 3, [OMNI] * 3)
        h2 = ctx.trace(pos, sc.listener, n, d, 3)
        assert np.array_equal(h0, h1) and np.array_equal(h0, h2) and h0.any()
    finally:
        ctx.close()


def _q(e):
    return int(np.float32(np.float32(e) * np.float32(4294967296.0)))


def test_noise_moments_of_the_weighted_values(fs, oracle, shoebox):
    """FS_FLAG_NOISE_STATS: the second moments are the squares of the weighted Q32.32 values that fs_trace_debug records"""
    from frequensee import capi
    sc = shoebox
    pats = _patterns()
    fwd, pat = _orient(2, omni_every=9)
    pos = POS5[1:3]
    n, depth, seed = 3000, 6, 21
    ctx = _ctx(fs, sc, flags=capi.FLAG_NOISE_STATS)
    try:
        ctx.set_directivity_patterns(pats)
        ctx.set_source_directivity(fwd, pat)
        h = ctx.trace(pos, sc.listener, n, depth, seed)
        m2 = ctx.histogram_m2()
        dbg = ctx.trace_debug(pos, sc.listener, n, 0, 2 * n, depth, seed)
    finally:
        ctx.close()
    D = _ref(sc)
    h_ref, _ = D.trace_sources_dir(oracle.default_config(), pos, n, depth, sc.listener, seed, pats, fwd, pat)
    assert np.array_equal(h, h_ref)
    B, K = 8, h.shape[2]
    s1 = np.zeros((2, B, K), object); s2 = np.zeros((2, B + 1, K), object)
    s1[:] = 0; s2[:] = 0
    for g, r in enumerate(dbg):
        if not r["connected"]:
            continue
        s, k = g // n, int(r["bin"])
        qs = [_q(r["energy"][b]) for b in range(B)]
        for b in range(B):
            s1[s, b, k] += qs[b]; s2[s, b, k] += qs[b] * qs[b]
        s2[s, B, k] += sum(qs) ** 2
    assert np.array_equal(h.astype(object), s1)
    got = m2[..., 0].astype(object) + (m2[..., 1].astype(object) << 64)
    assert np.array_equal(got, s2)


def test_multi_two_contexts_on_one_gpu(fs, oracle, shoebox):
    sc = shoebox
    pats = _patterns()
    fwd, pat = _orient(5, seed=4)
    m = fs.MultiContext([0, 0])
    single = _ctx(fs, sc)
    try:
        m.set_scene(sc.verts, sc.tri_mat, sc.absorption)
        for x in (m, single):
            x.set_directivity_patterns(pats)
            x.set_source_directivity(fwd, pat)
        a = m.trace(POS5, sc.listener, 3001, 8, 5)
        b = single.trace(POS5, sc.listener, 3001, 8, 5)
        assert np.array_equal(a, b) and a.any()
        a = m.trace_sources(POS5, N5, D5, sc.listener, 6)
        b = single.trace_sources(POS5, N5, D5, sc.listener, 6)
        assert np.array_equal(a, b)
        h_ref, _ = _ref(sc).trace_sources_dir(oracle.default_config(), POS5, N5, D5, sc.listener, 6, pats, fwd, pat)
        assert np.array_equal(a, h_ref)
        with pytest.raises(fs.FrequenSeeError):
            m.trace(POS5[:2], sc.listener, 100, 4, 5)      # 2 sources, 5 orientations installed
        m.set_source_directivity([], [])
        assert m.trace(POS5[:2], sc.listener, 100, 4, 5).any()
    finally:
        m.close(); single.close()


def test_error_and_state_rules(fs, shoebox):
    from frequensee import capi
    sc = shoebox
    L = capi.load()
    ctx = fs.Context(n_bands=4)
    ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption[:, :4])
    E = fs.FrequenSeeError
    try:
        pats = _patterns()
        # no table: only FS_OMNI is accepted
        with pytest.raises(E):
            ctx.set_source_directivity([[1, 0, 0]], [0])
        ctx.set_source_directivity([[1, 0, 0]], [OMNI])
        ctx.set_source_directivity([], [])
        # pattern tables
        for bad in (np.ones((0, 8, 33)), np.ones((257, 8, 33))):
            with pytest.raises(E):
                ctx.set_directivity_patterns(bad)
        for v in (-1.0, np.nan, np.inf):
            p = pats.copy(); p[1, 3, 7] = v
            with pytest.raises(E):
                ctx.set_directivity_patterns(p)
        p = pats.copy(); p[1, 6, 7] = np.nan                  # band 6 >= n_bands = 4: ignored
        ctx.set_directivity_patterns(p)
        assert L.fs_set_directivity_patterns(ctx.h, None, 1) == capi.FS_ERR_INVALID
        ctx.set_directivity_patterns(pats)
        # orientations
        for fwd, pat in (([[1, 0, 0]], [2]), ([[0, 0, 0]], [0]), ([[np.nan, 0, 1]], [0]), ([[np.inf, 0, 1]], [1])):
            with pytest.raises(E):
                ctx.set_source_directivity(fwd, pat)
        assert L.fs_set_source_directivity(ctx.h, None, 2) == capi.FS_ERR_INVALID
        pos = POS5[:3]
        fwd, pat = _orient(3)
        ctx.set_source_directivity(fwd, pat)
        ref = ctx.trace(pos, sc.listener, 2000, 6, 1)
        # a rejected orientation call changes nothing
        with pytest.raises(E):
            ctx.set_source_directivity([[1, 0, 0]] * 3, [0, 5, 0])
        assert np.array_equal(ctx.trace(pos, sc.listener, 2000, 6, 1), ref)
        # every trace entry point rejects another source count, before anything is enqueued: the histogram stays
        d_hist = __import__("torch").zeros(2 * 4 * ctx.cfg.n_bins, dtype=__import__("torch").int64, device="cuda")
        calls = [
            lambda: ctx.trace(pos[:2], sc.listener, 100, 4, 2),
            lambda: ctx.update(pos[:2], sc.listener, 100, 4, 2),
            lambda: ctx.trace_range(pos[:2], sc.listener, 100, 0, 200, 4, 2),
            lambda: ctx.trace_range_device(pos[:2], sc.listener, 100, 0, 200, 4, 2, d_hist.data_ptr()),
            lambda: ctx.trace_debug(pos[:2], sc.listener, 100, 0, 200, 4, 2),
            lambda: ctx.trace_sources(pos[:2], [100, 50], [4, 2], sc.listener, 2),
            lambda: ctx.update_sources(pos[:2], [100, 50], [4, 2], sc.listener, 2),
            lambda: ctx.trace_sources_range_device(pos[:2], [100, 50], [4, 2], sc.listener, 0, 150, 2, d_hist.data_ptr()),
        ]
        for i, call in enumerate(calls):
            with pytest.raises(E) as ei:
                call()
            assert ei.value.code == capi.FS_ERR_INVALID, i
            assert np.array_equal(ctx.get_histogram(), ref), i
        assert not d_hist.any()
        # a new pattern table clears the orientations: any source count, every source omni
        ctx.set_directivity_patterns(pats)
        h_omni = ctx.trace(pos[:2], sc.listener, 2000, 6, 1)
        ctx.set_source_directivity([[1, 0, 0]] * 2, [OMNI] * 2)
        assert np.array_equal(ctx.trace(pos[:2], sc.listener, 2000, 6, 1), h_omni)
        # stream order: a trace enqueued before a set call uses the orientations installed before it
        ctx.set_source_directivity(fwd, pat)
        ctx.trace(pos, sc.listener, 2000, 6, 1, want_hist=False)
        ctx.set_source_directivity(fwd, [OMNI] * 3)
        assert np.array_equal(ctx.get_histogram(), ref)
    finally:
        ctx.close()


def test_cpp_mirror_directivity(fs, oracle, tmp_path):
    from test_source_directivity import build_directivity_smoke
    exe = build_directivity_smoke(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    got = {l.split()[0]: [int(v) for v in re.findall(r"s\d+=(\d+)", l)] for l in r.stdout.splitlines()}
    X, Y, Z = 7.0, 5.0, 3.0
    quads = [[(0, 0, 0), (0, Y, 0), (0, Y, Z), (0, 0, Z)], [(X, 0, 0), (X, Y, 0), (X, Y, Z), (X, 0, Z)],
             [(0, 0, 0), (X, 0, 0), (X, 0, Z), (0, 0, Z)], [(0, Y, 0), (X, Y, 0), (X, Y, Z), (0, Y, Z)],
             [(0, 0, 0), (X, 0, 0), (X, Y, 0), (0, Y, 0)], [(0, 0, Z), (X, 0, Z), (X, Y, Z), (0, Y, Z)]]
    alpha = [0.02, 0.05, 0.12, 0.07, 0.37, 0.75]
    verts = np.array([[q[i] for i in t] for q in quads for t in ((0, 1, 2), (0, 2, 3))], np.float32)
    tri_mat, ab = np.repeat(np.arange(6, dtype=np.uint32), 2), np.repeat(np.array(alpha, np.float32)[:, None], 8, axis=1)
    D = directivity_oracle.Scene(verts, tri_mat, ab, use_bvh=True)
    cfg = oracle.default_config()
    pats = np.stack([fs.directivity_polar([0.5] * 8, [1.0] * 8), fs.directivity_polar([1.0] * 8, [1.0] * 8)])
    pos = np.array([[1.5, 1.2, 1.0], [6.0, 4.0, 2.0], [3.0, 2.5, 1.5]], np.float32)
    fwd = [[1, 0, 0], [0, -2, 0], [0, 0, 1]]
    n, d, lis = [3000, 4000, 5000], [8, 6, 4], [5.0, 3.5, 1.6]
    h, _ = D.trace_sources_dir(cfg, pos, n, d, lis, 0x5EED, pats, fwd, [0, 1, OMNI])
    assert got["sources"] == [int(x) for x in h.reshape(3, -1).sum(axis=1)]
    h, _ = D.trace_sources_dir(cfg, pos[:1], n[:1], d[:1], lis, 0x5EED + 1, pats, fwd[:1], [0])
    assert got["source0"] == [int(h.sum())]
    h, _ = sources_oracle.Scene(verts, tri_mat, ab, use_bvh=True).trace_sources(cfg, pos, n, d, lis, 0x5EED + 2)
    assert got["omni"] == [int(x) for x in h.reshape(3, -1).sum(axis=1)]
