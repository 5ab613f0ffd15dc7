"""Room-acoustic parameters on the GPU (fs_get_acoustic_params) against the float64 reference (tests/acoustics_oracle.py):
histograms of fs_trace, fs_trace_sources with mixed budgets and depths, FS_FLAG_CONNECT_ALL and FS_FLAG_MIS on the shoebox,
the furnished room and a tunnel slice with 1, 3 and 8 bands; edge histograms installed with fs_set_histogram (8 bands
near 2^64 in one bin, K = 2^16 and 2^20, silent sources, bin_ms = 2.5); the same bytes on every call, with and without
the EDC and on fs_multi context 0; the state and error rules; no side effects; physical sanity; the C++ mirror."""
import ctypes as C
import math
import re
import subprocess

import numpy as np
import pytest

import acoustics_oracle as A
from test_acoustics import build_acoustics_smoke, exp_decay
from test_gpu_source_budgets import _ctx

pytestmark = pytest.mark.gpu


def _check(ctx, hist=None):
    """the GPU records and EDC of ctx's current histogram against the reference; returns the records"""
    if hist is None:
        hist = ctx.get_histogram()
    arr, edc = ctx.acoustic_params(edc=True)
    ref, ref_edc = A.acoustic_params(hist, ctx.cfg.bin_ms)
    bad = A.compare(A.from_ctypes(arr, ctx.cfg.n_bands), ref)
    assert bad == [], bad[:10]
    assert A.edc_ulps(edc, ref_edc) <= 1
    plain = ctx.acoustic_params()
    assert bytes(plain) == bytes(arr)                    # the records do not depend on whether the EDC is requested
    return ref


def _scene(name, n_bands):
    from frequensee import scenes
    if name == "shoebox":
        return scenes.shoebox(n_bands=n_bands)
    if name == "room":
        return scenes.furnished_room(n_bands=n_bands)
    full = scenes.mine_tunnels(n_bands=n_bands)
    T = 250_000
    return scenes.Scene("tunnel_slice", full.verts[:T], full.tri_mat[:T], full.absorption, full.sources[:8], full.listener)


@pytest.mark.parametrize("n_bands", [1, 3, 8])
@pytest.mark.parametrize("scene", ["shoebox", "room", "tunnel"])
def test_traced_histograms_match_reference(fs, scene, n_bands):
    sc = _scene(scene, n_bands)
    pos = np.asarray(sc.sources, np.float32).reshape(-1, 3)
    lo, hi = sc.verts.reshape(-1, 3).min(0), sc.verts.reshape(-1, 3).max(0)
    rng = np.random.default_rng(n_bands)
    extra = (lo + (hi - lo) * rng.uniform(0.2, 0.8, (3, 3))).astype(np.float32)
    pos = np.concatenate([pos[:4], extra])
    lis = sc.listener if scene != "tunnel" else (0.5 * (lo + hi)).astype(np.float32)
    with _ctx(fs, sc, n_bands=n_bands) as ctx:
        ctx.trace(pos, lis, 1 << 15, 12, 0x5EED)
        ref = _check(ctx)
        assert any(r["broadband"]["valid"] for r in ref)
        n = rng.integers(2000, 40000, len(pos))
        d = rng.integers(1, 40, len(pos))
        ctx.trace_sources(pos, n, d, lis, 7)
        _check(ctx)


@pytest.mark.parametrize("n_bands", [1, 8])
def test_connect_all_and_mis_match_reference(fs, n_bands):
    from frequensee import capi
    sc = _scene("shoebox", n_bands)
    for flags in (capi.FLAG_CONNECT_ALL, capi.FLAG_MIS):
        with _ctx(fs, sc, flags=flags, n_bands=n_bands) as ctx:
            ctx.trace(sc.sources, sc.listener, 1 << 13, 6, 5)
            _check(ctx)
            ctx.trace_sources(np.array([[1.5, 1.2, 1.0], [3.0, 2.0, 2.0]], np.float32), [3000, 9000], [3, 6], sc.listener, 6)
            _check(ctx)


def test_edge_histograms(fs):
    # 8 bands each near 2^64 in one bin: the broadband sum needs 67 bits
    h = np.zeros((3, 8, 1000), np.uint64)
    h[0, :, 5] = np.uint64(2 ** 64 - 7)
    h[0, :, 6:400] = np.uint64(2 ** 63)
    h[0, 3, 7] = np.uint64(2 ** 64 - 1)
    h[2, 4, 999] = 1                                    # energy only in the overflow bin
    with fs.Context() as ctx:
        ctx.set_histogram(h, 1000)
        ref = _check(ctx, h)
        assert ref[0]["broadband"]["onset_bin"] == 5 and ref[1]["no_energy"] == 1 and ref[2]["band"][4]["onset_bin"] == 999
    # many bins per thread: K = 2^16 and 2^20 with a synthetic decay
    for K, bands, T in ((1 << 16, 2, 9.0), (1 << 20, 1, 60.0)):
        E = np.array(exp_decay(T, K, 1.0, amp=2 ** 40), np.uint64)
        h = np.stack([E, E[::-1].copy()][:bands])[None]
        with fs.Context(n_bins=K, n_bands=bands) as ctx:
            ctx.set_histogram(h, 1)
            ref = _check(ctx, h)
        assert ref[0]["band"][0]["valid"] & 7 == 7
        assert abs(ref[0]["band"][0]["t30"]["time_s"] / T - 1) < 1e-6
    # bin_ms = 2.5 (n50 = 20, n80 = 32) on a traced histogram
    from frequensee import scenes
    sc = scenes.shoebox()
    with _ctx(fs, sc, bin_ms=2.5, n_bins=500) as ctx:
        ctx.trace(sc.sources, sc.listener, 1 << 15, 16, 9)
        ref = _check(ctx)
        assert ref[0]["broadband"]["valid"] & (A.C50 | A.C80) == A.C50 | A.C80


def test_repeatable_and_multi_context_0(fs):
    from frequensee import scenes
    sc = scenes.shoebox()
    pos = np.array([[1.5, 1.2, 1.0], [6.0, 4.0, 2.0], [3.0, 2.5, 1.5]], np.float32)
    with _ctx(fs, sc) as ctx:
        ctx.trace_sources(pos, [20000, 5000, 9000], [16, 4, 9], sc.listener, 3)
        a1, e1 = ctx.acoustic_params(edc=True)
        a2, e2 = ctx.acoustic_params(edc=True)
        assert bytes(a1) == bytes(a2) and e1.tobytes() == e2.tobytes()
        m = fs.MultiContext([0, 0])
        try:
            m.set_scene(sc.verts, sc.tri_mat, sc.absorption)
            m.trace_sources(pos, [20000, 5000, 9000], [16, 4, 9], sc.listener, 3)
            b, eb = m.context(0).acoustic_params(edc=True)
        finally:
            m.close()
        assert bytes(b) == bytes(a1) and eb.tobytes() == e1.tobytes()


def test_state_errors_and_no_side_effects(fs):
    from frequensee import capi, scenes
    sc = scenes.shoebox()
    L = capi.load()
    with _ctx(fs, sc, flags=capi.FLAG_NOISE_STATS) as ctx:
        out = (capi.AcousticParams * 2)()
        C.memset(out, 0xAB, C.sizeof(out))
        before = bytes(out)
        assert L.fs_get_acoustic_params(ctx.h, out, 0, None) == capi.FS_ERR_STATE          # before any trace
        blocks = np.random.default_rng(8).uniform(-0.5, 0.5, (2, 1024, 2)).astype(np.float32)
        ctx.conv_init_source(0)
        ctx.conv_process(blocks[0], 0)
        ctx.update(sc.sources, sc.listener, 1 << 15, 12, 0x5EED)
        for n in (0, 2):
            assert L.fs_get_acoustic_params(ctx.h, out, n, None) == capi.FS_ERR_INVALID      # n_sources != 1
        assert L.fs_get_acoustic_params(ctx.h, None, 1, None) == capi.FS_ERR_INVALID
        assert bytes(out) == before
        h0, m0, ir0 = ctx.get_histogram(), ctx.histogram_m2(), ctx.build_ir(0)
        st0 = ctx.stats()
        ctx.acoustic_params(edc=True)
        st1 = ctx.stats()
        assert st1["kernel_launches"] == st0["kernel_launches"] + 1
        assert {k: v for k, v in st1.items() if k != "kernel_launches"} == {k: v for k, v in st0.items() if k != "kernel_launches"}
        y_with = ctx.conv_process(blocks[1], 0)
        assert np.array_equal(h0, ctx.get_histogram()) and np.array_equal(m0, ctx.histogram_m2())
        assert np.array_equal(ir0, ctx.build_ir(0))
    with _ctx(fs, sc, flags=capi.FLAG_NOISE_STATS) as ref_ctx:
        ref_ctx.conv_init_source(0)
        ref_ctx.conv_process(blocks[0], 0)
        ref_ctx.update(sc.sources, sc.listener, 1 << 15, 12, 0x5EED)
        ref_ctx.get_histogram(); ref_ctx.histogram_m2(); ref_ctx.build_ir(0)
        assert np.array_equal(y_with, ref_ctx.conv_process(blocks[1], 0))


def test_more_absorption_shortens_the_decay(fs):
    """shoebox, one absorption on every surface, FS_FLAG_MIS: 0.1 -> 0.3 lowers broadband T20 and T30 and raises C80"""
    from frequensee import capi, scenes
    sc = scenes.shoebox()
    res = []
    for alpha in (0.1, 0.3):
        absorption = np.full_like(sc.absorption, alpha)
        with fs.Context(flags=capi.FLAG_MIS) as ctx:
            ctx.set_scene(sc.verts, sc.tri_mat, absorption)
            ctx.trace(sc.sources, sc.listener, 1 << 18, 32, 21)
            res.append(ctx.acoustic_params()[0].broadband)
    lo, hi = res
    assert lo.valid & hi.valid & (A.T20 | A.T30 | A.C80) == A.T20 | A.T30 | A.C80
    assert hi.t20.time_s < lo.t20.time_s and hi.t30.time_s < lo.t30.time_s
    assert hi.c80_db > lo.c80_db


def test_cpp_mirror_update_acoustic_params(fs, oracle, tmp_path):
    import sources_oracle
    exe = build_acoustics_smoke(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "stale update refused" in r.stdout
    X, Y, Z = 7.0, 5.0, 3.0
    quads = [[(0, 0, 0), (0, Y, 0), (0, Y, Z), (0, 0, Z)], [(X, 0, 0), (X, Y, 0), (X, Y, Z), (X, 0, Z)],
             [(0, 0, 0), (X, 0, 0), (X, 0, Z), (0, 0, Z)], [(0, Y, 0), (X, Y, 0), (X, Y, Z), (0, Y, Z)],
             [(0, 0, 0), (X, 0, 0), (X, Y, 0), (0, Y, 0)], [(0, 0, Z), (X, 0, Z), (X, Y, Z), (0, Y, Z)]]
    alpha = [0.02, 0.05, 0.12, 0.07, 0.37, 0.75]
    verts = np.array([[q[i] for i in t] for q in quads for t in ((0, 1, 2), (0, 2, 3))], np.float32)
    R = sources_oracle.Scene(verts, np.repeat(np.arange(6, dtype=np.uint32), 2),
                             np.repeat(np.array(alpha, np.float32)[:, None], 8, axis=1), use_bvh=True)
    pos = np.array([[1.5, 1.2, 1.0], [6.0, 4.0, 2.0], [3.0, 2.5, 1.5]], np.float32)
    h = R.trace_sources(oracle.default_config(), pos, np.array([20000, 12000, 8000], np.uint64), [16, 8, 12],
                        [5.0, 3.5, 1.6], 0x5EED)[0]
    ref, _ = A.acoustic_params(h, 1.0)
    rows = re.findall(r"acoustics s(\d) (broadband|band0) onset=(\d+) valid=(\d+) edt=(\S+) t20=(\S+) t30=(\S+) r30=(\S+) "
                      r"c50=(\S+) c80=(\S+) d50=(\S+) ts=(\S+)", r.stdout)
    assert len(rows) == 6, r.stdout
    for s, which, onset, valid, *vals in rows:
        want = ref[int(s)]["broadband" if which == "broadband" else "band"]
        want = want if which == "broadband" else want[0]
        assert int(onset) == want["onset_bin"] and int(valid) == want["valid"], (s, which)
        exp = [want["edt"]["time_s"], want["t20"]["time_s"], want["t30"]["time_s"], want["t30"]["r"], want["c50_db"],
               want["c80_db"], want["d50"], want["ts_s"]]
        for g, w in zip(vals, exp):
            assert A._close(float(g), w), (s, which, g, w)
    assert any(int(x[3]) & 7 for x in rows)
