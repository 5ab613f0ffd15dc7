"""FS_FLAG_NOISE_STATS on the GPU: the histogram is unchanged by the flag, the second moments are bit-identical to the CPU
reference (fso_trace_sources_m2) in every kernel path, fs_get_noise matches the float64 statistics, fs_multi reduces
the moments exactly, the state and error rules hold, and one fs_allocate_paths step evens out the SNR of 16 emitters."""
import numpy as np
import pytest

import noise_oracle
import sources_oracle
from test_gpu_source_budgets import _ctx, _mm
from test_source_budgets import POS5, N5, D5

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def shoebox():
    from frequensee import scenes
    return scenes.shoebox()


@pytest.fixture(scope="module")
def room():
    from frequensee import scenes
    return scenes.furnished_room()


def _ref_scene(sc, mm=None):
    R = sources_oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=True)
    if mm is not None:
        R.set_material_model(*mm)
    return R


def _pos(sc, scene):
    return np.concatenate([np.asarray(sc.sources[:1], np.float32).reshape(-1, 3),
                           POS5[1:4] * np.float32(1.2 if scene == "room" else 1.0)])


@pytest.mark.parametrize("scene", ["shoebox", "room"])
def test_histogram_unchanged_by_the_flag(fs, shoebox, room, scene):
    from frequensee import capi
    sc = shoebox if scene == "shoebox" else room
    pos = _pos(sc, scene)
    for name, flags in (("default", 0), ("share", capi.FLAG_SHARE_LISTENER), ("model", capi.FLAG_MATERIAL_MODEL)):
        mm = _mm(sc) if flags & capi.FLAG_MATERIAL_MODEL else None
        a = _ctx(fs, sc, mm=mm, flags=flags)
        b = _ctx(fs, sc, mm=mm, flags=flags | capi.FLAG_NOISE_STATS)
        try:
            assert np.array_equal(a.trace(pos, sc.listener, 5000, 8, 11), b.trace(pos, sc.listener, 5000, 8, 11)), name
            d = [6] * 4 if flags & capi.FLAG_SHARE_LISTENER else [0, 3, 8, 16]
            n = [3000, 700, 5000, 64]
            assert np.array_equal(a.trace_sources(pos, n, d, sc.listener, 12), b.trace_sources(pos, n, d, sc.listener, 12)), name
            assert b.histogram_m2().any()
        finally:
            a.close(); b.close()


def _configs(capi):
    """(name, flags, FS_TUNE_* knobs, config overrides)"""
    return [("default", 0, {}, {}), ("mega_on", 0, {"FS_TUNE_MEGA": 1}, {}), ("mega_off", 0, {"FS_TUNE_MEGA": 0}, {}),
            ("small_batches", 0, {}, {"max_batch_paths": 1100}), ("no_splat_agg", capi.FLAG_NO_SPLAT_AGG, {}, {})]


@pytest.mark.parametrize("scene", ["shoebox", "room"])
def test_m2_bit_exact_vs_cpu_reference(fs, oracle, shoebox, room, scene):
    from frequensee import capi
    sc = shoebox if scene == "shoebox" else room
    R = _ref_scene(sc)
    cfg = oracle.default_config()
    pos = _pos(sc, scene)
    n_uni = 1 << 14
    h_u, m_u, _ = noise_oracle.trace_sources_m2(R, cfg, pos[:1], n_uni, 8, sc.listener, 0x5EED)
    pos5 = POS5 * np.float32(1.2 if scene == "room" else 1.0)
    h_s, m_s, _ = noise_oracle.trace_sources_m2(R, cfg, pos5, N5, D5, sc.listener, 77)
    for name, flags, env, over in _configs(capi):
        ctx = _ctx(fs, sc, env=env, flags=flags | capi.FLAG_NOISE_STATS, **over)
        try:
            assert np.array_equal(ctx.trace(pos[:1], sc.listener, n_uni, 8, 0x5EED), h_u), name
            assert np.array_equal(ctx.histogram_m2(), m_u), name
            st = ctx.noise_stats()
            ref = noise_oracle.noise_stats(h_u, m_u, n_uni)
            for k in ("signal", "variance", "band_signal", "band_variance"):
                np.testing.assert_allclose(st[k], ref[k], rtol=1e-12, atol=0, err_msg="%s %s" % (name, k))
            assert np.array_equal(st["no_energy"], ref["no_energy"])
            np.testing.assert_allclose(st["snr_db"], ref["snr_db"], rtol=1e-12, atol=1e-12)
            # per-source budgets with mixed depths (depth 0 included)
            assert np.array_equal(ctx.trace_sources(pos5, N5, D5, sc.listener, 77), h_s), name
            assert np.array_equal(ctx.histogram_m2(), m_s), name
            st = ctx.noise_stats()
            ref = noise_oracle.noise_stats(h_s, m_s, N5)
            assert list(st["n_paths"]) == N5
            for k in ("signal", "variance", "band_signal", "band_variance"):
                np.testing.assert_allclose(st[k], ref[k], rtol=1e-12, atol=0, err_msg="%s %s" % (name, k))
            np.testing.assert_allclose(st["band_snr_db"], ref["band_snr_db"], rtol=1e-12, atol=1e-12)
        finally:
            ctx.close()


def test_update_sources_and_shared_listener_vs_reference(fs, oracle, shoebox):
    """fs_update_sources leaves the same moments as fs_trace_sources; the shared-listener and material-model walks agree
    with the reference"""
    from frequensee import capi
    sc = shoebox
    for flags in (capi.FLAG_SHARE_LISTENER, capi.FLAG_MATERIAL_MODEL):
        mm = _mm(sc) if flags & capi.FLAG_MATERIAL_MODEL else None
        R = _ref_scene(sc, mm)
        cfg = oracle.default_config(flags=flags)
        d = [6] * 5 if flags == capi.FLAG_SHARE_LISTENER else D5
        h, m2, _ = noise_oracle.trace_sources_m2(R, cfg, POS5, N5, d, sc.listener, 5)
        ctx = _ctx(fs, sc, mm=mm, flags=flags | capi.FLAG_NOISE_STATS)
        try:
            hist = np.zeros_like(h)
            ctx.update_sources(POS5, N5, d, sc.listener, 5, hist_out=hist)
            assert np.array_equal(hist, h) and np.array_equal(ctx.histogram_m2(), m2)
        finally:
            ctx.close()


def test_multi_two_contexts_on_one_gpu(fs, shoebox):
    from frequensee import capi
    sc = shoebox
    pos = _pos(sc, "shoebox")
    one = _ctx(fs, sc, flags=capi.FLAG_NOISE_STATS)
    m = fs.MultiContext([0, 0], flags=capi.FLAG_NOISE_STATS)
    try:
        m.set_scene(sc.verts, sc.tri_mat, sc.absorption)
        c0 = m.context(0)
        for form in ("uniform", "sources"):
            if form == "uniform":
                h1 = one.trace(pos, sc.listener, 9001, 8, 3)
                h2 = m.trace(pos, sc.listener, 9001, 8, 3)
            else:
                h1 = one.trace_sources(POS5, N5, D5, sc.listener, 4)
                h2 = m.trace_sources(POS5, N5, D5, sc.listener, 4)
            assert np.array_equal(h1, h2), form
            assert np.array_equal(one.histogram_m2(), c0.histogram_m2()), form
            a, b = one.noise_stats(), c0.noise_stats()
            for k in a:
                assert np.array_equal(a[k], b[k]), (form, k)
    finally:
        m.close(); one.close()


def test_state_and_error_rules(fs, shoebox):
    from frequensee import capi
    sc = shoebox
    pos = _pos(sc, "shoebox")
    for bad in (capi.FLAG_CONNECT_ALL, capi.FLAG_MIS):
        with pytest.raises(fs.FrequenSeeError) as ei:
            fs.Context(flags=capi.FLAG_NOISE_STATS | bad)
        assert ei.value.code == capi.FS_ERR_INVALID
    plain = _ctx(fs, sc)
    try:
        plain.trace(pos, sc.listener, 1000, 4, 1)
        for f in (plain.noise_stats, plain.histogram_m2):
            with pytest.raises(fs.FrequenSeeError) as ei:
                f()
            assert ei.value.code == capi.FS_ERR_STATE
    finally:
        plain.close()
    ctx = _ctx(fs, sc, flags=capi.FLAG_NOISE_STATS)
    try:
        def state_error():
            for f in (ctx.noise_stats, ctx.histogram_m2):
                with pytest.raises(fs.FrequenSeeError) as ei:
                    f()
                assert ei.value.code == capi.FS_ERR_STATE
        state_error()                                                     # before any trace
        h = ctx.trace(pos, sc.listener, 1000, 4, 1)
        ctx.noise_stats()
        arr = (capi.NoiseStats * 8)()
        assert ctx.L.fs_get_noise(ctx.h, arr, 3) == capi.FS_ERR_INVALID   # wrong source count
        ctx.trace_range(pos, sc.listener, 1000, 0, 500, 4, 1, hist=np.zeros_like(h))
        state_error()
        ctx.trace(pos, sc.listener, 1000, 4, 1)
        ctx.set_histogram(h, 1000)
        state_error()
        ctx.trace_sources(POS5, N5, D5, sc.listener, 2)
        ctx.noise_stats()
        ctx.trace_debug(pos, sc.listener, 100, 0, 10, 4, 1)
        state_error()
    finally:
        ctx.close()


def test_closed_loop_on_the_tunnels(fs):
    """the 16 tunnel emitters nearest to the listener (most of the 64 are too far along the tunnel for any path to
    connect), budgets by distance rank (2 x 2^15 at depth 16, 4 x 2^14 at depth 12, 10 x 2^12 at depth 8); one
    fs_allocate_paths step at the same total must shrink the spread (std) of the broadband snr_db over the sources it
    leaves unclamped.  Measured on a B200 (the run is deterministic): 3.92 -> 2.62 dB, a factor 1.49, not the 2 one might
    hope for: each source's SNR comes from one update of at most 2^15 pairs, so the allocation also follows the noise of
    its own estimate.  The bound is 1.4."""
    from frequensee import capi, scenes
    tun = scenes.mine_tunnels()
    lis = np.asarray(tun.listener, np.float32)
    src = np.asarray(tun.sources, np.float32)
    src = src[np.sort(np.argsort(np.linalg.norm(src - lis, axis=1), kind="stable")[:16])]
    S = len(src)
    rank = np.argsort(np.linalg.norm(src - lis, axis=1), kind="stable")
    n = np.empty(S, np.uint64); d = np.empty(S, np.uint32)
    for r, s in enumerate(rank):
        n[s], d[s] = ((1 << 15, 16) if r < 2 else (1 << 14, 12) if r < 6 else (1 << 12, 8))
    total, lo, hi = int(n.sum()), 1 << 10, 1 << 17
    ctx = _ctx(fs, tun, flags=capi.FLAG_NOISE_STATS)
    try:
        ctx.trace_sources(src, n, d, lis, 100, want_hist=False)
        st0 = ctx.noise_stats()
        n1 = fs.allocate_paths(st0, total, lo, hi)
        assert int(n1.sum()) == total
        ctx.trace_sources(src, n1, d, lis, 101, want_hist=False)
        st1 = ctx.noise_stats()
    finally:
        ctx.close()
    free = (n1 > lo) & (n1 < hi) & ~st0["no_energy"] & ~st1["no_energy"]
    assert free.sum() >= 4
    s0, s1 = np.std(st0["snr_db"][free]), np.std(st1["snr_db"][free])
    print("closed loop: %d unclamped sources, std snr_db %.3f -> %.3f dB (factor %.2f)" % (free.sum(), s0, s1, s0 / s1))
    assert s1 <= s0 / 1.4


def test_cpp_mirror_total_rays_per_tick(fs, oracle, tmp_path):
    """UAudioRayTracingSubsystem::TotalRaysPerTick from plain C++: the first UpdateSources() splits 6000 pairs equally, the
    second by fs_allocate_paths from the first one's noise (NoiseWeight 1, 2, 0.5); each update's LastNoise equals the
    CPU reference's statistics of the same budgets and seed"""
    import re
    import subprocess
    from test_noise_stats import build_noise_smoke
    exe = build_noise_smoke(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("update=")]
    assert len(lines) == 2
    got = [{k: float(v) for k, v in re.findall(r"(\w+\d)=([-+0-9.eEinfa]+)", l)} for l in lines]
    X, Y, Z = 7.0, 5.0, 3.0
    quads = [[(0, 0, 0), (0, Y, 0), (0, Y, Z), (0, 0, Z)], [(X, 0, 0), (X, Y, 0), (X, Y, Z), (X, 0, Z)],
             [(0, 0, 0), (X, 0, 0), (X, 0, Z), (0, 0, Z)], [(0, Y, 0), (X, Y, 0), (X, Y, Z), (0, Y, Z)],
             [(0, 0, 0), (X, 0, 0), (X, Y, 0), (0, Y, 0)], [(0, 0, Z), (X, 0, Z), (X, Y, Z), (0, Y, Z)]]
    alpha = [0.02, 0.05, 0.12, 0.07, 0.37, 0.75]
    verts = np.array([[q[i] for i in t] for q in quads for t in ((0, 1, 2), (0, 2, 3))], np.float32)
    R = sources_oracle.Scene(verts, np.repeat(np.arange(6, dtype=np.uint32), 2),
                             np.repeat(np.array(alpha, np.float32)[:, None], 8, axis=1), use_bvh=True)
    cfg = oracle.default_config()
    pos = np.array([[1.5, 1.2, 1.0], [6.0, 4.0, 2.0], [3.0, 2.5, 1.5]], np.float32)
    depth, w, lis = [8, 4, 3], [1.0, 2.0, 0.5], [5.0, 3.5, 1.6]
    budget = np.array([2000, 2000, 2000], np.uint64)
    for u in range(2):
        assert [int(got[u]["n%d" % s]) for s in range(3)] == list(budget), u
        h, m2, _ = noise_oracle.trace_sources_m2(R, cfg, pos, budget, depth, lis, 0x5EED + u)
        ref = noise_oracle.noise_stats(h, m2, budget)
        for s in range(3):
            np.testing.assert_allclose(got[u]["sig%d" % s], ref["signal"][s], rtol=1e-12)
            np.testing.assert_allclose(got[u]["var%d" % s], ref["variance"][s], rtol=1e-12)
        budget = fs.allocate_paths(ref, 6000, 256, 4096, w)
    assert int(sum(got[1]["n%d" % s] for s in range(3))) == 6000


def test_broadband_sum_past_2_to_64(fs, shoebox):
    """2^26 direct-path pairs (depth 0) with the listener 0.1 m from the source: every pair splats the clamped value
    q = 10 * 2^32 into one bin of each of the 8 bands, so the broadband S1 = 5 * 2^62 passes 2^64 while no band does.
    The statistics must still be exact: broadband mean 80 per pair, signal 6400, variance 0"""
    from frequensee import capi
    sc = shoebox
    src = np.array([[3.0, 2.5, 1.5]], np.float32)
    lis = np.array([3.1, 2.5, 1.5], np.float32)
    ctx = _ctx(fs, sc, flags=capi.FLAG_NOISE_STATS)
    try:
        h = ctx.trace(src, lis, 1 << 26, 0, 9)
        k = int(np.flatnonzero(h[0, 0])[0])
        assert (h[0, :, k] == np.uint64(10 << 32) * np.uint64(1 << 26)).all()
        st = ctx.noise_stats()
    finally:
        ctx.close()
    assert st["signal"][0] == 6400.0 and st["variance"][0] == 0.0 and st["snr_db"][0] == np.inf
    assert (st["band_signal"][0] == 100.0).all() and (st["band_variance"][0] == 0.0).all()
