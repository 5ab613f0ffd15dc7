"""Per-source path budgets and depths on the GPU (fs_trace_sources, fs_update_sources, the shard and multi-device forms,
UpdateSources() of the C++ mirror): bit-exact against fs_trace in the uniform case, against the CPU reference of the
per-source form for mixed budgets and depths, and against fs_trace_range source by source."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import sources_oracle
from test_source_budgets import POS5, N5, D5, build_sources_smoke

pytestmark = pytest.mark.gpu


class _env:
    """FS_TUNE_* knobs are read by fs_create: set them around the creation of a context"""
    def __init__(self, **kv):
        self.kv = {k: str(v) for k, v in kv.items()}

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kv}
        os.environ.update(self.kv)

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _ctx(fs, sc, env=None, mm=None, **over):
    with _env(**(env or {})):
        ctx = fs.Context(**over)
    if mm is not None:
        ctx.set_scene_ex(sc.verts, sc.tri_mat, sc.absorption, *mm)
    else:
        ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption)
    return ctx


def _mm(sc, seed=3):
    rng = np.random.default_rng(seed)
    M, B = sc.absorption.shape
    return (rng.uniform(0, 0.5, (M, B)).astype(np.float32), rng.uniform(0, 1, (M, B)).astype(np.float32),
            rng.uniform(0.5, 10, M).astype(np.float32))


@pytest.fixture(scope="module")
def shoebox():
    from frequensee import scenes
    return scenes.shoebox()


@pytest.fixture(scope="module")
def room():
    from frequensee import scenes
    return scenes.furnished_room()


def _flags(capi):
    return [("default", 0, 3000, 8), ("fused", capi.FLAG_FUSED_EXTEND, 3000, 8), ("share", capi.FLAG_SHARE_LISTENER, 3000, 8),
            ("connect_all", capi.FLAG_CONNECT_ALL, 800, 6), ("mis", capi.FLAG_MIS, 800, 6),
            ("model", capi.FLAG_MATERIAL_MODEL, 3000, 8), ("count", capi.FLAG_COUNT_VISITS, 3000, 8)]


@pytest.mark.parametrize("scene", ["shoebox", "room"])
def test_uniform_budgets_bit_identical_to_fs_trace(fs, shoebox, room, scene):
    """identity 1 in every flag mode, with the persistent kernel on and off, three batch lanes and batch splits that cut
    a source's range in the middle"""
    from frequensee import capi
    sc = shoebox if scene == "shoebox" else room
    pos = np.array(sc.sources[:1] * 1, np.float32).reshape(-1, 3)
    pos = np.concatenate([pos, POS5[1:4] * np.float32(1.2 if scene == "room" else 1.0)])
    for name, flags, n, d in _flags(capi):
        mm = _mm(sc) if flags & capi.FLAG_MATERIAL_MODEL else None
        for env, over in (({}, {}), ({"FS_TUNE_MEGA": 0}, {"max_batch_paths": 1100}), ({"FS_TUNE_MEGA": 1}, {})):
            if env.get("FS_TUNE_MEGA") == 1 and flags & (capi.FLAG_CONNECT_ALL | capi.FLAG_MIS | capi.FLAG_COUNT_VISITS | capi.FLAG_FUSED_EXTEND):
                continue
            with _ctx(fs, sc, env, mm, flags=flags, **over) as ctx:
                a = ctx.trace(pos, sc.listener, n, d, 0x5EED)
                st_a = ctx.stats()
                b = ctx.trace_sources(pos, n, d, sc.listener, 0x5EED)
                st_b = ctx.stats()
            assert np.array_equal(a, b), (scene, name, env, over)
            assert a.any()
            assert st_a["paths"] == st_b["paths"] == 4 * n and st_a["connected"] == st_b["connected"], (scene, name, env)
    # three lanes: jobs of >= 3 x 2^17 pairs
    for flags in (0, capi.FLAG_SHARE_LISTENER):
        with _ctx(fs, sc, {"FS_TUNE_STREAMS": 3}, flags=flags) as ctx3, _ctx(fs, sc, {"FS_TUNE_STREAMS": 1}, flags=flags) as ctx1:
            a = ctx1.trace(pos, sc.listener, 1 << 17, 6, 11)
            b = ctx3.trace_sources(pos, 1 << 17, 6, sc.listener, 11)
            c = ctx1.trace_sources(pos, 1 << 17, 6, sc.listener, 11)
        assert np.array_equal(a, b) and np.array_equal(a, c), (scene, flags)


def _modes(capi, oracle):
    return [("default", 0, 0, {}), ("mega", 0, 0, {"FS_TUNE_MEGA": 1}), ("fused", capi.FLAG_FUSED_EXTEND, 0, {}),
            ("connect_all", capi.FLAG_CONNECT_ALL, oracle.FLAG_CONNECT_ALL, {}), ("mis", capi.FLAG_MIS, oracle.FLAG_MIS, {}),
            ("model", capi.FLAG_MATERIAL_MODEL, oracle.FLAG_MATERIAL_MODEL, {}), ("count", capi.FLAG_COUNT_VISITS, 0, {}),
            ("split", 0, 0, {}), ("share", capi.FLAG_SHARE_LISTENER, oracle.FLAG_SHARE_LISTENER, {})]


def test_mixed_budgets_bit_exact_vs_cpu_reference(fs, oracle, shoebox):
    """mixed budgets and depths (0, 1, 8, 3, 16) in every mode; shared listener with equal depths and mixed budgets"""
    from frequensee import capi
    sc = shoebox
    mm = _mm(sc)
    R = sources_oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=False)
    Rm = sources_oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=False)
    Rm.set_material_model(*mm)
    for name, gflags, oflags, env in _modes(capi, oracle):
        depths = [7] * 5 if name == "share" else D5
        over = {"max_batch_paths": 1000} if name == "split" else {}
        model = gflags & capi.FLAG_MATERIAL_MODEL
        ho, so = (Rm if model else R).trace_sources(oracle.default_config(flags=oflags), POS5, N5, depths, sc.listener, 21)
        with _ctx(fs, sc, env, mm if model else None, flags=gflags, **over) as ctx:
            h = ctx.trace_sources(POS5, N5, depths, sc.listener, 21)
            st = ctx.stats()
        assert np.array_equal(h, ho), name
        assert st["paths"] == sum(N5) and st["connected"] == so["connected"], name


def test_each_source_equals_fs_trace_range(fs, shoebox):
    """identity 2 on the device: source s of fs_trace_sources = fs_trace_range(pos_s, n_paths = o_s + n_s, g_first = o_s)"""
    sc = shoebox
    with _ctx(fs, sc) as ctx:
        h = ctx.trace_sources(POS5, N5, D5, sc.listener, 5)
        o = 0
        for s in range(5):
            hs = ctx.trace_range(POS5[s:s + 1], sc.listener, o + N5[s], o, N5[s], D5[s], 5)
            assert np.array_equal(h[s], hs[0]), s
            o += N5[s]


def test_update_sources_irs_and_histograms(fs, room):
    """fs_update_sources IRs = fs_set_histogram(single-source histogram, n_paths = n_s) + fs_build_ir; the returned
    histogram, fs_get_histogram and fs_build_ir after fs_trace_sources agree"""
    sc = room
    pos = np.array([[2.0, 1.8, 1.4], [9.0, 7.0, 1.2], [6.0, 4.5, 2.0], [1.0, 8.0, 1.0]], np.float32)
    n, d = [20000, 3000, 700, 9000], [12, 4, 0, 9]
    cfg = fs.default_config()
    hist = np.zeros((4, cfg.n_bands, cfg.n_bins), np.uint64)
    irs = np.zeros((4, cfg.n_channels, cfg.sample_rate), np.float32)
    with _ctx(fs, sc) as ctx:
        ctx.update_sources(pos, n, d, sc.listener, 3, hist_out=hist, ir_out=irs)
        assert np.array_equal(ctx.get_histogram(), hist)
        ir2 = ctx.build_ir(2)                         # single-source builder after a per-source trace: its own count
        ir_all = ctx.build_ir_all(4)
        assert np.array_equal(ir_all, irs) and np.array_equal(ir2, irs[2])
        h2 = ctx.trace_sources(pos, n, d, sc.listener, 3)
        assert np.array_equal(h2, hist)
        for s in range(4):
            ctx.set_histogram(hist[s], n[s])
            assert np.array_equal(ctx.build_ir(0), irs[s]), s
        # after a uniform trace the counts are uniform again
        h3 = ctx.trace(pos, sc.listener, 5000, 6, 3)
        ir3 = ctx.build_ir_all(4)
        ctx.set_histogram(h3, 5000)
        assert np.array_equal(ctx.build_ir_all(4), ir3)
    assert irs[0].any()


def test_multi_device_and_shards(fs, shoebox):
    import torch
    sc = shoebox
    cfg = fs.default_config()
    with _ctx(fs, sc) as ctx:
        ir_ref = np.zeros((5, cfg.n_channels, cfg.sample_rate), np.float32)
        h_ref = np.zeros((5, cfg.n_bands, cfg.n_bins), np.uint64)
        ctx.update_sources(POS5, N5, D5, sc.listener, 8, hist_out=h_ref, ir_out=ir_ref)
        # three shards of the flat range, summed on the device and installed with the per-source counts
        from frequensee import distributed
        G = sum(N5)
        acc = torch.zeros((5, cfg.n_bands, cfg.n_bins), dtype=torch.int64, device="cuda:0")
        part = torch.zeros_like(acc)
        for r in range(3):
            first, count = distributed.shard_range(G, r, 3)
            ctx.trace_sources_range_device(POS5, N5, D5, sc.listener, first, count, 8, part.data_ptr(), zero_first=True)
            ctx.synchronize()
            acc += part
        torch.cuda.synchronize()
        ctx.set_histogram_sources_device(acc.data_ptr(), N5)
        assert np.array_equal(ctx.get_histogram(), h_ref)
        assert np.array_equal(ctx.build_ir_all(5), ir_ref)
    devs = [[0, 0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])
    for dv in devs:
        for flags in (0, 128):
            depths = [6] * 5 if flags else D5
            with _ctx(fs, sc, flags=flags) as ctx:
                h1 = ctx.trace_sources(POS5, N5, depths, sc.listener, 8)
            m = fs.MultiContext(dv, flags=flags)
            try:
                m.set_scene(sc.verts, sc.tri_mat, sc.absorption)
                hm = m.trace_sources(POS5, N5, depths, sc.listener, 8)
                assert np.array_equal(hm, h1), (dv, flags)
                if not flags:
                    c0 = m.context(0)
                    assert np.array_equal(c0.build_ir_all(5), ir_ref), dv
            finally:
                m.close()


def test_errors_change_no_state(fs, shoebox):
    from frequensee import capi
    sc = shoebox
    L = capi.load()
    lis = np.array(sc.listener, np.float32)
    for flags, lim in ((0, 1024), (capi.FLAG_CONNECT_ALL, 63), (capi.FLAG_MIS, 32), (capi.FLAG_SHARE_LISTENER, 1024)):
        with _ctx(fs, sc, flags=flags) as ctx:
            h0 = ctx.trace_sources(POS5, N5, [min(x, 6) for x in D5] if not flags & capi.FLAG_SHARE_LISTENER else 6,
                                   sc.listener, 4)
            ir0 = ctx.build_ir(1)

            def unchanged():
                assert np.array_equal(ctx.get_histogram(), h0)
                assert np.array_equal(ctx.build_ir(1), ir0)

            bad = [([1, 0, 5, 5, 5], 3), ([10] * 5, [3, 3, lim + 1, 3, 3])]
            if flags & capi.FLAG_SHARE_LISTENER:
                bad.append(([10] * 5, [3, 3, 4, 3, 3]))
            for n, d in bad:
                with pytest.raises(fs.FrequenSeeError) as ei:
                    ctx.trace_sources(POS5, n, d, sc.listener, 4)
                assert ei.value.code == capi.FS_ERR_INVALID, (flags, n, d)
                with pytest.raises(fs.FrequenSeeError) as ei:
                    ctx.update_sources(POS5, n, d, sc.listener, 4)
                assert ei.value.code == capi.FS_ERR_INVALID
                unchanged()
            # n_sources * n_bins >= 2^32: rejected before the descriptors are read
            d1 = capi.source_descs(POS5[:1], 10, 3)
            S = (1 << 32) // ctx.cfg.n_bins + 1
            assert L.fs_trace_sources(ctx.h, C.addressof(d1), S, lis.ctypes.data, 4, None) == capi.FS_ERR_INVALID
            unchanged()
            # moved triangles without a refit
            ctx.update_vertices(sc.verts[:1], 0)
            with pytest.raises(fs.FrequenSeeError) as ei:
                ctx.trace_sources(POS5, N5, 3, sc.listener, 4)
            assert ei.value.code == capi.FS_ERR_STATE
            unchanged()
            ctx.refit()
            assert np.array_equal(ctx.trace_sources(POS5, N5, [min(x, 6) for x in D5] if not flags & capi.FLAG_SHARE_LISTENER else 6,
                                                    sc.listener, 4), h0)


def test_cpp_mirror_update_sources_matches_cpu_reference(fs, oracle, tmp_path):
    exe = build_sources_smoke(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    kv = dict(re.findall(r"(\w+)=([-+.\w]+)", r.stdout))
    X, Y, Z = 7.0, 5.0, 3.0
    quads = [[[0, 0, 0], [0, Y, 0], [0, Y, Z], [0, 0, Z]], [[X, 0, 0], [X, Y, 0], [X, Y, Z], [X, 0, Z]],
             [[0, 0, 0], [X, 0, 0], [X, 0, Z], [0, 0, Z]], [[0, Y, 0], [X, Y, 0], [X, Y, Z], [0, Y, Z]],
             [[0, 0, 0], [X, 0, 0], [X, Y, 0], [0, Y, 0]], [[0, 0, Z], [X, 0, Z], [X, Y, Z], [0, Y, Z]]]
    tris, mats = [], []
    for f, q in enumerate(quads):
        tris += [[q[0], q[1], q[2]], [q[0], q[2], q[3]]]
        mats += [f, f]
    alpha = np.repeat(np.array([[0.02], [0.05], [0.12], [0.07], [0.37], [0.75]], np.float32), 8, axis=1)
    R = sources_oracle.Scene(np.array(tris, np.float32), np.array(mats, np.uint32), alpha, use_bvh=False)
    cfg = oracle.default_config()
    pos = [[1.5, 1.2, 1.0], [6.0, 4.0, 2.0], [3.0, 2.5, 1.5]]
    n = [4096, 700, 1500]
    h, st = R.trace_sources(cfg, pos, n, [8, 0, 3], [5.0, 3.5, 1.6], 0x5EED)
    assert int(kv["connected"]) == st["connected"]
    for s in range(3):
        f = 1469598103934665603
        for b in h[s].astype("<u8").tobytes():
            f = ((f ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
        assert int(kv["hist%d" % s]) == f, s
        ir = oracle.build_ir(cfg, h[s], n[s])
        assert abs(float(kv["ir_energy%d" % s]) / float((ir[0].astype(np.float64) ** 2).sum()) - 1) < 1e-5, s
        assert int(kv["ir_peak%d" % s]) == int(np.argmax(ir[0])), s
