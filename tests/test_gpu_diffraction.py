"""First-order edge diffraction on the GPU (fs_diffraction): bit-identical to the CPU reference (fso_diffraction), every field
including the path count, on the panel, the shoebox, the furnished room (one source, a grid of listeners), door_rooms with the
door at 0/30/60/90 degrees and a slice of the tunnels with 64 sources, at thresholds 0/30/60/180; the edge set equal to the
reference's; the same bytes under every node format and builder; moving geometry and the edge cache; the legs clear under
fs_debug_any_hits and z and the gains against float64; no side effects; the error and state rules; fs_multi context 0; the
C++ mirror."""
import re
import subprocess

import numpy as np
import pytest

import diffraction_oracle as dor
from test_diffraction import PANEL, build_diffraction_smoke
from test_gpu_source_budgets import _ctx

pytestmark = pytest.mark.gpu

FOLDS = (0.0, 30.0, 60.0, 180.0)


class _Sc:
    def __init__(self, verts, tri_mat=None, absorption=None):
        self.verts = np.ascontiguousarray(verts, np.float32)
        self.tri_mat = np.zeros(len(self.verts), np.uint32) if tri_mat is None else tri_mat
        self.absorption = np.full((1, 8), 0.3, np.float32) if absorption is None else absorption


def _check(ctx, R, src, lis, folds=FOLDS):
    out = []
    for f in folds:
        got = ctx.diffraction(src, lis, f)
        ref = R.diffraction(src, lis, f)
        assert got.tobytes() == ref.tobytes(), (f, got, ref)
        assert np.array_equal(ctx.debug_diffraction_edges(f), R.edges(f)), f
        out.append(got)
    return out


def test_bit_identical_panel_and_shoebox(fs):
    from frequensee import scenes
    p = _Sc(PANEL)
    ctx = _ctx(fs, p)
    R = dor.Scene(p.verts)
    rng = np.random.default_rng(1)
    src = np.concatenate([[[-2, 0, 1]], rng.uniform([-4, -4, -1], [-0.1, 4, 5], (60, 3))]).astype(np.float32)
    got = _check(ctx, R, src, [2, 0, 1])
    assert got[1]["found"].sum() > 30
    sb = scenes.shoebox()
    ctx = _ctx(fs, sb)
    R = dor.Scene(sb.verts)
    src = rng.uniform([0.1, 0.1, 0.1], [6.9, 4.9, 2.9], (50, 3)).astype(np.float32)
    for g in _check(ctx, R, src, sb.listener):
        assert not g["found"].any()


def test_bit_identical_room_listener_grid(fs):
    """one source under the furniture's edges and a 5 x 3 grid of listeners around the room's listener"""
    from frequensee import scenes
    sc = scenes.furnished_room()
    ctx = _ctx(fs, sc)
    R = dor.Scene(sc.verts)
    src = np.array([[3.3777335, 2.8879292, 2.7426772]], np.float32)
    lx, ly, lz = sc.listener
    n_found = 0
    for dx in (-1.0, -0.5, 0.0, 0.5, 1.0):
        for dz in (-0.3, 0.0, 0.3):
            for g in _check(ctx, R, src, [lx + dx, ly, lz + dz], folds=(30.0, 60.0)):
                n_found += int(g["found"][0])
    assert n_found > 0


@pytest.mark.parametrize("angle", [0.0, 30.0, 60.0, 90.0])
def test_bit_identical_door(fs, angle):
    from frequensee import scenes
    sc = scenes.door_rooms()
    V = scenes.door_verts(sc, angle)
    ctx = fs.Context()
    ctx.set_scene(V, sc.tri_mat, sc.absorption)
    R = dor.Scene(V)
    src = np.asarray(sc.sources, np.float32)
    for lis in ([6.7, 3.2, 1.5], [9.0, 2.5, 1.5], [9.0, 5.0, 1.5], [10.0, 6.0, 1.6]):
        _check(ctx, R, src, lis)


def test_bit_identical_tunnel_slice_64_sources(fs):
    from frequensee import scenes
    full = scenes.mine_tunnels()
    T = 250_000
    sc = scenes.Scene("tunnel_slice", full.verts[:T], full.tri_mat[:T], full.absorption, full.sources[:8], full.listener)
    ctx = _ctx(fs, sc)
    R = dor.Scene(sc.verts)
    lo, hi = sc.verts.reshape(-1, 3).min(0), sc.verts.reshape(-1, 3).max(0)
    src = np.random.default_rng(3).uniform(lo, hi, (64, 3)).astype(np.float32)
    _check(ctx, R, src, (0.5 * (lo + hi)).astype(np.float32), folds=(30.0, 60.0))


def test_independent_of_tree(fs):
    from frequensee import scenes
    sc = scenes.door_rooms()
    V = scenes.door_verts(sc, 60.0)
    src = np.concatenate([sc.sources, [[3.0, 6.0, 1.0], [5.0, 3.8, 1.2]]]).astype(np.float32)
    out = []
    for env in ({}, {"FS_TUNE_WIDE": 0}, {"FS_TUNE_W8": 1}, {"FS_TUNE_BUILDER": 0}):
        ctx = _ctx(fs, _Sc(V, sc.tri_mat, sc.absorption), env=env)
        out.append(b"".join(ctx.diffraction(src, lis, f).tobytes() for f in (0.0, 30.0)
                            for lis in ([6.7, 3.2, 1.5], [9.0, 5.0, 1.5])))
        ctx.close()
    assert all(o == out[0] for o in out[1:])


def test_moving_geometry_and_edge_cache(fs):
    from frequensee import scenes
    sc = scenes.door_rooms()
    src = np.asarray(sc.sources, np.float32)
    grid = [[6.7, 3.2, 1.5], [9.0, 2.5, 1.5], [9.0, 5.0, 1.5], [10.0, 6.0, 1.6]]
    run = lambda c, f=30.0: b"".join(c.diffraction(src, lis, f).tobytes() for lis in grid)
    ctx = _ctx(fs, sc)
    closed = run(ctx)
    n30 = len(ctx.debug_diffraction_edges(30.0))
    moved = scenes.door_verts(sc, 60.0)
    first, cnt = sc.meta["door"]
    ctx.update_vertices(moved[first:first + cnt], first)
    with pytest.raises(fs.FrequenSeeError) as e:
        ctx.diffraction(src, grid[0], 30.0)
    assert e.value.code == fs.capi.FS_ERR_STATE
    with pytest.raises(fs.FrequenSeeError) as e:
        ctx.debug_diffraction_edges(30.0)
    assert e.value.code == fs.capi.FS_ERR_STATE
    ctx.refit()
    got = run(ctx)
    fresh = fs.Context()
    fresh.set_scene(moved, sc.tri_mat, sc.absorption)
    assert got == run(fresh)
    R = dor.Scene(moved)
    assert got == b"".join(R.diffraction(src, lis, 30.0).tobytes() for lis in grid)
    assert got != closed                                           # the door matters
    # a threshold change rebuilds the edge set, and going back gives the first set again
    assert len(ctx.debug_diffraction_edges(0.0)) > len(ctx.debug_diffraction_edges(60.0))
    assert np.array_equal(ctx.debug_diffraction_edges(30.0), dor.edges(moved, 30.0))
    assert n30 == len(dor.edges(sc.verts, 30.0))


def _fmaf():
    import ctypes as C
    libm = C.CDLL("libm.so.6")
    libm.fmaf.restype = C.c_float
    libm.fmaf.argtypes = [C.c_float, C.c_float, C.c_float]
    return lambda a, b, c: np.float32(libm.fmaf(float(a), float(b), float(c)))


def test_legs_clear_and_formula(fs):
    from frequensee import scenes
    sc = scenes.furnished_room()
    ctx = _ctx(fs, sc)
    rng = np.random.default_rng(6)
    src = rng.uniform([0.3, 0.3, 0.3], [11.7, 8.7, 3.3], (200, 3)).astype(np.float32)
    lis = np.asarray(sc.listener, np.float32)
    r = ctx.diffraction(src, lis, 30.0)
    k = np.nonzero(r["found"])[0]
    assert len(k) > 0
    rays, tmax = [], []
    eps = np.float32(ctx.cfg.eps_connect)
    fmaf = _fmaf()
    for i in k:
        for q in (src[i], lis):                                     # the leg as fs_diffraction.h builds it
            d = (r["apex"][i] - q).astype(np.float32)
            ln = np.float32(np.sqrt(fmaf(d[2], d[2], fmaf(d[1], d[1], np.float32(d[0] * d[0])))))
            inv = np.float32(1.0) / ln
            if ln - eps > 0:
                rays.append(np.concatenate([q, (d * inv).astype(np.float32)]))
                tmax.append(np.float32(ln - eps))
    hit = ctx.any_hits(np.array(rays, np.float32), np.array(tmax, np.float32))
    assert not hit.any()
    for i in k:
        a = r["apex"][i].astype(np.float64)
        L = np.linalg.norm(a - src[i]) + np.linalg.norm(a - lis)
        z = L - np.linalg.norm(lis.astype(np.float64) - src[i])
        assert abs(r["length"][i] - L) <= 1e-6 * L
        assert abs(r["path_difference"][i] - z) <= 1e-6 * L
        for b in range(8):
            g = max(1.0 / (3.0 + 40.0 * float(r["path_difference"][i]) * 62.5 * 2 ** b / 343.0), 0.01)
            assert abs(r["gain"][i][b] - g) <= 1e-6 * g


def test_no_side_effects(fs):
    from frequensee import scenes
    sc = scenes.shoebox()
    blocks = np.random.default_rng(8).uniform(-0.5, 0.5, (2, 1024, 2)).astype(np.float32)
    res = []
    for insert in (False, True):
        ctx = _ctx(fs, sc, flags=fs.capi.FLAG_NOISE_STATS)
        ctx.conv_init_source(0)
        ctx.conv_process(blocks[0], 0)
        ctx.update(sc.sources, sc.listener, 8192, 8, 0x5EED)
        st0 = ctx.stats()
        if insert:
            ctx.diffraction([[1, 1, 1], [-1, 2, 2]], sc.listener, 0.0)
            st1 = ctx.stats()
            assert st1["kernel_launches"] > st0["kernel_launches"]
            assert {k: v for k, v in st1.items() if k != "kernel_launches"} == \
                   {k: v for k, v in st0.items() if k != "kernel_launches"}
        out = [ctx.get_histogram(), ctx.histogram_m2(), ctx.noise_stats()["variance"], ctx.build_ir(0),
               ctx.conv_process(blocks[1], 0)]
        res.append(out)
        ctx.close()
    for a, b in zip(*res):
        assert np.array_equal(a, b)


def test_rejected_calls_change_nothing(fs):
    import ctypes as C
    L = fs.capi.load()
    empty = fs.Context()
    out = np.zeros(4097, fs.capi.DIFFRACTION_DTYPE)
    src = np.array([[-2, 0, 1]], np.float32)
    lis = np.array([2, 0, 1], np.float32)
    n = C.c_uint64(0)
    assert L.fs_diffraction(empty.h, src.ctypes.data, 1, lis.ctypes.data, 30.0, None, out.ctypes.data) == fs.capi.FS_ERR_STATE
    assert L.fs_debug_diffraction_edges(empty.h, 30.0, None, 0, C.byref(n)) == fs.capi.FS_ERR_STATE
    ctx = _ctx(fs, _Sc(PANEL))
    before = ctx.diffraction(src, lis, 30.0)
    hz = np.full(8, 500.0, np.float32)

    def call(s=src, n_src=1, lp=lis, fold=30.0, band=None, null=None):
        s = np.ascontiguousarray(s, np.float32)
        lp = np.ascontiguousarray(lp, np.float32)
        return L.fs_diffraction(ctx.h, None if null == "src" else s.ctypes.data, n_src, None if null == "lis" else lp.ctypes.data,
                                fold, None if band is None else band.ctypes.data, None if null == "out" else out.ctypes.data)

    assert call() == fs.capi.FS_OK and call(band=hz) == fs.capi.FS_OK
    bad = [dict(null="src"), dict(null="lis"), dict(null="out"), dict(n_src=0), dict(s=np.zeros((4097, 3)), n_src=4097),
           dict(s=[[np.nan, 0, 1]]), dict(s=[[0, np.inf, 1]]), dict(s=[[0, 0, 2e18]]), dict(lp=[np.nan, 0, 0]),
           dict(lp=[0, 0, -1e19]), dict(fold=-0.5), dict(fold=180.5), dict(fold=float("nan")), dict(fold=float("inf")),
           dict(band=np.array([500, 500, 0, 500, 500, 500, 500, 500], np.float32)),
           dict(band=np.array([500, -1, 500, 500, 500, 500, 500, 500], np.float32)),
           dict(band=np.array([500, 500, 500, 500, 500, 500, 500, np.inf], np.float32))]
    for kw in bad:
        assert call(**kw) == fs.capi.FS_ERR_INVALID, kw
        assert ctx.diffraction(src, lis, 30.0).tobytes() == before.tobytes(), kw
    assert L.fs_debug_diffraction_edges(ctx.h, 30.0, None, 0, None) == fs.capi.FS_ERR_INVALID
    assert L.fs_debug_diffraction_edges(ctx.h, 200.0, None, 0, C.byref(n)) == fs.capi.FS_ERR_INVALID
    assert L.fs_debug_diffraction_edges(ctx.h, 30.0, None, 0, C.byref(n)) == fs.capi.FS_OK and n.value == 4
    two = np.zeros((2, 2), np.uint32)
    assert L.fs_debug_diffraction_edges(ctx.h, 30.0, two.ctypes.data, 2, C.byref(n)) == fs.capi.FS_OK and n.value == 4
    assert np.array_equal(two, ctx.debug_diffraction_edges(30.0)[:2])
    many = ctx.diffraction(np.tile(src, (4096, 1)), lis, 30.0)
    assert len(many) == 4096 and np.all(many.view(np.uint8).reshape(4096, -1) == before.view(np.uint8))


def test_multi_context_0_equals_single(fs):
    from frequensee import scenes
    sc = scenes.door_rooms()
    V = scenes.door_verts(sc, 30.0)
    m = fs.MultiContext([0, 0])
    m.set_scene(V, sc.tri_mat, sc.absorption)
    src = np.concatenate([sc.sources, [[3.0, 6.0, 1.0]]]).astype(np.float32)
    got = m.context(0).diffraction(src, [9.0, 5.0, 1.5], 30.0)
    one = _ctx(fs, _Sc(V, sc.tri_mat, sc.absorption)).diffraction(src, [9.0, 5.0, 1.5], 30.0)
    assert got.tobytes() == one.tobytes()


def test_cpp_mirror_update_diffraction(fs, tmp_path):
    exe = build_diffraction_smoke(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    rows = re.findall(r"diffraction s(\d) found=(\d+) n=(\d+) edge=(\d+),(\d+) apex=(\S+) length=(\S+) z=(\S+) gain=(\S+)", r.stdout)
    assert len(rows) == 2, r.stdout
    ref = dor.Scene(PANEL).diffraction([[-2, 0, 1], [1, 1, 1]], [2, 0, 1], 30.0)
    for s, found, n, tri, k, apex, length, z, gain in rows:
        e = ref[int(s)]
        assert (int(found), int(n), int(tri), int(k)) == (e["found"], e["n_paths"], e["edge_tri"], e["edge_k"])
        assert np.array_equal(np.array([float(x) for x in apex.split(",")], np.float32), e["apex"])
        assert np.float32(float(length)) == e["length"] and np.float32(float(z)) == e["path_difference"]
        assert np.array_equal(np.array([float(x) for x in gain.split(",")], np.float32), e["gain"])
    assert ref["found"].tolist() == [1, 0]
