"""Direct-path occlusion on the GPU (fs_occlusion): bit-identical to the CPU reference (fso_occlusion) on the shoebox, the
furnished room with random Transmission / ThicknessCm and a slice of the tunnels, with mixed radii and ray counts and
max_crossings in {0, 1, 4, 16}; the same bytes under every node format and builder and with or without
FS_FLAG_MATERIAL_MODEL; moving geometry; agreement with fs_debug_any_hits; no side effects on the update, the noise moments,
the IRs and the convolver; the error and state rules; fs_multi context 0; the C++ mirror."""
import ctypes as C
import re
import subprocess

import numpy as np
import pytest

import occlusion_oracle
from test_gpu_source_budgets import _ctx, _mm
from test_occlusion import build_occlusion_smoke

pytestmark = pytest.mark.gpu

CROSSINGS = (0, 1, 4, 16)


@pytest.fixture(scope="module")
def shoebox():
    from frequensee import scenes
    return scenes.shoebox()


@pytest.fixture(scope="module")
def room():
    from frequensee import scenes
    return scenes.furnished_room()


@pytest.fixture(scope="module")
def door():
    from frequensee import scenes
    return scenes.door_rooms()


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _same(a, b):
    return np.array_equal(_bits(a[0]), _bits(b[0])) and np.array_equal(_bits(a[1]), _bits(b[1]))


def _ref(sc, mm=None):
    R = occlusion_oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=True)
    if mm is not None:
        R.set_material_model(mm[0], mm[1], mm[2])
    return R


def _sources(rng, lo, hi, S, big=False):
    """S emitters in the box [lo, hi]: a mix of points and balls with 1..700 rays (plus one of 65536 rays when big)"""
    pos = rng.uniform(lo, hi, (S, 3)).astype(np.float32)
    radius = np.where(rng.uniform(size=S) < 0.3, 0.0, rng.uniform(0.05, 1.5, S)).astype(np.float32)
    n = rng.integers(1, 700, S)
    if big:
        radius[S // 2], n[S // 2] = 0.75, 65536
    return pos, radius, n


def _check_against_ref(ctx, R, pos, radius, n, lis, seed):
    for mc in CROSSINGS:
        got = ctx.occlusion(pos, radius, n, lis, max_crossings=mc, seed=seed)
        ref = R.occlusion(pos, radius, n, lis, max_crossings=mc, seed=seed)
        assert _same(got, ref[:2]), mc
    return got


def test_bit_identical_shoebox(fs, shoebox):
    """emitters inside and outside the box (walls with random transmission in between), 300 sources with up to 700 rays
    and one of 65536: the CTAs span many sources"""
    sc = shoebox
    mm = _mm(sc)
    ctx = _ctx(fs, sc, mm=mm)
    R = _ref(sc, mm)
    pos, radius, n = _sources(np.random.default_rng(1), [-3, -3, -2], [10, 8, 5], 300, big=True)
    vis, tr = _check_against_ref(ctx, R, pos, radius, n, sc.listener, 0x5EED)
    assert 0.0 < vis.mean() < 1.0 and (tr > 0).any() and (tr < 1).any()


def test_bit_identical_room(fs, room):
    sc = room
    mm = _mm(sc, seed=8)
    ctx = _ctx(fs, sc, mm=mm)
    R = _ref(sc, mm)
    pos, radius, n = _sources(np.random.default_rng(2), [0.2, 0.2, 0.2], [11.8, 8.8, 3.4], 48)
    vis, _ = _check_against_ref(ctx, R, pos, radius, n, sc.listener, 7)
    assert 0.0 < vis.mean() < 1.0


def test_bit_identical_tunnel_slice(fs):
    from frequensee import scenes
    full = scenes.mine_tunnels()
    T = 250_000
    sc = scenes.Scene("tunnel_slice", full.verts[:T], full.tri_mat[:T], full.absorption, full.sources[:8], full.listener)
    mm = _mm(sc, seed=4)
    ctx = _ctx(fs, sc, mm=mm)
    R = _ref(sc, mm)
    lo, hi = sc.verts.reshape(-1, 3).min(0), sc.verts.reshape(-1, 3).max(0)
    rng = np.random.default_rng(3)
    pos = np.concatenate([full.sources[:8], rng.uniform(lo, hi, (8, 3))]).astype(np.float32)
    radius = np.tile(np.array([0.0, 0.5], np.float32), 8)
    n = np.tile([1, 256], 8)
    lis = (0.5 * (lo + hi)).astype(np.float32)
    _check_against_ref(ctx, R, pos, radius, n, lis, 11)


def test_independent_of_tree_and_material_flag(fs, room):
    sc = room
    mm = _mm(sc, seed=5)
    pos, radius, n = _sources(np.random.default_rng(4), [0.2, 0.2, 0.2], [11.8, 8.8, 3.4], 32)
    out = []
    for env, over in (({}, {}), ({"FS_TUNE_WIDE": 0}, {}), ({"FS_TUNE_W8": 1}, {}), ({"FS_TUNE_BUILDER": 0}, {}),
                      ({}, {"flags": fs.capi.FLAG_MATERIAL_MODEL})):
        ctx = _ctx(fs, sc, env=env, mm=mm, **over)
        out.append([ctx.occlusion(pos, radius, n, sc.listener, max_crossings=mc, seed=3) for mc in CROSSINGS])
        ctx.close()
    for o in out[1:]:
        for a, b in zip(out[0], o):
            assert _same(a, b)


def test_moving_geometry(fs, door):
    from frequensee import scenes
    sc = door
    pos, radius, n = np.asarray(sc.sources, np.float32).reshape(-1, 3), 0.4, 300
    ctx = _ctx(fs, sc)
    moved = scenes.door_verts(sc, 70.0)
    first, cnt = sc.meta["door"]
    ctx.update_vertices(moved[first:first + cnt], first)
    with pytest.raises(fs.FrequenSeeError) as e:
        ctx.occlusion(pos, radius, n, sc.listener)
    assert e.value.code == fs.capi.FS_ERR_STATE
    ctx.refit()
    got = ctx.occlusion(pos, radius, n, sc.listener, seed=5)
    fresh = fs.Context()
    fresh.set_scene(moved, sc.tri_mat, sc.absorption)
    assert _same(got, fresh.occlusion(pos, radius, n, sc.listener, seed=5))
    closed = _ctx(fs, sc).occlusion(pos, radius, n, sc.listener, seed=5)
    R = occlusion_oracle.Scene(moved, sc.tri_mat, sc.absorption)
    assert _same(got, R.occlusion(pos, radius, n, sc.listener, seed=5)[:2])
    assert not _same(got, closed)                      # the door matters


def _fmaf():
    libm = C.CDLL("libm.so.6")
    libm.fmaf.restype = C.c_float
    libm.fmaf.argtypes = [C.c_float, C.c_float, C.c_float]
    return lambda a, b, c: np.float32(libm.fmaf(float(a), float(b), float(c)))


def test_point_emitter_matches_any_hit(fs, room):
    """radius 0: visible == 1 - fs_debug_any_hits of the connection ray, built in numpy as the oracle builds it"""
    sc = room
    ctx = _ctx(fs, sc)
    rng = np.random.default_rng(6)
    pos = rng.uniform([0.2, 0.2, 0.2], [11.8, 8.8, 3.4], (400, 3)).astype(np.float32)
    lis = np.asarray(sc.listener, np.float32)
    fmaf = _fmaf()
    rays, tmax = [], []
    for q in pos:
        dl = (lis - q).astype(np.float32)
        ln = np.sqrt(fmaf(dl[2], dl[2], fmaf(dl[1], dl[1], np.float32(dl[0] * dl[0]))))
        inv = np.float32(1.0) / ln
        rays.append(np.concatenate([q, (dl * inv).astype(np.float32)]))
        tmax.append(np.float32(ln - np.float32(ctx.cfg.eps_connect)))
    assert min(tmax) > 0
    hit = ctx.any_hits(np.array(rays, np.float32), np.array(tmax, np.float32))
    vis, _ = ctx.occlusion(pos, 0.0, 1, lis, max_crossings=0)
    assert np.array_equal(vis, (~hit).astype(np.float32))
    assert 0 < hit.sum() < len(hit)


def test_no_side_effects(fs, shoebox):
    """an fs_occlusion call between fs_update and the calls that follow it changes none of their bytes"""
    sc = shoebox
    pos, radius, n = _sources(np.random.default_rng(7), [-2, -2, -1], [9, 7, 4], 20)
    blocks = np.random.default_rng(8).uniform(-0.5, 0.5, (2, 1024, 2)).astype(np.float32)
    res = []
    for insert in (False, True):
        ctx = _ctx(fs, sc, mm=_mm(sc), flags=fs.capi.FLAG_NOISE_STATS)
        ctx.conv_init_source(0)
        ctx.conv_process(blocks[0], 0)
        ctx.update(sc.sources, sc.listener, 8192, 8, 0x5EED)
        st0 = ctx.stats()
        if insert:
            ctx.occlusion(pos, radius, n, sc.listener, seed=1)
            st1 = ctx.stats()
            assert st1["kernel_launches"] == st0["kernel_launches"] + 1
            assert {k: v for k, v in st1.items() if k != "kernel_launches"} == \
                   {k: v for k, v in st0.items() if k != "kernel_launches"}
        out = [ctx.get_histogram(), ctx.histogram_m2(), ctx.noise_stats()["variance"], ctx.build_ir(0),
               ctx.conv_process(blocks[1], 0)]
        res.append(out)
        ctx.close()
    for a, b in zip(*res):
        assert np.array_equal(a, b)


def test_rejected_calls_change_nothing(fs, shoebox):
    sc = shoebox
    L = fs.capi.load()
    empty = fs.Context()
    src, S = fs.capi.occlusion_sources([[1, 1, 1]], 0.5, 16)
    out = (fs.capi.OcclusionResult * 1)()
    lis = np.asarray(sc.listener, np.float32)
    assert L.fs_occlusion(empty.h, src, 1, lis.ctypes.data, 4, 0, out) == fs.capi.FS_ERR_STATE
    ctx = _ctx(fs, sc, mm=_mm(sc))
    pos, radius, n = _sources(np.random.default_rng(9), [-2, -2, -1], [9, 7, 4], 12)
    before = ctx.occlusion(pos, radius, n, lis, seed=2)

    def call(src_pos=((1, 1, 1),), rad=0.5, rays=16, lis_pos=lis, mc=4, n_src=None, reserved=0, null=None):
        arr, S = fs.capi.occlusion_sources(src_pos, rad, rays)
        arr[0].reserved = reserved
        lp = np.asarray(lis_pos, np.float32)
        res = (fs.capi.OcclusionResult * max(S, 4097))()
        return L.fs_occlusion(ctx.h, None if null == "src" else arr, S if n_src is None else n_src,
                              None if null == "lis" else lp.ctypes.data, mc, 0, None if null == "out" else res)

    assert call() == fs.capi.FS_OK
    bad = [dict(null="src"), dict(null="lis"), dict(null="out"), dict(n_src=0), dict(mc=17),
           dict(src_pos=[[np.nan, 1, 1]]), dict(src_pos=[[1, np.inf, 1]]), dict(src_pos=[[1, 1, 2e18]]),
           dict(lis_pos=[np.nan, 0, 0]), dict(lis_pos=[0, 0, -1e19]), dict(rad=-0.1), dict(rad=np.nan), dict(rad=np.inf),
           dict(rays=0), dict(rays=65537), dict(reserved=1)]
    for kw in bad:
        assert call(**kw) == fs.capi.FS_ERR_INVALID, kw
        assert _same(before, ctx.occlusion(pos, radius, n, lis, seed=2)), kw
    many, S = fs.capi.occlusion_sources(np.zeros((4097, 3)), 0.0, 1)
    res = (fs.capi.OcclusionResult * 4097)()
    assert L.fs_occlusion(ctx.h, many, 4097, lis.ctypes.data, 4, 0, res) == fs.capi.FS_ERR_INVALID
    assert call(rad=0.0, rays=0) == fs.capi.FS_OK       # n_rays is ignored for a point emitter
    vis, tr = ctx.occlusion(np.zeros((4096, 3)) + [1, 1, 1], 0.0, 1, lis)
    assert vis.shape == (4096,) and np.all(vis == 1.0)


def test_multi_context_0_equals_single(fs, door):
    sc = door
    pos, radius, n = np.asarray(sc.sources, np.float32).reshape(-1, 3), 0.6, 500
    m = fs.MultiContext([0, 0])
    m.set_scene(sc.verts, sc.tri_mat, sc.absorption)
    got = m.context(0).occlusion(pos, radius, n, sc.listener, max_crossings=2, seed=4)
    one = _ctx(fs, sc).occlusion(pos, radius, n, sc.listener, max_crossings=2, seed=4)
    assert _same(got, one)


def test_cpp_mirror_update_occlusion(fs, tmp_path):
    exe = build_occlusion_smoke(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    rows = re.findall(r"occlusion s(\d) n=(\d+) visible=(\S+) tr=(\S+)", r.stdout)
    assert len(rows) == 3, r.stdout
    X, Y, Z, P, G = 7.0, 5.0, 3.0, 3.5, 3.0
    quads = [[[0, 0, 0], [0, Y, 0], [0, Y, Z], [0, 0, Z]], [[X, 0, 0], [X, Y, 0], [X, Y, Z], [X, 0, Z]],
             [[0, 0, 0], [X, 0, 0], [X, 0, Z], [0, 0, Z]], [[0, Y, 0], [X, Y, 0], [X, Y, Z], [0, Y, Z]],
             [[0, 0, 0], [X, 0, 0], [X, Y, 0], [0, Y, 0]], [[0, 0, Z], [X, 0, Z], [X, Y, Z], [0, Y, Z]],
             [[P, 0, 0], [P, G, 0], [P, G, Z], [P, 0, Z]]]
    verts = np.array([t for q in quads for t in ([q[0], q[1], q[2]], [q[0], q[2], q[3]])], np.float32)
    tri_mat = np.repeat(np.arange(7, dtype=np.uint32), 2)
    alpha = np.repeat(np.array([0.02, 0.05, 0.12, 0.07, 0.37, 0.75, 0.3], np.float32)[:, None], 8, 1)
    R = occlusion_oracle.Scene(verts, tri_mat, alpha)
    pos = np.array([[6.0, 1.0, 1.2], [1.5, 1.5, 1.5], [2.8, 2.9, 1.5]], np.float32)
    vis, tr, used = R.occlusion(pos, [0.0, 0.0, 0.8], 512, [5.0, 1.5, 1.6], max_crossings=8, seed=77)
    for s, nr, v, t in rows:
        s = int(s)
        assert int(nr) == used[s]
        assert np.float32(float(v)) == vis[s]
        assert np.array_equal(np.array([float(x) for x in t.split(",")], np.float32), tr[s])
    assert vis[0] == 1.0 and vis[1] == 0.0 and 0.0 < vis[2] < 1.0
