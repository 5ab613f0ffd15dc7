"""Direct-path occlusion, host side: known answers of the CPU reference (tests/oracle_ext/fso_occlusion.c, the per-ray
arithmetic of csrc/fs_occlusion.h) -- free field, one and two walls with hand-computed transmitted factors, shared edges and
vertices counted once, the crossing limit, the raw-hit cap, a half-plane shadow edge, tau_eff equal to the material model's
transmitted factor; brute force equal to the oracle BVH; the struct layouts; the C++ mirror's smoke program compiles and
fails loudly without a GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import occlusion_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B = 8


def quad(x, y0, y1, z0, z1):
    """two triangles in the plane x, diagonal from (y0, z0) to (y1, z1)"""
    v = np.array([[x, y0, z0], [x, y1, z0], [x, y1, z1], [x, y0, z1]], np.float32)
    return np.stack([v[[0, 1, 2]], v[[0, 2, 3]]])


def grid(x, lo, hi, n):
    """an n x n tessellated wall in the plane x over [lo, hi]^2 in (y, z)"""
    e = np.linspace(lo, hi, n + 1, dtype=np.float32)
    return np.concatenate([quad(x, e[i], e[i + 1], e[j], e[j + 1]) for i in range(n) for j in range(n)])


def scene(walls, mats, alpha, tau=None, thick=None, use_bvh=True):
    """walls: list of triangle arrays, mats: material id of each"""
    verts = np.concatenate(walls)
    tri_mat = np.concatenate([np.full(len(w), m, np.uint32) for w, m in zip(walls, mats)])
    S = occlusion_oracle.Scene(verts, tri_mat, np.asarray(alpha, np.float32), use_bvh=use_bvh)
    if tau is not None:
        S.set_material_model(tau, None, thick)
    return S


def tau_by_hand(alpha, tau, thick):
    """the material model's transmitted factor in float32: tau limited to 1 - Refl, raised to ThicknessCm / 2.5"""
    L = occlusion_oracle.lib()
    refl = np.float32(np.float32(1.0) - np.float32(alpha))
    t = np.float32(tau)
    if np.float32(refl + t) > np.float32(1.0):
        t = np.float32(np.float32(1.0) - refl)
    ex = np.float32(np.float32(thick) / np.float32(2.5))
    if not t > 0:
        return np.float32(0.0)
    return t if ex == np.float32(1.0) else np.float32(L.fso_powf(float(t), float(ex)))


def q32(g):
    """what one ray of gain g reports: trunc(g 2^32) 2^-32 (the Q32.32 sum), rounded to float"""
    return (np.floor(np.asarray(g, np.float64) * 2.0 ** 32) * 2.0 ** -32).astype(np.float32)


def _mats(rng, M):
    alpha = rng.uniform(0.0, 1.0, (M, B)).astype(np.float32)
    tau = rng.uniform(0.05, 1.0, (M, B)).astype(np.float32)
    return alpha, tau


SRC = np.array([[0.0, 0.3, 0.2]], np.float32)
LIS = np.array([4.0, 0.3, 0.2], np.float32)


def test_free_field_and_same_room():
    from frequensee import scenes
    sc = scenes.shoebox()
    S = occlusion_oracle.Scene(sc.verts, sc.tri_mat, sc.absorption)
    src = np.array([[1.0, 1.0, 1.0], [3.5, 2.5, 1.5], [6.0, 4.0, 2.0]], np.float32)
    for radius, n in ((0.0, 1), (0.5, 1000), (0.9, 64)):
        vis, tr, used = S.occlusion(src, radius, n, sc.listener, max_crossings=4, seed=3)
        assert np.all(vis == 1.0) and np.all(tr == 1.0) and np.all(used == n)
    empty = occlusion_oracle.Scene(np.zeros((0, 3, 3), np.float32), np.zeros(0, np.uint32), sc.absorption)
    vis, tr, _ = empty.occlusion(src, 0.5, 100, [0, 0, 0])
    assert np.all(vis == 1.0) and np.all(tr == 1.0)


@pytest.mark.parametrize("use_bvh", [False, True])
def test_one_wall_and_two_walls_known_answer(use_bvh):
    rng = np.random.default_rng(1)
    alpha, tau = _mats(rng, 2)
    tau[0, 0] = 0.999                 # (1 - alpha) + tau > 1: limited to alpha
    thick = np.array([2.5, 5.0], np.float32)
    hand = np.array([[tau_by_hand(alpha[m, b], tau[m, b], thick[m]) for b in range(B)] for m in range(2)], np.float32)
    assert hand[0, 0] == np.float32(np.float32(1.0) - np.float32(np.float32(1.0) - alpha[0, 0]))
    S1 = scene([quad(2.0, -5, 5, -5, 5)], [0], alpha, tau, thick, use_bvh)
    vis, tr, _ = S1.occlusion(SRC, 0.0, 1, LIS, max_crossings=4)
    assert vis[0] == 0.0 and np.array_equal(tr[0], q32(hand[0]))
    S2 = scene([quad(2.0, -5, 5, -5, 5), quad(3.0, -5, 5, -5, 5)], [0, 1], alpha, tau, thick, use_bvh)
    vis, tr, _ = S2.occlusion(SRC, 0.0, 1, LIS, max_crossings=4)
    assert vis[0] == 0.0 and np.array_equal(tr[0], q32((hand[0] * hand[1]).astype(np.float32)))
    vis, tr, _ = S2.occlusion(SRC, 0.0, 1, LIS, max_crossings=1)
    assert vis[0] == 0.0 and not tr.any()


def test_shared_diagonal_and_vertex_count_once():
    L = occlusion_oracle.lib()
    rng = np.random.default_rng(2)
    alpha, tau = _mats(rng, 1)
    S = scene([quad(2.0, -1, 1, -1, 1)], [0], alpha, tau)
    src, lis = np.array([[0.0, 0.25, 0.25]], np.float32), np.array([4.0, 0.25, 0.25], np.float32)
    t = C.c_float()
    d = np.array([1.0, 0.0, 0.0], np.float32)
    hits = 0
    for tri in quad(2.0, -1, 1, -1, 1):
        v0, e1, e2 = tri[0], tri[1] - tri[0], tri[2] - tri[0]
        hits += L.fso_intersect_tri(src[0].ctypes.data, d.ctypes.data, v0.ctypes.data, e1.ctypes.data, e2.ctypes.data, C.byref(t))
    assert hits == 2                                     # the ray does cross both triangles of the quad
    tau_eff = S.tau()[0]
    vis, tr, _ = S.occlusion(src, 0.0, 1, lis, max_crossings=1)
    assert vis[0] == 0.0 and np.array_equal(tr[0], q32(tau_eff))
    G = scene([grid(2.0, -2, 2, 4)], [0], alpha, tau)     # the ray through a vertex shared by 6 triangles
    vis, tr, _ = G.occlusion([[0.0, 0.0, 0.0]], 0.0, 1, [4.0, 0.0, 0.0], max_crossings=1)
    assert vis[0] == 0.0 and np.array_equal(tr[0], q32(tau_eff))


def test_walls_in_a_row_crossing_limit_and_raw_hit_cap():
    rng = np.random.default_rng(3)
    alpha, tau = _mats(rng, 1)
    tau[:] = np.maximum(tau, 0.6)
    alpha[:] = np.maximum(alpha, 0.5)
    k = 5
    S = scene([quad(1.0 + 0.5 * i, -5, 5, -5, 5) for i in range(k)], [0] * k, alpha, tau)
    te = S.tau()[0]
    prod = np.ones(B, np.float32)
    for _ in range(k):
        prod = (prod * te).astype(np.float32)
    vis, tr, _ = S.occlusion(SRC, 0.0, 1, LIS, max_crossings=k)
    assert vis[0] == 0.0 and np.array_equal(tr[0], q32(prod))
    vis, tr, _ = S.occlusion(SRC, 0.0, 1, LIS, max_crossings=k - 1)
    assert vis[0] == 0.0 and not tr.any()
    # pure occlusion: transmission == visible, for a blocked and a visible emitter
    vis, tr, _ = S.occlusion([[0.0, 0.3, 0.2], [3.5, 0.3, 0.2]], 0.0, 1, [3.6, 0.3, 0.2], max_crossings=0)
    assert list(vis) == [0.0, 1.0] and np.array_equal(tr, np.repeat(vis[:, None], B, 1))
    # three coincident copies of every wall: 3 raw hits per counted crossing; 10 walls (30 raw hits) pass, 11 (33) block
    for walls, expect_zero in ((10, False), (11, True)):
        W = scene([quad(0.5 + 0.25 * i, -5, 5, -5, 5) for i in range(walls) for _ in range(3)], [0] * (3 * walls), alpha, tau)
        vis, tr, _ = W.occlusion(SRC, 0.0, 1, LIS, max_crossings=16)
        assert vis[0] == 0.0
        assert (not tr.any()) if expect_zero else tr.all()


@pytest.mark.parametrize("seed", [1, 2, 3, 0x5EED])
def test_half_plane_shadow_edge(seed):
    """an absorbing wall over z < 0 between an emitter ball at the origin and a listener on the x axis: the plane z = 0
    through both holds the wall's edge, so half of the ball is in shadow"""
    alpha = np.full((1, B), 0.3, np.float32)
    S = scene([quad(2.0, -50, 50, -50, 0)], [0], alpha)
    n = 4096
    vis, tr, used = S.occlusion([[0.0, 0.0, 0.0]], 0.5, n, [4.0, 0.0, 0.0], max_crossings=8, seed=seed)
    assert used[0] == n
    assert abs(float(vis[0]) - 0.5) < 4.0 * np.sqrt(0.25 / n)
    assert np.array_equal(tr[0], np.full(B, vis[0]))    # tau = 0: only the visible rays transmit


def test_tau_table_equals_material_model():
    rng = np.random.default_rng(4)
    M = 12
    alpha, tau = _mats(rng, M)
    tau[::3] = rng.uniform(0.9, 1.0, (4, B))             # some limited to alpha
    tau[1, :2] = 0.0
    thick = rng.uniform(0.0, 12.0, M).astype(np.float32)
    thick[2] = 2.5
    thick[5] = 0.0
    S = scene([quad(2.0, -5, 5, -5, 5)], [0], alpha, tau, thick)
    hand = np.array([[tau_by_hand(alpha[m, b], tau[m, b], thick[m]) for b in range(B)] for m in range(M)], np.float32)
    assert np.array_equal(S.tau().view(np.uint32), hand.view(np.uint32))
    assert np.all(hand[5][tau[5] > 0] == 1.0)           # thickness 0: no loss
    none = scene([quad(2.0, -5, 5, -5, 5)], [0], alpha)
    assert not none.tau().any()                          # materials without Transmission block
    # a single wall of each material transmits exactly its row
    for m in (0, 1, 2, 7):
        W = scene([quad(2.0, -5, 5, -5, 5)], [m], alpha, tau, thick)
        _, tr, _ = W.occlusion(SRC, 0.0, 1, LIS)
        assert np.array_equal(tr[0], q32(hand[m])), m


def test_brute_force_equals_oracle_bvh():
    from frequensee import scenes
    sc = scenes.furnished_room(target_tris=20_000)
    rng = np.random.default_rng(5)
    M = sc.absorption.shape[0]
    tau = rng.uniform(0.0, 1.0, (M, B)).astype(np.float32)
    thick = rng.uniform(0.5, 10.0, M).astype(np.float32)
    res = []
    src = rng.uniform([0.5, 0.5, 0.3], [11.5, 8.5, 3.3], (7, 3)).astype(np.float32)
    radius = np.array([0.0, 0.5, 1.0, 0.25, 0.0, 2.0, 0.1], np.float32)
    n = np.array([1, 300, 200, 1, 9, 150, 64])
    for use_bvh in (False, True):
        S = occlusion_oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=use_bvh)
        S.set_material_model(tau, None, thick)
        res.append([S.occlusion(src, radius, n, sc.listener, max_crossings=mc, seed=9) for mc in (0, 1, 4, 16)])
    for a, b in zip(*res):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    vis, tr, used = res[1][2]
    assert list(used) == [1, 300, 200, 1, 1, 150, 64]
    assert 0.0 < vis.min() < 1.0 or tr.min() < 1.0      # the furniture occludes some of them


def test_struct_layouts(fs):
    cs, cr = fs.capi.OcclusionSource, fs.capi.OcclusionResult
    assert C.sizeof(cs) == 24 and C.sizeof(cr) == 44
    assert (cs.pos.offset, cs.radius.offset, cs.n_rays.offset, cs.reserved.offset) == (0, 12, 16, 20)
    assert (cr.visible.offset, cr.transmission.offset, cr.n_rays.offset, cr.reserved.offset) == (0, 4, 36, 40)
    arr, S = fs.capi.occlusion_sources([[1, 2, 3], [4, 5, 6]], [0.0, 0.5], 64)
    assert S == 2 and arr[1].radius == 0.5 and arr[1].n_rays == 64 and arr[0].reserved == 0


def build_occlusion_smoke(out_dir):
    exe = os.path.join(str(out_dir), "occlusion_smoke")
    libdir = os.path.join(ROOT, "audio-pathtracer_b200", "lib")
    env = dict(os.environ); env.pop("CC", None); env.pop("CXX", None)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "occlusion_smoke.cpp"), "-o", exe,
                           "-L", libdir, "-lfrequensee", "-Wl,-rpath," + libdir], env=env)
    return exe


def test_occlusion_smoke_compiles_and_fails_loudly_without_gpu(fs, tmp_path):
    """the mirror's OcclusionRadius / OcclusionRays / LastOcclusion / UpdateOcclusion build from plain C++"""
    import torch
    exe = build_occlusion_smoke(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([exe, "nogpu"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CPU fallback" in r.stdout
