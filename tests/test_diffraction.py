"""First-order edge diffraction, host side: known answers of the CPU reference (tests/oracle_ext/fso_diffraction.c, the
per-edge arithmetic of csrc/fs_diffraction.h) -- a thin screen worked out by hand, a lit receiver, the inside of a room, a
welded cube, tessellated edges and the tie-break at a shared vertex, the edge classification (T-junctions, three triangles on
one edge, degenerate triangles, -0.0, the folds of a uv sphere), the gain formula; brute force equal to the oracle BVH; the
result layout; the C++ mirror's smoke program compiles and fails loudly without a GPU."""
import math
import os
import subprocess

import numpy as np
import pytest

import diffraction_oracle as dor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C_AIR = 343.0


def quad(p0, p1, p2, p3):
    """two triangles (p0, p1, p2), (p0, p2, p3)"""
    v = np.array([p0, p1, p2, p3], np.float32)
    return np.stack([v[[0, 1, 2]], v[[0, 2, 3]]])


PANEL = quad([0, -2, 0], [0, 2, 0], [0, 2, 4], [0, -2, 4])     # 4 x 4 m in x = 0, y in [-2, 2], z in [0, 4]


def cube(lo=0.0, hi=1.0):
    """12 triangles of the cube [lo, hi]^3 on its 8 shared corner positions"""
    c = lambda i: [hi if i & 1 else lo, hi if i & 2 else lo, hi if i & 4 else lo]
    faces = [(0, 2, 6, 4), (1, 5, 7, 3), (0, 4, 5, 1), (2, 3, 7, 6), (0, 1, 3, 2), (4, 6, 7, 5)]
    return np.concatenate([quad(c(a), c(b), c(d), c(e)) for a, b, d, e in faces])


def hand_gain(z, f):
    return max(1.0 / (3.0 + 40.0 * z * f / C_AIR), 0.01)


def close(a, b, rel=1e-6):
    return abs(float(a) - float(b)) <= rel * max(abs(float(b)), 1e-6)


def test_thin_screen_known_answer():
    S = dor.Scene(PANEL)
    r = S.diffraction([[-2, 0, 1]], [2, 0, 1], 30.0)[0]
    assert r["found"] == 1 and r["n_paths"] == 4                  # the four rim edges; the diagonal is a flat seam
    assert (r["edge_tri"], r["edge_k"]) == (0, 0)                  # the bottom edge (0, -2, 0) -> (0, 2, 0)
    assert np.array_equal(r["apex"], np.zeros(3, np.float32))
    L = 2.0 * math.sqrt(5.0)
    assert close(r["length"], L) and close(r["path_difference"], L - 4.0)
    for b in range(8):
        assert close(r["gain"][b], hand_gain(L - 4.0, 62.5 * 2 ** b)), b
    assert close(r["gain"][0], 1.0 / (3.0 + 3.4413), 1e-4)        # 62.5 Hz
    assert abs(r["gain"][4] - 0.0172) < 1e-4                       # 1 kHz
    assert r["gain"][7] == np.float32(0.01)                        # 8 kHz: the 20 dB limit
    lit = S.diffraction([[-2, 0, 1], [-1, 1.5, 3]], [-1, 0.5, 2], 30.0)
    assert not lit["found"].any() and not lit.view(np.uint8).any()  # both in front: nothing, and every field 0


def test_shoebox_interior_never_diffracts():
    from frequensee import scenes
    sc = scenes.shoebox()
    S = dor.Scene(sc.verts)
    rng = np.random.default_rng(1)
    src = rng.uniform([0.1, 0.1, 0.1], [6.9, 4.9, 2.9], (40, 3)).astype(np.float32)
    for fold in (0.0, 30.0, 90.0):
        for lis in rng.uniform([0.1, 0.1, 0.1], [6.9, 4.9, 2.9], (5, 3)):
            assert not S.diffraction(src, lis, fold)["found"].any()
    assert len(S.edges(30.0)) == 12                                # the box's 12 wedges (concave from inside)


def _edge_of(verts, p, q):
    """lowest (tri, k) whose triangle edge has the endpoints {p, q}"""
    p, q = np.asarray(p, np.float32), np.asarray(q, np.float32)
    for t, tri in enumerate(verts):
        for k in range(3):
            a, b = tri[k], tri[(k + 1) % 3]
            if (np.array_equal(a, p) and np.array_equal(b, q)) or (np.array_equal(a, q) and np.array_equal(b, p)):
                return t, k
    raise AssertionError("no such edge")


def test_welded_cube():
    V = cube()
    S = dor.Scene(V)
    assert len(S.edges(30.0)) == 12
    opposite = S.diffraction([[-1.0, 0.5, 0.5]], [2.0, 0.5, 0.5], 30.0)[0]
    assert opposite["found"] == 0                                  # needs two edges
    r = S.diffraction([[0.5, -1.0, 0.5]], [1.5, 1.5, 0.5], 30.0)[0]
    assert r["found"] == 1
    assert (r["edge_tri"], r["edge_k"]) == _edge_of(V, [1, 0, 0], [1, 0, 1])
    assert np.allclose(r["apex"], [1.0, 0.0, 0.5], atol=1e-7)
    L = math.hypot(0.5, 1.0) + math.hypot(0.5, 1.5)
    assert close(r["length"], L)
    assert abs(r["path_difference"] - (L - math.hypot(1.0, 2.5))) < 1e-6     # a difference of float lengths near 2.7


def corner(n_seg, H=3.0):
    """two 4 m panels meeting at the vertical line x = y = 0 (a 90 degree corner, the solid in x < 0, y > 0), each split into
    n_seg strips along z that share their vertices on the corner"""
    from frequensee import scenes
    a = scenes.patch([-4, 0, 0], [4, 0, 0], [0, 0, H], 1, n_seg)
    b = scenes.patch([0, 0, 0], [0, 4, 0], [0, 0, H], 1, n_seg)
    return np.concatenate([a, b])


def test_tessellated_corner_and_shared_vertex_tie_break():
    src, lis = [[-2.0, -1.0, 1.3]], [1.0, 2.0, 1.3]
    one = dor.Scene(corner(1)).diffraction(src, lis, 30.0)[0]
    V = corner(24)
    many = dor.Scene(V).diffraction(src, lis, 30.0)[0]
    assert one["found"] == many["found"] == 1
    assert close(one["length"], 2.0 * math.sqrt(5.0)) and close(many["length"], one["length"])
    assert np.allclose(many["apex"], one["apex"], atol=1e-6) and np.allclose(one["apex"], [0, 0, 1.3], atol=1e-6)
    # S and L at the height of the vertex between strips 9 and 10 (z = 10 * 3 / 24): both segments reach it (x = |AB| and
    # x = 0), the lengths tie, the lower (tri, k) wins and both count
    z = np.float32(3.0 * 10 / 24)
    r = dor.Scene(V).diffraction([[-2.0, -1.0, z]], [1.0, 2.0, z], 30.0)[0]
    lo = _edge_of(V, [0, 0, np.float32(3.0 * 9 / 24)], [0, 0, z])
    hi = _edge_of(V, [0, 0, z], [0, 0, np.float32(3.0 * 11 / 24)])
    assert (r["edge_tri"], r["edge_k"]) == min(lo, hi)
    assert np.array_equal(r["apex"], np.array([0, 0, z], np.float32))
    edges = {tuple(e) for e in dor.edges(V, 30.0)}
    assert lo in edges and hi in edges


def test_edge_classification():
    # a T-junction: one long edge against two short ones -- three screens, whatever the threshold
    T = np.array([[[0, 0, 0], [0, 4, 0], [0, 2, 3]],
                  [[0, 0, 0], [0, 2, 0], [1, 1, -2]], [[0, 2, 0], [0, 4, 0], [1, 3, -2]]], np.float32)
    got = {tuple(e) for e in dor.edges(T, 180.0)}
    assert {(0, 0), (1, 0), (2, 0)} <= got
    # an edge held by three fins: never an edge, at any threshold
    F = np.array([[[0, 0, 0], [0, 0, 1], [1, 0, 0.5]], [[0, 0, 1], [0, 0, 0], [0, 1, 0.5]],
                  [[0, 0, 0], [0, 0, 1], [-1, -1, 0.5]]], np.float32)
    for fold in (0.0, 90.0, 180.0):
        assert (0, 0) not in {tuple(e) for e in dor.edges(F, fold)} and len(dor.edges(F, fold)) == 6
    # degenerate triangles hold no edge: the panel's bottom edge stays a screen
    D = np.concatenate([PANEL, np.array([[[0, -2, 0], [0, 2, 0], [0, 0, 0]], [[1, 1, 1], [1, 1, 1], [2, 2, 2]]], np.float32)])
    assert np.array_equal(dor.edges(D, 30.0), dor.edges(PANEL, 30.0))
    # -0.0 welds with +0.0: a 90 degree fold, one wedge, not two screens
    W = np.array([[[0, 0, 0], [0, 1, 0], [1, 0, 0]], [[-0.0, 1, -0.0], [0, 0, 0], [0, 0, 1]]], np.float32)
    assert np.signbit(W[1, 0, 0])
    assert len(dor.edges(W, 30.0)) == 5 and len(dor.edges(W, 100.0)) == 4
    # a uv sphere: its folds are a few degrees, so its edges appear only below that
    from frequensee import scenes
    U = scenes.uv_sphere([0, 0, 0], 1.0, 12, 24)
    U = np.where(np.abs(U) < 1e-6, 0.0, U).astype(np.float32)    # sin(pi) != 0: weld the south pole's points
    assert len(dor.edges(U, 30.0)) == 0
    assert len(dor.edges(U, 0.0)) > 0 and len(dor.edges(U, 5.0)) > 0
    e0 = {tuple(e) for e in dor.edges(U, 0.0)}
    assert {tuple(e) for e in dor.edges(U, 5.0)} <= e0


def test_gain_formula_and_default_bands():
    L = dor.lib()
    assert L.fso_diffraction_gain(0.0, 1000.0, 343.0) == np.float32(np.float32(1.0) / np.float32(3.0))
    assert L.fso_diffraction_gain(10.0, 8000.0, 343.0) == np.float32(0.01)
    for z, f in ((0.01, 125.0), (0.3, 500.0), (1.7, 63.0)):
        assert close(L.fso_diffraction_gain(z, f, 343.0), hand_gain(z, f), 1e-6)
    S = dor.Scene(PANEL)
    a = S.diffraction([[-2, 0.3, 1]], [2, -0.1, 1.5], 30.0)
    b = S.diffraction([[-2, 0.3, 1]], [2, -0.1, 1.5], 30.0, band_hz=[62.5 * 2 ** k for k in range(8)])
    assert a["found"][0] == 1 and a.tobytes() == b.tobytes()
    c = S.diffraction([[-2, 0.3, 1]], [2, -0.1, 1.5], 30.0, band_hz=[100.0] * 8)
    assert np.all(c["gain"][0] == c["gain"][0][0]) and c["gain"][0][0] > a["gain"][0][1]


def test_brute_force_equals_oracle_bvh():
    from frequensee import scenes
    sc = scenes.door_rooms()
    V = scenes.door_verts(sc, 60.0)
    lis = [[x, y, 1.5] for x in (6.7, 7.5, 9.0) for y in (1.0, 3.2, 5.0, 6.5)]
    found = 0
    for L in lis:
        outs = [dor.Scene(V, use_bvh=u).diffraction(sc.sources, L, 30.0, stats=True) for u in (False, True)]
        assert outs[0][0].tobytes() == outs[1][0].tobytes() and outs[0][1] == outs[1][1]
        found += int(outs[0][0]["found"][0])
    assert 0 < found < len(lis)                                    # the doorway's edges bend sound into the second room


def test_result_layout(fs):
    d = fs.capi.DIFFRACTION_DTYPE
    assert d.itemsize == 68 and d == dor.DTYPE
    assert [d.fields[k][1] for k in ("found", "n_paths", "edge_tri", "edge_k", "apex", "length", "path_difference", "gain")] \
        == [0, 4, 8, 12, 16, 28, 32, 36]


def build_diffraction_smoke(out_dir):
    exe = os.path.join(str(out_dir), "diffraction_smoke")
    libdir = os.path.join(ROOT, "audio-pathtracer_b200", "lib")
    env = dict(os.environ); env.pop("CC", None); env.pop("CXX", None)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "diffraction_smoke.cpp"), "-o", exe,
                           "-L", libdir, "-lfrequensee", "-Wl,-rpath," + libdir], env=env)
    return exe


def test_diffraction_smoke_compiles_and_fails_loudly_without_gpu(fs, tmp_path):
    """the mirror's LastDiffraction / UpdateDiffraction build from plain C++"""
    import torch
    exe = build_diffraction_smoke(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([exe, "nogpu"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CPU fallback" in r.stdout
