"""Moving geometry: fs_scene_update_vertices + fs_scene_refit.  The closest hit is min (t, original triangle id) of an
exact-sequence triangle test and the boxes only have to be conservative, so a refitted tree must give results bit-identical
to a tree freshly committed from the same moved triangles, and to the oracle; refitting unchanged triangles must reproduce
the committed traversal exactly (same node visits)."""
import contextlib
import os
import re
import subprocess
import threading
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROOM_WALL_TRIS = 6 * 2 * 24 * 24          # furnished_room: the tessellated shell comes first, the furniture after it


@contextlib.contextmanager
def _env(**kw):
    old = {k: os.environ.get(k) for k in kw}
    os.environ.update({k: str(v) for k, v in kw.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _ctx(fs, env=None, **over):
    with _env(**(env or {})):                 # FS_TUNE_* are read by fs_create
        return fs.Context(**over)


def _rays(rng, lo, hi, n):
    o = rng.uniform(lo, hi, size=(n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    return np.concatenate([o, d], axis=1)


def _door_rays(rng, n):
    """origins all over both rooms, a quarter of them around the doorway"""
    r = _rays(rng, [0.3, 0.3, 0.2], [11.9, 7.7, 2.8], n)
    q = n // 4
    r[:q] = _rays(rng, [5.0, 3.0, 0.2], [7.2, 5.0, 2.0], q)
    return r


def _rigid(v, deg, shift):
    a = np.deg2rad(deg)
    R = np.array([[np.cos(a), -np.sin(a), 0.0], [np.sin(a), np.cos(a), 0.0], [0.0, 0.0, 1.0]])
    return (np.asarray(v, np.float64) @ R.T + shift).astype(np.float32)


# ---- the scene helper (no GPU) -----------------------------------------------------------------------------------
def test_door_scene_helper(oracle):
    from frequensee import scenes
    sc = scenes.door_rooms()
    first, n = sc.meta["door"]
    assert first + n == sc.n_tris and sc.n_tris >= 4096
    assert np.array_equal(scenes.door_verts(sc, 0), sc.verts)
    hx, hy = sc.meta["hinge"]
    for deg in (15, 90, -40):
        v = scenes.door_verts(sc, deg)
        assert np.array_equal(v[:first], sc.verts[:first])          # only the door moves
        r0 = np.hypot(sc.verts[first:, :, 0] - hx, sc.verts[first:, :, 1] - hy)
        r1 = np.hypot(v[first:, :, 0] - hx, v[first:, :, 1] - hy)
        assert np.allclose(r0, r1, atol=1e-5) and np.array_equal(v[first:, :, 2], sc.verts[first:, :, 2])   # rigid, about z
    # a ray through the middle of the doorway: stopped by the closed door, through the open one
    o, d = [5.0, 4.0, 1.0], [1.0, 0.0, 0.0]
    hit, t, tri = oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=False).closest_hit(o, d)
    assert hit and first <= tri < first + n and abs(t - 1.08) < 1e-4
    hit, t, tri = oracle.Scene(scenes.door_verts(sc, 90), sc.tri_mat, sc.absorption, use_bvh=False).closest_hit(o, d)
    assert hit and not first <= tri < first + n and t > 1.3                 # past the dividing wall


# ---- device -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def room():
    from frequensee import scenes
    return scenes.furnished_room()


@pytest.fixture(scope="module")
def door():
    from frequensee import scenes
    return scenes.door_rooms()


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{}, {"FS_TUNE_BUILDER": 0}, {"FS_TUNE_COLLAPSE": 1}, {"FS_TUNE_COLLAPSE": 19}],
                         ids=["default", "lbvh", "greedy", "sparse"])
def test_noop_refit_reproduces_committed_traversal(fs, room, env):
    """Refitting unchanged triangles recomputes every box bit for bit (min / max unions of the same raw bounds, the same
    padding): same hits, same histogram, same surface-area cost.  The traversal counters are compared against the spread
    of repeated traces of the committed tree: they are not bit-reproducible even without a refit (on a B200 they vary by
    ~5e-4 between identical traces, with the order in which rays share warps)."""
    from frequensee import capi
    rays = _rays(np.random.default_rng(1), [0.3, 0.3, 0.2], [11.7, 8.7, 3.4], 60000)
    with _ctx(fs, env, flags=capi.FLAG_COUNT_VISITS) as ctx:
        ctx.set_scene(room.verts, room.tri_mat, room.absorption)
        t0, i0 = ctx.closest_hits(rays)
        h0 = ctx.trace(room.sources, room.listener, 1 << 18, 8, 21)
        visits = [ctx.stats()]
        for _ in range(2):
            assert np.array_equal(h0, ctx.trace(room.sources, room.listener, 1 << 18, 8, 21))
            visits.append(ctx.stats())
        ctx.update_vertices(room.verts)
        ratio = ctx.refit()
        t1, i1 = ctx.closest_hits(rays)
        h1 = ctx.trace(room.sources, room.listener, 1 << 18, 8, 21)
        s1 = ctx.stats()
    assert np.array_equal(h0, h1) and h0.any()
    assert np.array_equal(t0, t1) and np.array_equal(i0, i1)
    assert abs(ratio - 1.0) < 1e-6
    for k in ("node_visits", "tri_tests"):
        v = np.array([s[k] for s in visits], np.float64)
        assert v.min() > 0 and abs(s1[k] - v.mean()) <= max(v.max() - v.min(), 2e-3 * v.mean()), (k, v, s1[k])


VARIANTS = {
    "default": ({}, {}),                                         # persistent kernel: >= 2^17 pairs, >= 4096 triangles
    "per_bounce": ({"FS_TUNE_MEGA": 0}, {}),
    "fused": ({}, {"flags": 32}),                                # FLAG_FUSED_EXTEND: BVH2 float nodes
    "smem_treelet": ({}, {"flags": 32 | 4}),                     # + FLAG_SMEM_TREELET: the refitted treelet
    "w8": ({"FS_TUNE_W8": 1}, {}),                               # 8-wide nodes: refit = full commit
}


def _moves(room, door):
    from frequensee import scenes
    rng = np.random.default_rng(5)
    jit = room.verts.copy()
    nf = len(jit) - ROOM_WALL_TRIS
    jit[ROOM_WALL_TRIS:] += (rng.uniform(-0.15, 0.15, size=(nf, 1, 3)) + rng.normal(0, 0.01, size=(nf, 3, 3))).astype(np.float32)
    out = [("door %g" % a, door, scenes.door_verts(door, a), None) for a in (35.0, 90.0, 0.0)]
    out.append(("room_rigid", room, _rigid(room.verts, 17.0, [3.0, -2.0, 0.5]), (17.0, [3.0, -2.0, 0.5])))
    out.append(("room_jitter", room, jit, None))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_refit_equals_fresh_commit(fs, room, door, variant):
    from frequensee import capi
    env, over = VARIANTS[variant]
    rng = np.random.default_rng(11)
    live = {}
    try:
        for name, sc, verts, motion in _moves(room, door):
            if sc.name not in live:                                   # one context per scene, refitted move after move
                live[sc.name] = _ctx(fs, env, **over)
                live[sc.name].set_scene(sc.verts, sc.tri_mat, sc.absorption)
            ctx = live[sc.name]
            ctx.update_vertices(verts)
            ratio = ctx.refit()
            assert np.isfinite(ratio) and ratio > 0
            if sc.name == "door_rooms":
                rays, src, lis = _door_rays(rng, 60000), sc.sources, sc.listener
            else:
                rays = _rays(rng, [0.3, 0.3, 0.2], [11.7, 8.7, 3.4], 60000)
                src, lis = sc.sources, sc.listener
                if motion is not None:
                    rays[:, :3] = _rigid(rays[:, :3], *motion)
                    rays[:, 3:] = _rigid(rays[:, 3:], motion[0], [0.0, 0.0, 0.0])
                    src, lis = _rigid(src, *motion), _rigid(lis[None], *motion)[0]
            with _ctx(fs, env, **over) as fresh:
                fresh.set_scene(verts, sc.tri_mat, sc.absorption)
                t, i = ctx.closest_hits(rays)
                tf, i_f = fresh.closest_hits(rays)
                assert np.array_equal(t, tf) and np.array_equal(i, i_f), name
                assert (i != 0xffffffff).mean() > 0.5
                tmax = (t * rng.uniform(0.5, 1.5, len(t))).astype(np.float32)
                tmax[~np.isfinite(tmax)] = 10.0
                ha = ctx.any_hits(rays, tmax)
                assert np.array_equal(ha, fresh.any_hits(rays, tmax)), name
                h = ctx.trace(src, lis, 1 << 17, 8, 3)
                hf = fresh.trace(src, lis, 1 << 17, 8, 3)
                assert np.array_equal(h, hf), name
                assert h.any() == (name != "door 0"), name            # the closed door seals the listener's room
            if variant == "default":
                with fs.Context(flags=capi.FLAG_BRUTE_FORCE) as bf:
                    bf.set_scene(verts, sc.tri_mat, sc.absorption)
                    nb = 3000
                    tb, ib = bf.closest_hits(rays[:nb])
                    assert np.array_equal(t[:nb], tb) and np.array_equal(i[:nb], ib), name
                    assert np.array_equal(ha[:nb], bf.any_hits(rays[:nb], tmax[:nb])), name
    finally:
        for c in live.values():
            c.close()


@pytest.mark.gpu
def test_refit_matches_oracle_and_the_door_matters(fs, oracle, door):
    from frequensee import scenes
    cfg = oracle.default_config()
    hists = {}
    with fs.Context() as ctx:
        ctx.set_scene(scenes.door_verts(door, 60.0), door.tri_mat, door.absorption)     # committed open, then swung
        for ang in (0.0, 25.0, 90.0):
            v = scenes.door_verts(door, ang)
            ctx.update_vertices(v)
            ctx.refit()
            h = ctx.trace(door.sources, door.listener, 16384, 8, 0xD00D)
            st = ctx.stats()
            ho, so = oracle.Scene(v, door.tri_mat, door.absorption, use_bvh=True).trace(
                cfg, door.sources, door.listener, 16384, 8, 0xD00D, n_threads=16)
            assert np.array_equal(h, ho), ang
            assert (st["ext_rays"], st["shadow_rays"], st["connected"]) == (so["ext_rays"], so["shadow_rays"], so["connected"])
            hists[ang] = h
    assert not hists[0.0].any() and hists[25.0].any() and hists[90.0].any()   # the move really takes effect: closed = sealed


@pytest.mark.gpu
def test_grid_follows_geometry_leaving_the_committed_box(fs, door):
    """the door carried 40 m out of the scene box: with the committed quantisation grid its boxes would clamp to the grid
    edge and stop being conservative"""
    from frequensee import capi
    first, n = door.meta["door"]
    v = door.verts.copy()
    v[first:] += np.float32([40.0, 0.0, 0.0])
    rng = np.random.default_rng(8)
    m = 20000
    o = rng.uniform([44.0, 2.0, 0.2], [45.5, 6.0, 2.0], size=(m, 3)).astype(np.float32)
    target = rng.uniform([46.08, 3.5, 0.0], [46.12, 4.5, 2.1], size=(m, 3))
    d = target - o
    rays = np.concatenate([o, (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)], axis=1)
    with fs.Context(flags=capi.FLAG_BRUTE_FORCE) as bf:
        bf.set_scene(v, door.tri_mat, door.absorption)
        tb, ib = bf.closest_hits(rays)
    assert ((ib >= first) & (ib < first + n)).mean() > 0.99
    for over in ({}, {"flags": capi.FLAG_FUSED_EXTEND}):
        with fs.Context(**over) as ctx:
            ctx.set_scene(door.verts, door.tri_mat, door.absorption)
            ctx.update_vertices(v[first:], first)
            ctx.refit()
            t, i = ctx.closest_hits(rays)
        assert np.array_equal(t, tb) and np.array_equal(i, ib)


@pytest.mark.gpu
def test_partial_range_equals_fresh_commit_of_the_whole_scene(fs, door):
    from frequensee import scenes
    first, n = door.meta["door"]
    v = scenes.door_verts(door, 50.0)
    rays = _door_rays(np.random.default_rng(2), 40000)
    with fs.Context() as ctx, fs.Context() as fresh:
        ctx.set_scene(door.verts, door.tri_mat, door.absorption)
        ctx.update_vertices(v[first:first + n], first)
        ctx.refit()
        fresh.set_scene(v, door.tri_mat, door.absorption)
        t, i = ctx.closest_hits(rays)
        tf, i_f = fresh.closest_hits(rays)
        assert np.array_equal(t, tf) and np.array_equal(i, i_f)
        h = ctx.trace(door.sources, door.listener, 1 << 17, 8, 4)
        assert np.array_equal(h, fresh.trace(door.sources, door.listener, 1 << 17, 8, 4))


@pytest.mark.gpu
def test_tiny_scenes_and_several_updates_before_one_refit(fs, door):
    from frequensee import scenes
    ab = np.full((1, 8), 0.3, np.float32)
    one = np.array([[[0, 0, 2], [4, 0, 2], [0, 4, 2]]], np.float32)
    two = np.array([[[0, 0, 2], [4, 0, 2], [0, 4, 2]], [[-3, -1, 0], [3, -1, 0], [0, 5, 0]]], np.float32)
    rng = np.random.default_rng(6)
    for base in (one, two):
        moved = base + np.float32([0.7, -0.4, 0.9])
        moved[0, 1] += np.float32([1.5, 0.5, -0.3])                              # and one vertex of it non-rigidly
        mats = np.zeros(len(base), np.uint32)
        rays = _rays(rng, [-1, -1, -1], [3, 3, 4], 8000)
        with fs.Context() as ctx, fs.Context() as fresh:
            ctx.set_scene(base, mats, ab)
            ctx.update_vertices(moved)
            ctx.refit()
            fresh.set_scene(moved, mats, ab)
            t, i = ctx.closest_hits(rays)
            tf, i_f = fresh.closest_hits(rays)
            assert np.array_equal(t, tf) and np.array_equal(i, i_f) and (i != 0xffffffff).any()
            h = ctx.trace([[1, 1, 1]], [1.5, 1.2, 0.5], 4096, 4, 3)
            assert np.array_equal(h, fresh.trace([[1, 1, 1]], [1.5, 1.2, 0.5], 4096, 4, 3))
    first, n = door.meta["door"]
    final = scenes.door_verts(door, 75.0)
    final[100:140] += np.float32([0.0, 0.0, 0.05])                             # part of the shell lifted too
    with fs.Context() as ctx, fs.Context() as fresh:
        ctx.set_scene(door.verts, door.tri_mat, door.absorption)
        ctx.update_vertices(scenes.door_verts(door, 10.0)[first:], first)
        ctx.update_vertices(scenes.door_verts(door, 30.0)[first:], first)
        ctx.update_vertices(final[100:140], 100)
        ctx.update_vertices(final[first:], first)
        ctx.refit()
        fresh.set_scene(final, door.tri_mat, door.absorption)
        rays = _door_rays(rng, 30000)
        t, i = ctx.closest_hits(rays)
        tf, i_f = fresh.closest_hits(rays)
        assert np.array_equal(t, tf) and np.array_equal(i, i_f)
        h = ctx.trace(door.sources, door.listener, 1 << 17, 8, 5)
        assert np.array_equal(h, fresh.trace(door.sources, door.listener, 1 << 17, 8, 5))


@pytest.mark.gpu
def test_state_and_errors(fs, door):
    from frequensee import capi, scenes
    E = fs.FrequenSeeError
    first, n = door.meta["door"]
    v = scenes.door_verts(door, 40.0)
    with fs.Context() as ctx:
        with pytest.raises(E) as ei:
            ctx.update_vertices(v)
        assert ei.value.code == capi.FS_ERR_STATE                           # before fs_scene_set_triangles
        with pytest.raises(E) as ei:
            ctx.refit()
        assert ei.value.code == capi.FS_ERR_STATE                           # nothing committed
        tm = np.ascontiguousarray(door.tri_mat)
        ab = np.ascontiguousarray(door.absorption)
        verts = np.ascontiguousarray(door.verts)
        assert ctx.L.fs_scene_set_triangles(ctx.h, verts.ctypes.data, tm.ctypes.data, len(verts)) == 0
        assert ctx.L.fs_scene_set_materials(ctx.h, ab.ctypes.data, ab.shape[0], ab.shape[1]) == 0
        with pytest.raises(E) as ei:
            ctx.refit()
        assert ei.value.code == capi.FS_ERR_STATE                           # set, not committed
        assert ctx.L.fs_scene_commit(ctx.h) == 0
        rays = _door_rays(np.random.default_rng(3), 20000)
        t0, i0 = ctx.closest_hits(rays)
        h0 = ctx.trace(door.sources, door.listener, 1 << 16, 8, 9)
        bad_nan = v[first:].copy(); bad_nan[3, 1, 2] = np.nan
        bad_big = v[first:].copy(); bad_big[0, 0, 0] = 1e19
        for args in ((v[:1], door.n_tris), (v[:2], door.n_tris - 1), (v, 1), (bad_nan, first), (bad_big, first)):
            with pytest.raises(E) as ei:
                ctx.update_vertices(*args)
            assert ei.value.code == capi.FS_ERR_INVALID
        t1, i1 = ctx.closest_hits(rays)                                     # rejected calls changed nothing
        assert np.array_equal(t0, t1) and np.array_equal(i0, i1)
        assert np.array_equal(h0, ctx.trace(door.sources, door.listener, 1 << 16, 8, 9))
        ctx.update_vertices(v[first:], first)
        for call in (lambda: ctx.trace(door.sources, door.listener, 4096, 8, 9),
                     lambda: ctx.update(door.sources, door.listener, 4096, 8, 9),
                     lambda: ctx.closest_hits(rays[:10]),
                     lambda: ctx.any_hits(rays[:10], np.ones(10, np.float32))):
            with pytest.raises(E) as ei:
                call()
            assert ei.value.code == capi.FS_ERR_STATE and "refit" in str(ei.value)
        ctx.refit()
        h_refit = ctx.trace(door.sources, door.listener, 1 << 16, 8, 9)
        assert not np.array_equal(h_refit, h0)
    with fs.Context() as ctx:                                               # fs_scene_commit after an update = the refit
        ctx.set_scene(door.verts, door.tri_mat, door.absorption)
        ctx.update_vertices(v[first:], first)
        assert ctx.L.fs_scene_commit(ctx.h) == 0
        assert np.array_equal(h_refit, ctx.trace(door.sources, door.listener, 1 << 16, 8, 9))


@pytest.mark.gpu
def test_audio_thread_runs_through_door_moves(fs, door):
    from frequensee import scenes
    first, n = door.meta["door"]
    rng = np.random.default_rng(12)
    x = rng.uniform(-0.5, 0.5, size=(1024, 2)).astype(np.float32)
    angles = [10.0, 30.0, 50.0, 70.0, 90.0, 65.0]
    N = 1 << 16
    ir = np.zeros((1, 2, 48000), np.float32)
    with fs.Context(conv_clamp=0) as ctx:
        ctx.set_scene(door.verts, door.tri_mat, door.absorption)
        ctx.update(door.sources, door.listener, N, 8, 1, ir_out=ir)
        ctx.conv_init_source(0)
        stop, errors, blocks = threading.Event(), [], [0]

        def audio():
            try:
                while not stop.is_set():
                    ctx.conv_process(x, 0)
                    blocks[0] += 1
                    time.sleep(0.001)
            except Exception as e:                                          # pragma: no cover
                errors.append(e)

        th = threading.Thread(target=audio)
        th.start()
        try:
            for k, a in enumerate(angles):
                ctx.update_vertices(scenes.door_verts(door, a)[first:], first)
                ctx.refit()
                ctx.update(door.sources, door.listener, N, 8, 100 + k, ir_out=ir)
        finally:
            stop.set()
            th.join()
        assert not errors, errors
        assert blocks[0] > 0
    ir_ref = np.zeros_like(ir)
    with fs.Context(conv_clamp=0) as fresh:
        fresh.set_scene(scenes.door_verts(door, angles[-1]), door.tri_mat, door.absorption)
        fresh.update(door.sources, door.listener, N, 8, 100 + len(angles) - 1, ir_out=ir_ref)
    assert np.abs(ir).max() > 0 and np.array_equal(ir, ir_ref)


@pytest.mark.gpu
def test_multi_gpu_refit_equals_single_device(fs, door):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from frequensee import scenes
    first, n = door.meta["door"]
    with fs.MultiContext([0, 1]) as m, fs.Context(device=0) as one:
        m.set_scene(door.verts, door.tri_mat, door.absorption)
        one.set_scene(door.verts, door.tri_mat, door.absorption)
        for a in (20.0, 80.0):
            v = scenes.door_verts(door, a)[first:]
            m.update_vertices(v, first)
            one.update_vertices(v, first)
            assert m.refit() == one.refit()
            hm = m.trace(door.sources, door.listener, 1 << 18, 8, 31)
            assert np.array_equal(hm, one.trace(door.sources, door.listener, 1 << 18, 8, 31))


@pytest.mark.gpu
def test_cpp_mirror_move_geometry():
    exe = os.path.join(ROOT, "tests", "cpp", "dynamic_smoke")
    src = os.path.join(ROOT, "tests", "cpp", "dynamic_smoke.cpp")
    hpp = os.path.join(ROOT, "include", "frequensee.hpp")
    libdir = os.path.join(ROOT, "audio-pathtracer_b200", "lib")
    if not os.path.exists(exe) or os.path.getmtime(exe) < max(os.path.getmtime(src), os.path.getmtime(hpp)):
        env = dict(os.environ); env.pop("CC", None); env.pop("CXX", None)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
                               "-L", libdir, "-lfrequensee", "-Wl,-rpath," + libdir], env=env)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    kv = dict(re.findall(r"(\w+)=([-+.\w]+)", r.stdout))
    assert kv["same"] == "1", r.stdout
    assert kv["closed_differs"] == "1" and int(kv["connected_open"]) > 0
    assert int(kv["refits"]) == 3 and int(kv["rebuilds"]) == 1, r.stdout     # three refits after the first build
