"""BVH2 reinsertion (FS_TUNE_REINSERT): the pass only moves subtrees, so it must never make the surface-area cost worse, and
the results cannot depend on it -- the closest hit is min (t, original triangle id) and every box stays an exact min / max
union of its triangles' bounds."""
import contextlib
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_COST_LINE = re.compile(r"reinsertion: (\d+) iterations, (\d+) moves, surface-area cost ([0-9.e+-]+) -> ([0-9.e+-]+)")

_COMMIT_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
from frequensee import scenes, capi
sc = scenes.by_name(sys.argv[2], **eval(sys.argv[3]))
with capi.Context() as ctx:
    ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption)
"""


def _commit_log(scene, kw, env):
    e = dict(os.environ, FS_VERBOSE="1", **{k: str(v) for k, v in env.items()})
    r = subprocess.run([sys.executable, "-c", _COMMIT_SCRIPT, os.path.join(ROOT, "audio-pathtracer_b200"), scene, repr(kw)],
                       env=e, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("scene,kw", [("furnished_room", {}), ("door_rooms", {}), ("concert_hall", {"target_tris": 400_000})],
                         ids=["room", "door_rooms", "hall_400k"])
def test_reinsertion_never_raises_cost(scene, kw):
    m = _COST_LINE.search(_commit_log(scene, kw, {}))
    assert m, "no reinsertion report"
    iters, moves, c0, c1 = int(m.group(1)), int(m.group(2)), float(m.group(3)), float(m.group(4))
    assert iters >= 1 and c1 <= c0
    if scene == "furnished_room":
        assert moves > 0 and c1 < 0.99 * c0             # the room's PLOC tree has slack a reinsertion finds
    off = _commit_log(scene, kw, {"FS_TUNE_REINSERT": 0})
    assert not _COST_LINE.search(off)


@contextlib.contextmanager
def _reinsert(iters):
    """FS_TUNE_REINSERT is read when the scene is committed"""
    old = os.environ.get("FS_TUNE_REINSERT")
    if iters is not None:
        os.environ["FS_TUNE_REINSERT"] = str(iters)
    try:
        yield
    finally:
        if old is None:
            os.environ.pop("FS_TUNE_REINSERT", None)
        else:
            os.environ["FS_TUNE_REINSERT"] = old


def _rays(rng, lo, hi, n):
    o = rng.uniform(lo, hi, size=(n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    return np.concatenate([o, d], axis=1)


@pytest.mark.gpu
@pytest.mark.parametrize("scene,kw,paths,depth", [("furnished_room", {}, 1 << 18, 16),
                                                  ("concert_hall", {"target_tris": 400_000}, 1 << 17, 32)],
                         ids=["room", "hall_400k"])
def test_results_do_not_depend_on_reinsertion(fs, scene, kw, paths, depth):
    from frequensee import scenes, capi
    sc = scenes.by_name(scene, **kw)
    v = sc.verts.reshape(-1, 3)
    rays = _rays(np.random.default_rng(7), v.min(0), v.max(0), 100_000)
    out = {}
    for reinsert in (0, None):
        with _reinsert(reinsert), fs.Context(flags=capi.FLAG_COUNT_VISITS) as ctx:
            ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption)
            t, tri = ctx.closest_hits(rays)
            h = ctx.trace(sc.sources[:1], sc.listener, paths, depth, 5)
            out[reinsert] = (t, tri, h, ctx.stats())
    (t0, i0, h0, s0), (t1, i1, h1, s1) = out[0], out[None]
    assert h0.any() and np.array_equal(h0, h1)
    assert np.array_equal(t0, t1) and np.array_equal(i0, i1)
    if scene == "furnished_room":
        assert s1["node_visits"] < s0["node_visits"], (s0["node_visits"], s1["node_visits"])
