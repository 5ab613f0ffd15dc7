"""Cost of the direct-path occlusion query (fs_occlusion).  Writes one JSON (--out, default profiles/occlusion_<card>.json) with
the card name and power limit read in the same run.

Per case, after a warm-up: device ms (CUDA events on the context stream around the call's upload, zeroing, k_occlusion and
read-back) and wall ms (host clock around the call, which ends in a synchronisation), median / min / max over --rounds calls.
  tunnels  1 M triangles, the 64 emitters of the scene, radius 0.5 m, 1 / 64 / 256 / 1024 rays each, max_crossings 8
  room     furnished room (100 k triangles), 16 emitters at seeded positions, the same ray counts
Materials carry a seeded random Transmission (0..0.5) and ThicknessCm (0.5..10), so rays continue through the surfaces they
cross and every hit on the way is found.  The visible fraction and mean transmission are recorded with the times.

usage: python tools/bench_occlusion.py [--rounds N] [--out PATH]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(ROOT), "audio-pathtracer_b200"))
sys.path.insert(0, ROOT)
from bench_sources import gpu_info, summary  # noqa: E402

RAYS = (1, 64, 256, 1024)


def materials(sc, seed):
    rng = np.random.default_rng(seed)
    M, B = sc.absorption.shape
    return (rng.uniform(0.0, 0.5, (M, B)).astype(np.float32), None, rng.uniform(0.5, 10.0, M).astype(np.float32))


def run_case(fs, torch, sc, src, rounds, seed):
    out = {}
    with fs.Context() as ctx:
        ctx.set_scene_ex(sc.verts, sc.tri_mat, sc.absorption, *materials(sc, seed))
        stream = torch.cuda.Stream()
        ctx.set_stream(stream.cuda_stream)
        for n in RAYS:
            def call():
                return ctx.occlusion(src, 0.5, n, sc.listener, max_crossings=8, seed=seed)
            for _ in range(3):
                call()
            dev, wall = [], []
            for _ in range(rounds):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                t0 = time.perf_counter()
                vis, tr = call()
                wall.append(1e3 * (time.perf_counter() - t0))
                e1.record(stream)
                e1.synchronize()
                dev.append(e0.elapsed_time(e1))
            out["rays_%d" % n] = {"sources": len(src), "rays_total": len(src) * n, "device": summary(dev), "wall": summary(wall),
                                  "visible_mean": float(vis.mean()), "transmission_mean": float(tr.mean())}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import frequensee as fs
    from frequensee import scenes
    info = gpu_info()
    res = {"device": info, "rounds": args.rounds, "radius_m": 0.5, "max_crossings": 8}
    tun = scenes.mine_tunnels()
    res["tunnels"] = {"triangles": int(len(tun.verts)),
                      **run_case(fs, torch, tun, np.asarray(tun.sources, np.float32), args.rounds, 1)}
    room = scenes.furnished_room()
    src = np.random.default_rng(2).uniform([0.5, 0.5, 0.3], [11.5, 8.5, 3.3], (16, 3)).astype(np.float32)
    res["room"] = {"triangles": int(len(room.verts)), **run_case(fs, torch, room, src, args.rounds, 2)}
    out = args.out or os.path.join(os.path.dirname(ROOT), "profiles", "occlusion_%s.json" % info["gpu"].replace(" ", "_"))
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
