"""Cost of the first-order edge diffraction query (fs_diffraction).  Writes one JSON (--out, default
profiles/diffraction_<card>.json) with the card name and power limit read in the same run.

Per case and fold threshold (30 and 60 degrees), wall ms (host clock around the call, which ends in a synchronisation),
median / min / max over --rounds calls:
  first   the call right after a threshold change: edge extraction (hash, radix sort, grouping, compaction) and the query;
          the calls alternate between the two thresholds, so every one rebuilds
  steady  repeated calls at one threshold: the query alone on the cached edge set
  door     door_rooms (door open 60 degrees), its 1 source, listener in the second room
  room     furnished room (100 k triangles), 16 sources at seeded positions
  tunnels  mine tunnels (1 M triangles), their 64 sources
Edge counts, candidate pairs (source, edge) that pass the geometric tests, leg rays traced and paths found come from the CPU
reference (tests/oracle_ext/fso_diffraction.c), which makes the same choices; its single-thread time on the same inputs is
recorded for context.

usage: python tools/bench_diffraction.py [--rounds N] [--out PATH]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(ROOT)
for p in (os.path.join(REPO, "audio-pathtracer_b200"), os.path.join(REPO, "oracle"), os.path.join(REPO, "tests"), ROOT):
    sys.path.insert(0, p)
from bench_sources import gpu_info, summary  # noqa: E402

FOLDS = (30.0, 60.0)


def run_case(fs, dor, verts, tri_mat, absorption, src, lis, rounds):
    out = {"triangles": int(len(verts)), "sources": int(len(src))}
    with fs.Context() as ctx:
        ctx.set_scene(verts, tri_mat, absorption)
        ctx.diffraction(src, lis, FOLDS[1])
        first = {f: [] for f in FOLDS}
        for i in range(2 * rounds):
            f = FOLDS[i % 2]
            t0 = time.perf_counter()
            ctx.diffraction(src, lis, f)
            first[f].append(1e3 * (time.perf_counter() - t0))
        R = dor.Scene(verts)
        for f in FOLDS:
            for _ in range(3):
                r = ctx.diffraction(src, lis, f)
            steady = []
            for _ in range(rounds):
                t0 = time.perf_counter()
                r = ctx.diffraction(src, lis, f)
                steady.append(1e3 * (time.perf_counter() - t0))
            t0 = time.perf_counter()
            ref, (n_edges, n_cand, n_rays) = R.diffraction(src, lis, f, stats=True)
            ref_ms = 1e3 * (time.perf_counter() - t0)
            out["fold_%d" % f] = {"first": summary(first[f]), "steady": summary(steady), "edges": n_edges, "candidates": n_cand,
                                  "leg_rays": n_rays, "found": int(r["found"].sum()), "paths": int(r["n_paths"].sum()),
                                  "same_as_reference": r.tobytes() == ref.tobytes(), "cpu_reference_ms": ref_ms}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import frequensee as fs
    from frequensee import scenes
    import diffraction_oracle as dor
    info = gpu_info()
    res = {"device": info, "rounds": args.rounds}
    door = scenes.door_rooms()
    res["door"] = run_case(fs, dor, scenes.door_verts(door, 60.0), door.tri_mat, door.absorption,
                           np.asarray(door.sources, np.float32), [9.0, 2.5, 1.5], args.rounds)
    room = scenes.furnished_room()
    src = np.random.default_rng(2).uniform([0.5, 0.5, 0.3], [11.5, 8.5, 3.3], (16, 3)).astype(np.float32)
    res["room"] = run_case(fs, dor, room.verts, room.tri_mat, room.absorption, src, room.listener, args.rounds)
    tun = scenes.mine_tunnels()
    res["tunnels"] = run_case(fs, dor, tun.verts, tun.tri_mat, tun.absorption, np.asarray(tun.sources, np.float32),
                              tun.listener, args.rounds)
    out = args.out or os.path.join(REPO, "profiles", "diffraction_%s.json" % info["gpu"].replace(" ", "_"))
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
