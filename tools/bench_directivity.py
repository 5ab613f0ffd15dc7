"""Cost of directional sources (fs_set_directivity_patterns / fs_set_source_directivity).  Writes one JSON (--out, default
profiles/directivity_<card>.json) with the card name and power limit read in the same run.

Wall ms per update (host clock around a call that ends in a synchronisation), a context without orientations and one with
them alternating within every round after a warm-up of each:
  config 2  furnished room, one source with a cardioid facing a random direction, fs_update with 2^20 pairs at depth 16
  tunnels   1 M triangles, the 64 emitters of tools/bench_sources.py (budgets by distance rank to the listener: nearest 8
            2^15 pairs at depth 16, next 16 2^14 at depth 12, remaining 40 2^12 at depth 8), each with a cardioid facing
            a random direction, fs_update_sources
The walk is the same in both arms (directivity only weights the connected paths), so the extension- and connection-ray
counts must agree; they are recorded with the times.

usage: python tools/bench_directivity.py [--rounds N] [--out PATH]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "audio-pathtracer_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_sources import alternate, gpu_info, summary  # noqa: E402


def cardioids(fs, S, seed):
    rng = np.random.default_rng(seed)
    fwd = rng.normal(size=(S, 3)).astype(np.float32)
    return fs.directivity_polar([0.5] * 8, [1.0] * 8)[None], fwd, np.zeros(S, np.uint64)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import frequensee as fs
    from frequensee import capi, scenes
    info = gpu_info()
    res = {"device": info, "rounds": args.rounds}
    cfg = fs.default_config()
    C, K = cfg.n_channels, cfg.sample_rate

    room = scenes.furnished_room()
    rs = np.asarray(room.sources, np.float32)[:1]
    rl = np.asarray(room.listener, np.float32)
    with fs.Context() as off, fs.Context() as on:
        for c in (off, on):
            c.set_scene(room.verts, room.tri_mat, room.absorption)
        pats, fwd, pat = cardioids(fs, 1, 1)
        on.set_directivity_patterns(pats)
        on.set_source_directivity(fwd, pat)
        ir = capi.host_alloc((1, C, K))
        t = alternate({"directivity_off": lambda: off.update(rs, rl, 1 << 20, 16, 2, ir_out=ir),
                       "directivity_on": lambda: on.update(rs, rl, 1 << 20, 16, 2, ir_out=ir)}, args.rounds)
        res["config2_fs_update"] = {k: summary(v) for k, v in t.items()}
        so, sn = off.stats(), on.stats()
        res["config2_fs_update"]["rays_identical"] = bool(so["ext_rays"] == sn["ext_rays"] and so["shadow_rays"] == sn["shadow_rays"])
        print("config 2:", {k: round(res["config2_fs_update"][k]["median_ms"], 3) for k in t}, flush=True)
    del room

    tun = scenes.mine_tunnels()
    src = np.asarray(tun.sources, np.float32)
    lis = np.asarray(tun.listener, np.float32)
    S = len(src)
    rank = np.argsort(np.linalg.norm(src - lis, axis=1), kind="stable")
    n = np.empty(S, np.uint64); d = np.empty(S, np.uint32)
    for r, s in enumerate(rank):
        n[s], d[s] = ((1 << 15, 16) if r < 8 else (1 << 14, 12) if r < 24 else (1 << 12, 8))
    res["tunnels"] = {"triangles": int(len(tun.verts)), "sources": S, "pairs_per_update": int(n.sum())}
    with fs.Context() as off, fs.Context() as on:
        for c in (off, on):
            c.set_scene(tun.verts, tun.tri_mat, tun.absorption)
        pats, fwd, pat = cardioids(fs, S, 2)
        on.set_directivity_patterns(pats)
        on.set_source_directivity(fwd, pat)
        ir = capi.host_alloc((S, C, K))
        t = alternate({"directivity_off": lambda: off.update_sources(src, n, d, lis, 1, ir_out=ir),
                       "directivity_on": lambda: on.update_sources(src, n, d, lis, 1, ir_out=ir)}, args.rounds)
        res["tunnels"]["fs_update_sources"] = {k: summary(v) for k, v in t.items()}
        so, sn = off.stats(), on.stats()
        res["tunnels"]["rays_identical"] = bool(so["ext_rays"] == sn["ext_rays"] and so["shadow_rays"] == sn["shadow_rays"])
        print("tunnels:", {k: round(v["median_ms"], 3) for k, v in res["tunnels"]["fs_update_sources"].items()}, flush=True)

    out = args.out or os.path.join(ROOT, "profiles", "directivity_%s.json" % info["gpu"].replace(" ", "_"))
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
