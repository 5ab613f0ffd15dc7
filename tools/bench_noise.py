"""Cost and effect of FS_FLAG_NOISE_STATS.  Writes one JSON (--out, default profiles/noise_<card>.json) with the card name
and power limit read in the same run.

  cost: wall ms per update (host clock around a call that ends in a synchronisation), a context without the flag and one
  with it alternating within every round after a warm-up of each:
    config 2  furnished room, one source, fs_update with 2^20 pairs at depth 16
    tunnels   1 M triangles, 64 sources, fs_update_sources with budgets by distance rank to the listener (nearest 8: 2^15
              pairs at depth 16, next 16: 2^14 at depth 12, remaining 40: 2^12 at depth 8; 688 128 pairs)
  and the wall time of the C calls fs_get_noise + fs_allocate_paths for the 64 tunnel sources (preallocated buffers).
  loop: broadband snr_db (min / median / max over the sources with energy) of the tunnels with the distance-rank budgets,
  then after 1 and 4 updates whose budgets fs_allocate_paths chose from the previous update (same total, 2^10 .. 2^17 per
  source, depths kept, a new seed per update).

usage: python tools/bench_noise.py [--rounds N] [--out PATH]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "audio-pathtracer_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_sources import alternate, gpu_info, summary  # noqa: E402


def snr_summary(st):
    v = st["snr_db"][~st["no_energy"]]
    return {"min_db": float(v.min()), "median_db": float(np.median(v)), "max_db": float(v.max()),
            "std_db": float(np.std(v)), "sources_with_energy": int(len(v))}


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
    with fs.Context() as off, fs.Context(flags=capi.FLAG_NOISE_STATS) as on:
        ir = capi.host_alloc((1, C, K))
        for c in (off, on):
            c.set_scene(room.verts, room.tri_mat, room.absorption)
        h_off = np.zeros((1, cfg.n_bands, cfg.n_bins), np.uint64); h_on = np.zeros_like(h_off)
        t = alternate({"flag_off": lambda: off.update(rs, rl, 1 << 20, 16, 2, ir_out=ir),
                       "flag_on": lambda: on.update(rs, rl, 1 << 20, 16, 2, ir_out=ir)}, args.rounds)
        off.update(rs, rl, 1 << 20, 16, 2, hist_out=h_off); on.update(rs, rl, 1 << 20, 16, 2, hist_out=h_on)
        res["config2_fs_update"] = {k: summary(v) for k, v in t.items()}
        res["config2_fs_update"]["histograms_identical"] = bool(np.array_equal(h_off, h_on))
        res["config2_fs_update"]["snr"] = snr_summary(on.noise_stats())
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
    total, lo, hi = int(n.sum()), 1 << 10, 1 << 17
    res["tunnels"] = {"triangles": int(len(tun.verts)), "sources": S, "pairs_per_update": total}
    with fs.Context() as off, fs.Context(flags=capi.FLAG_NOISE_STATS) as on:
        for c in (off, on):
            c.set_scene(tun.verts, tun.tri_mat, tun.absorption)
        ir = capi.host_alloc((S, C, K))
        t = alternate({"flag_off": lambda: off.update_sources(src, n, d, lis, 1, ir_out=ir),
                       "flag_on": lambda: on.update_sources(src, n, d, lis, 1, ir_out=ir)}, args.rounds)
        res["tunnels"]["fs_update_sources"] = {k: summary(v) for k, v in t.items()}
        ho = np.zeros((S, cfg.n_bands, cfg.n_bins), np.uint64); hn = np.zeros_like(ho)
        off.update_sources(src, n, d, lis, 1, hist_out=ho); on.update_sources(src, n, d, lis, 1, hist_out=hn)
        res["tunnels"]["histograms_identical"] = bool(np.array_equal(ho, hn))
        # the two C entry points a game calls, with preallocated arrays (ctypes call overhead only, no Python loops)
        L = capi.load()
        arr = (capi.NoiseStats * S)()
        nxt = np.zeros(S, np.uint64)
        ms = []
        for _ in range(args.rounds):
            t0 = time.perf_counter()
            rc = L.fs_get_noise(on.h, arr, S)
            rc |= L.fs_allocate_paths(arr, S, total, lo, hi, None, nxt.ctypes.data)
            ms.append(1e3 * (time.perf_counter() - t0))
            assert rc == 0
        res["tunnels"]["get_noise_plus_allocate"] = summary(ms)
        print("tunnels:", {k: round(v["median_ms"], 3) for k, v in res["tunnels"]["fs_update_sources"].items()},
              "noise + allocate %.3f ms" % res["tunnels"]["get_noise_plus_allocate"]["median_ms"], flush=True)
        # the allocation loop
        loop = []
        budgets = n.copy()
        for step in range(5):
            on.update_sources(src, budgets, d, lis, 1000 + step, ir_out=ir)
            st = on.noise_stats()
            loop.append(dict(snr_summary(st), update=step, allocated=step > 0,
                             clamped_min=int((budgets == lo).sum()), clamped_max=int((budgets == hi).sum())))
            print("loop", loop[-1], flush=True)
            budgets = fs.allocate_paths(st, total, lo, hi)
        res["tunnels"]["allocation_loop"] = {"min_paths": lo, "max_paths": hi, "total": total, "updates": loop}

    out = args.out or os.path.join(ROOT, "profiles", "noise_%s.json" % info["gpu"].replace(" ", "_"))
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
