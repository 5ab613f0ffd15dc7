"""Per-source budgets in one call (fs_update_sources) against the alternatives an integrator has without it.  Writes one
JSON (--out, default profiles/sources_<card>.json) with the card name and power limit read in the same run.

  tunnels (1 M triangles, 64 sources, one listener), budgets by distance rank to the listener: nearest 8 sources 2^15 pairs
  at depth 16, next 16 2^14 at depth 12, remaining 40 2^12 at depth 8 (688 128 pairs).  Wall ms per update of all 64 IRs
  (host clock around the call, which ends in a synchronisation):
    A  64 fs_update calls with one source each, each with its own budget (what ForceUpdateSources does)
    B  one fs_update_sources
    C  one uniform fs_update with 2^14 pairs at depth 16 for all 64 sources
  table cost: fs_update_sources with equal budgets against fs_update with the same arguments, on the furnished room
  (config 2: one source, 2^20 pairs, depth 16) and on the tunnels (64 x 2^14 pairs, depth 16).
Arms alternate within every round after a warm-up of each.

usage: python tools/bench_sources.py [--rounds N] [--out PATH]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "audio-pathtracer_b200"))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.strip().split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def wall_ms(fn):
    t0 = time.perf_counter()
    fn()
    return 1e3 * (time.perf_counter() - t0)


def alternate(arms, rounds, warmup=2):
    """arms: {name: fn}; every fn ends in a host synchronisation.  Returns {name: [ms per round]}"""
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    out = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            out[k].append(wall_ms(fn))
    return out


def summary(times):
    a = np.asarray(times, np.float64)
    return {"median_ms": float(np.median(a)), "min_ms": float(a.min()), "max_ms": float(a.max()), "runs": len(a)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import frequensee as fs
    from frequensee import scenes
    info = gpu_info()
    res = {"device": info, "rounds": args.rounds}
    cfg = fs.default_config()
    C, K = cfg.n_channels, cfg.sample_rate

    tun = scenes.mine_tunnels()
    src = np.asarray(tun.sources, np.float32)
    lis = np.asarray(tun.listener, np.float32)
    S = len(src)
    rank = np.argsort(np.linalg.norm(src - lis, axis=1), kind="stable")
    n = np.empty(S, np.uint64); d = np.empty(S, np.uint32)
    for r, s in enumerate(rank):
        n[s], d[s] = ((1 << 15, 16) if r < 8 else (1 << 14, 12) if r < 24 else (1 << 12, 8))
    res["tunnels"] = {"triangles": int(len(tun.verts)), "sources": S, "pairs_per_update": int(n.sum())}
    with fs.Context() as ctx:
        ctx.set_scene(tun.verts, tun.tri_mat, tun.absorption)
        ir_all = fs.capi.host_alloc((S, C, K))
        ir_one = fs.capi.host_alloc((1, C, K))
        seed = [1]

        def arm_a():
            for s in range(S):
                ctx.update(src[s:s + 1], lis, int(n[s]), int(d[s]), seed[0], ir_out=ir_one)

        def arm_b():
            ctx.update_sources(src, n, d, lis, seed[0], ir_out=ir_all)

        def arm_c():
            ctx.update(src, lis, 1 << 14, 16, seed[0], ir_out=ir_all)

        t = alternate({"A_per_source_updates": arm_a, "B_update_sources": arm_b, "C_uniform_update": arm_c}, args.rounds)
        res["tunnels"]["budgets"] = {k: summary(v) for k, v in t.items()}
        print("tunnels budgets:", {k: round(v["median_ms"], 3) for k, v in res["tunnels"]["budgets"].items()}, flush=True)

        def eq_update():
            ctx.update(src, lis, 1 << 14, 16, 2, ir_out=ir_all)

        def eq_sources():
            ctx.update_sources(src, 1 << 14, 16, lis, 2, ir_out=ir_all)

        t = alternate({"fs_update": eq_update, "fs_update_sources": eq_sources, "fs_update_again": eq_update}, args.rounds)
        res["tunnels"]["table_cost"] = {k: summary(v) for k, v in t.items()}
        print("tunnels table cost:", {k: round(v["median_ms"], 3) for k, v in res["tunnels"]["table_cost"].items()}, flush=True)
    del tun

    room = scenes.furnished_room()
    rs = np.asarray(room.sources, np.float32)[:1]
    rl = np.asarray(room.listener, np.float32)
    with fs.Context() as ctx:
        ctx.set_scene(room.verts, room.tri_mat, room.absorption)
        ir1 = fs.capi.host_alloc((1, C, K))

        def u():
            ctx.update(rs, rl, 1 << 20, 16, 2, ir_out=ir1)

        def us():
            ctx.update_sources(rs, 1 << 20, 16, rl, 2, ir_out=ir1)

        t = alternate({"fs_update": u, "fs_update_sources": us, "fs_update_again": u}, args.rounds)
        res["room_table_cost"] = {k: summary(v) for k, v in t.items()}
        print("room table cost:", {k: round(v["median_ms"], 3) for k, v in res["room_table_cost"].items()}, flush=True)

    out = args.out or os.path.join(ROOT, "profiles", "sources_%s.json" % info["gpu"].replace(" ", "_"))
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
