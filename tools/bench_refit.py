"""Moving geometry on the device: fs_scene_refit against fs_scene_commit, what a refitted tree costs the trace, and the
interactive loop of a swinging door.  Writes one JSON (--out, default profiles/refit_<card>.json) with the card name and
power limit read in the same run.

  per scene (room 99 k, tunnels 1 M, hall 5 M triangles): fs_scene_commit (median of repeated commits), fs_scene_refit wall
    clock around the call (it ends in a host synchronisation; median after warm-up) and refit device time (CUDA events on
    the context stream around the call)
  degradation (room): cost ratio and trace time of the refitted tree against the size of the motion -- a rigid rotation of
    the whole room, then per-triangle jitter of the furniture -- with the trace time after a full commit of the same geometry
  interactive loop (door_rooms): 60 frames of update_vertices(door) + refit + update, against 60 static update frames

usage: python tools/bench_refit.py [--scenes room,tunnels,hall] [--out PATH]
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

ROOM_WALL_TRIS = 6 * 2 * 24 * 24          # furnished_room: the shell comes first, the furniture after it
N_PAIRS, DEPTH = 1 << 20, 16              # one IR update of BASELINE configs[1]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.strip().split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def med(x):
    return float(np.median(np.asarray(x, np.float64)))


def timed_refit(ctx, torch, reps, warmup=3):
    """wall clock (ms) around fs_scene_refit, and device time between CUDA events recorded on the context stream"""
    wall, dev = [], []
    for r in range(warmup + reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        ratio = ctx.refit()
        t1 = time.perf_counter()
        e1.record()
        e1.synchronize()
        if r >= warmup:
            wall.append(1e3 * (t1 - t0))
            dev.append(e0.elapsed_time(e1))
    return med(wall), med(dev), ratio


def commit_ms(ctx, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        ctx._ck(ctx.L.fs_scene_commit(ctx.h))         # ends in a host synchronisation
        out.append(1e3 * (time.perf_counter() - t0))
    return med(out)


def trace_ms(ctx, sc, reps=5, seed=1):
    ctx.trace(sc.sources, sc.listener, N_PAIRS, DEPTH, seed, want_hist=False)
    ctx.synchronize()
    out = []
    for r in range(reps):
        ctx.trace(sc.sources[:1], sc.listener, N_PAIRS, DEPTH, seed + r)
        out.append(ctx.stats()["last_trace_ms"])
    return med(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", default="room,tunnels,hall")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import frequensee as fs
    from frequensee import scenes
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    info = gpu_info()
    torch.cuda.init()
    stream = torch.cuda.current_stream()
    res = {"tool": "tools/bench_refit.py", **info, "trace": {"pairs": N_PAIRS, "depth": DEPTH}, "scenes": {}}
    build = {"room": lambda: scenes.furnished_room(), "tunnels": lambda: scenes.mine_tunnels(),
             "hall": lambda: scenes.concert_hall()}
    for key in args.scenes.split(","):
        sc = build[key]()
        with fs.Context(device=0) as ctx:
            ctx.set_stream(stream.cuda_stream)          # the CUDA events below are recorded on the context's stream
            ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption)
            c_ms = commit_ms(ctx, 3 if sc.n_tris > 2_000_000 else 7)
            ctx.update_vertices(sc.verts)
            w_ms, d_ms, ratio = timed_refit(ctx, torch, args.reps)
            row = {"n_tris": sc.n_tris, "commit_ms": c_ms, "refit_wall_ms": w_ms, "refit_device_ms": d_ms,
                   "commit_over_refit": c_ms / w_ms, "noop_cost_ratio": ratio}
            print(key, json.dumps(row), flush=True)
            res["scenes"][key] = row
    # degradation: room, rigid rotation of everything, then furniture jitter of growing amplitude
    sc = scenes.furnished_room()
    rng = np.random.default_rng(1)
    nf = sc.n_tris - ROOM_WALL_TRIS
    dirs = rng.normal(size=(nf, 1, 3))
    dirs /= np.linalg.norm(dirs, axis=2, keepdims=True)
    curve = []
    with fs.Context(device=0) as ctx:
        ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption)
        base = trace_ms(ctx, sc)
        c = np.array([6.0, 4.5, 1.8])
        moves = []
        for deg in (2.0, 5.0, 15.0, 45.0):
            a = np.deg2rad(deg)
            R = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1.0]])
            moves.append(("rigid_rotation_deg", deg, ((sc.verts - c) @ R.T + c).astype(np.float32)))
        for amp in (0.01, 0.03, 0.1, 0.3, 1.0):
            v = sc.verts.copy()
            v[ROOM_WALL_TRIS:] += (amp * dirs * rng.uniform(0, 1, size=(nf, 1, 1))).astype(np.float32)
            moves.append(("furniture_jitter_m", amp, v))
        for kind, size, v in moves:
            ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption)           # every move starts from the committed room
            ctx.update_vertices(v)
            ratio = ctx.refit()
            t_refit = trace_ms(ctx, sc)
            ctx._ck(ctx.L.fs_scene_commit(ctx.h))                        # full build of the same geometry
            t_full = trace_ms(ctx, sc)
            row = {"motion": kind, "size": size, "cost_ratio": ratio, "trace_ms_refit": t_refit, "trace_ms_rebuilt": t_full,
                   "slowdown": t_refit / t_full}
            print(json.dumps(row), flush=True)
            curve.append(row)
    res["degradation"] = {"scene": "furnished_room", "trace_ms_committed": base, "rows": curve}
    # the interactive loop: a door swinging over 60 frames
    sc = scenes.door_rooms()
    first, n = sc.meta["door"]
    frames = [scenes.door_verts(sc, 90.0 * k / 59)[first:] for k in range(60)]
    ir = np.zeros((1, 2, 48000), np.float32)
    with fs.Context(device=0) as ctx:
        ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption)
        for k in range(5):
            ctx.update(sc.sources, sc.listener, N_PAIRS, DEPTH, k, ir_out=ir)
        static, moving, refit_part, ratios = [], [], [], []
        for k in range(60):
            t0 = time.perf_counter()
            ctx.update(sc.sources, sc.listener, N_PAIRS, DEPTH, 100 + k, ir_out=ir)
            static.append(1e3 * (time.perf_counter() - t0))
        for k in range(60):
            t0 = time.perf_counter()
            ctx.update_vertices(frames[k], first)
            ratios.append(ctx.refit())
            t1 = time.perf_counter()
            ctx.update(sc.sources, sc.listener, N_PAIRS, DEPTH, 200 + k, ir_out=ir)
            moving.append(1e3 * (time.perf_counter() - t0))
            refit_part.append(1e3 * (t1 - t0))
    res["door_loop"] = {"scene": "door_rooms", "n_tris": sc.n_tris, "door_tris": n, "frames": 60,
                        "static_update_ms_median": med(static), "moving_frame_ms_median": med(moving),
                        "update_vertices_plus_refit_ms_median": med(refit_part), "max_cost_ratio": float(max(ratios))}
    print(json.dumps(res["door_loop"]), flush=True)
    out = args.out or os.path.join(ROOT, "profiles", "refit_%s.json" % info["gpu"].replace(" ", "_"))
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", out)


if __name__ == "__main__":
    main()
