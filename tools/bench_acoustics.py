"""Cost of the room-acoustic parameters (fs_get_acoustic_params), and the shoebox decay times next to Eyring's formula.
Writes one JSON (--out, default profiles/acoustics_<card>.json) with the card name and power limit read in the same run.

Per case, after a warm-up: device ms (CUDA events on the context stream around the call: k_acoustics and the read-back of
the records, plus the EDC when it is requested) and wall ms (host clock around the call, which ends in a synchronisation),
median / min / max over --rounds calls, with and without the EDC.
  room     furnished room (config 2), its one source, 2^20 path pairs, depth 16: 9 slots x 1000 bins
  tunnels  the 64 emitters of the tunnel scene, 2^14 pairs each, depth 16: 576 slots x 1000 bins
For comparison, host ms of what a host does without the call: fs_get_histogram (the copy) plus the same parameters in
vectorised numpy float64 (not exact integers; timing only).
Decay check: the 7 x 5 x 3 m shoebox with one absorption alpha on every surface and band, FS_FLAG_MIS, 2^18 pairs, depth
32, and the default endpoint mode at depth 200: broadband T20 / T30 next to Eyring's T = 24 ln 10 V / (c S (-ln(1 - alpha))).

usage: python tools/bench_acoustics.py [--rounds N] [--out PATH]
"""
import argparse
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(ROOT), "audio-pathtracer_b200"))
sys.path.insert(0, ROOT)
from bench_sources import gpu_info, summary  # noqa: E402

C_HI = (1.0, 10 ** -0.5, 10 ** -0.5)
C_LO = (0.1, 10 ** -2.5, 10 ** -3.5)


def numpy_params(hist, bin_ms):
    """the host-side alternative: EDC, the three fits, C50 / C80 / D50 / Ts of every slot, float64, vectorised"""
    S, B, K = hist.shape
    E = np.concatenate([hist.astype(np.float64), hist.astype(np.float64).sum(1, keepdims=True)], 1)   # [S][B+1][K]
    R = np.cumsum(E[..., ::-1], -1)[..., ::-1]
    S0 = R[..., :1]
    with np.errstate(divide="ignore", invalid="ignore"):
        L = 10 * np.log10(R / S0)
    d = bin_ms * 1e-3
    k = np.arange(K, dtype=np.float64)
    nz = E > 0
    k0 = np.where(nz.any(-1), nz.argmax(-1), 0)[..., None]
    out = {}
    for i, name in enumerate(("edt", "t20", "t30")):
        after = (R <= S0 * C_HI[i]) & (k >= k0)
        ka = after.argmax(-1)[..., None]
        keep = (R >= S0 * C_LO[i]) & (k <= K - 2)
        kb = K - 1 - keep[..., ::-1].argmax(-1)[..., None]
        m = (k >= ka) & (k <= kb)
        n = m.sum(-1)
        w = np.where(m, 2 * k - ka - kb, 0.0)
        sw = (w * np.where(m, L, 0.0)).sum(-1)
        with np.errstate(divide="ignore", invalid="ignore"):
            out[name] = -60.0 / (6 * sw / (d * n * (n * n - 1.0)))
    t = (k - k0) * d
    for ms, name in ((50, "c50"), (80, "c80")):
        nw = int(ms / bin_ms + 0.5)
        early = (E * ((k >= k0) & (k < k0 + nw))).sum(-1)
        with np.errstate(divide="ignore", invalid="ignore"):
            out[name] = 10 * np.log10(early / (S0[..., 0] - early))
            if name == "c50":
                out["d50"] = early / S0[..., 0]
    with np.errstate(divide="ignore", invalid="ignore"):
        out["ts"] = (E * np.maximum(t, 0)).sum(-1) / S0[..., 0]
    return out, L


def time_call(torch, ctx, stream, rounds, edc):
    for _ in range(3):
        ctx.acoustic_params(edc=edc)
    dev, wall = [], []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        t0 = time.perf_counter()
        ctx.acoustic_params(edc=edc)
        wall.append(1e3 * (time.perf_counter() - t0))
        e1.record(stream)
        e1.synchronize()
        dev.append(e0.elapsed_time(e1))
    return {"device": summary(dev), "wall": summary(wall)}


def run_case(fs, torch, ctx, rounds):
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    res = {"sources": ctx.n_sources, "slots": ctx.n_sources * (ctx.cfg.n_bands + 1), "bins": ctx.cfg.n_bins,
           "call": time_call(torch, ctx, stream, rounds, False), "call_with_edc": time_call(torch, ctx, stream, rounds, True)}
    host = []
    for _ in range(rounds):
        t0 = time.perf_counter()
        h = ctx.get_histogram()
        numpy_params(h, ctx.cfg.bin_ms)
        host.append(1e3 * (time.perf_counter() - t0))
    res["host_copy_and_numpy"] = summary(host)
    res["histogram_bytes"] = int(h.nbytes)
    p = ctx.acoustic_params()
    bb = [p[s].broadband for s in range(ctx.n_sources)]
    res["broadband_t30_median_s"] = float(np.nanmedian([b.t30.time_s for b in bb]))
    res["broadband_t30_valid"] = int(sum(1 for b in bb if b.valid & 4))
    return res


def eyring(fs, scenes, flags, depth, alpha):
    sc = scenes.shoebox()
    X, Y, Z = sc.meta["size"]
    V, A = X * Y * Z, 2 * (X * Y + X * Z + Y * Z)
    with fs.Context(flags=flags) as ctx:
        ctx.set_scene(sc.verts, sc.tri_mat, np.full_like(sc.absorption, alpha))
        ctx.trace(sc.sources, sc.listener, 1 << 18, depth, 0x5EED)
        b = ctx.acoustic_params()[0].broadband
        c = ctx.cfg.sound_speed
    return {"alpha": alpha, "depth": depth, "t20_s": b.t20.time_s, "t30_s": b.t30.time_s, "t30_r": b.t30.r,
            "edt_s": b.edt.time_s, "c80_db": b.c80_db, "valid": int(b.valid),
            "eyring_s": 24 * math.log(10) * V / (c * A * -math.log(1 - alpha))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import frequensee as fs
    from frequensee import capi, scenes
    info = gpu_info()
    res = {"device": info, "rounds": args.rounds}
    room = scenes.furnished_room()
    with fs.Context() as ctx:
        ctx.set_scene(room.verts, room.tri_mat, room.absorption)
        ctx.trace(room.sources[:1], room.listener, 1 << 20, 16, 0x5EED, want_hist=False)
        res["room"] = run_case(fs, torch, ctx, args.rounds)
    tun = scenes.mine_tunnels()
    with fs.Context() as ctx:
        ctx.set_scene(tun.verts, tun.tri_mat, tun.absorption)
        src = np.asarray(tun.sources, np.float32)
        ctx.trace(src, tun.listener, 1 << 14, 16, 0x5EED, want_hist=False)
        res["tunnels"] = run_case(fs, torch, ctx, args.rounds)
    res["shoebox_vs_eyring"] = [eyring(fs, scenes, capi.FLAG_MIS, 32, a) for a in (0.1, 0.3)] + \
                               [eyring(fs, scenes, 0, 200, a) for a in (0.1, 0.3)]
    res["shoebox_vs_eyring"][0]["mode"] = res["shoebox_vs_eyring"][1]["mode"] = "mis"
    res["shoebox_vs_eyring"][2]["mode"] = res["shoebox_vs_eyring"][3]["mode"] = "endpoint"
    out = args.out or os.path.join(os.path.dirname(ROOT), "profiles", "acoustics_%s.json" % info["gpu"].replace(" ", "_"))
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
