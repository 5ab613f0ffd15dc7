"""Cost and effect of the convolver's IR cross-fade (FS_FLAG_CONV_CROSSFADE).  Prints one JSON line and writes it to --out
(default profiles/crossfade_<card>.json), with the card name and power limit read in the same run.

  device_ms_per_callback  last_conv_ms (CUDA events around the k_conv_blocks launch on the convolver's stream), medians
                          over rounds in which the cases alternate, for one source (fs_conv_process) and for 64 sources
                          in one fs_conv_process_multi, each with its own 1 s stereo IR:
                            off     flag off
                            steady  flag on, no IR published since the previous callback (plain kernel)
                            fade    flag on, a new IR published (fs_set_ir) before every callback: the worst case
  roofline                algorithmic bytes of one callback, S * C * [(P+1)(Bk+1) * 16 + 2 Bk * 8] for a plain block and
                          S * C * [(P+1)(Bk+1) * 24 + 2 Bk * 8] for a fade block (X_{k-p} read once against two spectra
                          sets), over the measured device time, against the HBM peak as in tools/bench_conv.py
  click                   furnished room (config 2 scene), one source, a real re-trace (2^20 pairs, depth 16, new seed,
                          listener moved 1 cm) and IR rebuild every 800 frames (60 Hz) with its IR read back, so the
                          block at which each IR takes effect is known; dry input a 250 Hz sine of amplitude 0.5 plus
                          noise 40 dB below it.  metric = RMS(y[k Bk] - y[k Bk - 1] over the boundaries where a new IR
                          took effect) / RMS(y[n] - y[n-1] inside blocks), flag off and on, and each output's rel-L2
                          against the float64 model of tests/crossfade_model.py

usage: python tools/bench_conv_crossfade.py [--rounds N] [--seconds S] [--out PATH]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "audio-pathtracer_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import frequensee as fs                       # noqa: E402
from frequensee import capi, scenes           # noqa: E402
import crossfade_model as cm                  # noqa: E402

BK, C, FS = 1024, 2, 48000


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.strip().split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def summary(ms):
    a = np.asarray(ms, np.float64)
    return {"median_ms": float(np.median(a)), "min_ms": float(a.min()), "max_ms": float(a.max()), "runs": len(a)}


def callback_costs(S, rounds, rng):
    """device ms per callback of the three cases, alternating within every round"""
    irs = (rng.normal(size=(2, S, C, FS)) * np.exp(-np.arange(FS) / 7000.0) * 0.02).astype(np.float32)
    ids = np.arange(S, dtype=np.uint32)
    x = rng.uniform(-0.5, 0.5, size=(S, BK, C)).astype(np.float32)
    ctx_off = fs.Context(conv_clamp=0)
    ctx_on = fs.Context(conv_clamp=0, flags=capi.FLAG_CONV_CROSSFADE)
    try:
        for ctx in (ctx_off, ctx_on):
            for s in range(S):
                ctx.set_ir(irs[0, s], s); ctx.conv_init_source(s)

        def callback(ctx):
            if S == 1:
                ctx.conv_process(x[0], 0)
            else:
                ctx.conv_process_multi(x, ids)
            return ctx.stats()["last_conv_ms"]

        out = {"off": [], "steady": [], "fade": []}
        for r in range(rounds + 5):                  # the first 5 rounds warm every case up
            t_off = callback(ctx_off)
            for s in range(S):
                ctx_on.set_ir(irs[(r + 1) % 2, s], s)
            t_fade = callback(ctx_on)
            t_steady = callback(ctx_on)
            if r >= 5:
                out["off"].append(t_off); out["fade"].append(t_fade); out["steady"].append(t_steady)
        return {k: summary(v) for k, v in out.items()}
    finally:
        ctx_off.close(); ctx_on.close()


def click(seconds, rng):
    sc = scenes.furnished_room()
    NB = int(seconds * FS) // BK
    n = NB * BK
    t = np.arange(n) / float(FS)
    x = (0.5 * np.sin(2 * np.pi * 250.0 * t)[:, None] + 0.005 * rng.standard_normal((n, C))).astype(np.float32)
    lis = np.array(sc.listener, np.float32)
    res = {}
    for name, flags in (("off", 0), ("on", capi.FLAG_CONV_CROSSFADE)):
        y = np.zeros((NB, BK, C), np.float32)
        irs, sched, boundaries = {}, [], []
        with fs.Context(conv_clamp=0, flags=flags) as ctx:
            ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption)
            ctx.conv_init_source(0)
            next_refresh, q, cur = 0, 0, None
            for k in range(NB):
                heard = None
                if k * BK >= next_refresh:               # every 800 frames of audio time: one refresh per callback or none
                    l2 = lis + np.float32(0.01 * (q % 16)) * np.array([1, 0, 0], np.float32)
                    ctx.trace(sc.sources[:1], l2, 1 << 20, 16, 5000 + q, want_hist=False)
                    irs[q] = ctx.build_ir(0)
                    if cur is not None:
                        boundaries.append(k)
                        heard = cur if flags else None
                    cur = q
                    q += 1
                    while next_refresh <= k * BK:
                        next_refresh += 800
                sched.append((heard, cur))
                y[k] = ctx.conv_process(x[k * BK:(k + 1) * BK])
        want = cm.run(x, irs, sched, BK, clamp=False)
        res[name] = {"metric": cm.click_metric(y.reshape(-1, C), BK, boundaries),
                     "rel_l2_vs_float64_model": float(np.linalg.norm(y - want) / np.linalg.norm(want)),
                     "ir_changes": len(boundaries), "blocks": NB}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=60)
    ap.add_argument("--seconds", type=float, default=3.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = gpu_info()
    rng = np.random.default_rng(3)
    res = dict(info)
    res["config"] = ("1 s 48 kHz stereo IRs, 1024-frame callbacks (P = 47 partitions), conv_clamp 0; fade = new IR "
                     "published before every callback")
    peak = 6545.9
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    P = (FS + BK - 1) // BK
    res["device_ms_per_callback"] = {}
    res["roofline"] = {"bound": "hbm", "peak_gbs": peak}
    for S in (1, 64):
        d = callback_costs(S, args.rounds * (4 if S == 1 else 1), rng)
        res["device_ms_per_callback"]["sources_%d" % S] = d
        plain = S * C * ((P + 1) * (BK + 1) * 16 + 2 * BK * 8)
        fade = S * C * ((P + 1) * (BK + 1) * 24 + 2 * BK * 8)
        r = {}
        for case, b in (("off", plain), ("steady", plain), ("fade", fade)):
            ms = d[case]["median_ms"]
            r[case] = {"bytes": b, "achieved_gbs": b / (ms * 1e-3) / 1e9, "frac_of_peak": b / (ms * 1e-3) / 1e9 / peak}
        res["roofline"]["sources_%d" % S] = r
    res["click"] = click(args.seconds, rng)
    out = args.out or os.path.join(ROOT, "profiles", "crossfade_%s.json" % info["gpu"].replace(" ", "_"))
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
