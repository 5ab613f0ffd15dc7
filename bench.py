#!/usr/bin/env python
"""bench.py -- headline benchmark of the BDPT -> histogram -> IR hot path.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): procedural furnished room (~100 k triangles, 8 materials,
8 absorption bands), 1 source / 1 listener, 2^20 BDPT path pairs per IR update, max depth 16,
1000 x 1 ms bins, 1 s 48 kHz IR.  A step = one IR update = fs_trace + fs_build_ir (histogram ->
IR -> convolver partition spectra).  N GPUs: weak scaling, every rank traces 2^20 pairs of a
global N * 2^20 work range against a replicated BVH, one NCCL integer reduce per step.

One JSON line on stdout (rank 0).  `value` = path pairs/s with everything resident in HBM;
`e2e` = the same through the C-ABI with host buffers (positions in, histogram + IR out; at N > 1 the shard
histograms stay on the devices, rank 0 reads the reduced histogram and the IR back);
`roofline` = the traversal kernel that ran (k_path_q for this workload: every bounce of a batch in one persistent
launch; k_trace_q per bounce for small jobs): algorithmic bytes / its CUDA-event time vs the measured HBM peak, with
the binding resource, the L2-relative figure and an instruction roofline; `cpu_baseline` = the CPU oracle (a port of the
reference's loop) on a bounded sample; `parity` = GPU histogram == oracle on that sample (and NCCL-reduced shards == one
GPU at N > 1); `north_star` (N = 8) = the 10.5 M-pair / 5 M-triangle hall update; `cabi_multi` = all N GPUs from one
process through fs_multi_*.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "audio-pathtracer_b200"))

import numpy as np  # noqa: E402

METRIC = "bdpt_path_pairs_per_second"
UNIT = "paths/s"
WORKLOAD = "furnished_room_100k_tris_1M_paths_depth16_8bands"
SEED0 = 1000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--paths", type=int, default=1 << 20)
    ap.add_argument("--depth", type=int, default=16)
    ap.add_argument("--scene", default="furnished_room", choices=["furnished_room", "mine_tunnels", "concert_hall", "shoebox"],
                    help="default furnished_room = BASELINE.json configs[1]; the others are extra measurements")
    ap.add_argument("--sources", type=int, default=1,
                    help="emitters (BASELINE configs[3]: 64 in the mine tunnels); --paths stays the path pairs per GPU per step, "
                         "split evenly over the sources")
    ap.add_argument("--share-listener", action="store_true",
                    help="FS_FLAG_SHARE_LISTENER: listener subpaths keyed by the path index, traced once per update and shared "
                         "by all sources (SURVEY 8f rank 4; different random numbers than the default mode)")
    ap.add_argument("--cpu-sample-paths", type=int, default=1 << 19)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--strong", action="store_true",
                    help="strong scaling: --paths is the TOTAL per step, cut into N shards (default: weak, --paths per GPU)")
    ap.add_argument("--north-star", choices=["auto", "on", "off"], default="auto",
                    help="after the headline measurement also time BASELINE north_star's point (concert hall ~5 M triangles, "
                         "10 485 760 path pairs, depth 32, sharded over the N GPUs) and report it under 'north_star'; auto = at N = 8")
    ap.add_argument("--north-star-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the last one computed to DIR (either --impl): histogram.npy "
                         "(float64 energies, [sources][bands][bins]) and ir.npy (float32 impulse responses, "
                         "[sources][channels][samples])")
    return ap.parse_args()


def config_dict(args, n):
    wl = WORKLOAD if (args.scene == "furnished_room" and args.paths == 1 << 20 and args.depth == 16 and args.sources == 1) else \
        "%s_%d_paths_depth%d_8bands%s" % (args.scene, args.paths, args.depth, "_%dsources" % args.sources if args.sources > 1 else "")
    return {"workload": wl, "scene": "%s (seeded procedural)" % args.scene,
            "paths_per_gpu_per_step": (args.paths // n) if args.strong else args.paths,
            "max_depth": args.depth, "bands": 8, "bins": 1000, "sources": args.sources, "rr_prob": 0.9,
            "parallelism": "path-range sharding x%d, replicated BVH, one int64 reduce" % n,
            "share_listener": bool(args.share_listener),
            "l2": "no explicit flush: per-step wavefront state+records (~0.6 GB) exceed the 126 MB L2; "
                  "the ~11 MB BVH is L2-resident by design, as in steady-state 60 Hz refresh"}


# ---------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:                                   # one long-lived nvidia-smi in loop mode (-lms), parsed at the end
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.3)                    # first sample lands before the timed region starts
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is None:
            return
        time.sleep(0.1)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        for line in out.strip().splitlines():
            self.rows.append([c.strip() for c in line.split(",")])

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md, MEASURED_PEAKS.json absent)"


# ---------------------------------------------------------------------------------------------
# reference arm: the CPU oracle (port of the reference's BDPT loop) on all host threads
# ---------------------------------------------------------------------------------------------
def cpu_oracle_rate(args, n_paths, threads, repeats=1, seed=SEED0):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle as po
    from frequensee import scenes
    sc = scenes.by_name(args.scene)
    sc.sources = sc.sources[:args.sources]
    S = po.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=True)
    cfg = po.default_config(flags=po.FLAG_SHARE_LISTENER) if args.share_listener else po.default_config()
    times = []
    for r in range(repeats):
        t0 = time.perf_counter()
        per_source = max(1, n_paths // len(sc.sources))      # n_paths = path pairs over all sources
        h, st = S.trace(cfg, sc.sources, sc.listener, per_source, args.depth, seed + r, n_threads=threads)
        irs = [po.build_ir(cfg, h[si], per_source) for si in range(len(sc.sources))]
        times.append(time.perf_counter() - t0)
    st["hist"], st["ir"] = h, np.stack(irs)                  # of the last repeat (seed + repeats - 1): parity check, dump
    return times, st


def write_outputs(out_dir, hist, ir):
    """--dump-outputs: histogram.npy = the Q32.32 histogram / 2^32 (float64, [sources][bands][bins]), ir.npy = the impulse
    responses (float32, [sources][channels][samples]).  At most 64 sources x (64 KB + 384 KB), well under 64 MB."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "histogram.npy"), np.asarray(hist, dtype=np.uint64).astype(np.float64) / 2.0 ** 32)
    np.save(os.path.join(out_dir, "ir.npy"), np.ascontiguousarray(ir, dtype=np.float32))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    sample = min(args.paths, 1 << 17)
    cpu_oracle_rate(args, sample, threads, repeats=max(1, min(args.warmup, 1)))
    times, st = cpu_oracle_rate(args, sample, threads, repeats=args.steps)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, st["hist"], st["ir"])
    total = sum(times)
    v = sample * args.steps / total
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 + u64 Q32.32", "data": "synthetic",
            "config": dict(config_dict(args, args.gpus), sample_paths_per_step=sample),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": "%d path pairs per step of the same workload (oracle/fs_oracle.c: the reference's "
                                       "BDPT loop restated in C; the UE plugin itself cannot be built)" % sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "mrays_per_s": (st["ext_rays"] + st["shadow_rays"]) / (total / args.steps) / 1e6}
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
def profile_counters(args, kernel="k_trace_q"):
    """per-launch ncu counters of the traversal kernel on this workload from the committed `ncu --set full` capture
    (profiles/*_traffic.json: dram bytes, lts throughput, thread instructions); {} for workloads that were not captured"""
    out = {}
    pdir = os.path.join(ROOT, "profiles")
    want = "hall" if args.scene == "concert_hall" else ("room" if args.scene == "furnished_room" else None)
    for f in sorted(os.listdir(pdir)) if (want and os.path.isdir(pdir)) else []:
        if f.endswith("_traffic.json"):
            try:
                j = json.load(open(os.path.join(pdir, f)))
            except Exception:
                continue
            if j.get("scene", "room") == want and j.get("kernel", "k_trace_q").startswith(kernel):
                out = j
    return out


class Workload:
    """one scene + job size on this rank: contexts, the device step and every measurement taken of it"""

    def __init__(self, env, scene, paths_total_or_per_gpu, depth, n_sources, share_listener, strong):
        import frequensee as fs
        from frequensee import scenes, capi
        from frequensee.distributed import shard_range
        self.env, self.fs, self.capi = env, fs, capi
        torch = env["torch"]
        N, rank, local = env["N"], env["rank"], env["local"]
        sc = scenes.by_name(scene)
        sc.sources = sc.sources[:n_sources]
        self.sc, self.D, self.NS = sc, depth, len(sc.sources)
        self.P_total = paths_total_or_per_gpu if strong else paths_total_or_per_gpu * N     # path pairs per step, whole job
        if self.P_total % self.NS:
            raise SystemExit("--paths x --gpus must be a multiple of --sources")
        self.base_flags = capi.FLAG_SHARE_LISTENER if share_listener else 0
        self.ctx = fs.Context(device=local, flags=self.base_flags)   # production configuration: no per-kernel events, batch lanes on
        self.ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption)
        self.ctx.set_stream(env["stream"].cuda_stream)
        self.B, self.Kb = self.ctx.cfg.n_bands, self.ctx.cfg.n_bins
        self.d_hist = torch.zeros((self.NS, self.B, self.Kb), dtype=torch.int64, device="cuda")
        self.n_global = self.P_total // self.NS                  # per-source path count of the whole job
        self.g_first, self.g_count = shard_range(self.n_global * self.NS, rank, N)   # contiguous range of g = source * n + i

    def step_device(self, seed):
        env, ctx, sc = self.env, self.ctx, self.sc
        ctx.trace_range_device(sc.sources, sc.listener, self.n_global, self.g_first, self.g_count, self.D, seed,
                               self.d_hist.data_ptr(), True)
        if env["N"] > 1:
            env["dist"].reduce(self.d_hist, dst=0, op=env["dist"].ReduceOp.SUM)
        if env["rank"] == 0:
            ctx.set_histogram_device(self.d_hist.data_ptr(), self.NS, self.n_global)
            if self.NS == 1:
                ctx.build_ir(0, want_ir=False)
            else:
                ctx.build_ir_all(self.NS, want_ir=False)

    def time_device(self, K, W, seed0=SEED0):
        """W warm-up steps, then K steps between a barrier + synchronize on both sides; CUDA events; max over ranks"""
        env = self.env
        torch = env["torch"]
        for w in range(W):
            self.step_device(seed0 - 1 - w)
        env["barrier"]()
        launches0 = self.ctx.stats()["kernel_launches"]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with Clocks(env["local"]) as clk:
            env["barrier"]()
            e0.record(env["stream"])
            for k in range(K):
                self.step_device(seed0 + k)
            e1.record(env["stream"])
            env["barrier"]()
            dev_ms = e0.elapsed_time(e1)
        launches = self.ctx.stats()["kernel_launches"] - launches0
        t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
        if env["N"] > 1:
            env["dist"].all_reduce(t, op=env["dist"].ReduceOp.MAX)
        return float(t.item()), int(launches), clk.summary()

    def stage_times(self, n_steps, seed0=SEED0):
        """per-kernel-class device time: the same steps (same seeds) re-run on a second context with FS_FLAG_TIME_KERNELS,
        i.e. CUDA events on the launching stream around every stage and every traversal launch (k_trace_q per bounce, or the
        one k_path_q of a batch).  That context runs its batches on ONE lane, so each kernel is timed alone."""
        torch = self.env["torch"]
        tctx = self.fs.Context(device=self.env["local"], flags=self.capi.FLAG_TIME_KERNELS | self.base_flags)
        tctx.set_scene(self.sc.verts, self.sc.tri_mat, self.sc.absorption)
        tctx.set_stream(self.env["stream"].cuda_stream)
        per = []
        for k in range(-1, n_steps):
            tctx.trace_range_device(self.sc.sources, self.sc.listener, self.n_global, self.g_first, self.g_count, self.D,
                                    seed0 + k, self.d_hist.data_ptr(), True)
            torch.cuda.synchronize()
            if k >= 0:
                per.append(tctx.stats())
        tctx.close()
        m = lambda key: float(np.mean([s[key] for s in per]))       # noqa: E731
        return {"extend_ms": m("extend_ms"), "connect_ms": m("connect_ms"), "trace_ms": m("trace_ms"), "eval_ms": m("eval_ms"),
                "extend_launches": per[0]["extend_launches"], "persistent": per[0].get("persistent_launches", 0),
                "rays": m("ext_rays") + m("shadow_rays"),
                "ext_rays": m("ext_rays"), "connected": m("connected")}

    def visit_counts(self, n_steps, seed0=SEED0):
        """algorithmic bytes: visit counts of the same rays from the instrumented build of the same kernels"""
        cctx = self.fs.Context(device=self.env["local"], flags=self.capi.FLAG_COUNT_VISITS | self.base_flags)
        cctx.set_scene(self.sc.verts, self.sc.tri_mat, self.sc.absorption)
        cnt = []
        for k in range(n_steps):
            cctx.trace_range(self.sc.sources, self.sc.listener, self.n_global, self.g_first, self.g_count, self.D, seed0 + k)
            cnt.append(cctx.stats())
        cctx.close()
        en = float(np.mean([c["node_visits"] - c["shadow_node_visits"] for c in cnt]))
        et = float(np.mean([c["tri_tests"] - c["shadow_tri_tests"] for c in cnt]))
        er = float(np.mean([c["ext_rays"] for c in cnt]))
        return en, et, er

    def roofline(self, args_like, st, clocks):
        """SURVEY.md 8(d): bytes_ray = 64 * n_node (one 4-wide node) + 48 * n_tri (v0, e1, e2) + 32 (ray record read) + 8 (hit
        write), n_node / n_tri measured; achieved = bytes / CUDA-event time of the traversal launches; peak = measured HBM copy
        bandwidth.  `bound` names the resource that actually limits the kernel on this scene (ncu evidence under profiles/)."""
        en, et, er = self.visit_counts(2)
        ext_bytes = 64.0 * en + 48.0 * et + 40.0 * er
        peak, peak_src = measured_peak()
        trc_ms, nl = st["trace_ms"], max(st["extend_launches"], 1)
        achieved = ext_bytes / (trc_ms * 1e-3) / 1e9 if trc_ms > 0 else None
        bvh_mb = (self.sc.n_tris * 0.5 * 64 + self.sc.n_tris * 64) / 1e6      # reachable 4-wide nodes (~T/2 x 64 B) + triangles (64 B)
        in_l2 = bvh_mb < 100
        persistent = st.get("persistent", 0) > 0
        prof = profile_counters(args_like, "k_path_q" if persistent else "k_trace_q")
        kname = ("k_path_q (persistent per-batch kernel: every bounce of the batch -- 4-wide BVH closest-hit traversal with the "
                 "warp-shared triangle queue AND in-kernel shading / ray generation -- in %d launch(es) per step; bytes counted "
                 "are the traversal's only" % st["extend_launches"]) if persistent else \
                ("k_trace_q<closest> (persistent 4-wide BVH closest-hit traversal, warp-shared triangle queue), %d launches "
                 "per step on the one-lane timing context" % st["extend_launches"])
        r = {"bound": "issue" if in_l2 else "hbm",
             "binding_resource": ("issue slots / ALU pipe: the %.0f MB of nodes + triangles are L2/L1-resident (DRAM traffic is a few %% of "
                                  "the algorithmic bytes), the kernel is limited by instruction issue at ~2/3 lane occupancy" % bvh_mb) if in_l2
                                 else ("memory latency / L2+HBM fetch of the %.0f MB of nodes + triangles (larger than the 126 MB L2): "
                                       "a third of the stall samples wait for the node fetch" % bvh_mb),
             "kernel": kname,
             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
             "traffic": prof.get("dram_bytes_per_launch"), "peak_source": peak_src,
             "bytes_per_launch": ext_bytes / nl, "ms_per_launch": trc_ms / nl,
             "nodes_per_ray": en / er, "tris_per_ray": et / er,
             "note": "achieved = ALGORITHMIC fetch bytes (SURVEY.md 8d) / kernel time, normalised by the measured HBM copy peak as "
                     "prescribed; with an L2-resident BVH it is served by L2/L1, so frac is not a distance to a physical limit -- "
                     "l2_frac and inst below are"}
        # L2-relative figure and instruction roofline (ncu counters of the committed capture of this scene, per launch)
        if prof.get("lts_throughput_pct") is not None:
            r["l2_frac"] = prof["lts_throughput_pct"] / 100.0
        if prof.get("thread_inst_per_step") and prof.get("launches") == st["extend_launches"]:
            # the capture covers one step of this workload on one lane: thread-level instructions per extension ray
            tipr = prof["thread_inst_per_step"] / er
            sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
            peak_inst = 148 * 4 * 32 * sm_mhz * 1e6                       # thread-instructions/s: SMs x schedulers x lanes x clock
            ach_inst = tipr * er / (trc_ms * 1e-3) if trc_ms > 0 else None
            r["inst"] = {"thread_inst_per_ray": tipr, "achieved": ach_inst, "peak": peak_inst,
                         "unit": "thread-inst/s", "frac": (ach_inst / peak_inst) if ach_inst else None,
                         "active_lanes_per_inst": prof.get("active_lanes_per_inst"),
                         "source": prof.get("source")}
        return r

    def dump_outputs(self, out_dir):
        """rank 0, after time_device: the context's copy of the last timed step's histogram (summed over the ranks at N > 1)
        and the impulse responses rebuilt from it by the same IR kernels (deterministic: the floats the step left on the
        device, which the timed step does not read back)"""
        ir = self.ctx.build_ir(0)[None] if self.NS == 1 else self.ctx.build_ir_all(self.NS)
        write_outputs(out_dir, self.ctx.get_histogram(), ir)

    def close(self):
        self.ctx.close()


def run_b200(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: anything native code prints there (e.g. "NCCL version ...") goes to stderr
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    host_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        host_group = dist.new_group(backend="gloo")        # host-side barrier (no kernel spinning on the idle GPUs)
    N, K, W = world, args.steps, args.warmup
    stream = torch.cuda.Stream()                            # a real (non-NULL) stream: the C-ABI treats NULL as "own stream"
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0

    def barrier():
        if N > 1:
            dist.barrier()
        torch.cuda.synchronize()

    env = {"torch": torch, "dist": dist, "N": N, "rank": rank, "local": local, "stream": stream, "barrier": barrier}
    wl = Workload(env, args.scene, args.paths, args.depth, args.sources, args.share_listener, args.strong)
    sc, ctx, D, NS_, B, Kb = wl.sc, wl.ctx, wl.D, wl.NS, wl.B, wl.Kb
    P_total = wl.P_total
    dev_ms, launches, clocks = wl.time_device(K, W)
    if args.dump_outputs and rank == 0:
        wl.dump_outputs(args.dump_outputs)
    value = P_total * K / (dev_ms * 1e-3)
    st = wl.stage_times(min(K, 5))
    roofline = wl.roofline(args, st, clocks)

    # ---- parity inside the driver-run line ---------------------------------------------------------------------------
    # N > 1: the NCCL-reduced histogram of the N shards == rank 0's own single-GPU trace of the same global range
    # (one step's worth of one GPU: wl.P_total / N pairs in total, cut into N shards).  Outside the timed region.
    parity = {}
    from frequensee.distributed import shard_range
    n_chk = max(NS_, (P_total // N) // NS_ * NS_) // NS_   # per-source path count of the check job
    if N > 1:
        gf, gc = shard_range(n_chk * NS_, rank, N)
        ctx.trace_range_device(sc.sources, sc.listener, n_chk, gf, gc, D, SEED0 + 77, wl.d_hist.data_ptr(), True)
        dist.reduce(wl.d_hist, dst=0, op=dist.ReduceOp.SUM)
        torch.cuda.synchronize()
        if rank == 0:
            reduced = wl.d_hist.clone()
            ctx.trace_range_device(sc.sources, sc.listener, n_chk, 0, n_chk * NS_, D, SEED0 + 77, wl.d_hist.data_ptr(), True)
            torch.cuda.synchronize()
            parity["nccl_reduce_bit_exact"] = bool(torch.equal(reduced, wl.d_hist))
            parity["nccl_reduce_check"] = "%d path pairs x %d sources, %d shards reduced over NCCL vs one GPU" % (n_chk, NS_, N)
        barrier()

    # e2e: the public C-ABI calls with host buffers in (positions) and out (histogram, impulse responses), copies inside the
    # timed region.  N = 1: fs_trace + fs_build_ir*.  N > 1: every rank traces its shard into device memory
    # (fs_trace_range_device, positions from the host), one NCCL reduce, rank 0 adopts the sum (fs_set_histogram_device) and
    # reads the results back (fs_get_histogram + fs_build_ir*) -- the shard histograms never visit the host
    e2e = None
    g_first, g_count, n_global = wl.g_first, wl.g_count, wl.n_global
    d_hist = wl.d_hist
    if N == 1:
        ctx.set_stream(None)
    if rank == 0 or N > 1:
        # the host keeps ONE set of page-locked result buffers (fs_host_alloc) and reuses it every update, as a plugin would:
        # the copy engine writes them directly and no update pays for a fresh allocation
        ir_buf = wl.capi.host_alloc((NS_, ctx.cfg.n_channels, ctx.cfg.sample_rate)) if rank == 0 else None
        h_buf = wl.capi.host_alloc((NS_, B, Kb), np.uint64) if (rank == 0 and N == 1) else None
        def step_host(seed):
            if N == 1:
                # one call = one update (UpdateSource): positions H2D, trace, IR rebuild, histogram + IR D2H, one synchronisation
                return ctx.update(sc.sources, sc.listener, n_global, D, seed, hist_out=h_buf, ir_out=ir_buf)
            ctx.trace_range_device(sc.sources, sc.listener, n_global, g_first, g_count, D, seed, d_hist.data_ptr(), True)
            dist.reduce(d_hist, dst=0, op=dist.ReduceOp.SUM)
            if rank != 0:
                return None, None
            ctx.set_histogram_device(d_hist.data_ptr(), NS_, n_global)
            h = ctx.get_histogram()                                          # reduced histogram D2H
            ir = ctx.build_ir(0, out=ir_buf[0]) if NS_ == 1 else ctx.build_ir_all(NS_, out=ir_buf)      # IR D2H
            return h, ir
        step_host(SEED0 - 1)
        barrier()
        t0 = time.perf_counter()
        for k in range(K):
            h, ir = step_host(SEED0 + k)
        barrier()
        wall = time.perf_counter() - t0
        tw = torch.tensor([wall], dtype=torch.float64, device="cuda")
        if N > 1:
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        wall = float(tw.item())
        hb = NS_ * B * Kb * 8
        e2e = {"value": P_total * K / wall, "unit": UNIT, "h2d_bytes_per_step": int(sc.sources.nbytes + sc.listener.nbytes),
               "d2h_bytes_per_step": int(hb + NS_ * ctx.cfg.n_channels * ctx.cfg.sample_rate * 4), "ms_per_step": 1e3 * wall / K}
    cpu = cpu1 = None
    if rank == 0 and N == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        times, so = cpu_oracle_rate(args, args.cpu_sample_paths, threads, repeats=1)
        cpu = {"value": args.cpu_sample_paths / times[0], "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "%d path pairs of the same workload (oracle/fs_oracle.c, pthreads, %d threads), %.2f s"
                         % (args.cpu_sample_paths, threads, times[0])}
        # the same sample on the GPU through the C-ABI: the integers must be the oracle's (the oracle only as the checker)
        per_src = max(1, args.cpu_sample_paths // NS_)
        hg = ctx.trace(sc.sources, sc.listener, per_src, D, SEED0)
        parity["oracle_bit_exact"] = bool(np.array_equal(hg, so["hist"]))
        parity["oracle_check"] = "%d path pairs of this workload, GPU histogram == CPU oracle histogram" % (per_src * NS_)
        # one host thread: what the reference has, its whole update runs on the game thread (SUB.cpp:55-85)
        n1 = max(NS_, min(args.cpu_sample_paths, 1 << 15))
        t1, _ = cpu_oracle_rate(args, n1, 1, repeats=1)
        cpu1 = {"value": n1 / t1[0], "unit": UNIT, "cores": 1, "kind": "port",
                "sample": "%d path pairs of the same workload on ONE host thread, %.2f s" % (n1, t1[0])}
    wl.close()

    # ---- BASELINE north_star's point, in the same driver-run line -------------------------------------------------------
    north = None
    want_ns = args.north_star == "on" or (args.north_star == "auto" and N == 8 and args.scene == "furnished_room" and not args.strong)
    if want_ns:
        NS_PAIRS = 10 * (1 << 20)                                            # 10 485 760 >= 10 M bidirectional path pairs
        hall = Workload(env, "concert_hall", NS_PAIRS, 32, 1, False, strong=True)
        h_ms, h_launches, h_clocks = hall.time_device(args.north_star_steps, 2, seed0=SEED0 + 500)
        hst = hall.stage_times(2, seed0=SEED0 + 500)
        class _A: scene = "concert_hall"; paths = NS_PAIRS // N; depth = 32     # noqa: E701
        hroof = hall.roofline(_A, hst, h_clocks)
        if rank == 0:
            per = h_ms / args.north_star_steps
            north = {"workload": "concert_hall_%d_tris_%d_pairs_depth32_8bands" % (hall.sc.n_tris, NS_PAIRS), "n_gpus": N,
                     "ms_per_ir_update": per, "target_ms": 16.0, "paths_per_s": NS_PAIRS / (per * 1e-3),
                     "mrays_per_s": hst["rays"] * N / (per * 1e-3) / 1e6, "steps": args.north_star_steps, "warmup": 2,
                     "roofline_frac": hroof["frac"], "roofline": hroof, "clocks": h_clocks, "gpu_launches": h_launches,
                     "stage_ms_rank0_one_lane": {"trace_closest": hst["trace_ms"], "shade_gen": hst["extend_ms"] - hst["trace_ms"],
                                                 "connect": hst["connect_ms"], "eval_splat": hst["eval_ms"]}}
        hall.close()
    # ---- the same update through the C-ABI's own multi-GPU path (fs_multi_*: one process, one context per device, peer-store
    # reduce on device 0 -- no NCCL, no torch on the data path), run by rank 0 alone while the other ranks wait on the host
    cabi_multi = None
    if N > 1 and args.scene == "furnished_room" and not args.strong:
        if rank == 0:
            import frequensee as fs2
            from frequensee import scenes as scenes2
            try:
                sc2 = scenes2.by_name(args.scene); sc2.sources = sc2.sources[:args.sources]
                per_src = args.paths * N // len(sc2.sources)
                # NCCL reduce of one histogram, alone (CUDA events), for comparison
                with fs2.MultiContext(list(range(N))) as mc:
                    mc.set_scene(sc2.verts, sc2.tri_mat, sc2.absorption)
                    c0 = mc.context(0)
                    for w in range(3):
                        mc.trace(sc2.sources, sc2.listener, per_src, args.depth, SEED0 - 1 - w, want_hist=False)
                        c0.build_ir(0, want_ir=False)
                    mc.synchronize()
                    t0 = time.perf_counter()
                    for k in range(K):
                        mc.trace(sc2.sources, sc2.listener, per_src, args.depth, SEED0 + k, want_hist=False)
                        c0.build_ir(0, want_ir=False) if len(sc2.sources) == 1 else c0.build_ir_all(len(sc2.sources), want_ir=False)
                    mc.synchronize()
                    wall_m = time.perf_counter() - t0
                    tot_ms, red_ms = mc.last_ms()
                    hm = mc.trace(sc2.sources, sc2.listener, n_chk, args.depth, SEED0 + 77)
                cabi_multi = {"ms_per_step": 1e3 * wall_m / K, "value": args.paths * N * K / wall_m, "unit": UNIT,
                              "device_ms_last_update": tot_ms, "device_ms_wait_for_peers_and_sum": red_ms,
                              "bit_exact_vs_nccl_reduce": bool(parity.get("nccl_reduce_bit_exact")) and
                              bool(np.array_equal(hm.view(np.int64), reduced.cpu().numpy())),
                              "what": "fs_multi_trace + fs_build_ir on %d devices from ONE process (wall clock around enqueue + synchronise)" % N}
            except Exception as e:                                          # never lose the headline line over the extra measurement
                cabi_multi = {"error": str(e)[:300]}
        dist.barrier(group=host_group)
    if rank == 0:
        ext_ms_all, trc_ms = st["extend_ms"], st["trace_ms"]
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": N, "steps": K, "warmup": W,
                "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
                "dtype": "f32 + u64 Q32.32", "data": "synthetic", "config": config_dict(args, N),
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
                "roofline": roofline, "cpu_baseline": cpu, "cpu_baseline_1thread": cpu1, "parity": parity, "north_star": north, "cabi_multi": cabi_multi,
                "mrays_per_s": st["rays"] * N / (dev_ms / K * 1e-3) / 1e6,
                "ms_per_ir_update": dev_ms / K,
                "stage_ms": {"trace_closest": trc_ms, "shade_gen": ext_ms_all - trc_ms, "connect": st["connect_ms"], "eval_splat": st["eval_ms"]},
                "rays_per_step_per_gpu": st["rays"], "ext_rays_per_step_per_gpu": st["ext_rays"],
                "connected_per_step_per_gpu": st["connected"], "triangles": int(sc.n_tris)}
        json_out.write(json.dumps(line) + "\n")
        json_out.flush()
    if N > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
