"""FS_FLAG_CONV_CROSSFADE on the device against the float64 model of tests/crossfade_model.py (1e-5 relative L2 per
callback block), and bit-identity with a flag-off context wherever no fade happens."""
import threading
import time

import numpy as np
import pytest

import crossfade_model as cm

pytestmark = pytest.mark.gpu
TOL = 1e-5
BK, C, FS = 1024, 2, 48000


def _rel(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _irs(rng, n, scale=0.05, tau=3000.0):
    return (rng.normal(size=(n, C, FS)) * np.exp(-np.arange(FS) / tau) * scale).astype(np.float32)


def _ctx(fs, flag, **over):
    from frequensee import capi
    return fs.Context(flags=capi.FLAG_CONV_CROSSFADE if flag else 0, **over)


def _assert_blocks(y, want, what):
    for k in range(len(want)):
        r = _rel(y[k], want[k])
        assert r < TOL, "%s: block %d rel-L2 %g" % (what, k, r)


def test_no_republish_is_bit_identical_to_flag_off(fs):
    """flag on, IR published once before the first callback: conv_process, conv_process_many and conv_process_multi give
    exactly the flag-off output (no block fades, so the plain kernel runs)"""
    rng = np.random.default_rng(1)
    irs = _irs(rng, 4)
    x = rng.uniform(-0.5, 0.5, size=(4, 8, BK, C)).astype(np.float32)
    outs = []
    for flag in (False, True):
        with _ctx(fs, flag) as ctx:
            for s in range(4):
                ctx.set_ir(irs[s], s); ctx.conv_init_source(s)
            y0 = np.stack([ctx.conv_process(x[0, k], 0) for k in range(8)])
            y1 = ctx.conv_process_many(x[1], 1)
            y23 = np.stack([ctx.conv_process_multi(x[2:, k], [2, 3]) for k in range(8)])
            outs.append((y0, y1, y23))
    for a, b in zip(*outs):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("clamp,wet", [(1, 1.0), (0, 1.0), (1, 0.25)])
def test_single_source_switches(fs, clamp, wet):
    """a -> b at block 20; b -> c -> d published between two callbacks (the fade is b -> d, c is never heard); d
    republished unchanged at block 30 (a fade between equal IRs)"""
    rng = np.random.default_rng(2)
    a, b, c, d = _irs(rng, 4)
    NB = 36
    x = (rng.uniform(-0.6, 0.6, size=(NB * BK, C))).astype(np.float32)
    y = np.zeros((NB, BK, C), np.float32)
    sched = []
    with _ctx(fs, True, conv_clamp=clamp, conv_wet=wet) as ctx:
        ctx.set_ir(a); ctx.conv_init_source(0)
        cur = "a"
        for k in range(NB):
            heard = None
            if k == 20:
                ctx.set_ir(b); heard, cur = cur, "b"
            elif k == 25:
                ctx.set_ir(c); ctx.set_ir(d); heard, cur = cur, "d"
            elif k == 30:
                ctx.set_ir(d); heard = "d"
            y[k] = ctx.conv_process(x[k * BK:(k + 1) * BK])
            sched.append((heard, cur))
    want = cm.run(x, {"a": a, "b": b, "c": c, "d": d}, sched, BK, clamp=bool(clamp), wet=wet)
    _assert_blocks(y, want, "clamp %d wet %g" % (clamp, wet))
    # the fade really is a blend: block 20 differs from both hard switches
    ys = cm.wet_outputs(x, {"a": a, "b": b})
    for k_ir in ("a", "b"):
        assert _rel(y[20], cm.block(x, ys, 20, BK, k_ir, None, bool(clamp), wet)) > 1e-2


def test_process_many_fades_block_zero_only(fs):
    rng = np.random.default_rng(3)
    a, b = _irs(rng, 2)
    NB = 5
    x = rng.uniform(-0.5, 0.5, size=(2 * NB * BK, C)).astype(np.float32)
    with _ctx(fs, True, conv_clamp=0) as ctx:
        ctx.set_ir(a); ctx.conv_init_source(0)
        y0 = ctx.conv_process_many(x[:NB * BK].reshape(NB, BK, C))
        ctx.set_ir(b)
        y1 = ctx.conv_process_many(x[NB * BK:].reshape(NB, BK, C))
    sched = [(None, "a")] * NB + [("a", "b")] + [(None, "b")] * (NB - 1)
    want = cm.run(x, {"a": a, "b": b}, sched, BK, clamp=False)
    _assert_blocks(np.concatenate([y0, y1]), want, "process_many")


def test_multi_64_sources_every_third_switches(fs):
    """one conv_process_multi launch in which sources 0, 3, 6, ... fade and the others do not: every source matches its
    model, and the sources that did not switch are bit-identical to a flag-off context"""
    S, NB, SW = 64, 6, 3
    rng = np.random.default_rng(4)
    irs_a = _irs(rng, S, scale=0.02)
    irs_b = _irs(rng, S, scale=0.02)
    x = rng.uniform(-0.5, 0.5, size=(S, NB * BK, C)).astype(np.float32)
    ids = np.arange(S, dtype=np.uint32)
    switched = ids % 3 == 0
    outs = {}
    for flag in (False, True):
        y = np.zeros((S, NB, BK, C), np.float32)
        with _ctx(fs, flag, conv_clamp=0) as ctx:
            for s in range(S):
                ctx.set_ir(irs_a[s], s); ctx.conv_init_source(s)
            for k in range(NB):
                if k == SW:
                    for s in ids[switched]:
                        ctx.set_ir(irs_b[s], int(s))
                y[:, k] = ctx.conv_process_multi(x[:, k * BK:(k + 1) * BK], ids)
        outs[flag] = y
    for s in range(S):
        if switched[s]:
            sched = [(None, "a")] * SW + [("a", "b")] + [(None, "b")] * (NB - SW - 1)
        else:
            sched = [(None, "a")] * NB
            assert np.array_equal(outs[True][s], outs[False][s]), "source %d" % s
        want = cm.run(x[s], {"a": irs_a[s], "b": irs_b[s]}, sched, BK, clamp=False)
        _assert_blocks(outs[True][s], want, "source %d" % s)


def test_reinit_never_fades(fs):
    rng = np.random.default_rng(5)
    a, b = _irs(rng, 2)
    x = rng.uniform(-0.5, 0.5, size=(4, BK, C)).astype(np.float32)
    with _ctx(fs, True, conv_clamp=0) as ctx:
        ctx.set_ir(a); ctx.conv_init_source(0)
        for k in range(3):
            ctx.conv_process(x[k])
        ctx.set_ir(b)
        ctx.conv_release_source(0); ctx.conv_init_source(0)
        y = ctx.conv_process(x[3])
    want = cm.run(x[3], {"b": b}, [(None, "b")], BK, clamp=False)
    _assert_blocks(y[None], want, "after re-init")


def test_async_publication_never_switches_without_fade(fs):
    """the game thread publishes a cycle of K identifiable IRs through the asynchronous path (set_histogram + build_ir
    without read-back: spectra finished on the context stream, handed over by h_ready) while the audio thread runs
    callbacks.  Every block must be exactly one (heard, cur) candidate of the model, heard = the previous block's cur,
    cur never goes back in publication order, and a block fades exactly when heard != cur."""
    K, NB = 6, 200
    bins = [2 + 3 * j for j in range(K)]                 # IR j starts at 48 * bins[j] samples: inside block 0, so every
                                                          # candidate's output is non-zero in every block
    rng = np.random.default_rng(6)
    x = rng.uniform(-0.5, 0.5, size=(NB * BK, C)).astype(np.float32)
    with _ctx(fs, True, conv_clamp=0) as ctx:
        cfg = ctx.cfg
        hists = []
        for j in range(K):
            h = np.zeros((1, cfg.n_bands, cfg.n_bins), np.uint64)
            h[0, 0, bins[j]] = np.uint64(int(0.01 * 2 ** 32))
            hists.append(h)
        irs = {}
        for j in list(range(1, K)) + [0]:                  # ends with IR 0 published, synchronously
            ctx.set_histogram(hists[j], 1)
            irs[j] = ctx.build_ir(0)
        ctx.conv_init_source(0)
        started = [0]                                     # publication index q (IR q % K) last started by the game thread
        stop = threading.Event()
        err = []

        def game():
            try:
                prng = np.random.default_rng(8)
                q = 0
                while not stop.is_set():
                    q += 1
                    started[0] = q
                    ctx.set_histogram(hists[q % K], 1)
                    ctx.build_ir(0, want_ir=False)
                    time.sleep(float(prng.uniform(1e-3, 4e-3)))
            except Exception as e:                        # reported by the audio thread's assertions below
                err.append(e)

        t = threading.Thread(target=game)
        t.start()
        y = np.zeros((NB, BK, C), np.float32)
        upper = np.zeros(NB, np.int64)
        try:
            for k in range(NB):
                y[k] = ctx.conv_process(x[k * BK:(k + 1) * BK])
                upper[k] = started[0]
                time.sleep(5e-4)
        finally:
            stop.set()
            t.join()
        assert not err, err
    ys = cm.wet_outputs(x, irs)
    q_prev, cur_prev, fades = 0, None, 0
    for k in range(NB):
        cands = [(h, c) for h in range(K) for c in range(K)]
        match = [(h, c) for h, c in cands
                 if _rel(y[k], cm.block(x, ys, k, BK, c, None if h == c else h, False)) < TOL]
        assert len(match) == 1, "block %d: candidates %r" % (k, match)
        h, c = match[0]
        if cur_prev is None:                              # the first callback after fs_conv_init_source never fades
            assert h == c, "block 0 fades"
        else:
            assert h == cur_prev, "block %d fades from %d, previous block ended on %d" % (k, h, cur_prev)
        q = q_prev + (c - q_prev) % K                     # first publication of IR c at or after the previous one
        assert q <= upper[k], "block %d: IR %d is not a publication at or after %d" % (k, c, q_prev)
        fades += h != c
        q_prev, cur_prev = q, c
    assert fades >= 10, "only %d fade blocks: the schedule did not exercise the hand-off" % fades


# Click metric (tests/crossfade_model.click_metric) of the float64 model on the same workload, with IRs from the CPU
# oracle's shoebox traces (4096 pairs, depth 8, seeds 101..120, a new IR every 2nd block over 40 blocks, 250 Hz sine of
# amplitude 0.5 plus noise 40 dB below it, no clamp): hard swap 28.3, cross-fade 0.99.
CLICK_THRESHOLD = 3.0


def test_click_metric_on_device_output(fs):
    from frequensee import scenes
    sc = scenes.shoebox()
    NB, EVERY = 40, 2
    n = NB * BK
    t = np.arange(n) / float(FS)
    rng = np.random.default_rng(7)
    x = (0.5 * np.sin(2 * np.pi * 250 * t)[:, None] + 0.005 * rng.standard_normal((n, C))).astype(np.float32)
    bnd = list(range(EVERY, NB, EVERY))
    metric = {}
    for flag in (False, True):
        y = np.zeros((NB, BK, C), np.float32)
        with _ctx(fs, flag, conv_clamp=0) as ctx:
            ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption)
            ctx.conv_init_source(0)
            for k in range(NB):
                if k % EVERY == 0:
                    ctx.trace(sc.sources[:1], sc.listener, 4096, 8, 101 + k // EVERY, want_hist=False)
                    ctx.build_ir(0)
                y[k] = ctx.conv_process(x[k * BK:(k + 1) * BK])
        metric[flag] = cm.click_metric(y.reshape(-1, C), BK, bnd)
    assert metric[False] > CLICK_THRESHOLD > metric[True], metric
