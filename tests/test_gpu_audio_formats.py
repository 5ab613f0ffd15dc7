"""IR reconstruction and partitioned convolution on the device at every audio format of tests/audio_reference.FORMATS
(sample rates 8 - 96 kHz, 1 - 8 channels, conv_block 32 - 2048, rounded and truncating bin widths, warm-up windows up
to 8128 taps), against the float64 references of tests/audio_reference.py and tests/crossfade_model.py.
Tolerance: BASELINE.json's 1e-5 relative L2, per IR and per callback block.  The largest relative L2 of each test is
recorded as the junit property max_rel_l2."""
import numpy as np
import pytest

import audio_reference as ar
import crossfade_model as cm

pytestmark = pytest.mark.gpu
TOL = 1e-5
N_PATHS = 4096
SRCS = np.array([[1.5, 1.2, 1.0], [3.0, 2.0, 1.5], [5.5, 4.0, 2.0]], np.float32)


@pytest.fixture(scope="module")
def shoebox():
    from frequensee import scenes
    return scenes.shoebox()


class _Worst:
    def __init__(self):
        self.v = 0.0

    def check(self, got, want, what):
        r = ar.rel_l2(got, want)
        self.v = max(self.v, r)
        assert r < TOL, "%s: rel-L2 %g" % (what, r)


@pytest.fixture
def worst(request):
    w = _Worst()
    yield w
    request.node.user_properties.append(("max_rel_l2", "%.3e" % w.v))


def _irs(rng, fmt, keys, scale=0.05):
    """decaying noise IRs [C][sample_rate], distinct per channel, with a last tap so that the last partition counts"""
    C, ns = fmt["n_channels"], fmt["sample_rate"]
    out = {}
    for k in keys:
        ir = (rng.normal(size=(C, ns)) * np.exp(-np.arange(ns) / (ns / 16.0)) * scale).astype(np.float32)
        ir[:, -1] = 0.02
        out[k] = ir
    return out


def _check_blocks(worst, y, want, what):
    """every block with a non-zero reference to TOL; the others must be silent.  A block whose exact output is zero (the
    IR has not started yet) holds the FFT round-off of the float64 reference, ~1e-16 of the signal: that counts as zero."""
    silent = max(1e-9 * np.abs(want).max(), 1e-12)
    for k in range(len(want)):
        if np.abs(want[k]).max() > silent:
            worst.check(y[k], want[k], "%s block %d" % (what, k))
        else:
            assert np.abs(y[k]).max() < 1e-6, "%s block %d" % (what, k)


@pytest.mark.parametrize("fid", list(ar.FORMATS))
def test_ir_from_trace(fs, fid, shoebox, worst):
    """build_ir, build_ir_all, build_ir_bands (two seeds) and build_ir under FS_FLAG_IR_NORMALIZE on a traced histogram"""
    from frequensee import capi
    fmt = ar.FORMATS[fid]
    sc = shoebox
    with fs.Context(**fmt) as ctx:
        ctx.set_scene(sc.verts, sc.tri_mat, sc.absorption)
        h = ctx.trace(SRCS, sc.listener, N_PATHS, 8, 0x5EED)
        one = np.stack([ctx.build_ir(s) for s in range(len(SRCS))])
        allir = ctx.build_ir_all(len(SRCS))
        bands = {seed: ctx.build_ir_bands(seed, hist_source=1, conv_source=1) for seed in (5, 6)}
    with fs.Context(flags=capi.FLAG_IR_NORMALIZE, **fmt) as ctx:
        ctx.set_histogram(h, N_PATHS)
        normed = np.stack([ctx.build_ir(s) for s in range(len(SRCS))])
    C, ns = fmt["n_channels"], fmt["sample_rate"]
    assert one.shape == (len(SRCS), C, ns)
    assert np.array_equal(allir, one)
    for s in range(len(SRCS)):
        ref = ar.build_ir(fmt, h[s], N_PATHS)
        assert np.abs(ref).max() > 0
        worst.check(one[s], ref, "build_ir source %d" % s)
        worst.check(normed[s], ar.build_ir(fmt, h[s], N_PATHS, normalize=True), "normalised source %d" % s)
        for c in range(1, C):
            assert np.array_equal(one[s, c], one[s, 0]) and np.array_equal(normed[s, c], normed[s, 0])
    assert not np.array_equal(bands[5], bands[6])
    for seed, ir in bands.items():
        worst.check(ir, ar.build_ir_bands(fmt, h[1], N_PATHS, seed), "bands seed %d" % seed)
    end = fmt["n_bins"] * ar.spb(fmt)
    if end < ns:                                                 # past the last bin: no envelope, no low-pass tail
        assert not bands[5][:, end:].any() and not bands[6][:, end:].any()


@pytest.mark.parametrize("fid", list(ar.FORMATS))
def test_ir_from_energy(fs, fid, worst):
    """the edge energies of test_ir_from_energy_seam_and_edge_histograms at this format, and one bin exactly at the float32
    threshold next to one a rounding step below it"""
    fmt = ar.FORMATS[fid]
    K = fmt["n_bins"]
    rng = np.random.default_rng(2)
    thr = np.float32(ar.IR_THRESHOLD)
    edge = np.zeros(K, np.float32)
    edge[K // 50] = thr
    edge[K // 3] = np.nextafter(thr, np.float32(0))
    last = np.where(np.arange(K) == K - 1, 0.02, 0).astype(np.float32)
    cases = {"zero": np.zeros(K, np.float32),
             "sparse": (rng.uniform(0, 0.05, K) * (rng.uniform(size=K) < 0.3)).astype(np.float32),
             "last bin": last,
             "below threshold": np.full(K, 5e-7, np.float32),
             "threshold edge": edge}
    end = K * ar.spb(fmt)
    with fs.Context(**fmt) as ctx:
        for name, e in cases.items():
            ir = ctx.build_ir_from_energy(e)
            ref = ar.build_ir_from_energy(fmt, e)
            for c in range(1, fmt["n_channels"]):
                assert np.array_equal(ir[c], ir[0])
            if not ref.any():
                assert not ir.any(), name
                continue
            worst.check(ir, ref, name)
            if name == "last bin" and end < fmt["sample_rate"]:    # the low-pass's decaying tail after the ramp
                worst.check(ir[:, end:], ref[:, end:], "tail after the ramp")


@pytest.mark.parametrize("fid", list(ar.FORMATS))
def test_convolution_stream(fs, fid, worst):
    """2P + 8 blocks (the frequency-domain delay line wraps twice) with IR switches before and after the first wrap, through
    conv_process_many in chunks and block by block; then a unit impulse gives the IR back over P blocks and silence after"""
    fmt = ar.FORMATS[fid]
    bk, C = fmt["conv_block"], fmt["n_channels"]
    P = ar.partitions(fmt)
    nb = 2 * P + 8
    s1, s2 = max(1, P // 3), P + P // 3 + 1
    switch = {0: "a", s1: "b", s2: "c"}
    rng = np.random.default_rng(10)
    irs = _irs(rng, fmt, "abc")
    x = rng.uniform(-0.5, 0.5, size=(nb * bk, C)).astype(np.float32)
    blocks = x.reshape(nb, bk, C)
    with fs.Context(conv_clamp=0, **fmt) as ctx:
        for src in (0, 1, 2):
            ctx.set_ir(irs["a"], src); ctx.conv_init_source(src)
        bounds = sorted(switch) + [nb]
        many = []
        for i in range(len(bounds) - 1):
            ctx.set_ir(irs[switch[bounds[i]]], 0)
            many.append(ctx.conv_process_many(blocks[bounds[i]:bounds[i + 1]], 0))
        many = np.concatenate(many)
        stream = np.zeros_like(many)
        for k in range(nb):
            if k in switch:
                ctx.set_ir(irs[switch[k]], 1)
            stream[k] = ctx.conv_process(blocks[k], 1)
        imp = np.zeros((P + 4, bk, C), np.float32)
        imp[0, 0, :] = 1.0
        y_imp = ctx.conv_process_many(imp, 2)
    sched, cur = [], None
    for k in range(nb):
        cur = switch.get(k, cur)
        sched.append((None, cur))
    want = cm.run(x, irs, sched, bk, clamp=False)
    _check_blocks(worst, many, want, "many")
    assert np.array_equal(stream, many)
    back = np.zeros((P * bk, C), np.float64)
    back[:fmt["sample_rate"]] = irs["a"].T
    worst.check(y_imp[:P].reshape(-1, C), back, "impulse response")
    assert np.abs(y_imp[P:]).max() < 1e-6


@pytest.mark.parametrize("fid", ["F4", "F5", "F7", "F9"])
def test_crossfade_switches(fs, fid, worst):
    """FS_FLAG_CONV_CROSSFADE at conv_block 32 and 2048, mono and 8 channels: a -> b at block 20; b -> c -> d published
    between two callbacks (the fade is b -> d); d republished unchanged at block 30"""
    from frequensee import capi
    fmt = ar.FORMATS[fid]
    bk, C = fmt["conv_block"], fmt["n_channels"]
    NB = 36
    rng = np.random.default_rng(11)
    irs = _irs(rng, fmt, "abcd")
    x = rng.uniform(-0.6, 0.6, size=(NB * bk, C)).astype(np.float32)
    y = np.zeros((NB, bk, C), np.float32)
    sched = []
    with fs.Context(flags=capi.FLAG_CONV_CROSSFADE, conv_wet=0.75, **fmt) as ctx:
        ctx.set_ir(irs["a"]); ctx.conv_init_source(0)
        cur = "a"
        for k in range(NB):
            heard = None
            if k == 20:
                ctx.set_ir(irs["b"]); heard, cur = cur, "b"
            elif k == 25:
                ctx.set_ir(irs["c"]); ctx.set_ir(irs["d"]); heard, cur = cur, "d"
            elif k == 30:
                ctx.set_ir(irs["d"]); heard = "d"
            y[k] = ctx.conv_process(x[k * bk:(k + 1) * bk])
            sched.append((heard, cur))
    want = cm.run(x, irs, sched, bk, clamp=True, wet=0.75)
    _check_blocks(worst, y, want, fid)


def _many_source_hist(fmt, S, rng):
    """source 0 empty, every other source a distinct sparse decaying histogram whose first bin (2..8) varies"""
    K = fmt["n_bins"]
    h = np.zeros((S, 8, K), np.uint64)
    env = np.exp(-np.arange(K) / 150.0)
    for s in range(1, S):
        v = rng.uniform(0, 2.0 ** 33, size=(8, K)) * env * (rng.uniform(size=(8, K)) < 0.4)
        v[:, : 2 + s % 7] = 0
        h[s] = v.astype(np.uint64)
    return h


def test_more_than_64_sources(fs, worst):
    """F3 (5.1, 44.1 kHz, conv_block 256) with 130 sources, three chunks of the 64-entry pointer tables, the last one
    partial: build_ir_all against the reference source by source, then conv_process_multi over 2P blocks"""
    fmt = ar.FORMATS["F3"]
    S, bk, C = 130, fmt["conv_block"], fmt["n_channels"]
    nb = 2 * ar.partitions(fmt)
    rng = np.random.default_rng(12)
    h = _many_source_hist(fmt, S, rng)
    x = rng.uniform(-0.5, 0.5, size=(nb, S, bk, C)).astype(np.float32)
    ids = np.arange(S, dtype=np.uint32)
    y = np.zeros_like(x)
    with fs.Context(conv_clamp=0, **fmt) as ctx:
        ctx.set_histogram(h, 1000)
        irs = ctx.build_ir_all(S)
        for s in range(S):
            ctx.conv_init_source(s)
        for k in range(nb):
            y[k] = ctx.conv_process_multi(x[k], ids)
    assert not irs[0].any() and not y[:, 0].any()
    for s in range(1, S):
        worst.check(irs[s], ar.build_ir(fmt, h[s], 1000), "build_ir_all source %d" % s)
    for s in range(1, S):
        want = cm.run(x[:, s].reshape(-1, C), {"a": irs[s]}, [(None, "a")] * nb, bk, clamp=False)
        _check_blocks(worst, y[:, s], want, "source %d" % s)


def test_crossfade_across_the_chunk_boundary(fs, worst):
    """F3 with FS_FLAG_CONV_CROSSFADE and 130 sources: sources 63 and 64 (last of the first chunk, first of the second)
    switch IR in the same callback; every source matches its own model"""
    from frequensee import capi
    fmt = ar.FORMATS["F3"]
    S, bk, C = 130, fmt["conv_block"], fmt["n_channels"]
    NB, SW = 6, 3
    rng = np.random.default_rng(13)
    h = _many_source_hist(fmt, S, rng)
    x = rng.uniform(-0.5, 0.5, size=(S, NB * bk, C)).astype(np.float32)
    ids = np.arange(S, dtype=np.uint32)
    y = np.zeros((S, NB, bk, C), np.float32)
    with fs.Context(flags=capi.FLAG_CONV_CROSSFADE, conv_clamp=0, **fmt) as ctx:
        ctx.set_histogram(h, 1000)
        irs = ctx.build_ir_all(S)
        for s in range(S):
            ctx.conv_init_source(s)
        new = {63: irs[129], 64: irs[1]}
        for k in range(NB):
            if k == SW:
                for s, ir in new.items():
                    ctx.set_ir(ir, s)
            y[:, k] = ctx.conv_process_multi(x[:, k * bk:(k + 1) * bk], ids)
    for s in range(1, S):
        if s in new:
            sched = [(None, "a")] * SW + [("a", "b")] + [(None, "b")] * (NB - SW - 1)
            want = cm.run(x[s], {"a": irs[s], "b": new[s]}, sched, bk, clamp=False)
        else:
            want = cm.run(x[s], {"a": irs[s]}, [(None, "a")] * NB, bk, clamp=False)
        _check_blocks(worst, y[s], want, "source %d" % s)


def test_refused_threshold_and_energy(fs):
    """fs_create refuses an ir_threshold that is not finite and > 0; fs_build_ir_from_energy refuses a negative or
    non-finite entry and leaves the source's IR and convolver exactly as a context that never saw the call"""
    from frequensee import capi
    for bad in (0.0, -1e-6, float("nan"), float("inf")):
        with pytest.raises(fs.FrequenSeeError) as ei:
            fs.Context(ir_threshold=bad)
        assert ei.value.code == capi.FS_ERR_INVALID, bad
    rng = np.random.default_rng(14)
    e = (rng.uniform(0, 0.05, 1000) * (rng.uniform(size=1000) < 0.3)).astype(np.float32)
    x = rng.uniform(-0.5, 0.5, size=(4, 1024, 2)).astype(np.float32)

    def run(bad):
        with fs.Context(conv_clamp=0) as ctx:
            ctx.build_ir_from_energy(e)
            ctx.conv_init_source(0)
            y0 = ctx.conv_process_many(x[:2])
            if bad is not None:
                with pytest.raises(fs.FrequenSeeError) as ei:
                    ctx.build_ir_from_energy(bad)
                assert ei.value.code == capi.FS_ERR_INVALID
            return np.concatenate([y0, ctx.conv_process_many(x[2:])])

    clean = run(None)
    assert np.abs(clean).max() > 0
    for v in (-1e-3, np.nan, np.inf):
        bad = e.copy()
        bad[500] = v
        assert np.array_equal(run(bad), clean), v
