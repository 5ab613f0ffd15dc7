"""Pins oracle/fs_oracle.c against the REFERENCE'S OWN CODE for the BDPT and IR stages.

oracle/_ref/libref_ue_bodies.so holds the unmodified bodies of UAudioRayTracingSubsystem::{UpdateSource,
GenerateFullPaths, ConnectSubpaths, GeneratePath, EvaluatePath} (SUB.cpp:128-420), UFrequenSeeAudioComponent::
{FlushEnergyBuffer, AddEnergyAtDelay, ReconstructImpulseResponse} (COMP.h:76-91, COMP.cpp:320-380) and the reverb plugin's
Initialize / ConvolveFFT / FCircularAudioBuffer (REV.cpp:74-102, 172-213, CIRC.cpp), compiled from /root/reference against
the engine stand-in oracle/ue_shim (scene query, random numbers; see oracle/ref_ue_bodies.cpp).  The oracle runs with the
reference's own constants (pyoracle.ue_pin_config: one band = Absorption[2] used as reflectivity, distances / 1000,
"NodeDistance < 1" skip, air 0.05, offsets 0.1 units, 49 samples per bin).

Tolerances: the reference computes geometry in double (FVector) and calls libm exp/powf, the oracle is float with
polynomial exp/log -- agreement is to float rounding, not bit for bit, except where the arithmetic is identical
(bin index, IR reconstruction: bit-exact).
"""
import os

import numpy as np
import pytest


@pytest.fixture(scope="module")
def po(oracle):
    if oracle.ref_ue_lib() is None:
        pytest.skip("oracle/_ref/libref_ue_bodies.so not built (reference tree absent)")
    return oracle


def pin_scene():
    """shoebox 7 x 5 x 3 m with a partition wall, a low table block and a cabinet: about half of the end-point pairs occluded"""
    from frequensee import scenes
    t, face = scenes.box((0, 0, 0), (7.0, 5.0, 3.0), 1)
    parts, mats = [t], [np.array([0, 6, 2, 1, 3, 4], np.uint32)[face]]
    for lo, hi, m in (((3.2, 0.0, 0.0), (3.5, 3.2, 2.4), 1), ((4.4, 2.6, 0.0), (5.8, 3.6, 0.8), 7), ((0.8, 3.4, 0.0), (1.6, 4.6, 1.9), 5)):
        b, _ = scenes.box(lo, hi, 1)
        parts.append(b); mats.append(np.full(len(b), m, np.uint32))
    return np.concatenate(parts), np.concatenate(mats), scenes.absorption_table(8), [1.5, 1.2, 1.0], [5.0, 3.5, 1.6]


def closet_scene():
    """2 x 2 x 2 m box, source and listener 1.2 m apart: direct paths put bins above the reference's 1e-6 IR threshold"""
    from frequensee import scenes
    t, face = scenes.box((0, 0, 0), (2.0, 2.0, 2.0), 1)
    return t, np.array([0, 6, 2, 1, 3, 4], np.uint32)[face], scenes.absorption_table(8), [0.4, 1.0, 1.0], [1.6, 1.0, 1.0]


def test_evaluate_path_body(po):
    """EvaluatePath (SUB.cpp:360-420): node order, which node's material / probability a segment uses, the < 1 skip,
    1/(4 pi d^2), exp(-0.05 d), pow(p, 0.1), clamp-then-gain, delay = sum d / 343"""
    rng = np.random.default_rng(11)
    cfg = po.ue_pin_config()
    refl = np.linspace(0.05, 0.95, 8).astype(np.float32)
    S = po.Scene(np.zeros((0, 3, 3), np.float32), np.zeros(0, np.uint32), (1.0 - refl)[:, None].copy(), use_bvh=False)
    worst_d = worst_g = 0.0
    n_clamped = n_skipped = 0
    for trial in range(400):
        n = int(rng.integers(2, 40))
        step = rng.uniform(0.2, 1.6) if trial % 3 == 0 else rng.uniform(1.0, 12.0)      # every third path has short segments
        pos = np.cumsum(rng.normal(size=(n, 3)) * step, axis=0).astype(np.float32)
        mat = rng.integers(-1, 8, size=n).astype(np.int32)
        prob = rng.uniform(0.005, 1.0, size=n).astype(np.float32)
        if trial % 7 == 0:                                                               # short, loud path: exercises the clamp
            p0 = rng.uniform(-3, 3, 3).astype(np.float32)
            pos = np.stack([p0, p0 + np.float32([1.01, 0, 0]), p0 + np.float32([1.01, 1.02, 0])]).astype(np.float32)
            mat = rng.integers(-1, 8, size=3).astype(np.int32); prob = np.full(3, 1e-25, np.float32)
        seg = np.linalg.norm(np.diff(pos.astype(np.float64), axis=0), axis=1)
        if np.abs(seg - 1.0).min() < 1e-4:
            continue                                                                     # float vs double could disagree on "< 1"
        n_skipped += int((seg < 1.0).sum())
        d_o, e_o = po.evaluate_nodes(S, cfg, pos, mat, prob)
        v2 = np.where(mat >= 0, refl[np.maximum(mat, 0)], -1.0).astype(np.float32)
        d_r, g_r = po.ref_ue_evaluate_path(pos.astype(np.float64) * po.UE_UNIT, v2, prob)
        n_clamped += int(g_r == 10.0)
        worst_d = max(worst_d, abs(d_o / d_r - 1.0))
        if g_r > 1e-30:
            worst_g = max(worst_g, abs(float(e_o[0]) / g_r - 1.0))
        else:
            assert e_o[0] < 1e-30
    assert n_clamped >= 20 and n_skipped > 200
    assert worst_d < 2e-6 and worst_g < 5e-5, (worst_d, worst_g)


def test_add_energy_at_delay_body(po):
    """AddEnergyAtDelay (COMP.h:87-91): FloorToInt(delay * 1000 / BinSizeMs) clamped into [0, NumBins - 1] -- exact.
    (Delays beyond 2^31 ms = 24 days overflow the reference's int32 conversion and land in bin 0; the harness keeps them in
    the last bin.  Path delays are bounded by depth x scene size / 343 m/s: never reached, not tested.)"""
    rng = np.random.default_rng(5)
    cfg = po.ue_pin_config()
    delays = np.concatenate([rng.uniform(-0.1, 1.3, 3000), np.arange(0, 1001) / 1000.0, [2e6, -2e6, 5.0, 0.9989999, 0.999, 0.9999999]]).astype(np.float32)
    for d in delays:
        buf = po.ref_ue_add_energy([d], [1.0])
        assert list(np.flatnonzero(buf)) == [po.bin_index(cfg, d)], float(d)
    # accumulation: the float EnergyBuffer equals the sum of what lands in each bin
    e = rng.uniform(0, 1e-3, len(delays)).astype(np.float32)
    buf = po.ref_ue_add_energy(delays, e)
    acc = np.zeros(1000)
    for d, x in zip(delays, e):
        acc[po.bin_index(cfg, d)] += float(x)
    assert np.allclose(buf, acc, rtol=1e-5, atol=1e-9)


def test_reconstruct_impulse_response_body_bit_exact(po):
    """ReconstructImpulseResponse (COMP.cpp:320-380): the oracle with the reference's 49 samples per bin reproduces it BIT FOR
    BIT (same float operations in the same order); the harness default (48, the FIX of SURVEY A7) differs exactly there"""
    rng = np.random.default_rng(7)
    cfg49 = po.ue_pin_config(bin_ms=49.0 / 48.0)
    cfg48 = po.ue_pin_config()
    for trial in range(6):
        e = (rng.uniform(0, 1, 1000) ** 4 * 10.0 ** rng.uniform(-7, -2)).astype(np.float32)     # values on both sides of the 1e-6 threshold
        e[rng.integers(0, 1000, 300)] = 0.0
        if trial == 0:
            e[:] = 0.0; e[17] = 3e-4                                                            # single-bin KAT
        ir, spb = po.ref_ue_reconstruct_ir(e)
        assert spb == 49                                                                        # ceil(0.001f * 48000) on this host too
        o49 = po.build_ir_from_energy(cfg49, e)
        assert np.array_equal(o49, ir)
        assert np.array_equal(ir[0], ir[1])                                                     # both channels read the same mono histogram
        # the reference never writes the bins past 48000 / 49 = 979.6; the FIXed harness does (48 samples per bin)
        e_tail = np.zeros(1000, np.float32); e_tail[990] = 1e-3
        assert not ref_nonzero(po, e_tail) and po.build_ir_from_energy(cfg48, e_tail).any()
    # same envelope, different time axis: sample j of bin k sits at 49 k + j in the reference and at 48 k + j in the harness
    e = np.zeros(1000, np.float32); e[100] = 2e-4
    ir, _ = po.ref_ue_reconstruct_ir(e)
    o48 = po.build_ir_from_energy(cfg48, e)
    assert int(np.flatnonzero(ir[0])[0]) == 100 * 49 + 1 and int(np.flatnonzero(o48[0])[0]) == 100 * 48 + 1
    assert abs(float(ir[0].max()) / float(o48[0].max()) - 1.0) < 0.02


def ref_nonzero(po, e):
    return bool(po.ref_ue_reconstruct_ir(e)[0].any())


@pytest.mark.parametrize("scene_fn, seeds", [(pin_scene, (1, 2, 3, 4)), (closet_scene, (5, 6))])
def test_update_source_whole_reference_loop(po, scene_fn, seeds):
    """The reference's UpdateSource, whole and unmodified (1000 path pairs): GenerateFullPaths -> GeneratePath x 2 +
    ConnectSubpaths -> EvaluatePath -> AddEnergyAtDelay -> ReconstructImpulseResponse, against the oracle's fso_trace +
    fso_build_ir on the same scene, seeds and constants."""
    verts, tri_mat, ab, src, lis = scene_fn()
    W = po.RefUEWorld(verts, tri_mat, 1.0 - ab[:, 2])
    S = po.Scene(verts, tri_mat, ab[:, 2:3].copy(), use_bvh=False)
    cfg = po.ue_pin_config()
    n = 1000
    any_ir = False
    for seed in seeds:
        e_ref, ir_ref, n_traces = W.update_source(src, lis, seed)
        h, st, dbg = S.trace(cfg, [src], lis, n, 512, seed, debug=True)
        # every ray the reference traces, the oracle traces (Russian roulette and the walk order are the same)
        assert n_traces == st["ext_rays"] + st["shadow_rays"]
        rec = W.paths(src, lis, seed, n)
        assert np.array_equal(rec["n_src_nodes"], dbg["n_src_nodes"]) and np.array_equal(rec["n_lis_nodes"], dbg["n_lis_nodes"])
        assert int(rec["n_src_nodes"].max()) < 512                                   # the oracle's max_depth never cut a walk
        same = rec["connected"] == dbg["connected"]
        short = (rec["n_src_nodes"] + rec["n_lis_nodes"]) <= 8
        assert same[short].all() and same.mean() >= 0.995                            # long walks amplify float-vs-double rounding
        m = short & (rec["connected"] == 1)
        assert m.sum() > 30
        assert np.abs(rec["delay_s"][m] / dbg["delay_s"][m] - 1.0).max() < 1e-5
        assert np.allclose(rec["gain"][m], dbg["energy"][m, 0], rtol=5e-5, atol=1e-30)
        assert np.allclose(rec["src_end"][m] / po.UE_UNIT, dbg["src_end"][m], atol=2e-4)
        # the histogram: float EnergyBuffer (1/1000 applied per path) vs Q32.32 integers / 2^32 / 1000
        e_or = h[0, 0].astype(np.float64) / 2.0 ** 32 / n
        assert e_ref.sum() > 0 and np.abs(e_ref - e_or).sum() / e_or.sum() < 2e-5
        # the IR of that histogram (49 samples per bin, as the reference computes)
        ir_or = po.build_ir_from_energy(po.ue_pin_config(bin_ms=49.0 / 48.0), e_or.astype(np.float32))
        if ir_ref.any():
            any_ir = True
            assert np.linalg.norm(ir_or - ir_ref) / np.linalg.norm(ir_ref) < 1e-5
        else:
            assert not ir_or.any()                                                   # every bin below kEnergyThreshold = 1e-6
    if scene_fn is closet_scene:
        assert any_ir


@pytest.mark.parametrize("scene_fn, seed, tag", [(pin_scene, 1, "pin_seed1"), (closet_scene, 5, "closet_seed5")])
def test_update_source_against_stored_reference_output(oracle, scene_fn, seed, tag):
    """The same comparison without the reference tree: the oracle against the output of the reference's UpdateSource stored
    in tests/golden/ref_ue_v1.npz (ray count, EnergyBuffer, and the IR where the reference produced one)."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_ue_v1.npz"))
    verts, tri_mat, ab, src, lis = scene_fn()
    S = oracle.Scene(verts, tri_mat, ab[:, 2:3].copy(), use_bvh=False)
    h, st = S.trace(oracle.ue_pin_config(), [src], lis, 1000, 512, seed)
    assert st["ext_rays"] + st["shadow_rays"] == int(g[tag + "_traces"])
    e_ref = g[tag + "_energy"]
    e_or = h[0, 0].astype(np.float64) / 2.0 ** 32 / 1000
    assert e_ref.sum() > 0 and np.abs(e_ref - e_or).sum() / e_or.sum() < 2e-5
    if tag + "_ir0" in g:
        ir_ref = g[tag + "_ir0"]
        ir_or = oracle.build_ir_from_energy(oracle.ue_pin_config(bin_ms=49.0 / 48.0), e_or.astype(np.float32))
        assert ir_ref.any() and np.linalg.norm(ir_or[0] - ir_ref) / np.linalg.norm(ir_ref) < 1e-5


def test_flush_energy_buffer_keeps_old_energy_in_the_engine(po):
    """FlushEnergyBuffer is EnergyBuffer.SetNumZeroed(NumBins) (COMP.h:76-79): the engine zero-fills only NEW elements, so once
    the buffer has its size a 'flush' clears nothing -- which is why the second flush at SUB.cpp:191 does not blank the IR in
    the reference, and why consecutive updates accumulate there.  The harness clears (the evident intent): documented FIX."""
    verts, tri_mat, ab, src, lis = closet_scene()
    W = po.RefUEWorld(verts, tri_mat, 1.0 - ab[:, 2])
    e, ir, _ = W.update_source(src, lis, 5)
    assert e.any() and ir.any()                                                      # not blanked by the flush before Reconstruct


def test_reverb_bodies_against_direct_form(po, oracle):
    """ConvolveFFT + Initialize (REV.cpp:74-102, 172-213) + FCircularAudioBuffer (CIRC.cpp) + KissFFT, all the reference's own
    code, against the oracle's double-precision direct form; and identical to the restated driver oracle/ref_kissfft_conv.c"""
    rng = np.random.default_rng(2)
    ir = (rng.normal(size=(2, 48000)) * np.exp(-np.arange(48000) / 6000.0) * 0.01).astype(np.float32)
    x = rng.uniform(-0.5, 0.5, size=(4, 1024, 2)).astype(np.float32)
    cfg = oracle.default_config()
    cv = oracle.Conv(cfg); cv.set_ir(ir)
    ue = po.RefUEConv(); ue.set_ir(ir)
    assert ue.fft_size == 65536
    rk = oracle.RefKissConv() if oracle.ref_lib() is not None else None
    if rk is not None:
        rk.set_ir(ir)
    for b in range(4):
        y = ue.process(x[b])
        yo = cv.process(x[b])
        assert np.linalg.norm(y - yo) / np.linalg.norm(yo) < 1e-5
        if rk is not None:
            assert np.array_equal(y, rk.process(x[b]))


def test_reference_golden_fixture_is_current(po):
    """tests/golden/ref_ue_v1.npz (made by tests/golden/make_ref_ue_golden.py from the reference bodies) still equals what
    the library computes -- the fixture is what the GPU parity test falls back to when oracle/_ref did not travel"""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_ue_v1.npz"))
    verts, tri_mat, ab, src, lis = pin_scene()
    W = po.RefUEWorld(verts, tri_mat, 1.0 - ab[:, 2])
    e, ir, n_traces = W.update_source(src, lis, 1)
    assert np.array_equal(e, g["pin_seed1_energy"]) and int(g["pin_seed1_traces"]) == n_traces
    verts, tri_mat, ab, src, lis = closet_scene()
    W = po.RefUEWorld(verts, tri_mat, 1.0 - ab[:, 2])
    e, ir, n_traces = W.update_source(src, lis, 5)
    assert np.array_equal(e, g["closet_seed5_energy"]) and np.array_equal(ir[0], g["closet_seed5_ir0"])
