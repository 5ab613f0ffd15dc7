"""The float64 IR references of tests/audio_reference.py and the convolution model of tests/crossfade_model.py against the
CPU oracle, at every audio format the GPU tests use: they restate the library's semantics before they judge the device."""
import numpy as np
import pytest

import audio_reference as ar
import crossfade_model as cm

TOL = 1e-5


def _hist(fmt, seed, n_paths):
    """[8][n_bins] decaying sparse histogram: empty bins, bins near the threshold and bins far above it"""
    rng = np.random.default_rng(seed)
    k = fmt["n_bins"]
    at_thr = n_paths * 2.0 ** 32 * 1e-6                        # integer sum of a bin at the threshold energy
    env = np.exp(-np.arange(k) / (0.3 * k))
    h = rng.uniform(0.0, 50.0, size=(8, k)) * env * at_thr * (rng.uniform(size=(8, k)) < 0.6)
    h[:, : k // 50] = 0                                        # nothing before the direct path
    near = rng.choice(k, size=k // 20, replace=False)          # band sums within a few per cent of the threshold
    h[:, near] = at_thr / 8 * rng.uniform(0.95, 1.05, size=(1, len(near)))
    return h.astype(np.uint64)


@pytest.mark.parametrize("fid", list(ar.FORMATS))
def test_ir_references_match_oracle(oracle, fid):
    fmt = ar.FORMATS[fid]
    n_paths = 4096
    h = _hist(fmt, 1, n_paths)
    for norm in (False, True):
        cfg = oracle.default_config(**fmt, flags=ar.FLAG_IR_NORMALIZE if norm else 0)
        r = ar.rel_l2(oracle.build_ir(cfg, h, n_paths), ar.build_ir(fmt, h, n_paths, norm))
        assert r < TOL, (fid, norm, r)
        e = ar.energy_f32(h[3], n_paths)
        r = ar.rel_l2(oracle.build_ir_from_energy(cfg, e), ar.build_ir_from_energy(fmt, e, norm))
        assert r < TOL, (fid, norm, r)
    cfg = oracle.default_config(**fmt)
    ref = ar.build_ir_bands(fmt, h, n_paths, 9)
    assert ar.rel_l2(oracle.build_ir_bands(cfg, h, n_paths, 9), ref) < TOL
    if fmt["n_bins"] * ar.spb(fmt) < fmt["sample_rate"]:       # the ramp ends before the IR does
        assert not ref[:, fmt["n_bins"] * ar.spb(fmt):].any()


def test_spb_rounding_and_band_caps():
    assert [ar.spb(ar.FORMATS[f]) for f in ("F1", "F2", "F6", "F10")] == [48, 44, 60, 64]
    assert ar.band_centre(ar.FORMATS["F7"], 6) == 3600.0 and ar.band_centre(ar.FORMATS["F7"], 5) == 2000.0
    assert ar.band_centre(ar.FORMATS["F5"], 7) == 7200.0 and ar.band_centre(ar.FORMATS["F2"], 7) == 8000.0
    assert [ar.partitions(ar.FORMATS[f]) for f in ar.FORMATS] == [47, 87, 173, 3000, 125, 11, 4, 750, 24, 1000]


def test_philox_matches_oracle(oracle):
    rng = np.random.default_rng(5)
    for _ in range(20):
        ctr = [int(v) for v in rng.integers(0, 2 ** 32, 4, dtype=np.uint64)]
        key = [int(v) for v in rng.integers(0, 2 ** 32, 2, dtype=np.uint64)]
        got = [int(v) for v in ar.philox4x32_10(*ctr, *key)]
        assert got == oracle.philox(ctr, key)


def test_convolution_model_matches_oracle(oracle):
    """8 kHz, conv_block 32, two channels: the model over 2P + 8 blocks with two IR switches, against the oracle's
    direct-form convolver"""
    fmt = dict(ar.FORMATS["F7"], conv_block=32)
    bk, C, ns = 32, 2, fmt["sample_rate"]
    P = ar.partitions(fmt)
    nb = 2 * P + 8
    rng = np.random.default_rng(3)
    irs = {k: (rng.normal(size=(C, ns)) * np.exp(-np.arange(ns) / 500.0) * 0.05).astype(np.float32) for k in "abc"}
    for ir in irs.values():
        ir[:, -1] = 0.02
    x = rng.uniform(-0.5, 0.5, size=(nb * bk, C)).astype(np.float32)
    switch = {0: "a", P // 3: "b", P + P // 3 + 1: "c"}
    cfg = oracle.default_config(**fmt, conv_clamp=0)
    cv = oracle.Conv(cfg)
    sched, got, cur = [], [], None
    for k in range(nb):
        if k in switch:
            cur = switch[k]
            cv.set_ir(irs[cur])
        sched.append((None, cur))
        got.append(cv.process(x[k * bk:(k + 1) * bk]))
    want = cm.run(x, irs, sched, bk, clamp=False)
    for k in range(nb):
        assert ar.rel_l2(got[k], want[k]) < TOL, k


def test_fs_create_refuses_a_threshold_that_is_not_finite_and_positive(fs):
    """checked before any device is looked for, so this holds on a machine without a GPU as well"""
    for bad in (0.0, -1e-6, float("nan"), float("inf")):
        with pytest.raises(fs.FrequenSeeError) as ei:
            fs.Context(ir_threshold=bad)
        assert ei.value.code == fs.capi.FS_ERR_INVALID, bad
        assert "ir_threshold" in str(ei.value)
