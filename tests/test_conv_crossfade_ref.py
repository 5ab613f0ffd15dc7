"""The float64 cross-fade model of tests/crossfade_model.py checked on the CPU: without an IR switch it is the oracle's
streaming convolver, and its window table has the documented end values."""
import numpy as np

import crossfade_model as cm


def test_model_without_switch_equals_oracle_conv(oracle):
    cfg = oracle.default_config()
    bk, C, L = cfg.conv_block, cfg.n_channels, cfg.sample_rate
    rng = np.random.default_rng(11)
    ir = (rng.normal(size=(C, L)) * np.exp(-np.arange(L) / 2000.0) * 0.05).astype(np.float32)
    NB = 4
    x = rng.uniform(-0.6, 0.6, size=(NB * bk, C)).astype(np.float32)
    cv = oracle.Conv(cfg)
    cv.set_ir(ir)
    want = np.stack([cv.process(x[k * bk:(k + 1) * bk]) for k in range(NB)])
    got = cm.run(x, {"a": ir}, [(None, "a")] * NB, bk, clamp=bool(cfg.conv_clamp), wet=cfg.conv_wet)
    assert np.linalg.norm(got - want) / np.linalg.norm(want) < 1e-6


def test_window_table_end_values():
    w = cm.window(1024)
    assert w.dtype == np.float32 and w.shape == (1024,)
    assert w[-1] == 1.0 and 0.0 < w[0] < 1e-5
    assert np.all(np.diff(w) >= 0)
    for bk in (32, 2048):
        assert cm.window(bk)[-1] == 1.0


def test_fade_between_equal_outputs_is_plain():
    rng = np.random.default_rng(12)
    bk = 64
    x = rng.uniform(-0.5, 0.5, size=(3 * bk, 2)).astype(np.float32)
    ir = (rng.normal(size=(2, 200)) * 0.1).astype(np.float32)
    plain = cm.run(x, {"a": ir}, [(None, "a")] * 3, bk, clamp=False)
    faded = cm.run(x, {"a": ir, "b": ir.copy()}, [(None, "a"), ("a", "b"), (None, "b")], bk, clamp=False)
    assert np.allclose(plain, faded, rtol=0, atol=1e-12)
