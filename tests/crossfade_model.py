"""float64 model of the convolver with FS_FLAG_CONV_CROSSFADE.

Every IR a source was given is convolved with the source's whole input history (since fs_conv_init_source, zero before)
in double precision; a callback block is then either the plain output of one IR or, on a fade block, the window blend of
the output of the IR heard before and of the newly adopted one, followed by the clamp and wet/dry mix of
fso_conv_process."""
import numpy as np
from scipy.signal import fftconvolve


def window(bk):
    """the fade-in table the library uploads: w[i] = 0.5 - 0.5 cos(pi (i+1) / Bk), computed in double, stored as float"""
    i = np.arange(bk, dtype=np.float64)
    return (0.5 - 0.5 * np.cos(np.pi * (i + 1.0) / bk)).astype(np.float32)


def wet_outputs(x, irs):
    """x: [n][C] input history; irs: {key: [C][L] IR} -> {key: [n][C] float64 history (*) IR, first n samples}"""
    x = np.asarray(x, np.float64)
    n, C = x.shape
    return {k: np.stack([fftconvolve(x[:, c], np.asarray(ir[c], np.float64))[:n] for c in range(C)], axis=1)
            for k, ir in irs.items()}


def block(x, ys, k, bk, cur, heard=None, clamp=True, wet=1.0):
    """expected output of callback block k: plain with IR `cur` (heard None), or the fade from `heard` to `cur`"""
    s = slice(k * bk, (k + 1) * bk)
    v = ys[cur][s]
    if heard is not None:
        w = window(bk).astype(np.float64)[:, None]
        v = (1.0 - w) * ys[heard][s] + w * v
    if clamp:
        v = np.clip(v, -1.0, 1.0)
    return v * wet + np.asarray(x[s], np.float64) * (1.0 - wet)


def run(x, irs, schedule, bk, clamp=True, wet=1.0):
    """x: [n_blocks * bk][C]; schedule[k] = (heard or None, cur) -> expected [n_blocks][bk][C]"""
    ys = wet_outputs(x, irs)
    return np.stack([block(x, ys, k, bk, cur, heard, clamp, wet) for k, (heard, cur) in enumerate(schedule)])


def click_metric(y, bk, boundaries):
    """RMS of the sample step across the block boundaries where a new IR took effect over the RMS of the steps between
    neighbouring samples inside blocks.  y: [n][C]; boundaries: block indices k (the step y[k Bk] - y[k Bk - 1])."""
    y = np.asarray(y, np.float64)
    d = np.diff(y, axis=0)                      # d[j] = y[j + 1] - y[j]
    at = np.zeros(len(d), bool)
    at[[k * bk - 1 for k in boundaries]] = True
    interior = np.ones(len(d), bool)
    interior[np.arange(bk - 1, len(d), bk)] = False
    return float(np.sqrt(np.mean(d[at] ** 2)) / np.sqrt(np.mean(d[interior] ** 2)))
