"""float64 restatements of the IR reconstruction (fs_build_ir, fs_build_ir_all, fs_build_ir_bands, fs_build_ir_from_energy)
at any audio format fs_create accepts, and the audio formats the tests run them at.

Only the threshold decision is taken on the float32 energy the library computes; everything after it is double:
  spb      = (uint32)(bin_ms * 1e-3 * sample_rate + 0.5), bin_ms as the float the config holds
  a_k      = E_k / sqrt(E_k sqrt(4 pi)) where |E_k| >= ir_threshold, else 0              (COMP.cpp:339-346)
  ramp[i]  = (1 - w) a_{k-1} + w a_k, k = i / spb, w = (i % spb) / spb, a_{-1} = a_0; 0 from n_bins * spb on
                                                                                       (COMP.cpp:347-363)
  y        = exact one-pole low-pass y_i = a x_i + (1 - a) y_{i-1}, y_0 = x_0, over all sample_rate samples, with the
             coefficients a and 1 - a as the float values the library multiplies by     (COMP.cpp:366-375)
  bands    = sum_b ramp_b * carrier_{c,b}: Philox4x32-10 noise through two RBJ band-pass sections at 62.5 2^b Hz
             (capped at 0.45 fs), unit RMS; no low-pass
  normalise: each channel divided by its L2 norm unless that norm is below 1e-4 (FS_FLAG_IR_NORMALIZE)
The convolver's reference is tests/crossfade_model.py."""
import numpy as np
from scipy.signal import lfilter

FLAG_IR_NORMALIZE = 1024

# id -> fs_config overrides.  P = ceil(sample_rate / conv_block) partitions of the convolver.
FORMATS = {
    "F1": dict(sample_rate=48000, n_channels=2, conv_block=1024, n_bins=1000, bin_ms=1.0, ir_lowpass=0.25),    # default
    "F2": dict(sample_rate=44100, n_channels=2, conv_block=512, n_bins=1000, bin_ms=1.0, ir_lowpass=0.25),     # spb 44.1 -> 44
    "F3": dict(sample_rate=44100, n_channels=6, conv_block=256, n_bins=1000, bin_ms=1.0, ir_lowpass=0.25),     # 5.1
    "F4": dict(sample_rate=96000, n_channels=8, conv_block=32, n_bins=1000, bin_ms=1.0, ir_lowpass=0.25),      # P = 3000
    "F5": dict(sample_rate=16000, n_channels=1, conv_block=128, n_bins=1000, bin_ms=1.0, ir_lowpass=0.25),     # mono
    "F6": dict(sample_rate=22050, n_channels=3, conv_block=2048, n_bins=400, bin_ms=2.7, ir_lowpass=0.9),      # spb 59.5 -> 60
    "F7": dict(sample_rate=8000, n_channels=2, conv_block=2048, n_bins=1000, bin_ms=1.0, ir_lowpass=1.0),      # P = 4
    "F8": dict(sample_rate=48000, n_channels=1, conv_block=64, n_bins=2000, bin_ms=1.0, ir_lowpass=0.0034),   # W = 8128 taps
    "F9": dict(sample_rate=48000, n_channels=8, conv_block=2048, n_bins=1000, bin_ms=1.0, ir_lowpass=0.25),    # 96 KB smem fade
    "F10": dict(sample_rate=32000, n_channels=4, conv_block=32, n_bins=500, bin_ms=2.0, ir_lowpass=0.25),     # spb 64
}

IR_THRESHOLD = 1e-6
N_BANDS = 8
PI4 = np.sqrt(4.0 * np.pi)


def partitions(fmt):
    return -(-fmt["sample_rate"] // fmt["conv_block"])


def spb(fmt):
    """samples per bin, rounded exactly as fs_ir.cu does it"""
    return int(float(np.float32(fmt["bin_ms"])) * 1e-3 * fmt["sample_rate"] + 0.5)


def energy_f32(hist_bk, n_paths):
    """the float32 energy of one histogram row (or of the band sum): (float)((double)sum * 2^-32 / n_paths)"""
    s = np.asarray(hist_bk, np.uint64)
    return (s.astype(np.float64) * (1.0 / 4294967296.0) / float(n_paths)).astype(np.float32)


def amplitudes(e32, threshold=IR_THRESHOLD):
    """COMP.cpp:339-346 in double, the threshold taken on the float32 energy"""
    keep = np.abs(e32) >= np.float32(threshold)
    e = np.where(keep, e32.astype(np.float64), 0.0)
    out = np.zeros_like(e)
    out[keep] = e[keep] / np.sqrt(e[keep] * PI4)
    return out


def ramp(amp, fmt):
    """COMP.cpp:347-363: [sample_rate] piecewise-linear envelope, 0 from n_bins * spb on"""
    ns, k, n = fmt["sample_rate"], len(amp), spb(fmt)
    i = np.arange(ns)
    b = i // n
    w = (i - b * n) / float(n)
    inside = b < k
    bc = np.minimum(b, k - 1)
    e = amp[bc]
    pe = np.where(bc > 0, amp[np.maximum(bc - 1, 0)], amp[0])
    return np.where(inside, (1.0 - w) * pe + w * e, 0.0)


def lowpass(x, a):
    """y_i = a x_i + (1 - a) y_{i-1}, y_0 = x_0, exact over all samples; a and 1 - a are the floats the library uses"""
    a = float(np.float32(a))
    c = float(np.float32(1.0) - np.float32(a))
    if len(x) == 0:
        return x
    y, _ = lfilter([a], [1.0, -c], x, zi=[x[0] - a * x[0]])
    return y


def normalise(ir):
    out = ir.copy()
    for c in range(len(out)):
        n = np.sqrt(np.sum(out[c] ** 2))
        if np.float32(n) >= np.float32(1e-4):
            out[c] /= n
    return out


def build_ir_from_energy(fmt, energy, normalize=False):
    """fs_build_ir_from_energy: energy float32 [n_bins] -> float64 [n_channels][sample_rate]"""
    e32 = np.asarray(energy, np.float32)
    y = lowpass(ramp(amplitudes(e32), fmt), fmt["ir_lowpass"])
    ir = np.repeat(y[None], fmt["n_channels"], axis=0)
    return normalise(ir) if normalize else ir


def build_ir(fmt, hist, n_paths, normalize=False):
    """fs_build_ir of one source: hist uint64 [n_bands][n_bins], summed over the bands in integers"""
    h = np.asarray(hist, np.uint64)
    return build_ir_from_energy(fmt, energy_f32(h.sum(axis=0, dtype=np.uint64), n_paths), normalize)


# ---- Philox4x32-10, vectorised over counters (the library's and the oracle's generator) ------------------------------
_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_U32 = 0xFFFFFFFF


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """counters (uint arrays or scalars, broadcast) and key -> four uint32 arrays"""
    c = [np.asarray(v, np.uint64) & _U32 for v in (c0, c1, c2, c3)]
    c = np.broadcast_arrays(*c)
    c0, c1, c2, c3 = (v.copy() for v in c)
    k0, k1 = np.uint64(k0 & _U32), np.uint64(k1 & _U32)
    for r in range(10):
        p0 = np.uint64(_M0) * c0
        p1 = np.uint64(_M1) * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & np.uint64(_U32)
        hi1, lo1 = p1 >> np.uint64(32), p1 & np.uint64(_U32)
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0 = (k0 + np.uint64(_W0)) & np.uint64(_U32)
        k1 = (k1 + np.uint64(_W1)) & np.uint64(_U32)
    return c0, c1, c2, c3


def white_noise(seed, ch, band, n):
    """x[t] = r[t % 4] * 2^-31 - 1, r = Philox(counter (t / 4, 'IRNZ', ch, band), key = seed)"""
    q = np.arange((n + 3) // 4, dtype=np.uint64)
    r = philox4x32_10(q, 0x49524E5A, ch, band, seed & _U32, seed >> 32)
    u = np.stack(r, axis=1).reshape(-1)[:n]
    return u.astype(np.float64) * (2.0 / 4294967296.0) - 1.0


def band_centre(fmt, b):
    return min(62.5 * 2.0 ** b, 0.45 * fmt["sample_rate"])


def band_carriers(fmt, seed, n_bands=N_BANDS):
    """[n_channels][n_bands][sample_rate] float64 unit-RMS band-limited noise"""
    ns, fsr = fmt["sample_rate"], float(fmt["sample_rate"])
    out = np.zeros((fmt["n_channels"], n_bands, ns))
    for b in range(n_bands):
        w0 = 2.0 * np.pi * band_centre(fmt, b) / fsr
        alpha = np.sin(w0) / (2.0 * np.sqrt(2.0))
        a0 = 1.0 + alpha
        num = [alpha / a0, 0.0, -alpha / a0]
        den = [1.0, -2.0 * np.cos(w0) / a0, (1.0 - alpha) / a0]
        for c in range(fmt["n_channels"]):
            v = lfilter(num, den, lfilter(num, den, white_noise(seed, c, b, ns)))
            rms = np.sqrt(np.mean(v * v))
            out[c, b] = v / rms if rms > 0 else 0.0
    return out


def build_ir_bands(fmt, hist, n_paths, seed, normalize=False, carriers=None):
    """fs_build_ir_bands: ir[c][t] = sum_b ramp_b[t] carrier[c][b][t]"""
    h = np.asarray(hist, np.uint64)
    car = band_carriers(fmt, seed, len(h)) if carriers is None else carriers
    env = np.stack([ramp(amplitudes(energy_f32(h[b], n_paths)), fmt) for b in range(len(h))])
    ir = np.einsum("bt,cbt->ct", env, car)
    return normalise(ir) if normalize else ir


def rel_l2(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))
