"""Room-acoustic parameters of the energy histogram (fs_get_acoustic_params), without a GPU: the reference
(tests/acoustics_oracle.py) against answers worked out by hand -- exponential decays give T20 / T30 back, the EDT of a
two-slope curve, C50 / D50 / Ts of a sparse 12-bin histogram -- every validity rule, the rounded 50 / 80 ms windows, the
thresholds of csrc/fs_acoustics.h against 10^(x/10), the ctypes layouts, and the C++ mirror's smoke program."""
import ctypes as C
import math
import os
import subprocess
from decimal import Decimal, getcontext
from fractions import Fraction

import numpy as np
import pytest

import acoustics_oracle as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def exp_decay(T, K, bin_ms, amp=2 ** 44):
    """E_k = round(amp 10^(-6 k delta / T)) with the remainder of the infinite tail in the overflow bin: the EDC is a line"""
    d = float(np.float32(bin_ms)) * 1e-3
    q = 10.0 ** (-6.0 * d / T)
    E = [round(amp * q ** k) for k in range(K)]
    E[K - 1] = round(amp * q ** (K - 1) / (1.0 - q))
    return E


def test_thresholds_are_the_nearest_doubles():
    getcontext().prec = 60
    for x, v in A.constants().items():
        exact = Fraction(Decimal(10) ** (Decimal(int(x)) / 10))
        assert v == float(exact), x                    # Fraction -> float rounds to nearest
    assert set(A.constants()) == {"0", "-5", "-10", "-25", "-35"}


@pytest.mark.parametrize("T,K,bin_ms", [(0.8, 1000, 1.0), (0.35, 1000, 1.0), (2.0, 4000, 1.0), (1.3, 700, 2.5), (0.63, 300, 5.0)])
def test_exponential_decay_gives_t20_t30_edt_back(T, K, bin_ms):
    E = exp_decay(T, K, bin_ms)
    rec, edc = A.slot(E, bin_ms)
    assert rec["valid"] & (A.EDT | A.T20 | A.T30) == A.EDT | A.T20 | A.T30
    for name in A.FITS:
        assert abs(rec[name]["time_s"] / T - 1.0) < 1e-6, (name, rec[name])
        assert -1.0 - 1e-12 < rec[name]["r"] < -1.0 + 1e-9
    assert bool(rec["valid"] & A.TS) == (E[-1] == 0)  # energy in the overflow bin: no centre time
    assert rec["onset_bin"] == 0 and edc[0] == 0.0
    d = float(np.float32(bin_ms)) * 1e-3
    k = np.arange(K - 1)
    top = -60.0 * k * d / T > -80.0                   # below that the rounded integer energies are no longer a line
    np.testing.assert_allclose(edc[:-1][top], -60.0 * k[top] * d / T, atol=1e-3)
    # T20 starts at the first bin at or below -5 dB and ends at the last one at or above -25 dB
    t = k * d
    assert rec["t20"]["first_bin"] == int(np.flatnonzero(-60 * t / T <= -5.0 + 1e-9)[0])
    assert rec["t20"]["first_bin"] + rec["t20"]["n_points"] - 1 == int(np.flatnonzero(-60 * t / T >= -25.0 - 1e-9)[-1])


def test_edt_of_a_two_slope_curve():
    """R_k falls with T1 = 0.4 s to -15 dB, then with T2 = 2.0 s: EDT (0 .. -10 dB) is T1, T20 and T30 lie between"""
    K, d, T1, T2, A0 = 3000, 1e-3, 0.4, 2.0, 2 ** 50
    knee = 0.4 * 15 / 60
    def level(t):
        return -60 * t / T1 if t <= knee else -15 - 60 * (t - knee) / T2
    R = [round(A0 * 10 ** (level(k * d) / 10)) for k in range(K)]
    E = [R[k] - R[k + 1] for k in range(K - 1)] + [R[K - 1]]
    rec, _ = A.slot(E, 1.0)
    assert rec["valid"] & 7 == 7
    assert abs(rec["edt"]["time_s"] / T1 - 1.0) < 1e-6
    assert T1 < rec["t20"]["time_s"] < rec["t30"]["time_s"] < T2
    assert rec["edt"]["r"] < -0.999999 and rec["t30"]["r"] > rec["edt"]["r"]


def test_sparse_histogram_by_hand():
    """bin_ms = 10: 50 ms = 5 bins, 80 ms = 8 bins.  E = 8, 4, 2, 1, 1 at bins 2, 4, 6, 7, 9 of 12; S0 = 16.
    early50 = bins 2..6 = 14, late50 = 2: C50 = 10 log10 7, D50 = 14/16.  early80 = bins 2..9 = 16: C80 = +inf (valid).
    Ts = 10 ms (0 8 + 2 4 + 4 2 + 5 1 + 7 1) / 16 = 17.5 ms."""
    E = [0] * 12
    for k, v in ((2, 8), (4, 4), (6, 2), (7, 1), (9, 1)):
        E[k] = v
    rec, edc = A.slot(E, 10.0)
    assert rec["onset_bin"] == 2
    assert rec["valid"] & (A.C50 | A.C80 | A.TS) == A.C50 | A.C80 | A.TS
    assert rec["c50_db"] == pytest.approx(10 * math.log10(7), rel=1e-15)
    assert rec["d50"] == 0.875
    assert rec["c80_db"] == math.inf
    assert rec["ts_s"] == pytest.approx(0.0175, rel=1e-15)
    # decay curve: R = 16 16 16 8 8 4 4 2 1 1 0 0
    want = [0, 0, 0, 10 * math.log10(0.5)] * 1 + [10 * math.log10(0.5), 10 * math.log10(0.25), 10 * math.log10(0.25),
                                                  10 * math.log10(0.125), 10 * math.log10(1 / 16), 10 * math.log10(1 / 16),
                                                  -math.inf, -math.inf]
    assert np.array_equal(edc, np.array(want, np.float32))
    # EDT: points 2 .. the last bin with R >= 1.6 (bin 7, R = 2): L = 0, -3.01, -3.01, -6.02, -6.02, -9.03 at t = 0 .. 50 ms
    L = 10 * np.log10(np.array([16, 8, 8, 4, 4, 2]) / 16)
    t = np.arange(6) * 0.01
    slope = np.polyfit(t, L, 1)[0]
    assert rec["edt"]["first_bin"] == 2 and rec["edt"]["n_points"] == 6
    assert rec["edt"]["time_s"] == pytest.approx(-60 / slope, rel=1e-12)
    assert rec["edt"]["r"] == pytest.approx(np.corrcoef(t, L)[0, 1], rel=1e-12)


def test_range_not_reached_before_the_overflow_bin():
    """a decay that ends at -20 dB with the rest in the overflow bin: EDT valid, T20 / T30 not"""
    E = exp_decay(0.5, 200, 1.0)
    K = len(E)
    R = sum(E)
    cut = next(k for k in range(K) if sum(E[k:]) <= R * 10 ** -2.0)     # -20 dB
    E2 = E[:cut] + [0] * (K - 1 - cut) + [sum(E[cut:])]
    rec, _ = A.slot(E2, 1.0)
    assert rec["valid"] & 7 == A.EDT
    assert math.isnan(rec["t20"]["time_s"]) and math.isnan(rec["t30"]["r"])
    assert rec["t30"]["n_points"] > 3                  # points are reported even though the fit is not valid


def test_fewer_than_three_points():
    E = [10 ** 6, 10 ** 4, 100, 1] + [0] * 8
    rec, _ = A.slot(E, 1.0)
    assert rec["valid"] & 7 == 0
    assert rec["edt"]["n_points"] == 1 and rec["t20"]["n_points"] == 1 and rec["t20"]["first_bin"] == 1


def test_energy_only_in_the_overflow_bin():
    K = 50
    rec, edc = A.slot([0] * (K - 1) + [12345], 1.0)
    assert rec["onset_bin"] == K - 1 and rec["valid"] == 0
    assert all(rec[n]["n_points"] == 0 for n in A.FITS)
    assert all(math.isnan(rec[k]) for k in ("c50_db", "c80_db", "d50", "ts_s"))
    assert np.all(edc == 0.0)


def test_energy_only_in_the_onset_bin_is_free_field():
    E = [0] * 200
    E[17] = 2 ** 63 + 5
    rec, edc = A.slot(E, 1.0)
    assert rec["onset_bin"] == 17
    assert rec["valid"] == A.C50 | A.C80 | A.TS
    assert rec["c50_db"] == math.inf and rec["c80_db"] == math.inf and rec["d50"] == 1.0 and rec["ts_s"] == 0.0
    assert rec["edt"]["first_bin"] == 17 and rec["t20"]["first_bin"] == 18 and rec["t20"]["n_points"] == 0
    assert edc[17] == 0.0 and np.all(np.isneginf(edc[18:]))


def test_band_without_energy_and_broadband_past_2_to_64():
    B, K = 8, 64
    h = np.zeros((2, B, K), np.uint64)
    h[0, :, 3] = np.uint64(2 ** 64 - 1)                 # every band near 2^64 in one bin: the broadband sum needs 67 bits
    h[0, :, 9] = np.uint64(2 ** 60)
    h[0, 5] = 0                                       # band 5 is silent
    out, edc = A.acoustic_params(h, 1.0)
    bb = out[0]["broadband"]
    assert out[0]["no_energy"] == 0 and bb["onset_bin"] == 3
    s0 = 7 * (2 ** 64 - 1) + 7 * 2 ** 60
    assert bb["d50"] == A.to_double(s0) / A.to_double(s0)
    assert bb["ts_s"] == pytest.approx(1e-3 * (6 * 7 * 2 ** 60) / s0, rel=1e-15)
    assert out[0]["band"][5]["onset_bin"] == A.NO_ONSET and out[0]["band"][5]["valid"] == 0
    assert np.all(np.isnan(edc[0, 5]))
    assert out[1]["no_energy"] == 1 and all(b["valid"] == 0 for b in out[1]["band"])
    assert np.all(np.isnan(edc[1]))


@pytest.mark.parametrize("bin_ms,n50,n80", [(1.0, 50, 80), (2.5, 20, 32), (3.0, 17, 27), (0.7, 71, 114), (7.0, 7, 11),
                                            (60.0, 1, 1), (120.0, 0, 1), (170.0, 0, 0)])
def test_window_lengths_round_to_the_nearest_bin(bin_ms, n50, n80):
    assert (A.window(50.0, bin_ms), A.window(80.0, bin_ms)) == (n50, n80)
    E = [0, 0, 5] + [1] * 200 + [0]
    rec, _ = A.slot(E, bin_ms)
    for nw, key, bit in ((n50, "c50_db", A.C50), (n80, "c80_db", A.C80)):
        if nw == 0:
            assert not rec["valid"] & bit and math.isnan(rec[key])
        else:
            early = 5 + (nw - 1)
            assert rec["valid"] & bit
            assert rec[key] == pytest.approx(10 * math.log10(early / (205 - early)), rel=1e-14)


def test_early_window_must_end_before_the_overflow_bin():
    # k0 = 2, n50 = 5: valid iff k0 + 5 <= K - 1
    for K, ok in ((8, True), (7, False)):
        E = [0, 0] + [1] * (K - 2)
        E[K - 1] = 0
        rec, _ = A.slot(E, 10.0)
        assert bool(rec["valid"] & A.C50) == ok, K


def test_struct_layouts(fs):
    f, s, p = fs.capi.DecayFit, fs.capi.AcousticSlot, fs.capi.AcousticParams
    assert (C.sizeof(f), C.sizeof(s), C.sizeof(p)) == (24, 112, 1016)
    assert (f.time_s.offset, f.r.offset, f.first_bin.offset, f.n_points.offset) == (0, 8, 16, 20)
    assert (s.edt.offset, s.t20.offset, s.t30.offset, s.c50_db.offset, s.c80_db.offset, s.d50.offset, s.ts_s.offset,
            s.onset_bin.offset, s.valid.offset) == (0, 24, 48, 72, 80, 88, 96, 104, 108)
    assert (p.no_energy.offset, p.reserved.offset, p.broadband.offset, p.band.offset) == (0, 4, 8, 120)
    assert (fs.capi.AP_EDT, fs.capi.AP_T20, fs.capi.AP_T30, fs.capi.AP_C50, fs.capi.AP_C80, fs.capi.AP_TS) == \
           (A.EDT, A.T20, A.T30, A.C50, A.C80, A.TS)


def build_acoustics_smoke(out_dir):
    exe = os.path.join(str(out_dir), "acoustics_smoke")
    libdir = os.path.join(ROOT, "audio-pathtracer_b200", "lib")
    env = dict(os.environ); env.pop("CC", None); env.pop("CXX", None)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "acoustics_smoke.cpp"), "-o", exe,
                           "-L", libdir, "-lfrequensee", "-Wl,-rpath," + libdir], env=env)
    return exe


def test_acoustics_smoke_compiles_and_fails_loudly_without_gpu(fs, tmp_path):
    """the mirror's LastAcoustics / UpdateAcousticParams build from plain C++"""
    import torch
    exe = build_acoustics_smoke(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([exe, "nogpu"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CPU fallback" in r.stdout
