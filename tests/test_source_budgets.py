"""Per-source path budgets and depths (fs_trace_sources), host side: the CPU reference of the per-source form agrees with
the oracle's fso_trace in the uniform case and, source by source, with an fso_trace range; the C struct layout; the C++
mirror's UpdateSources() compiles and fails loudly without a GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import sources_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
POS5 = np.array([[1.0, 1.0, 1.0], [6.0, 4.0, 2.0], [3.5, 2.5, 1.5], [0.5, 4.5, 2.5], [5.0, 1.0, 0.5]], np.float32)
N5 = [1, 700, 4096, 33, 2000]
D5 = [0, 1, 8, 3, 16]


def _shoebox(oracle, model=False):
    from frequensee import scenes
    sc = scenes.shoebox()
    S = oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=True)
    R = sources_oracle.Scene(sc.verts, sc.tri_mat, sc.absorption, use_bvh=True)
    if model:
        rng = np.random.default_rng(3)
        M, B = sc.absorption.shape
        mm = (rng.uniform(0, 0.5, (M, B)).astype(np.float32), rng.uniform(0, 1, (M, B)).astype(np.float32),
              rng.uniform(0.5, 10, M).astype(np.float32))
        S.set_material_model(*mm)
        R.set_material_model(*mm)
    return sc, S, R


@pytest.mark.parametrize("flags", [0, 128, 64])        # default, FS_FLAG_SHARE_LISTENER, FS_FLAG_CONNECT_ALL
def test_uniform_budgets_equal_fso_trace(oracle, flags):
    sc, S, R = _shoebox(oracle)
    cfg = oracle.default_config(flags=flags)
    pos = POS5[:3]
    h0, s0 = S.trace(cfg, pos, sc.listener, 900, 6, 0x5EED)
    h1, s1 = R.trace_sources(cfg, pos, 900, 6, sc.listener, 0x5EED)
    assert np.array_equal(h0, h1)
    assert s0["paths"] == s1["paths"] == 2700 and s0["connected"] == s1["connected"] and s0["ext_rays"] == s1["ext_rays"]


@pytest.mark.parametrize("mode", ["default", "connect_all", "material_model"])
def test_each_source_equals_its_fso_trace_range(oracle, mode):
    """identity 2: outside FS_FLAG_SHARE_LISTENER the histogram of source s is fso_trace(pos_s, 1 source,
    n_paths = o_s + n_s, g in [o_s, o_s + n_s), depth_s)"""
    sc, S, R = _shoebox(oracle, model=(mode == "material_model"))
    flags = {"default": 0, "connect_all": oracle.FLAG_CONNECT_ALL, "material_model": oracle.FLAG_MATERIAL_MODEL}[mode]
    cfg = oracle.default_config(flags=flags)
    h, st = R.trace_sources(cfg, POS5, N5, D5, sc.listener, 77)
    assert st["paths"] == sum(N5)
    o = 0
    for s in range(5):
        hs, _ = S.trace(cfg, POS5[s:s + 1], sc.listener, o + N5[s], D5[s], 77, g_first=o, g_count=N5[s])
        assert np.array_equal(h[s], hs[0]), "source %d" % s
        o += N5[s]
    assert h[2].any() and h[4].any()
    # depth 0: the direct-path pair only -- every pair of source 0 lands in one bin per band
    assert (h[0] != 0).sum(axis=1).max() <= 1


def test_shared_listener_keys_by_the_path_index(oracle):
    """with FS_FLAG_SHARE_LISTENER and equal depths, a source's histogram does not depend on where its range starts:
    the listener walk of pair i is keyed by i = g - o_s, the source walk by g"""
    sc, S, R = _shoebox(oracle)
    cfg = oracle.default_config(flags=oracle.FLAG_SHARE_LISTENER)
    pos = POS5[:3]
    h, _ = R.trace_sources(cfg, pos, [300, 500, 200], 5, sc.listener, 9)
    # source 1 alone, its range shifted to start at 0, differs in its source walks ...
    h1, _ = R.trace_sources(cfg, pos[1:2], 500, 5, sc.listener, 9)
    # ... but source 0 (o_0 = 0) is the uniform single-source trace of fso_trace
    h0, _ = S.trace(cfg, pos[0:1], sc.listener, 300, 5, 9)
    assert np.array_equal(h[0], h0[0])
    assert not np.array_equal(h[1], h1[0])


def test_source_desc_layout(fs):
    from frequensee import capi
    D = capi.SourceDesc
    assert C.sizeof(D) == 24
    assert (D.pos.offset, D.max_depth.offset, D.n_paths.offset) == (0, 12, 16)
    src = ('#include <stddef.h>\n#include "frequensee.h"\n'
           '_Static_assert(sizeof(fs_source_desc) == 24, "size");\n'
           '_Static_assert(offsetof(fs_source_desc, max_depth) == 12, "max_depth");\n'
           '_Static_assert(offsetof(fs_source_desc, n_paths) == 16, "n_paths");\n')
    subprocess.run(["gcc", "-std=c11", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), "-x", "c", "-"],
                   input=src, text=True, check=True)


def build_sources_smoke(out_dir):
    exe = os.path.join(str(out_dir), "sources_smoke")
    libdir = os.path.join(ROOT, "audio-pathtracer_b200", "lib")
    env = dict(os.environ); env.pop("CC", None); env.pop("CXX", None)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "sources_smoke.cpp"), "-o", exe,
                           "-L", libdir, "-lfrequensee", "-Wl,-rpath," + libdir], env=env)
    return exe


def test_sources_smoke_compiles_and_fails_loudly_without_gpu(fs, tmp_path):
    import torch
    exe = build_sources_smoke(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([exe, "nogpu"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CPU fallback" in r.stdout
