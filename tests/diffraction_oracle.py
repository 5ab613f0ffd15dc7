"""CPU reference of first-order edge diffraction: fso_diffraction (tests/oracle_ext/fso_diffraction.c, the per-edge arithmetic
of audio-pathtracer_b200/csrc/fs_diffraction.h with its own edge grouping and the oracle's any-hit rays), compiled together
with the oracle into a temporary directory on first use, with the oracle's own compiler flags."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import pyoracle

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None

# fso_diff_result == fs_diffraction_result (68 bytes)
DTYPE = np.dtype([
    ("found", np.uint32), ("n_paths", np.uint32), ("edge_tri", np.uint32), ("edge_k", np.uint32),
    ("apex", np.float32, (3,)), ("length", np.float32), ("path_difference", np.float32), ("gain", np.float32, (8,))])


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="fso_diffraction_"), "libfso_diffraction.so")
        cmd = ["gcc", "-O2", "-std=gnu99", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-fPIC", "-w", "-shared",
               "-o", out, os.path.join(HERE, "oracle_ext", "fso_diffraction.c"), "-lm"]
        if pyoracle._has_fma():
            cmd.insert(1, "-mfma")
        subprocess.check_call(cmd)
        L = C.CDLL(out)
        L.fso_scene_create.restype = C.c_void_p
        L.fso_scene_create.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int]
        L.fso_scene_destroy.argtypes = [C.c_void_p]
        L.fso_diffraction_edges.restype = C.c_uint64
        L.fso_diffraction_edges.argtypes = [C.c_void_p, C.c_uint64, C.c_float, C.c_void_p, C.c_uint64]
        L.fso_diffraction.restype = None
        L.fso_diffraction.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p,
                                      C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
        L.fso_diffraction_gain.restype = C.c_float
        L.fso_diffraction_gain.argtypes = [C.c_float, C.c_float, C.c_float]
        _lib = L
    return _lib


def edges(verts, min_fold_deg):
    """the edge set as (tri, k) pairs [n][2], ascending"""
    v = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3, 3)
    n = lib().fso_diffraction_edges(v.ctypes.data, len(v), min_fold_deg, None, 0)
    out = np.zeros((n, 2), np.uint32)
    lib().fso_diffraction_edges(v.ctypes.data, len(v), min_fold_deg, out.ctypes.data, n)
    return out


class Scene:
    """triangles with one material each; use_bvh=False: every leg ray by brute force over all triangles"""

    def __init__(self, verts, tri_mat=None, absorption=None, use_bvh=True):
        self.verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3, 3)
        self.tri_mat = np.ascontiguousarray(np.zeros(len(self.verts), np.uint32) if tri_mat is None else tri_mat, np.uint32)
        self.absorption = np.ascontiguousarray(np.full((1, 8), 0.5, np.float32) if absorption is None else absorption, np.float32)
        self.n_mats, self.n_bands = self.absorption.shape
        self.h = lib().fso_scene_create(self.verts.ctypes.data, self.tri_mat.ctypes.data, len(self.verts),
                                        self.absorption.ctypes.data, self.n_mats, self.n_bands, int(use_bvh))
        assert self.h

    def close(self):
        if self.h:
            lib().fso_scene_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def edges(self, min_fold_deg):
        return edges(self.verts, min_fold_deg)

    def diffraction(self, src_pos, lis_pos, min_fold_deg=30.0, band_hz=None, eps_offset=1e-3, eps_connect=1e-3,
                    sound_speed=343.0, n_bands=None, stats=False):
        """DTYPE array [S] as fs_diffraction returns it (and, with stats, (edges, candidates, leg rays traced))"""
        B = self.n_bands if n_bands is None else n_bands
        src = np.ascontiguousarray(src_pos, dtype=np.float32).reshape(-1, 3)
        lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
        hz = None if band_hz is None else np.ascontiguousarray(band_hz, np.float32).reshape(B)
        out = np.zeros(len(src), DTYPE)
        st = np.zeros(3, np.uint64)
        lib().fso_diffraction(self.h, self.verts.ctypes.data, min_fold_deg, src.ctypes.data, len(src), lis.ctypes.data,
                              None if hz is None else hz.ctypes.data, B, eps_offset, eps_connect, sound_speed,
                              out.ctypes.data, st.ctypes.data)
        return (out, tuple(int(x) for x in st)) if stats else out
