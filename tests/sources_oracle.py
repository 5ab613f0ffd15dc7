"""CPU reference of per-source path budgets and depths (fso_trace_sources in tests/oracle_ext/fso_sources.c), compiled
together with the oracle into a temporary directory on first use, with the oracle's own compiler flags."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import pyoracle

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="fso_sources_"), "libfso_sources.so")
        cmd = ["gcc", "-O2", "-std=gnu99", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-fPIC", "-w", "-shared",
               "-o", out, os.path.join(HERE, "oracle_ext", "fso_sources.c"), "-lm"]
        if pyoracle._has_fma():
            cmd.insert(1, "-mfma")
        subprocess.check_call(cmd)
        L = C.CDLL(out)
        L.fso_scene_create.restype = C.c_void_p
        L.fso_scene_create.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int]
        L.fso_scene_destroy.argtypes = [C.c_void_p]
        L.fso_scene_set_material_model.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.fso_trace_sources.restype = C.c_int
        L.fso_trace_sources.argtypes = [C.c_void_p, C.POINTER(pyoracle.Config), C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_uint32, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p,
                                        C.POINTER(pyoracle.Stats)]
        _lib = L
    return _lib


class Scene:
    def __init__(self, verts, tri_mat, absorption, use_bvh=True):
        self.verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3, 3)
        self.tri_mat = np.ascontiguousarray(tri_mat, dtype=np.uint32)
        self.absorption = np.ascontiguousarray(absorption, dtype=np.float32)
        n_mats, n_bands = self.absorption.shape
        self.h = lib().fso_scene_create(self.verts.ctypes.data, self.tri_mat.ctypes.data, len(self.verts),
                                        self.absorption.ctypes.data, n_mats, n_bands, int(use_bvh))
        assert self.h

    def set_material_model(self, transmission, scattering, thickness_cm):
        """transmission [M][B], scattering [M][B], thickness_cm [M], as pyoracle.Scene.set_material_model"""
        self._mm = [np.ascontiguousarray(a, np.float32) for a in (transmission, scattering, thickness_cm)]
        lib().fso_scene_set_material_model(self.h, *[a.ctypes.data for a in self._mm])

    def trace_sources(self, cfg, src_pos, n_paths, depths, lis_pos, seed, g_first=0, g_count=None):
        src = np.ascontiguousarray(src_pos, dtype=np.float32).reshape(-1, 3)
        S = len(src)
        n = np.ascontiguousarray(np.broadcast_to(np.asarray(n_paths, np.uint64), (S,)))
        d = np.ascontiguousarray(np.broadcast_to(np.asarray(depths, np.uint32), (S,)))
        lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
        if g_count is None:
            g_count = int(n.sum()) - g_first
        hist = np.zeros((S, cfg.n_bands, cfg.n_bins), dtype=np.uint64)
        st = pyoracle.Stats()
        rc = lib().fso_trace_sources(self.h, C.byref(cfg), src.ctypes.data, n.ctypes.data, d.ctypes.data, S,
                                     lis.ctypes.data, g_first, g_count, seed, hist.ctypes.data, C.byref(st))
        if rc != 0:
            raise RuntimeError("fso_trace_sources failed: %d" % rc)
        return hist, st.as_dict()

    def close(self):
        if self.h:
            lib().fso_scene_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
