"""CPU reference of directional sources: fso_trace_sources_dir (tests/oracle_ext/fso_directivity.c, the pair loop of
fso_trace_sources with every path weighted by its source pattern's gain at the emission direction), compiled together with
the oracle into a temporary directory on first use, with the oracle's own compiler flags."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import pyoracle
import sources_oracle

HERE = os.path.dirname(os.path.abspath(__file__))
OMNI = 0xFFFFFFFF
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="fso_directivity_"), "libfso_directivity.so")
        cmd = ["gcc", "-O2", "-std=gnu99", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-fPIC", "-w", "-shared",
               "-o", out, os.path.join(HERE, "oracle_ext", "fso_directivity.c"), "-lm"]
        if pyoracle._has_fma():
            cmd.insert(1, "-mfma")
        subprocess.check_call(cmd)
        L = C.CDLL(out)
        L.fso_scene_create.restype = C.c_void_p
        L.fso_scene_create.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int]
        L.fso_scene_destroy.argtypes = [C.c_void_p]
        L.fso_scene_set_material_model.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.fso_trace_sources_dir.restype = C.c_int
        L.fso_trace_sources_dir.argtypes = [C.c_void_p, C.POINTER(pyoracle.Config), C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(pyoracle.Stats)]
        _lib = L
    return _lib


class Scene(sources_oracle.Scene):
    """an fso_scene of this library (the handle of sources_oracle.Scene belongs to another compiled copy of the oracle)"""

    def __init__(self, verts, tri_mat, absorption, use_bvh=True):
        self.verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3, 3)
        self.tri_mat = np.ascontiguousarray(tri_mat, dtype=np.uint32)
        self.absorption = np.ascontiguousarray(absorption, dtype=np.float32)
        n_mats, n_bands = self.absorption.shape
        self.h = lib().fso_scene_create(self.verts.ctypes.data, self.tri_mat.ctypes.data, len(self.verts),
                                        self.absorption.ctypes.data, n_mats, n_bands, int(use_bvh))
        assert self.h

    def set_material_model(self, transmission, scattering, thickness_cm):
        self._mm = [np.ascontiguousarray(a, np.float32) for a in (transmission, scattering, thickness_cm)]
        lib().fso_scene_set_material_model(self.h, *[a.ctypes.data for a in self._mm])

    def close(self):
        if self.h:
            lib().fso_scene_destroy(self.h)
            self.h = None

    def trace_sources_dir(self, cfg, src_pos, n_paths, depths, lis_pos, seed, gains, forward, pattern, want_dbg=False):
        """gains [P][B][33] (B <= 8), forward [S][3], pattern [S] (OMNI = omni).  Returns (hist [S][B][K], stats) or, with
        want_dbg (endpoint mode only), (hist, stats, dbg [G] records like pyoracle's)"""
        src = np.ascontiguousarray(src_pos, dtype=np.float32).reshape(-1, 3)
        S = len(src)
        n = np.ascontiguousarray(np.broadcast_to(np.asarray(n_paths, np.uint64), (S,)))
        d = np.ascontiguousarray(np.broadcast_to(np.asarray(depths, np.uint32), (S,)))
        lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
        g = np.asarray(gains, np.float32)
        if g.ndim == 2:
            g = g[None]
        full = np.zeros((max(len(g), 1), 8, 33), np.float32)
        full[:len(g), :g.shape[1]] = g
        f = np.ascontiguousarray(np.asarray(forward, np.float32).reshape(S, 3))
        pat = np.ascontiguousarray(np.broadcast_to(np.asarray(pattern, np.uint64), (S,)).astype(np.uint32))
        hist = np.zeros((S, cfg.n_bands, cfg.n_bins), dtype=np.uint64)
        dbg = np.zeros(int(n.sum()), dtype=pyoracle.PATH_DBG_DTYPE) if want_dbg else None
        st = pyoracle.Stats()
        rc = lib().fso_trace_sources_dir(self.h, C.byref(cfg), src.ctypes.data, n.ctypes.data, d.ctypes.data, S,
                                         lis.ctypes.data, seed, full.ctypes.data, len(g), f.ctypes.data, pat.ctypes.data,
                                         hist.ctypes.data, dbg.ctypes.data if want_dbg else None, C.byref(st))
        if rc != 0:
            raise RuntimeError("fso_trace_sources_dir failed: %d" % rc)
        return (hist, st.as_dict(), dbg) if want_dbg else (hist, st.as_dict())
