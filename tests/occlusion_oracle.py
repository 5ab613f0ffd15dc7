"""CPU reference of direct-path occlusion: fso_occlusion (tests/oracle_ext/fso_occlusion.c, the per-ray arithmetic of
audio-pathtracer_b200/csrc/fs_occlusion.h over the oracle's brute-force or BVH hit search), compiled together with the oracle
into a temporary directory on first use, with the oracle's own compiler flags."""
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
        out = os.path.join(tempfile.mkdtemp(prefix="fso_occlusion_"), "libfso_occlusion.so")
        cmd = ["gcc", "-O2", "-std=gnu99", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-fPIC", "-w", "-shared",
               "-o", out, os.path.join(HERE, "oracle_ext", "fso_occlusion.c"), "-lm"]
        if pyoracle._has_fma():
            cmd.insert(1, "-mfma")
        subprocess.check_call(cmd)
        L = C.CDLL(out)
        L.fso_scene_create.restype = C.c_void_p
        L.fso_scene_create.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int]
        L.fso_scene_destroy.argtypes = [C.c_void_p]
        L.fso_scene_set_material_model.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.fso_occlusion_tau.argtypes = [C.c_void_p, C.c_void_p]
        L.fso_occlusion.restype = C.c_int
        L.fso_occlusion.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32,
                                    C.c_uint64, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
        L.fso_powf.restype = C.c_float
        L.fso_powf.argtypes = [C.c_float, C.c_float]
        _lib = L
    return _lib


class Scene:
    """an fso_scene of this library; use_bvh=False: brute force over all triangles"""

    def __init__(self, verts, tri_mat, absorption, use_bvh=True):
        self.verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3, 3)
        self.tri_mat = np.ascontiguousarray(tri_mat, dtype=np.uint32)
        self.absorption = np.ascontiguousarray(absorption, dtype=np.float32)
        self.n_mats, self.n_bands = self.absorption.shape
        self.h = lib().fso_scene_create(self.verts.ctypes.data, self.tri_mat.ctypes.data, len(self.verts),
                                        self.absorption.ctypes.data, self.n_mats, self.n_bands, int(use_bvh))
        assert self.h

    def set_material_model(self, transmission=None, scattering=None, thickness_cm=None):
        """transmission [M][B], scattering [M][B], thickness_cm [M] (None: the defaults 0, 1, 2.5 cm)"""
        self._mm = [None if a is None else np.ascontiguousarray(a, np.float32) for a in (transmission, scattering, thickness_cm)]
        lib().fso_scene_set_material_model(self.h, *[None if a is None else a.ctypes.data for a in self._mm])

    def tau(self):
        out = np.zeros((self.n_mats, self.n_bands), np.float32)
        lib().fso_occlusion_tau(self.h, out.ctypes.data)
        return out

    def close(self):
        if self.h:
            lib().fso_scene_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def occlusion(self, src_pos, radius, n_rays, lis_pos, max_crossings=4, seed=0, eps_connect=1e-3, eps_offset=1e-3):
        """(visible [S] float32, transmission [S][B] float32, rays used [S]) as fs_occlusion returns them"""
        src = np.ascontiguousarray(src_pos, dtype=np.float32).reshape(-1, 3)
        S = len(src)
        r = np.ascontiguousarray(np.broadcast_to(np.asarray(radius, np.float32), (S,)))
        n = np.ascontiguousarray(np.broadcast_to(np.asarray(n_rays, np.uint64), (S,)).astype(np.uint32))
        lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
        vis = np.zeros(S, np.float32)
        tr = np.zeros((S, 8), np.float32)
        used = np.zeros(S, np.uint32)
        rc = lib().fso_occlusion(self.h, src.ctypes.data, r.ctypes.data, n.ctypes.data, S, lis.ctypes.data, max_crossings,
                                 seed, eps_connect, eps_offset, vis.ctypes.data, tr.ctypes.data, used.ctypes.data)
        if rc != 0:
            raise ValueError("fso_occlusion rejected the arguments")
        return vis, tr[:, :self.n_bands], used
