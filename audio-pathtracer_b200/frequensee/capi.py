"""ctypes binding of the C-ABI in include/frequensee.h (libfrequensee.so, CUDA sm_100a).

This is the only way Python reaches the product: there is no CPU fallback.  Loading fails loudly
if the shared library is missing (run `python -c "import __graft_entry__ as g; g.build()"` or
`make -C audio-pathtracer_b200/csrc`), and fs_create fails loudly if no B200-class GPU is usable.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FS_LIB_PATH") or os.path.join(os.path.dirname(HERE), "lib", "libfrequensee.so")   # FS_LIB_PATH: A/B builds (tools/)
MAX_BANDS = 8

FS_OK = 0
FS_ERR_INVALID, FS_ERR_CUDA, FS_ERR_NOMEM, FS_ERR_STATE, FS_ERR_OVERFLOW = -1, -2, -3, -4, -5
FLAG_COUNT_VISITS, FLAG_NO_SPLAT_AGG, FLAG_SMEM_TREELET, FLAG_BRUTE_FORCE, FLAG_TIME_KERNELS, FLAG_FUSED_EXTEND = 1, 2, 4, 8, 16, 32
FLAG_CONNECT_ALL = 64
FLAG_SHARE_LISTENER = 128
FLAG_MATERIAL_MODEL = 256
FLAG_MIS = 512
FLAG_IR_NORMALIZE = 1024
FLAG_CONV_CROSSFADE = 2048
FLAG_NOISE_STATS = 4096
DIR_POINTS = 33          # FS_DIR_POINTS: directivity tables are sampled at cos = -1 + i/16
OMNI = 0xFFFFFFFF        # FS_OMNI: a source without a pattern

# every symbol include/frequensee.h declares (tests/test_abi.py checks the library exports them all)
ABI_SYMBOLS = [
    "fs_default_config", "fs_create", "fs_destroy", "fs_last_error", "fs_set_stream", "fs_synchronize",
    "fs_scene_set_triangles", "fs_scene_set_materials", "fs_scene_set_materials_ex", "fs_scene_commit",
    "fs_scene_update_vertices", "fs_scene_refit",
    "fs_trace", "fs_update", "fs_trace_range_device", "fs_trace_range", "fs_trace_debug",
    "fs_trace_sources", "fs_update_sources", "fs_trace_sources_range_device", "fs_set_histogram_sources_device",
    "fs_get_noise", "fs_get_histogram_m2", "fs_allocate_paths",
    "fs_debug_closest_hits", "fs_debug_any_hits",
    "fs_build_ir", "fs_build_ir_to", "fs_build_ir_all", "fs_build_ir_bands", "fs_build_ir_from_energy", "fs_set_histogram", "fs_set_histogram_device",
    "fs_get_histogram", "fs_get_histogram_sources", "fs_set_ir", "fs_load_float_array", "fs_save_float_array",
    "fs_host_alloc", "fs_host_free",
    "fs_conv_init_source", "fs_conv_release_source", "fs_conv_process", "fs_conv_process_many", "fs_conv_process_multi",
    "fs_debug_rfft", "fs_get_stats",
    "fs_multi_create", "fs_multi_destroy", "fs_multi_last_error", "fs_multi_device_count", "fs_multi_context",
    "fs_multi_scene_set_triangles", "fs_multi_scene_set_materials", "fs_multi_scene_set_materials_ex", "fs_multi_scene_commit",
    "fs_multi_scene_update_vertices", "fs_multi_scene_refit",
    "fs_multi_trace", "fs_multi_trace_sources", "fs_multi_last_ms", "fs_multi_synchronize",
    "fs_set_directivity_patterns", "fs_set_source_directivity", "fs_directivity_polar",
    "fs_multi_set_directivity_patterns", "fs_multi_set_source_directivity",
    "fs_occlusion",
    "fs_get_acoustic_params",
    "fs_diffraction", "fs_debug_diffraction_edges",
]


class _Pinned:
    """owner of one fs_host_alloc() block; numpy views keep it alive through their .base chain"""

    def __init__(self, nbytes):
        self.p = C.c_void_p()
        rc = load().fs_host_alloc(nbytes, C.byref(self.p))
        if rc != 0 or not self.p.value:
            raise MemoryError("fs_host_alloc(%d) failed" % nbytes)
        self.buf = (C.c_char * nbytes).from_address(self.p.value)

    def __del__(self):
        try:
            if self.p.value:
                load().fs_host_free(self.p)
                self.p = C.c_void_p()
        except Exception:
            pass


def host_alloc(shape, dtype=np.float32):
    """page-locked numpy array (fs_host_alloc): IR / histogram destinations the copy engine writes directly"""
    dt = np.dtype(dtype)
    n = int(np.prod(shape)) * dt.itemsize
    own = _Pinned(max(n, 1))
    a = np.frombuffer(own.buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)
    return _PinnedArray(a, own)


class _PinnedArray(np.ndarray):
    def __new__(cls, arr, owner):
        obj = arr.view(cls)
        obj._fs_owner = owner
        return obj

    def __array_finalize__(self, obj):
        self._fs_owner = getattr(obj, "_fs_owner", None)


class Config(C.Structure):
    """fs_config"""
    _fields_ = [
        ("n_bands", C.c_uint32), ("n_bins", C.c_uint32), ("bin_ms", C.c_float),
        ("rr_prob", C.c_float), ("eps_offset", C.c_float), ("eps_connect", C.c_float),
        ("min_seg", C.c_float), ("sound_speed", C.c_float), ("pdf_exponent", C.c_float),
        ("energy_clamp", C.c_float), ("energy_gain", C.c_float),
        ("air_absorption", C.c_float * MAX_BANDS),
        ("sample_rate", C.c_uint32), ("n_channels", C.c_uint32),
        ("ir_threshold", C.c_float), ("ir_lowpass", C.c_float),
        ("conv_block", C.c_uint32), ("conv_clamp", C.c_uint32), ("conv_wet", C.c_float),
        ("max_batch_paths", C.c_uint32), ("flags", C.c_uint32), ("device", C.c_int32),
    ]


class Stats(C.Structure):
    """fs_stats"""
    _fields_ = [("paths", C.c_uint64), ("ext_rays", C.c_uint64), ("shadow_rays", C.c_uint64),
                ("connected", C.c_uint64), ("node_visits", C.c_uint64), ("tri_tests", C.c_uint64),
                ("shadow_node_visits", C.c_uint64), ("shadow_tri_tests", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("bvh_nodes", C.c_uint64), ("bvh_max_leaf", C.c_uint64),
                ("last_trace_ms", C.c_float), ("last_ir_ms", C.c_float),
                ("extend_ms", C.c_float), ("connect_ms", C.c_float), ("eval_ms", C.c_float),
                ("extend_launches", C.c_uint32), ("trace_ms", C.c_float), ("persistent_launches", C.c_uint32),
                ("last_conv_ms", C.c_float)]

    def as_dict(self):
        return {k: (float(getattr(self, k)) if t is C.c_float else int(getattr(self, k)))
                for k, t in self._fields_}


PATH_DBG_DTYPE = np.dtype([
    ("n_src_nodes", np.uint32), ("n_lis_nodes", np.uint32), ("connected", np.uint32),
    ("bin", np.int32), ("delay_s", np.float32), ("total_dist", np.float32),
    ("energy", np.float32, (MAX_BANDS,)), ("src_end", np.float32, (3,)), ("lis_end", np.float32, (3,)),
])


class SourceDesc(C.Structure):
    """fs_source_desc: one emitter of a per-source-budget update (RaycastsPerTick / RaycastBounces, COMP.h:35-66)"""
    _fields_ = [("pos", C.c_float * 3), ("max_depth", C.c_uint32), ("n_paths", C.c_uint64)]


def source_descs(src_pos, n_paths, depths):
    """fs_source_desc[S] from positions [S][3], budgets [S] and depths [S]"""
    src = np.ascontiguousarray(src_pos, dtype=np.float32).reshape(-1, 3)
    n = np.broadcast_to(np.asarray(n_paths, dtype=np.uint64), (len(src),))
    d = np.broadcast_to(np.asarray(depths, dtype=np.uint32), (len(src),))
    arr = (SourceDesc * len(src))()
    for s in range(len(src)):
        arr[s].pos[:] = [float(v) for v in src[s]]
        arr[s].max_depth = int(d[s])
        arr[s].n_paths = int(n[s])
    return arr


class SourceOrient(C.Structure):
    """fs_source_orient: forward axis and pattern index (or OMNI) of one directional source"""
    _fields_ = [("forward", C.c_float * 3), ("pattern", C.c_uint32)]


def _patterns(gains):
    """fs_directivity[P] from energy gains [P][B][33] (B <= 8; missing bands are zero and ignored)"""
    g = np.asarray(gains, dtype=np.float32)
    if g.ndim == 2:
        g = g[None]
    if g.ndim != 3 or g.shape[1] > MAX_BANDS or g.shape[2] != DIR_POINTS:
        raise ValueError("gains must be [P][B][%d] with B <= %d" % (DIR_POINTS, MAX_BANDS))
    full = np.zeros((g.shape[0], MAX_BANDS, DIR_POINTS), np.float32)
    full[:, :g.shape[1]] = g
    return full


def _orients(forward, pattern):
    """fs_source_orient[S] from forward axes [S][3] and pattern indices [S] (OMNI for an omni source)"""
    f = np.asarray(forward, dtype=np.float32).reshape(-1, 3)
    pat = np.broadcast_to(np.asarray(pattern, dtype=np.uint64), (len(f),))
    arr = (SourceOrient * max(len(f), 1))()
    for s in range(len(f)):
        arr[s].forward[:] = [float(v) for v in f[s]]
        arr[s].pattern = int(pat[s])
    return arr, len(f)


class NoiseStats(C.Structure):
    """fs_noise_stats: Monte Carlo noise of one source in the last update (FS_FLAG_NOISE_STATS)"""
    _fields_ = [("n_paths", C.c_uint64), ("no_energy", C.c_uint32), ("reserved", C.c_uint32),
                ("signal", C.c_double), ("variance", C.c_double), ("snr_db", C.c_double),
                ("band_signal", C.c_double * MAX_BANDS), ("band_variance", C.c_double * MAX_BANDS),
                ("band_snr_db", C.c_double * MAX_BANDS)]


def noise_stats_array(d):
    """fs_noise_stats[S] from the dict Context.noise_stats() returns (keys n_paths, no_energy, signal, variance, band_signal,
    band_variance; snr values are not read by fs_allocate_paths)"""
    S = len(d["n_paths"])
    arr = (NoiseStats * S)()
    for s in range(S):
        arr[s].n_paths = int(d["n_paths"][s])
        arr[s].no_energy = int(d["no_energy"][s])
        arr[s].signal = float(d["signal"][s])
        arr[s].variance = float(d["variance"][s])
        arr[s].snr_db = float(d["snr_db"][s]) if "snr_db" in d else 0.0
    return arr


class OcclusionSource(C.Structure):
    """fs_occlusion_source: one emitter of a direct-path occlusion query (radius 0 = a point: one ray)"""
    _fields_ = [("pos", C.c_float * 3), ("radius", C.c_float), ("n_rays", C.c_uint32), ("reserved", C.c_uint32)]


class OcclusionResult(C.Structure):
    """fs_occlusion_result: visible fraction and mean per-band transmitted gain of one emitter's sample rays"""
    _fields_ = [("visible", C.c_float), ("transmission", C.c_float * MAX_BANDS), ("n_rays", C.c_uint32),
                ("reserved", C.c_uint32)]


def occlusion_sources(src_pos, radius, n_rays):
    """fs_occlusion_source[S] from centres [S][3], radii [S] and ray counts [S] (scalars broadcast)"""
    src = np.ascontiguousarray(src_pos, dtype=np.float32).reshape(-1, 3)
    r = np.broadcast_to(np.asarray(radius, dtype=np.float32), (len(src),))
    n = np.broadcast_to(np.asarray(n_rays, dtype=np.uint64), (len(src),))
    arr = (OcclusionSource * max(len(src), 1))()
    for s in range(len(src)):
        arr[s].pos[:] = [float(v) for v in src[s]]
        arr[s].radius = float(r[s])
        arr[s].n_rays = int(n[s])
    return arr, len(src)


AP_EDT, AP_T20, AP_T30, AP_C50, AP_C80, AP_TS = 1, 2, 4, 8, 16, 32    # FS_AP_*: valid bits of an AcousticSlot
NO_ONSET = 0xFFFFFFFF


class DecayFit(C.Structure):
    """fs_decay_fit: one least-squares fit of the Schroeder decay curve (time_s = -60 / slope; NaN unless valid)"""
    _fields_ = [("time_s", C.c_double), ("r", C.c_double), ("first_bin", C.c_uint32), ("n_points", C.c_uint32)]


class AcousticSlot(C.Structure):
    """fs_acoustic_slot: EDT / T20 / T30, C50 / C80 / D50 and centre time of one band or the broadband sum"""
    _fields_ = [("edt", DecayFit), ("t20", DecayFit), ("t30", DecayFit), ("c50_db", C.c_double), ("c80_db", C.c_double),
                ("d50", C.c_double), ("ts_s", C.c_double), ("onset_bin", C.c_uint32), ("valid", C.c_uint32)]


class AcousticParams(C.Structure):
    """fs_acoustic_params: the room-acoustic parameters of one source, broadband and per band"""
    _fields_ = [("no_energy", C.c_uint32), ("reserved", C.c_uint32), ("broadband", AcousticSlot),
                ("band", AcousticSlot * MAX_BANDS)]


# fs_diffraction_result (68 bytes): the shortest first-order diffraction path of one source
DIFFRACTION_DTYPE = np.dtype([
    ("found", np.uint32), ("n_paths", np.uint32), ("edge_tri", np.uint32), ("edge_k", np.uint32),
    ("apex", np.float32, (3,)), ("length", np.float32), ("path_difference", np.float32),
    ("gain", np.float32, (MAX_BANDS,))])


class FrequenSeeError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("frequensee error %d: %s" % (code, msg))
        self.code = code


_lib = None


def load():
    """dlopen libfrequensee.so and declare prototypes; raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libfrequensee.so not built at %s -- the product has no CPU fallback; "
                          "run __graft_entry__.build()" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    L.fs_default_config.argtypes = [C.POINTER(Config)]
    L.fs_default_config.restype = None
    L.fs_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.fs_destroy.argtypes = [vp]
    L.fs_destroy.restype = None
    L.fs_last_error.argtypes = [vp]
    L.fs_last_error.restype = C.c_char_p
    L.fs_set_stream.argtypes = [vp, vp]
    L.fs_synchronize.argtypes = [vp]
    L.fs_scene_set_triangles.argtypes = [vp, vp, vp, u64]
    L.fs_scene_set_materials.argtypes = [vp, vp, u32, u32]
    L.fs_scene_set_materials_ex.argtypes = [vp, vp, vp, vp, vp, u32, u32]
    L.fs_scene_commit.argtypes = [vp]
    L.fs_scene_update_vertices.argtypes = [vp, vp, u64, u64]
    L.fs_scene_refit.argtypes = [vp, C.POINTER(C.c_float)]
    L.fs_trace.argtypes = [vp, vp, u32, vp, u64, u32, u64, vp]
    L.fs_update.argtypes = [vp, vp, u32, vp, u64, u32, u64, vp, vp]
    L.fs_trace_range_device.argtypes = [vp, vp, u32, vp, u64, u64, u64, u32, u64, vp, i32]
    L.fs_trace_range.argtypes = [vp, vp, u32, vp, u64, u64, u64, u32, u64, vp]
    L.fs_trace_debug.argtypes = [vp, vp, u32, vp, u64, u64, u64, u32, u64, vp]
    L.fs_trace_sources.argtypes = [vp, vp, u32, vp, u64, vp]
    L.fs_update_sources.argtypes = [vp, vp, u32, vp, u64, vp, vp]
    L.fs_trace_sources_range_device.argtypes = [vp, vp, u32, vp, u64, u64, u64, vp, i32]
    L.fs_set_histogram_sources_device.argtypes = [vp, vp, u32, vp]
    L.fs_get_noise.argtypes = [vp, vp, u32]
    L.fs_get_histogram_m2.argtypes = [vp, vp]
    L.fs_allocate_paths.argtypes = [vp, u32, u64, u64, u64, vp, vp]
    L.fs_debug_closest_hits.argtypes = [vp, vp, u64, vp, vp]
    L.fs_debug_any_hits.argtypes = [vp, vp, vp, u64, vp]
    L.fs_build_ir.argtypes = [vp, u32, vp]
    L.fs_build_ir_to.argtypes = [vp, u32, u32, vp]
    L.fs_build_ir_from_energy.argtypes = [vp, u32, vp, vp]
    L.fs_set_histogram.argtypes = [vp, vp, u32, u64]
    L.fs_set_histogram_device.argtypes = [vp, vp, u32, u64]
    L.fs_get_histogram.argtypes = [vp, vp]
    L.fs_get_histogram_sources.argtypes = [vp, C.POINTER(u32)]
    L.fs_set_ir.argtypes = [vp, u32, vp]
    L.fs_build_ir_bands.argtypes = [vp, u32, u32, u64, vp]
    L.fs_build_ir_all.argtypes = [vp, u32, vp]
    L.fs_load_float_array.argtypes = [C.c_char_p, vp, u64, C.POINTER(u64)]
    L.fs_save_float_array.argtypes = [C.c_char_p, vp, u64]
    L.fs_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.fs_host_free.argtypes = [vp]
    L.fs_host_free.restype = None
    L.fs_conv_init_source.argtypes = [vp, u32]
    L.fs_conv_release_source.argtypes = [vp, u32]
    L.fs_conv_process.argtypes = [vp, u32, vp, vp, u32]
    L.fs_conv_process_many.argtypes = [vp, u32, vp, vp, u32, u32]
    L.fs_conv_process_multi.argtypes = [vp, vp, u32, vp, vp, u32]
    L.fs_debug_rfft.argtypes = [vp, vp, u32, vp]
    L.fs_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.fs_multi_create.argtypes = [C.POINTER(Config), vp, u32, C.POINTER(vp)]
    L.fs_multi_destroy.argtypes = [vp]
    L.fs_multi_destroy.restype = None
    L.fs_multi_last_error.argtypes = []
    L.fs_multi_last_error.restype = C.c_char_p
    L.fs_multi_device_count.argtypes = [vp]
    L.fs_multi_device_count.restype = u32
    L.fs_multi_context.argtypes = [vp, u32]
    L.fs_multi_context.restype = vp
    L.fs_multi_scene_set_triangles.argtypes = [vp, vp, vp, u64]
    L.fs_multi_scene_set_materials.argtypes = [vp, vp, u32, u32]
    L.fs_multi_scene_set_materials_ex.argtypes = [vp, vp, vp, vp, vp, u32, u32]
    L.fs_multi_scene_commit.argtypes = [vp]
    L.fs_multi_scene_update_vertices.argtypes = [vp, vp, u64, u64]
    L.fs_multi_scene_refit.argtypes = [vp, C.POINTER(C.c_float)]
    L.fs_multi_trace.argtypes = [vp, vp, u32, vp, u64, u32, u64, vp]
    L.fs_multi_trace_sources.argtypes = [vp, vp, u32, vp, u64, vp]
    L.fs_multi_last_ms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    L.fs_multi_synchronize.argtypes = [vp]
    L.fs_set_directivity_patterns.argtypes = [vp, vp, u32]
    L.fs_set_source_directivity.argtypes = [vp, vp, u32]
    L.fs_directivity_polar.argtypes = [vp, vp, u32, vp]
    L.fs_multi_set_directivity_patterns.argtypes = [vp, vp, u32]
    L.fs_multi_set_source_directivity.argtypes = [vp, vp, u32]
    L.fs_occlusion.argtypes = [vp, vp, u32, vp, u32, u64, vp]
    L.fs_get_acoustic_params.argtypes = [vp, vp, u32, vp]
    L.fs_diffraction.argtypes = [vp, vp, u32, vp, C.c_float, vp, vp]
    L.fs_debug_diffraction_edges.argtypes = [vp, C.c_float, vp, u64, C.POINTER(C.c_uint64)]
    for n in ABI_SYMBOLS:
        if n not in ("fs_default_config", "fs_destroy", "fs_last_error", "fs_multi_destroy", "fs_multi_last_error",
                     "fs_multi_device_count", "fs_multi_context"):
            getattr(L, n).restype = C.c_int
    _lib = L
    return L


def default_config(**over):
    cfg = Config()
    load().fs_default_config(C.byref(cfg))
    for k, v in over.items():
        if k == "air_absorption":
            for i, a in enumerate(v):
                cfg.air_absorption[i] = a
        else:
            setattr(cfg, k, v)
    return cfg


class Context:
    """Owns one fs_ctx.  Thin: argument marshalling + error codes -> exceptions."""

    def __init__(self, cfg=None, **over):
        self.L = load()
        self.cfg = cfg if cfg is not None else default_config(**over)
        h = C.c_void_p()
        rc = self.L.fs_create(C.byref(self.cfg), C.byref(h))
        if rc != FS_OK:
            raise FrequenSeeError(rc, (self.L.fs_last_error(None) or b"").decode())
        self.h = h
        self.n_sources = 0

    def close(self):
        if getattr(self, "h", None):
            self.L.fs_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc != FS_OK:
            raise FrequenSeeError(rc, (self.L.fs_last_error(self.h) or b"").decode())

    # -- scene --
    def set_scene(self, verts, tri_mat, absorption):
        verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3, 3)
        tri_mat = np.ascontiguousarray(tri_mat, dtype=np.uint32)
        absorption = np.ascontiguousarray(absorption, dtype=np.float32)
        if len(verts) != len(tri_mat):
            raise ValueError("verts / tri_mat length mismatch")
        self._ck(self.L.fs_scene_set_triangles(self.h, verts.ctypes.data, tri_mat.ctypes.data, len(verts)))
        self._ck(self.L.fs_scene_set_materials(self.h, absorption.ctypes.data, absorption.shape[0],
                                                absorption.shape[1]))
        self._ck(self.L.fs_scene_commit(self.h))

    def set_scene_ex(self, verts, tri_mat, absorption, transmission=None, scattering=None, thickness_cm=None):
        """the whole UAcousticMaterial asset (MAT.h:16-34); used by the tracer only with FLAG_MATERIAL_MODEL"""
        verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3, 3)
        tri_mat = np.ascontiguousarray(tri_mat, dtype=np.uint32)
        absorption = np.ascontiguousarray(absorption, dtype=np.float32)
        opt = [None if a is None else np.ascontiguousarray(a, dtype=np.float32) for a in (transmission, scattering, thickness_cm)]
        self._ck(self.L.fs_scene_set_triangles(self.h, verts.ctypes.data, tri_mat.ctypes.data, len(verts)))
        self._ck(self.L.fs_scene_set_materials_ex(self.h, absorption.ctypes.data, *[a.ctypes.data if a is not None else None for a in opt],
                                                   absorption.shape[0], absorption.shape[1]))
        self._ck(self.L.fs_scene_commit(self.h))

    def update_vertices(self, verts, first_tri=0):
        """moves triangles [first_tri, first_tri + len(verts)) of the scene (same count, same materials); on a committed
        scene the move takes effect at refit() (or a full commit)"""
        verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3, 3)
        self._ck(self.L.fs_scene_update_vertices(self.h, verts.ctypes.data, first_tri, len(verts)))

    def refit(self):
        """refits the committed BVH to the moved triangles; returns its surface-area cost over that of the tree as committed"""
        r = C.c_float(1.0)
        self._ck(self.L.fs_scene_refit(self.h, C.byref(r)))
        return r.value

    def set_stream(self, stream_ptr):
        self._ck(self.L.fs_set_stream(self.h, C.c_void_p(stream_ptr)))

    def synchronize(self):
        self._ck(self.L.fs_synchronize(self.h))

    # -- trace --
    @staticmethod
    def _pos(src_pos, lis_pos):
        src = np.ascontiguousarray(src_pos, dtype=np.float32).reshape(-1, 3)
        lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
        return src, lis

    def trace(self, src_pos, lis_pos, n_paths, max_depth, seed, want_hist=True, out=None):
        """`out`: a caller-owned uint64 [S][B][K] array that receives the histogram (page-locked if it came from host_alloc():
        written by the copy engine directly, and no fresh allocation per update)"""
        src, lis = self._pos(src_pos, lis_pos)
        S = len(src)
        self.n_sources = S
        shape = (S, self.cfg.n_bands, self.cfg.n_bins)
        if out is not None:
            if out.shape != shape or out.dtype != np.uint64 or not out.flags.c_contiguous:
                raise ValueError("out must be a C-contiguous uint64 array of shape %r" % (shape,))
            hist = out
        else:
            hist = np.zeros(shape, dtype=np.uint64) if want_hist else None
        self._ck(self.L.fs_trace(self.h, src.ctypes.data, S, lis.ctypes.data, n_paths, max_depth, seed,
                                 hist.ctypes.data if hist is not None else None))
        return hist

    def update(self, src_pos, lis_pos, n_paths, max_depth, seed, hist_out=None, ir_out=None):
        """fs_update: trace + IR rebuild of every source in one call with one synchronisation (UpdateSource, SUB.cpp:128-195).
        hist_out: uint64 [S][B][K] or None; ir_out: float32 [S][C][fs] or None (caller-owned, ideally from host_alloc())"""
        src, lis = self._pos(src_pos, lis_pos)
        S = len(src)
        self.n_sources = S
        for a, shape, dt in ((hist_out, (S, self.cfg.n_bands, self.cfg.n_bins), np.uint64),
                             (ir_out, (S, self.cfg.n_channels, self.cfg.sample_rate), np.float32)):
            if a is not None and (a.shape != shape or a.dtype != dt or not a.flags.c_contiguous):
                raise ValueError("buffer must be C-contiguous %s of shape %r" % (np.dtype(dt).name, shape))
        self._ck(self.L.fs_update(self.h, src.ctypes.data, S, lis.ctypes.data, n_paths, max_depth, seed,
                                  hist_out.ctypes.data if hist_out is not None else None,
                                  ir_out.ctypes.data if ir_out is not None else None))
        return hist_out, ir_out

    def trace_range(self, src_pos, lis_pos, n_paths, g_first, g_count, max_depth, seed, hist=None):
        src, lis = self._pos(src_pos, lis_pos)
        S = len(src)
        self.n_sources = S
        if hist is None:
            hist = np.zeros((S, self.cfg.n_bands, self.cfg.n_bins), dtype=np.uint64)
        self._ck(self.L.fs_trace_range(self.h, src.ctypes.data, S, lis.ctypes.data, n_paths, g_first, g_count,
                                       max_depth, seed, hist.ctypes.data))
        return hist

    def trace_range_device(self, src_pos, lis_pos, n_paths, g_first, g_count, max_depth, seed, d_hist_ptr,
                           zero_first=True):
        src, lis = self._pos(src_pos, lis_pos)
        self.n_sources = len(src)
        self._ck(self.L.fs_trace_range_device(self.h, src.ctypes.data, len(src), lis.ctypes.data, n_paths,
                                              g_first, g_count, max_depth, seed, C.c_void_p(d_hist_ptr),
                                              int(zero_first)))

    # -- per-source budgets (fs_trace_sources*): n_paths[S] pairs and depths[S] per source; scalars broadcast --
    def trace_sources(self, src_pos, n_paths, depths, lis_pos, seed, want_hist=True):
        d = source_descs(src_pos, n_paths, depths)
        lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
        S = len(d)
        self.n_sources = S
        hist = np.zeros((S, self.cfg.n_bands, self.cfg.n_bins), dtype=np.uint64) if want_hist else None
        self._ck(self.L.fs_trace_sources(self.h, C.addressof(d), S, lis.ctypes.data, seed,
                                         hist.ctypes.data if hist is not None else None))
        return hist

    def update_sources(self, src_pos, n_paths, depths, lis_pos, seed, hist_out=None, ir_out=None):
        """fs_update_sources: one trace with per-source budgets + the IR of every source, one synchronisation"""
        d = source_descs(src_pos, n_paths, depths)
        lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
        S = len(d)
        self.n_sources = S
        for a, shape, dt in ((hist_out, (S, self.cfg.n_bands, self.cfg.n_bins), np.uint64),
                             (ir_out, (S, self.cfg.n_channels, self.cfg.sample_rate), np.float32)):
            if a is not None and (a.shape != shape or a.dtype != dt or not a.flags.c_contiguous):
                raise ValueError("buffer must be C-contiguous %s of shape %r" % (np.dtype(dt).name, shape))
        self._ck(self.L.fs_update_sources(self.h, C.addressof(d), S, lis.ctypes.data, seed,
                                          hist_out.ctypes.data if hist_out is not None else None,
                                          ir_out.ctypes.data if ir_out is not None else None))
        return hist_out, ir_out

    def trace_sources_range_device(self, src_pos, n_paths, depths, lis_pos, g_first, g_count, seed, d_hist_ptr,
                                   zero_first=True):
        d = source_descs(src_pos, n_paths, depths)
        lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
        self.n_sources = len(d)
        self._ck(self.L.fs_trace_sources_range_device(self.h, C.addressof(d), len(d), lis.ctypes.data, g_first, g_count,
                                                      seed, C.c_void_p(d_hist_ptr), int(zero_first)))

    def set_histogram_sources_device(self, d_ptr, n_paths):
        n = np.ascontiguousarray(n_paths, dtype=np.uint64)
        self.n_sources = len(n)
        self._ck(self.L.fs_set_histogram_sources_device(self.h, C.c_void_p(d_ptr), len(n), n.ctypes.data))

    def trace_debug(self, src_pos, lis_pos, n_paths, g_first, g_count, max_depth, seed):
        src, lis = self._pos(src_pos, lis_pos)
        dbg = np.zeros(g_count, dtype=PATH_DBG_DTYPE)
        self._ck(self.L.fs_trace_debug(self.h, src.ctypes.data, len(src), lis.ctypes.data, n_paths, g_first,
                                       g_count, max_depth, seed, dbg.ctypes.data))
        return dbg

    def closest_hits(self, rays):
        rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 6)
        t = np.zeros(len(rays), dtype=np.float32)
        tri = np.zeros(len(rays), dtype=np.uint32)
        self._ck(self.L.fs_debug_closest_hits(self.h, rays.ctypes.data, len(rays), t.ctypes.data, tri.ctypes.data))
        return t, tri

    def any_hits(self, rays, tmax):
        rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 6)
        tmax = np.ascontiguousarray(tmax, dtype=np.float32)
        out = np.zeros(len(rays), dtype=np.uint8)
        self._ck(self.L.fs_debug_any_hits(self.h, rays.ctypes.data, tmax.ctypes.data, len(rays), out.ctypes.data))
        return out.astype(bool)

    # -- histogram / IR --
    def set_histogram(self, hist, n_paths):
        hist = np.ascontiguousarray(hist, dtype=np.uint64)
        if hist.ndim == 2:
            hist = hist[None]
        self.n_sources = hist.shape[0]
        self._ck(self.L.fs_set_histogram(self.h, hist.ctypes.data, hist.shape[0], n_paths))

    def set_histogram_device(self, d_ptr, n_sources, n_paths):
        self.n_sources = n_sources
        self._ck(self.L.fs_set_histogram_device(self.h, C.c_void_p(d_ptr), n_sources, n_paths))

    def get_histogram(self):
        n = C.c_uint32(0)
        self._ck(self.L.fs_get_histogram_sources(self.h, C.byref(n)))
        hist = np.zeros((n.value, self.cfg.n_bands, self.cfg.n_bins), dtype=np.uint64)
        self._ck(self.L.fs_get_histogram(self.h, hist.ctypes.data))
        return hist

    # -- directional sources --
    def set_directivity_patterns(self, gains):
        """fs_set_directivity_patterns: energy gains [P][B][33] at cos = -1 + i/16 (B <= 8); replaces the table and clears the
        source orientations"""
        full = _patterns(gains)
        self._ck(self.L.fs_set_directivity_patterns(self.h, full.ctypes.data, len(full)))

    def set_source_directivity(self, forward, pattern):
        """fs_set_source_directivity: forward axes [S][3] and pattern indices [S] (OMNI: omni); S = 0 (forward = []) clears"""
        arr, S = _orients(forward, pattern)
        self._ck(self.L.fs_set_source_directivity(self.h, arr, S))

    def occlusion(self, src_pos, radius, n_rays, lis_pos, max_crossings=4, seed=0):
        """fs_occlusion: direct-path occlusion of every emitter (centres [S][3], radii [S], ray counts [S]; scalars
        broadcast).  Returns (visible [S] float32, transmission [S][B] float32)"""
        arr, S = occlusion_sources(src_pos, radius, n_rays)
        lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
        out = (OcclusionResult * max(S, 1))()
        self._ck(self.L.fs_occlusion(self.h, arr, S, lis.ctypes.data, max_crossings, seed, out))
        B = self.cfg.n_bands
        vis = np.array([out[s].visible for s in range(S)], np.float32)
        tr = np.array([list(out[s].transmission)[:B] for s in range(S)], np.float32).reshape(S, B)
        return vis, tr

    def diffraction(self, src_pos, lis_pos, min_fold_deg=30.0, band_hz=None):
        """fs_diffraction: the shortest first-order diffraction path of every source (positions [S][3]) to the listener
        around the scene's edges whose fold is at least min_fold_deg; band_hz [B] centre frequencies (None: 62.5 2^b Hz).
        Returns a DIFFRACTION_DTYPE array [S]"""
        src = np.ascontiguousarray(src_pos, dtype=np.float32).reshape(-1, 3)
        lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
        hz = None if band_hz is None else np.ascontiguousarray(band_hz, dtype=np.float32).reshape(self.cfg.n_bands)
        out = np.zeros(max(len(src), 1), DIFFRACTION_DTYPE)
        self._ck(self.L.fs_diffraction(self.h, src.ctypes.data, len(src), lis.ctypes.data, float(min_fold_deg),
                                       None if hz is None else hz.ctypes.data, out.ctypes.data))
        return out[:len(src)]

    def debug_diffraction_edges(self, min_fold_deg=30.0):
        """fs_debug_diffraction_edges: the edge set for a fold threshold as (tri, k) pairs [n][2] uint32, ascending"""
        n = C.c_uint64(0)
        self._ck(self.L.fs_debug_diffraction_edges(self.h, float(min_fold_deg), None, 0, C.byref(n)))
        out = np.zeros((n.value, 2), np.uint32)
        if n.value:
            self._ck(self.L.fs_debug_diffraction_edges(self.h, float(min_fold_deg), out.ctypes.data, n.value, C.byref(n)))
        return out

    def noise_stats(self):
        """fs_get_noise: per-source noise of the last update as a dict of numpy arrays -- n_paths [S], no_energy [S] bool,
        signal / variance / snr_db [S] (broadband) and band_signal / band_variance / band_snr_db [S][B]"""
        n = C.c_uint32(0)
        self._ck(self.L.fs_get_histogram_sources(self.h, C.byref(n)))
        S, B = n.value, self.cfg.n_bands
        arr = (NoiseStats * max(S, 1))()
        self._ck(self.L.fs_get_noise(self.h, arr, S))
        return {
            "n_paths": np.array([arr[s].n_paths for s in range(S)], np.uint64),
            "no_energy": np.array([bool(arr[s].no_energy) for s in range(S)]),
            "signal": np.array([arr[s].signal for s in range(S)]),
            "variance": np.array([arr[s].variance for s in range(S)]),
            "snr_db": np.array([arr[s].snr_db for s in range(S)]),
            "band_signal": np.array([list(arr[s].band_signal)[:B] for s in range(S)]).reshape(S, B),
            "band_variance": np.array([list(arr[s].band_variance)[:B] for s in range(S)]).reshape(S, B),
            "band_snr_db": np.array([list(arr[s].band_snr_db)[:B] for s in range(S)]).reshape(S, B),
        }

    def acoustic_params(self, edc=False):
        """fs_get_acoustic_params: the AcousticParams[S] of the current histogram, and with edc=True also the decay curves as
        float32 [S][B+1][K] in dB (slot B is broadband)"""
        n = C.c_uint32(0)
        self._ck(self.L.fs_get_histogram_sources(self.h, C.byref(n)))
        S = n.value
        arr = (AcousticParams * max(S, 1))()
        curves = np.empty((S, self.cfg.n_bands + 1, self.cfg.n_bins), np.float32) if edc else None
        self._ck(self.L.fs_get_acoustic_params(self.h, arr, S, curves.ctypes.data if edc else None))
        return (arr, curves) if edc else arr

    def histogram_m2(self):
        """fs_get_histogram_m2: second moments of the last update, uint64 [S][B+1][K][2] (lo, hi); slot B is broadband"""
        n = C.c_uint32(0)
        self._ck(self.L.fs_get_histogram_sources(self.h, C.byref(n)))
        out = np.zeros((n.value, self.cfg.n_bands + 1, self.cfg.n_bins, 2), dtype=np.uint64)
        self._ck(self.L.fs_get_histogram_m2(self.h, out.ctypes.data))
        return out

    def build_ir(self, source=0, want_ir=True, out=None):
        shape = (self.cfg.n_channels, self.cfg.sample_rate)
        if out is not None:
            if out.shape != shape or out.dtype != np.float32 or not out.flags.c_contiguous:
                raise ValueError("out must be a C-contiguous float32 array of shape %r" % (shape,))
            ir = out
        else:
            ir = np.zeros(shape, dtype=np.float32) if want_ir else None
        self._ck(self.L.fs_build_ir(self.h, source, ir.ctypes.data if ir is not None else None))
        return ir

    def build_ir_to(self, hist_source, conv_source, want_ir=True):
        ir = np.zeros((self.cfg.n_channels, self.cfg.sample_rate), dtype=np.float32) if want_ir else None
        self._ck(self.L.fs_build_ir_to(self.h, hist_source, conv_source, ir.ctypes.data if want_ir else None))
        return ir

    def build_ir_all(self, n_sources, want_ir=True, out=None):
        """all sources of a multi-emitter update, IR kernels launched once per 64 sources.  `out`: a caller-owned float32
        [n_sources][C][fs] array (page-locked if it came from host_alloc(): written by the copy engine directly)"""
        shape = (n_sources, self.cfg.n_channels, self.cfg.sample_rate)
        if out is None:
            out = np.zeros(shape, dtype=np.float32) if want_ir else None
        elif out.shape != shape or out.dtype != np.float32 or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous float32 array of shape %r" % (shape,))
        self._ck(self.L.fs_build_ir_all(self.h, n_sources, out.ctypes.data if out is not None else None))
        return out

    def build_ir_bands(self, noise_seed, hist_source=0, conv_source=0, want_ir=True):
        """per-band synthesis: band envelopes x octave-band noise carriers (SURVEY 8f rank 2)"""
        out = np.zeros((self.cfg.n_channels, self.cfg.sample_rate), dtype=np.float32) if want_ir else None
        self._ck(self.L.fs_build_ir_bands(self.h, hist_source, conv_source, noise_seed, out.ctypes.data if want_ir else None))
        return out

    def build_ir_from_energy(self, energy, source=0):
        energy = np.ascontiguousarray(energy, dtype=np.float32)
        if energy.shape != (self.cfg.n_bins,):
            raise ValueError("energy must have n_bins entries")
        ir = np.zeros((self.cfg.n_channels, self.cfg.sample_rate), dtype=np.float32)
        self._ck(self.L.fs_build_ir_from_energy(self.h, source, energy.ctypes.data, ir.ctypes.data))
        return ir

    def set_ir(self, ir, source=0):
        ir = np.ascontiguousarray(ir, dtype=np.float32)
        if ir.shape != (self.cfg.n_channels, self.cfg.sample_rate):
            raise ValueError("ir must be [n_channels][sample_rate]")
        self._ck(self.L.fs_set_ir(self.h, source, ir.ctypes.data))

    # -- convolution --
    def conv_init_source(self, source=0):
        self._ck(self.L.fs_conv_init_source(self.h, source))

    def conv_release_source(self, source=0):
        self._ck(self.L.fs_conv_release_source(self.h, source))

    def conv_process(self, block, source=0):
        block = np.ascontiguousarray(block, dtype=np.float32)
        out = np.zeros_like(block)
        self._ck(self.L.fs_conv_process(self.h, source, block.ctypes.data, out.ctypes.data, block.shape[0]))
        return out

    def conv_process_many(self, blocks, source=0):
        """blocks: [n_blocks][frames][C]"""
        blocks = np.ascontiguousarray(blocks, dtype=np.float32)
        out = np.zeros_like(blocks)
        self._ck(self.L.fs_conv_process_many(self.h, source, blocks.ctypes.data, out.ctypes.data,
                                             blocks.shape[1], blocks.shape[0]))
        return out

    def conv_process_multi(self, blocks, sources):
        """blocks: [n_sources][frames][C], one callback of every listed source in one launch"""
        blocks = np.ascontiguousarray(blocks, dtype=np.float32)
        src = np.ascontiguousarray(sources, dtype=np.uint32)
        assert blocks.shape[0] == len(src)
        out = np.zeros_like(blocks)
        self._ck(self.L.fs_conv_process_multi(self.h, src.ctypes.data, len(src), blocks.ctypes.data, out.ctypes.data,
                                              blocks.shape[1]))
        return out

    def rfft(self, x):
        x = np.ascontiguousarray(x, dtype=np.float32)
        out = np.zeros((len(x) // 2 + 1, 2), dtype=np.float32)
        self._ck(self.L.fs_debug_rfft(self.h, x.ctypes.data, len(x), out.ctypes.data))
        return out[:, 0] + 1j * out[:, 1]

    def stats(self):
        st = Stats()
        self._ck(self.L.fs_get_stats(self.h, C.byref(st)))
        return st.as_dict()


class MultiContext:
    """fs_multi: one context per device inside this process, peer-store histogram reduce on device 0"""

    def __init__(self, devices, cfg=None, **over):
        self.L = load()
        self.cfg = cfg if cfg is not None else default_config(**over)
        devs = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        rc = self.L.fs_multi_create(C.byref(self.cfg), devs, len(devices), C.byref(h))
        if rc != FS_OK:
            raise FrequenSeeError(rc, (self.L.fs_multi_last_error() or b"").decode())
        self.h = h
        self.n = len(devices)

    def _ck(self, rc):
        if rc != FS_OK:
            raise FrequenSeeError(rc, (self.L.fs_multi_last_error() or b"").decode())

    def context(self, i=0):
        """the per-device context as a (non-owning) Context: build_ir / conv / stats continue on it"""
        c = Context.__new__(Context)
        c.L, c.cfg, c.n_sources = self.L, self.cfg, 0
        c.h = C.c_void_p(self.L.fs_multi_context(self.h, i))
        c.close = lambda: None
        return c

    def set_scene(self, verts, tri_mat, absorption):
        verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3, 3)
        tri_mat = np.ascontiguousarray(tri_mat, dtype=np.uint32)
        absorption = np.ascontiguousarray(absorption, dtype=np.float32)
        self._ck(self.L.fs_multi_scene_set_triangles(self.h, verts.ctypes.data, tri_mat.ctypes.data, len(verts)))
        self._ck(self.L.fs_multi_scene_set_materials(self.h, absorption.ctypes.data, absorption.shape[0], absorption.shape[1]))
        self._ck(self.L.fs_multi_scene_commit(self.h))

    def update_vertices(self, verts, first_tri=0):
        verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3, 3)
        self._ck(self.L.fs_multi_scene_update_vertices(self.h, verts.ctypes.data, first_tri, len(verts)))

    def refit(self):
        """every device refits its copy; returns device 0's cost ratio"""
        r = C.c_float(1.0)
        self._ck(self.L.fs_multi_scene_refit(self.h, C.byref(r)))
        return r.value

    def trace(self, src_pos, lis_pos, n_paths, max_depth, seed, want_hist=True):
        src, lis = Context._pos(src_pos, lis_pos)
        hist = np.zeros((len(src), self.cfg.n_bands, self.cfg.n_bins), dtype=np.uint64) if want_hist else None
        self._ck(self.L.fs_multi_trace(self.h, src.ctypes.data, len(src), lis.ctypes.data, n_paths, max_depth, seed,
                                       hist.ctypes.data if want_hist else None))
        return hist

    def trace_sources(self, src_pos, n_paths, depths, lis_pos, seed, want_hist=True):
        d = source_descs(src_pos, n_paths, depths)
        lis = np.ascontiguousarray(lis_pos, dtype=np.float32).reshape(3)
        hist = np.zeros((len(d), self.cfg.n_bands, self.cfg.n_bins), dtype=np.uint64) if want_hist else None
        self._ck(self.L.fs_multi_trace_sources(self.h, C.addressof(d), len(d), lis.ctypes.data, seed,
                                               hist.ctypes.data if want_hist else None))
        return hist

    def set_directivity_patterns(self, gains):
        """fs_multi_set_directivity_patterns: Context.set_directivity_patterns on every device"""
        full = _patterns(gains)
        self._ck(self.L.fs_multi_set_directivity_patterns(self.h, full.ctypes.data, len(full)))

    def set_source_directivity(self, forward, pattern):
        """fs_multi_set_source_directivity: Context.set_source_directivity on every device"""
        arr, S = _orients(forward, pattern)
        self._ck(self.L.fs_multi_set_source_directivity(self.h, arr, S))

    def last_ms(self):
        a, b = C.c_float(), C.c_float()
        self._ck(self.L.fs_multi_last_ms(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def synchronize(self):
        self._ck(self.L.fs_multi_synchronize(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.L.fs_multi_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def allocate_paths(stats, total, min_paths, max_paths, weight=None):
    """fs_allocate_paths: ray budgets [S] (uint64, sum == total) for the next update from Context.noise_stats() of the last
    one (a dict, or a NoiseStats array); host only, no context"""
    L = load()
    arr = stats if isinstance(stats, C.Array) else noise_stats_array(stats)
    S = len(arr)
    w = None if weight is None else np.ascontiguousarray(np.broadcast_to(np.asarray(weight, np.float32), (S,)))
    out = np.zeros(S, np.uint64)
    rc = L.fs_allocate_paths(arr, S, int(total), int(min_paths), int(max_paths), w.ctypes.data if w is not None else None,
                             out.ctypes.data)
    if rc != FS_OK:
        raise FrequenSeeError(rc, "fs_allocate_paths: invalid argument")
    return out


def directivity_polar(dipole_weight, power):
    """fs_directivity_polar: energy gains [B][33] of |(1 - w_b) + w_b c| ^ p_b at c = -1 + i/16 (B = len(w)); host only"""
    w = np.ascontiguousarray(np.atleast_1d(dipole_weight), dtype=np.float32)
    p = np.ascontiguousarray(np.broadcast_to(np.asarray(power, np.float32), w.shape))
    out = np.zeros((MAX_BANDS, DIR_POINTS), np.float32)
    rc = load().fs_directivity_polar(w.ctypes.data, p.ctypes.data, len(w), out.ctypes.data)
    if rc != FS_OK:
        raise FrequenSeeError(rc, "fs_directivity_polar: invalid argument")
    return out[:len(w)]


def load_float_array(path):
    """one float per line (the reference's saved_ir.txt, COMP.cpp:454-490); host only, no context"""
    L = load()
    n = C.c_uint64(0)
    rc = L.fs_load_float_array(os.fsencode(path), None, 0, C.byref(n))
    if rc != FS_OK:
        raise FrequenSeeError(rc, "cannot read %s" % path)
    out = np.zeros(n.value, np.float32)
    rc = L.fs_load_float_array(os.fsencode(path), out.ctypes.data, n.value, C.byref(n))
    if rc != FS_OK:
        raise FrequenSeeError(rc, "cannot read %s" % path)
    return out


def save_float_array(path, data):
    """COMP.cpp:492-505: one float per line, shortest form that reads back exactly"""
    L = load()
    data = np.ascontiguousarray(data, dtype=np.float32).ravel()
    rc = L.fs_save_float_array(os.fsencode(path), data.ctypes.data, data.size)
    if rc != FS_OK:
        raise FrequenSeeError(rc, "cannot write %s" % path)
