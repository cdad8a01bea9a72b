"""Host-side mirror of the reference's interface for the detail-transfer hot path.

The reference (horizon-research/3D-Reconstruction-From-Point-Cloud) exposes this path as
C++ objects in ``src/pointsTransfer.cpp``:

* ``Tree tree(points.begin(), points.end());``            (:259, typedefs :37-40)
* ``K_neighbor_search search(tree, query, K);``           (:474)
* iteration over ``(Point, squared distance)`` results    (:475-478)

with ``Point`` (src/Point.h) as the record type and ``Distance`` (src/Distance.h) as the
metric.  This module keeps those names and argument meanings and forwards everything to the
C ABI in ``include/points_transfer.h`` (``libpoints_transfer_b200.so``, hand-written sm_100a
CUDA).  There is no CPU fallback: if the library is missing or no CUDA device is present the
calls raise.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# PT_LIB_NAME selects a diagnosis build of the same library (e.g. the -DPT_STATS one of `make stats`)
LIB_PATH = os.path.join(_HERE, os.environ.get("PT_LIB_NAME", "libpoints_transfer_b200.so"))

# Byte-for-byte mirror of the reference ``struct Point`` (src/Point.h:1-6), 80 bytes.
POINT_DTYPE = np.dtype(
    [("ver", "<f8", 3), ("normal", "<f8", 3), ("color", "<i4", 3), ("pad_", "<i4"),
     ("U", "<f8"), ("V", "<f8")]
)
assert POINT_DTYPE.itemsize == 80
ATTR_DTYPE = np.dtype([("nx", "<f4"), ("ny", "<f4"), ("nz", "<f4"), ("rgba", "u1", 4)])
CAND_DTYPE = np.dtype([("d2", "<f8"), ("id", "<i4"), ("rgba", "u1", 4), ("nx", "<f4"),
                       ("ny", "<f4"), ("nz", "<f4"), ("pad_", "<i4")])
assert ATTR_DTYPE.itemsize == 16 and CAND_DTYPE.itemsize == 32

PT_OK = 0
PT_ERR_NO_DEVICE = 3
PT_ERR_UNSUPPORTED = 5
PT_ERR_NOT_REPRESENTABLE = 6
PT_ERR_NON_FINITE = 7
PT_MAX_K = 32
COORD_AUTO, COORD_F32, COORD_F64 = 0, 1, 2
SYNTH_HEIGHTFIELD, SYNTH_SKEWED = 0, 1

# Every symbol include/points_transfer.h declares (the drop-in library) ...
ABI_SYMBOLS = (
    "pt_version", "pt_status_string", "pt_device_count", "pt_index_build", "pt_index_free",
    "pt_index_get_info", "pt_index_fallback_counts", "pt_knn", "pt_transfer", "pt_texture_render", "pt_transfer_slab", "pt_index_build_device", "pt_query_device",
    "pt_merge_device", "pt_halo_route_device", "pt_halo_prepare_device",
    "pt_halo_merge_device", "pt_ghost_check_device", "pt_route_samples_device",
    "pt_scatter_rows_device", "pt_sharded_build", "pt_sharded_free", "pt_sharded_get_info", "pt_sharded_knn",
    "pt_sharded_transfer", "pt_texture_render_lists", "pt_set_option", "pt_get_option", "pt_debug_stats", "pt_debug_stats_n", "pt_kernel_launch_count",
    "pt_texture_bake", "pt_bake_texels_device", "pt_bake_compose_device",
    "pt_texture_bake_ex", "pt_bake_samples_device", "pt_bake_frames_device", "pt_bake_compose_tangent_device",
    "pt_texture_bake_height", "pt_bake_compose_height_device", "pt_sharded_bake",
    "pt_index_estimate_normals", "pt_estimate_normals_device", "pt_index_orient_normals",
    "pt_sharded_estimate_normals", "pt_sharded_orient_normals",
)
# ... and include/pt_synth.h (bench / test scaffolding, its own library)
SYNTH_SYMBOLS = ("pt_synth_cloud_device", "pt_synth_samples_device", "pt_synth_pack_points_device",
                 "pt_synth_pack_queries_device")
SYNTH_LIB_PATH = os.path.join(_HERE, "libpt_synth_b200.so")


class PointsTransferError(RuntimeError):
    def __init__(self, status, where):
        self.status = status
        super().__init__(f"{where}: status {status} ({status_string(status)})")


class BuildOpts(ctypes.Structure):
    _fields_ = [("device", ctypes.c_int), ("coord_mode", ctypes.c_int),
                ("ids", ctypes.c_void_p), ("reserved", ctypes.c_int * 8)]


class IndexInfo(ctypes.Structure):
    _fields_ = [("n_points", ctypes.c_uint64), ("n_leaves", ctypes.c_uint64),
                ("n_levels", ctypes.c_int), ("coord_mode", ctypes.c_int),
                ("device", ctypes.c_int), ("last_fallback_samples", ctypes.c_int),
                ("bbox_lo", ctypes.c_double * 3), ("bbox_hi", ctypes.c_double * 3),
                ("device_bytes", ctypes.c_uint64), ("build_ms", ctypes.c_float),
                ("last_query_ms", ctypes.c_float), ("last_h2d_ms", ctypes.c_float),
                ("last_d2h_ms", ctypes.c_float)]


class TextureStats(ctypes.Structure):
    _fields_ = [("triangles", ctypes.c_uint64), ("inside_points", ctypes.c_uint64),
                ("knn_ms", ctypes.c_float), ("draw_ms", ctypes.c_float), ("pad_ms", ctypes.c_float)]


class BakeStats(ctypes.Structure):
    _fields_ = [("texels", ctypes.c_uint64), ("empty", ctypes.c_uint64), ("raster_ms", ctypes.c_float),
                ("knn_ms", ctypes.c_float), ("pad_ms", ctypes.c_float)]


class BakeOutputs(ctypes.Structure):
    _fields_ = [("bgra", ctypes.c_void_p), ("normal_bgra", ctypes.c_void_p), ("normal", ctypes.c_void_p),
                ("tangent_bgra", ctypes.c_void_p), ("tangent_normal", ctypes.c_void_p),
                ("vertex_tangents", ctypes.c_void_p)]


class BakeHeight(ctypes.Structure):
    _fields_ = [("height", ctypes.c_void_p), ("height_u16", ctypes.c_void_p), ("range", ctypes.c_double * 2),
                ("range_used", ctypes.c_double * 2), ("texels", ctypes.c_uint64)]


class NormalsStats(ctypes.Structure):
    _fields_ = [("estimated", ctypes.c_uint64), ("knn_ms", ctypes.c_float), ("pca_ms", ctypes.c_float)]


class OrientStats(ctypes.Structure):
    _fields_ = [("oriented", ctypes.c_uint64), ("flipped", ctypes.c_uint64), ("components", ctypes.c_uint64),
                ("edges", ctypes.c_uint64), ("knn_ms", ctypes.c_float), ("mst_ms", ctypes.c_float)]


class ShardedOpts(ctypes.Structure):
    _fields_ = [("n_devices", ctypes.c_int), ("devices", ctypes.POINTER(ctypes.c_int)), ("halo", ctypes.c_double),
                ("k_hint", ctypes.c_int), ("coord_mode", ctypes.c_int), ("reserved", ctypes.c_int * 8)]


class ShardedInfo(ctypes.Structure):
    _fields_ = [("n_slabs", ctypes.c_int), ("rebuilds", ctypes.c_int), ("halo", ctypes.c_double),
                ("n_points", ctypes.c_uint64), ("slab_points", ctypes.c_uint64 * 64),
                ("slab_ghosts", ctypes.c_uint64 * 64), ("slab_device", ctypes.c_int * 64)]


class SynthParams(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int), ("seed", ctypes.c_uint64),
                ("first_index", ctypes.c_uint64), ("u0", ctypes.c_double),
                ("u1", ctypes.c_double), ("v0", ctypes.c_double), ("v1", ctypes.c_double),
                ("sigma", ctypes.c_double)]


_lib = None


def lib():
    """Load the CUDA library.  Fails loudly: there is no fallback implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a).  points_transfer_b200 has no CPU fallback.")
    L = ctypes.CDLL(LIB_PATH)
    vp, sz, i32, dbl = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_double
    L.pt_version.restype = ctypes.c_char_p
    L.pt_status_string.restype = ctypes.c_char_p
    L.pt_status_string.argtypes = [i32]
    L.pt_device_count.restype = i32
    L.pt_index_build.restype = i32
    L.pt_index_build.argtypes = [vp, sz, ctypes.POINTER(BuildOpts), ctypes.POINTER(vp)]
    L.pt_index_free.restype = i32
    L.pt_index_free.argtypes = [vp]
    L.pt_index_get_info.restype = i32
    L.pt_index_get_info.argtypes = [vp, ctypes.POINTER(IndexInfo)]
    L.pt_index_fallback_counts.restype = i32
    L.pt_index_fallback_counts.argtypes = [vp, ctypes.POINTER(ctypes.c_uint32 * 2)]
    L.pt_knn.restype = i32
    L.pt_knn.argtypes = [vp, vp, sz, i32, dbl, vp, vp]
    L.pt_transfer.restype = i32
    L.pt_transfer.argtypes = [vp, vp, sz, i32, dbl, vp, vp, vp, vp]
    L.pt_texture_render.restype = i32
    L.pt_texture_render.argtypes = [vp, vp, sz, vp, sz, i32, dbl, i32, i32, vp, ctypes.POINTER(TextureStats)]
    L.pt_transfer_slab.restype = i32
    L.pt_transfer_slab.argtypes = [vp, vp, i32, sz, i32, dbl, vp, i32, i32, dbl, vp, vp, vp, vp,
                                   ctypes.POINTER(i32)]
    L.pt_index_build_device.restype = i32
    L.pt_index_build_device.argtypes = [vp, i32, vp, vp, sz, i32, ctypes.POINTER(vp)]
    L.pt_query_device.restype = i32
    L.pt_query_device.argtypes = [vp, vp, sz, i32, dbl, vp, vp, vp, vp, vp, vp, vp]
    L.pt_merge_device.restype = i32
    L.pt_merge_device.argtypes = [vp, i32, sz, i32, vp, vp, vp, vp, vp, i32, vp]
    u32 = ctypes.c_uint32
    L.pt_halo_route_device.restype = i32
    L.pt_halo_route_device.argtypes = [vp, vp, sz, i32, dbl, vp, i32, i32, u32, vp, vp, vp, vp, vp]
    L.pt_halo_prepare_device.restype = i32
    L.pt_halo_prepare_device.argtypes = [vp, i32, u32, vp, vp, vp]
    L.pt_halo_merge_device.restype = i32
    L.pt_halo_merge_device.argtypes = [vp, vp, vp, vp, u32, i32, vp, vp, vp, vp, vp]
    L.pt_ghost_check_device.restype = i32
    L.pt_ghost_check_device.argtypes = [vp, vp, sz, i32, dbl, vp, i32, i32, dbl, vp, vp]
    L.pt_route_samples_device.restype = i32
    L.pt_route_samples_device.argtypes = [vp, sz, vp, i32, u32, vp, vp, vp, vp, vp]
    L.pt_scatter_rows_device.restype = i32
    L.pt_scatter_rows_device.argtypes = [vp, vp, sz, u32, vp, vp]
    L.pt_sharded_build.restype = i32
    L.pt_sharded_build.argtypes = [vp, sz, ctypes.POINTER(ShardedOpts), ctypes.POINTER(vp)]
    L.pt_sharded_free.restype = i32
    L.pt_sharded_free.argtypes = [vp]
    L.pt_sharded_get_info.restype = i32
    L.pt_sharded_get_info.argtypes = [vp, ctypes.POINTER(ShardedInfo)]
    L.pt_sharded_knn.restype = i32
    L.pt_sharded_knn.argtypes = [vp, vp, sz, i32, dbl, vp, vp]
    L.pt_sharded_transfer.restype = i32
    L.pt_sharded_transfer.argtypes = [vp, vp, sz, i32, dbl, vp, vp, vp, vp]
    L.pt_texture_render_lists.restype = i32
    L.pt_texture_render_lists.argtypes = [vp, sz, vp, sz, vp, sz, vp, i32, i32, i32, i32, vp,
                                          ctypes.POINTER(TextureStats)]
    L.pt_texture_bake.restype = i32
    L.pt_texture_bake.argtypes = [vp, vp, sz, vp, sz, i32, dbl, i32, i32, vp, vp, vp, ctypes.POINTER(BakeStats)]
    L.pt_bake_texels_device.restype = i32
    L.pt_bake_texels_device.argtypes = [vp, sz, vp, sz, i32, vp, vp, ctypes.POINTER(sz), i32, vp]
    L.pt_bake_compose_device.restype = i32
    L.pt_bake_compose_device.argtypes = [vp, sz, vp, vp, i32, i32, vp, vp, vp, i32, vp]
    L.pt_texture_bake_ex.restype = i32
    L.pt_texture_bake_ex.argtypes = [vp, vp, sz, vp, sz, i32, dbl, i32, i32, ctypes.POINTER(BakeOutputs),
                                     ctypes.POINTER(BakeStats)]
    L.pt_bake_samples_device.restype = i32
    L.pt_bake_samples_device.argtypes = [vp, sz, vp, sz, i32, vp, vp, vp, ctypes.POINTER(sz), i32, vp]
    L.pt_bake_frames_device.restype = i32
    L.pt_bake_frames_device.argtypes = [vp, sz, vp, sz, vp, vp, i32, vp]
    L.pt_bake_compose_tangent_device.restype = i32
    L.pt_bake_compose_tangent_device.argtypes = [vp, vp, sz, vp, sz, vp, vp, sz, vp, vp, i32, i32, vp, vp, i32, vp]
    L.pt_texture_bake_height.restype = i32
    L.pt_texture_bake_height.argtypes = [vp, vp, sz, vp, sz, i32, dbl, i32, i32, ctypes.POINTER(BakeOutputs),
                                         ctypes.POINTER(BakeHeight), ctypes.POINTER(BakeStats)]
    L.pt_sharded_bake.restype = i32
    L.pt_sharded_bake.argtypes = [vp, vp, sz, vp, sz, i32, dbl, i32, i32, ctypes.POINTER(BakeOutputs),
                                  ctypes.POINTER(BakeHeight), ctypes.POINTER(BakeStats)]
    L.pt_bake_compose_height_device.restype = i32
    L.pt_bake_compose_height_device.argtypes = [vp, vp, sz, vp, sz, vp, vp, vp, sz, vp, i32, vp, sz, i32, i32, vp, vp,
                                                vp, vp, i32, vp]
    L.pt_index_estimate_normals.restype = i32
    L.pt_index_estimate_normals.argtypes = [vp, i32, dbl, vp, i32, vp, vp, ctypes.POINTER(NormalsStats)]
    L.pt_estimate_normals_device.restype = i32
    L.pt_estimate_normals_device.argtypes = [vp, i32, dbl, vp, i32, vp, vp, vp]
    L.pt_sharded_estimate_normals.restype = i32
    L.pt_sharded_estimate_normals.argtypes = [vp, i32, dbl, vp, i32, vp, vp, ctypes.POINTER(NormalsStats)]
    L.pt_index_orient_normals.restype = i32
    L.pt_index_orient_normals.argtypes = [vp, i32, dbl, vp, i32, vp, vp, ctypes.POINTER(OrientStats)]
    L.pt_sharded_orient_normals.restype = i32
    L.pt_sharded_orient_normals.argtypes = [vp, i32, dbl, vp, i32, vp, vp, ctypes.POINTER(OrientStats)]
    L.pt_set_option.restype = i32
    L.pt_set_option.argtypes = [ctypes.c_char_p, i32]
    L.pt_get_option.restype = i32
    L.pt_get_option.argtypes = [ctypes.c_char_p, ctypes.POINTER(i32)]
    L.pt_kernel_launch_count.restype = ctypes.c_uint64
    _lib = L
    return L


_synth_lib = None


def synth_lib():
    """The synthetic-workload generators (bench / test scaffolding, libpt_synth_b200.so)."""
    global _synth_lib
    if _synth_lib is not None:
        return _synth_lib
    if not os.path.exists(SYNTH_LIB_PATH):
        raise ImportError(f"{SYNTH_LIB_PATH} is missing: run __graft_entry__.build()")
    L = ctypes.CDLL(SYNTH_LIB_PATH)
    vp, sz, i32, dbl = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_double
    L.pt_synth_cloud_device.restype = i32
    L.pt_synth_cloud_device.argtypes = [vp, vp, sz, ctypes.POINTER(SynthParams), vp]
    L.pt_synth_samples_device.restype = i32
    L.pt_synth_samples_device.argtypes = [vp, sz, sz, dbl, dbl, dbl, dbl, i32, vp]
    L.pt_synth_pack_points_device.restype = i32
    L.pt_synth_pack_points_device.argtypes = [vp, vp, sz, vp, vp]
    L.pt_synth_pack_queries_device.restype = i32
    L.pt_synth_pack_queries_device.argtypes = [vp, sz, vp, vp]
    _synth_lib = L
    return L


def version():
    return lib().pt_version().decode()


def status_string(status):
    return lib().pt_status_string(int(status)).decode()


def device_count():
    return lib().pt_device_count()


def kernel_launch_count():
    return int(lib().pt_kernel_launch_count())


def debug_stats(reset=True):
    """Work counters of the query kernel (zeros unless the library was built with -DPT_STATS)."""
    names = ("expansions", "leaves", "pushes", "pops", "compactions", "heap_inserts", "parked",
             "warp_rounds", "overflowed", "samples", "warp_drain_iters", "warp_expand_iters",
             "grid_attempts", "grid_candidates", "grid_exact_selects", "grid_handed_over",
             "span_lookups", "span_copies", "span_copies_mergeable", "span_warps", "span_warp_busy_ns_sum",
             "span_warp_busy_ns_max", "span_first_start_ns_inv", "span_last_finish_ns", "span_redo_halves")
    buf = (ctypes.c_uint64 * len(names))()
    _check(lib().pt_debug_stats_n(buf, len(names), 1 if reset else 0), "pt_debug_stats_n")
    return {n: int(buf[i]) for i, n in enumerate(names)}


def set_option(name, value):
    _check(lib().pt_set_option(name.encode(), int(value)), f"pt_set_option({name})")


def get_option(name):
    v = ctypes.c_int(0)
    _check(lib().pt_get_option(name.encode(), ctypes.byref(v)), f"pt_get_option({name})")
    return v.value


def _check(status, where):
    if status != PT_OK:
        raise PointsTransferError(status, where)


def make_points(xyz, normal=None, color=None, uv=None):
    """Pack arrays into the reference's 80-byte AoS ``Point`` records (src/Point.h)."""
    xyz = np.asarray(xyz, dtype=np.float64).reshape(-1, 3)
    p = np.zeros(xyz.shape[0], dtype=POINT_DTYPE)
    p["ver"] = xyz
    if normal is not None:
        p["normal"] = np.asarray(normal, dtype=np.float64).reshape(-1, 3)
    if color is not None:
        p["color"] = np.asarray(color, dtype=np.int32).reshape(-1, 3)
    if uv is not None:
        uv = np.asarray(uv, dtype=np.float64).reshape(-1, 2)
        p["U"], p["V"] = uv[:, 0], uv[:, 1]
    return p


def _as_points(a, what):
    a = np.ascontiguousarray(a)
    if a.dtype != POINT_DTYPE:
        raise TypeError(f"{what} must be an array of 80-byte Point records (POINT_DTYPE)")
    return a.reshape(-1)


def _radius(radius):
    return -1.0 if radius is None else float(radius)


def _viewpoint(viewpoint):
    return None if viewpoint is None else ctypes.cast((ctypes.c_double * 3)(*map(float, viewpoint)), ctypes.c_void_p)


def _np_ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class Distance:
    """The reference's metric (src/Distance.h).  Only the radius transform is needed on the
    host; the metric itself is evaluated on the device in the same operation order."""

    @staticmethod
    def transformed_distance(d):
        """``Distance::transformed_distance(double d)`` -- src/Distance.h:97."""
        return d * d

    @staticmethod
    def inverse_of_transformed_distance(d):
        """src/Distance.h:99."""
        return float(np.sqrt(d))


class Tree:
    """``Tree tree(points.begin(), points.end())`` -- src/pointsTransfer.cpp:259.

    ``points`` is an array of ``Point`` records on the host.  The spatial index is built
    on the GPU immediately (the reference builds lazily inside the first query)."""

    def __init__(self, points, device=-1, coord_mode=COORD_AUTO, ids=None):
        self._h = ctypes.c_void_p()
        pts = _as_points(points, "points")
        opts = BuildOpts()
        opts.device, opts.coord_mode = int(device), int(coord_mode)
        self._ids = None
        if ids is not None:
            self._ids = np.ascontiguousarray(ids, dtype=np.int32)
            if self._ids.shape[0] != pts.shape[0]:
                raise ValueError("ids must have one entry per point")
            opts.ids = self._ids.ctypes.data
        _check(lib().pt_index_build(_np_ptr(pts), pts.shape[0], ctypes.byref(opts),
                                    ctypes.byref(self._h)), "pt_index_build")

    @classmethod
    def _from_handle(cls, handle):
        t = cls.__new__(cls)
        t._h = handle
        t._ids = None
        return t

    @property
    def handle(self):
        return self._h

    def info(self):
        info = IndexInfo()
        _check(lib().pt_index_get_info(self._h, ctypes.byref(info)), "pt_index_get_info")
        return info

    def size(self):
        return int(self.info().n_points)

    def fallback_counts(self):
        """(samples re-run by the warp kernel, samples the grid kernel handed over) of the last
        query launch on this index."""
        out = (ctypes.c_uint32 * 2)()
        _check(lib().pt_index_fallback_counts(self._h, ctypes.byref(out)), "pt_index_fallback_counts")
        return int(out[0]), int(out[1])

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().pt_index_free(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- host-buffer calls (the reference-facing plugin surface) -----------------------
    def knn(self, queries, k, radius=None, want_d2=True, out_idx=None, out_d2=None):
        """Batched ``K_neighbor_search``: returns ``(idx[m,k] int32, d2[m,k] float64)``
        in ascending ``(d2, index)`` order, padded with ``-1`` / ``+inf``."""
        q = _as_points(queries, "queries")
        m = q.shape[0]
        idx = out_idx if out_idx is not None else np.empty((m, k), dtype=np.int32)
        d2 = out_d2 if out_d2 is not None else (np.empty((m, k), dtype=np.float64) if want_d2 else None)
        _check(lib().pt_knn(self._h, _np_ptr(q), m, int(k), _radius(radius), _np_ptr(idx),
                            _np_ptr(d2)), "pt_knn")
        return idx, d2

    def transfer(self, queries, k, radius=None, want_idx=True, want_d2=False, out=None):
        """k-NN + fused colour/normal blend for every sample.  Returns a dict with ``rgba``
        ``[m,4] uint8``, ``normal`` ``[m,3] float32`` and optionally ``idx`` / ``d2``."""
        q = _as_points(queries, "queries")
        m = q.shape[0]
        out = {} if out is None else out
        if "rgba" not in out:
            out["rgba"] = np.empty((m, 4), dtype=np.uint8)
        if "normal" not in out:
            out["normal"] = np.empty((m, 3), dtype=np.float32)
        if want_idx and "idx" not in out:
            out["idx"] = np.empty((m, k), dtype=np.int32)
        if want_d2 and "d2" not in out:
            out["d2"] = np.empty((m, k), dtype=np.float64)
        _check(lib().pt_transfer(self._h, _np_ptr(q), m, int(k), _radius(radius),
                                 _np_ptr(out.get("idx")), _np_ptr(out.get("d2")),
                                 _np_ptr(out["rgba"]), _np_ptr(out["normal"])), "pt_transfer")
        return out


    def texture(self, vertices, faces, k=20, resolution=8192, radius=None, pad=True):
        """The reference's output image (src/pointsTransfer.cpp:462-611): per-face transfer of the
        cloud's colours into the mesh's UV space.  vertices: Point records (position, U, V,
        colour), faces: int32 [F,3].  Returns (bgra uint8 [res,res,4] as cv::Mat CV_8UC4, stats)."""
        v = _as_points(vertices, "vertices")
        f = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
        img = np.empty((resolution, resolution, 4), dtype=np.uint8)
        st = TextureStats()
        _check(lib().pt_texture_render(self._h, _np_ptr(v), v.shape[0], _np_ptr(f), f.shape[0], int(k),
                                       _radius(radius), int(resolution), 1 if pad else 0, _np_ptr(img),
                                       ctypes.byref(st)), "pt_texture_render")
        return img, {"triangles": int(st.triangles), "inside_points": int(st.inside_points),
                     "knn_ms": st.knn_ms, "draw_ms": st.draw_ms, "pad_ms": st.pad_ms}

    def bake(self, vertices, faces, k=20, resolution=2048, radius=None, pad=True,
             want=("bgra", "normal_bgra", "normal"), height_range=None):
        """Per-texel bake (DESIGN.md section 8): colour and normal maps of the cloud on the mesh's
        UV atlas.  vertices: Point records (position, normal, U, V), faces: int32 [F,3].  Returns a
        dict with the requested outputs -- ``bgra`` uint8 [res,res,4] (B G R 255), ``normal_bgra``
        uint8 [res,res,4] (object-space normal map, RGB = xyz), ``normal`` float32 [res,res,3]
        (never padded), ``tangent_bgra`` uint8 [res,res,4] (tangent-space normal map, glTF / OpenGL
        convention), ``tangent_normal`` float32 [res,res,3] (never padded), ``tangents`` float32
        [n_vertices,4] (the per-vertex tangent and handedness the tangent maps are expressed in, glTF
        TANGENT layout), ``height`` float32 [res,res] (the cloud's signed height above the mesh along
        the interpolated mesh normal, NaN without a value, never padded), ``height_u16`` uint16
        [res,res] (its 16-bit code over ``height_range`` = (lo, hi) when finite with lo < hi, else
        over the heights' min and max; decode with lo + E * (hi - lo) / 65535) -- and ``stats``
        (texels, empty, raster_ms, knn_ms, pad_ms).  With a height output the result also carries
        ``height_range`` (the (lo, hi) used) and ``stats["height_texels"]`` (texels with a value).
        All outputs come from one k-NN pass."""
        return _bake(lib().pt_texture_bake_height, "pt_texture_bake_height", self._h, vertices, faces, k, resolution,
                     radius, pad, want, height_range)

    def estimate_normals(self, k=16, radius=None, viewpoint=None, store=False):
        """PCA normal estimation over each point's k nearest neighbours (DESIGN.md section 8, "Normal
        estimation").  Returns a dict with ``normal`` float32 [n,3] ((0, 0, 0) without an estimate),
        ``variation`` float32 [n] (surface variation, NaN without an estimate), both in the order of
        the points the tree was built from, and ``stats`` (estimated, knn_ms, pca_ms).  Orientation:
        the point's own normal where it is usable, else towards ``viewpoint`` (x, y, z) when given,
        else the largest component positive.  ``store=True`` also replaces the tree's normals with
        the estimates, so later ``transfer`` / ``bake`` calls blend them."""
        return _estimate_normals(lib().pt_index_estimate_normals, "pt_index_estimate_normals", self._h, self.size(),
                                 k, radius, viewpoint, store)

    def orient_normals(self, k=18, radius=None, viewpoint=None, store=False):
        """Orients the tree's normals consistently by propagation along the minimum spanning forest of
        the k-NN graph (DESIGN.md section 8, "Normal orientation").  Returns a dict with ``normal``
        float32 [n,3] (the stored normal, negated where its sign flips; unchanged where it is not
        usable), ``root`` int32 [n] (the id of the point's component root, -1 where it does not take
        part), both in the order of the points the tree was built from, and ``stats`` (oriented,
        flipped, components, edges, knn_ms, mst_ms).  Each component's root, its highest point, faces
        ``viewpoint`` (x, y, z) when given, else +z.  ``store=True`` also replaces the tree's normals
        with the oriented ones, so later ``transfer`` / ``bake`` calls blend them."""
        return _orient_normals(lib().pt_index_orient_normals, "pt_index_orient_normals", self._h, self.size(), k,
                               radius, viewpoint, store)

    def transfer_slab(self, queries_ptr, queries_are_xyz, m, k, radius, boxes6, rank, halo,
                      idx_ptr, rgba_ptr, normal_ptr, d2_ptr=None):
        """pt_transfer_slab on raw host pointers (ints): one slab's pipelined host-buffer step
        with the ghost-zone check fused in.  boxes6: float64 numpy [R,6].  Returns True when the
        results are final (no sample may leave the ghost zone towards another slab)."""
        boxes6 = np.ascontiguousarray(boxes6, dtype=np.float64)
        need = ctypes.c_int32(0)
        _check(lib().pt_transfer_slab(self._h, queries_ptr, 1 if queries_are_xyz else 0, int(m),
                                      int(k), _radius(radius), _np_ptr(boxes6), boxes6.shape[0],
                                      int(rank), float(halo), idx_ptr, d2_ptr, rgba_ptr,
                                      normal_ptr, ctypes.byref(need)), "pt_transfer_slab")
        return need.value == 0


_BAKE_OUTPUTS = ("bgra", "normal_bgra", "normal", "tangent_bgra", "tangent_normal", "tangents")
_HEIGHT_OUTPUTS = ("height", "height_u16")


def _bake(fn, name, handle, vertices, faces, k, resolution, radius, pad, want, height_range):
    """Arguments, output arrays and result dict of ``Tree.bake`` and ``ShardedTree.bake``: ``fn`` is
    ``pt_texture_bake_height`` or ``pt_sharded_bake``, which take the same arguments after the handle."""
    v = _as_points(vertices, "vertices")
    f = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    names = _BAKE_OUTPUTS + _HEIGHT_OUTPUTS
    unknown = set(want) - set(names)
    if unknown or not want:
        raise ValueError(f"want must name some of {', '.join(names)} (got {want!r})")
    res = int(resolution)
    shapes = {"bgra": ((res, res, 4), np.uint8), "normal_bgra": ((res, res, 4), np.uint8),
              "normal": ((res, res, 3), np.float32), "tangent_bgra": ((res, res, 4), np.uint8),
              "tangent_normal": ((res, res, 3), np.float32), "tangents": ((v.shape[0], 4), np.float32),
              "height": ((res, res), np.float32), "height_u16": ((res, res), np.uint16)}
    out = {n: np.empty(*shapes[n]) for n in names if n in want}
    o = BakeOutputs(*[out[n].ctypes.data if n in out else None for n in _BAKE_OUTPUTS])
    hb = None
    if any(n in out for n in _HEIGHT_OUTPUTS):
        lo, hi = (float("nan"), float("nan")) if height_range is None else map(float, height_range)
        hb = BakeHeight(*[out[n].ctypes.data if n in out else None for n in _HEIGHT_OUTPUTS],
                        (ctypes.c_double * 2)(lo, hi))
    st = BakeStats()
    _check(fn(handle, _np_ptr(v), v.shape[0], _np_ptr(f), f.shape[0], int(k), _radius(radius), res, 1 if pad else 0,
              ctypes.byref(o), None if hb is None else ctypes.byref(hb), ctypes.byref(st)), name)
    out["stats"] = {"texels": int(st.texels), "empty": int(st.empty), "raster_ms": st.raster_ms,
                    "knn_ms": st.knn_ms, "pad_ms": st.pad_ms}
    if hb is not None:
        out["height_range"] = (hb.range_used[0], hb.range_used[1])
        out["stats"]["height_texels"] = int(hb.texels)
    return out


def _estimate_normals(fn, name, handle, n, k, radius, viewpoint, store):
    """Output arrays and result dict of ``Tree.estimate_normals`` and ``ShardedTree.estimate_normals``:
    ``fn`` is ``pt_index_estimate_normals`` or ``pt_sharded_estimate_normals``, which take the same
    arguments after the handle."""
    out = {"normal": np.empty((n, 3), dtype=np.float32), "variation": np.empty(n, dtype=np.float32)}
    st = NormalsStats()
    _check(fn(handle, int(k), _radius(radius), _viewpoint(viewpoint), 1 if store else 0, _np_ptr(out["normal"]),
              _np_ptr(out["variation"]), ctypes.byref(st)), name)
    out["stats"] = {"estimated": int(st.estimated), "knn_ms": st.knn_ms, "pca_ms": st.pca_ms}
    return out


def _orient_normals(fn, name, handle, n, k, radius, viewpoint, store):
    """Output arrays and result dict of ``Tree.orient_normals`` and ``ShardedTree.orient_normals``:
    ``fn`` is ``pt_index_orient_normals`` or ``pt_sharded_orient_normals``, which take the same
    arguments after the handle."""
    out = {"normal": np.empty((n, 3), dtype=np.float32), "root": np.empty(n, dtype=np.int32)}
    st = OrientStats()
    _check(fn(handle, int(k), _radius(radius), _viewpoint(viewpoint), 1 if store else 0, _np_ptr(out["normal"]),
              _np_ptr(out["root"]), ctypes.byref(st)), name)
    out["stats"] = {"oriented": int(st.oriented), "flipped": int(st.flipped), "components": int(st.components),
                    "edges": int(st.edges), "knn_ms": st.knn_ms, "mst_ms": st.mst_ms}
    return out


class ShardedTree:
    """The cloud sharded over several GPUs of one box by the C++ host (``pt_sharded_*``,
    csrc/pt_sharded.cu): same calls as ``Tree``, ids index the caller's ``points``."""

    def __init__(self, points, devices, halo=0.0, k_hint=20, coord_mode=COORD_AUTO):
        self._points = _as_points(points, "points")          # must outlive the handle
        self._h = ctypes.c_void_p()
        devs = (ctypes.c_int * len(devices))(*[int(d) for d in devices])
        o = ShardedOpts()
        o.n_devices, o.devices, o.halo, o.k_hint, o.coord_mode = len(devices), devs, float(halo), int(k_hint), int(coord_mode)
        _check(lib().pt_sharded_build(_np_ptr(self._points), self._points.shape[0], ctypes.byref(o),
                                      ctypes.byref(self._h)), "pt_sharded_build")

    def info(self):
        i = ShardedInfo()
        _check(lib().pt_sharded_get_info(self._h, ctypes.byref(i)), "pt_sharded_get_info")
        n = i.n_slabs
        return {"n_slabs": n, "rebuilds": i.rebuilds, "halo": i.halo, "slab_points": list(i.slab_points[:n]),
                "slab_ghosts": list(i.slab_ghosts[:n]), "slab_device": list(i.slab_device[:n])}

    def knn(self, queries, k, radius=None, want_d2=True):
        q = _as_points(queries, "queries")
        m = q.shape[0]
        idx = np.empty((m, k), dtype=np.int32)
        d2 = np.empty((m, k), dtype=np.float64) if want_d2 else None
        _check(lib().pt_sharded_knn(self._h, _np_ptr(q), m, int(k), _radius(radius), _np_ptr(idx), _np_ptr(d2)),
               "pt_sharded_knn")
        return idx, d2

    def transfer(self, queries, k, radius=None, want_idx=True, want_d2=False):
        q = _as_points(queries, "queries")
        m = q.shape[0]
        out = {"rgba": np.empty((m, 4), dtype=np.uint8), "normal": np.empty((m, 3), dtype=np.float32)}
        if want_idx:
            out["idx"] = np.empty((m, k), dtype=np.int32)
        if want_d2:
            out["d2"] = np.empty((m, k), dtype=np.float64)
        _check(lib().pt_sharded_transfer(self._h, _np_ptr(q), m, int(k), _radius(radius), _np_ptr(out.get("idx")),
                                         _np_ptr(out.get("d2")), _np_ptr(out["rgba"]), _np_ptr(out["normal"])),
               "pt_sharded_transfer")
        return out

    def bake(self, vertices, faces, k=20, resolution=2048, radius=None, pad=True,
             want=("bgra", "normal_bgra", "normal"), height_range=None):
        """``Tree.bake`` on the sharded cloud (``pt_sharded_bake``): same arguments and result, every
        output byte-identical to ``Tree.bake`` on one index of the same cloud.  The raster, frames and
        composition run on slab 0's device and each slab answers the texels in its x-range on its
        own device; ``stats["knn_ms"]`` is the host wall time of that part."""
        return _bake(lib().pt_sharded_bake, "pt_sharded_bake", self._h, vertices, faces, k, resolution, radius, pad,
                     want, height_range)

    def estimate_normals(self, k=16, radius=None, viewpoint=None, store=False):
        """``Tree.estimate_normals`` on the sharded cloud (``pt_sharded_estimate_normals``): same
        arguments and result, ``normal``, ``variation`` and ``stats["estimated"]`` byte-identical to
        ``Tree.estimate_normals`` on one index of the same cloud.  Each slab estimates the points it
        owns on its own device; ``stats["knn_ms"]`` is the host wall time of that stage and
        ``stats["pca_ms"]`` the PCA kernels' device time summed over the slabs.  ``store=True`` also
        replaces the normals in every slab that holds the point, so later ``transfer`` / ``bake``
        calls blend them, and keeps them across rebuilds of the slabs."""
        return _estimate_normals(lib().pt_sharded_estimate_normals, "pt_sharded_estimate_normals", self._h,
                                 self._points.shape[0], k, radius, viewpoint, store)

    def orient_normals(self, k=18, radius=None, viewpoint=None, store=False):
        """``Tree.orient_normals`` on the sharded cloud (``pt_sharded_orient_normals``): same arguments
        and result, ``normal``, ``root`` and the four counts of ``stats`` byte-identical to
        ``Tree.orient_normals`` on one index of the same cloud.  Each slab builds the edges of the points
        it owns and the spanning forest of the edges between them on its own device; slab 0's device
        joins them into the cloud's forest.  ``stats["knn_ms"]`` is the host wall time of the slab
        stage and ``stats["mst_ms"]`` that of the rest.  ``store=True`` also replaces the normals in
        every slab that holds the point, so later ``transfer`` / ``bake`` calls blend them, and keeps
        them across rebuilds of the slabs."""
        return _orient_normals(lib().pt_sharded_orient_normals, "pt_sharded_orient_normals", self._h,
                               self._points.shape[0], k, radius, viewpoint, store)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().pt_sharded_free(self._h)
            self._h = ctypes.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def texture_from_lists(points, vertices, faces, idx, resolution=8192, pad=True, device=0):
    """``pt_texture_render_lists``: the texture stage for neighbour lists computed elsewhere."""
    p, v = _as_points(points, "points"), _as_points(vertices, "vertices")
    f = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    img = np.empty((resolution, resolution, 4), dtype=np.uint8)
    st = TextureStats()
    _check(lib().pt_texture_render_lists(_np_ptr(p), p.shape[0], _np_ptr(v), v.shape[0], _np_ptr(f), f.shape[0],
                                         _np_ptr(idx), idx.shape[1], int(resolution), 1 if pad else 0, int(device),
                                         _np_ptr(img), ctypes.byref(st)), "pt_texture_render_lists")
    return img, {"triangles": int(st.triangles), "inside_points": int(st.inside_points)}


class K_neighbor_search:
    """``K_neighbor_search search(tree, query, K)`` -- src/pointsTransfer.cpp:474.

    Iterating yields ``(point_index, squared_distance)`` in ascending order, like the
    reference's ``search.begin() .. search.end()`` over ``(Point, d2)`` pairs (:475-478);
    the caller indexes its own ``points`` array with ``point_index``."""

    def __init__(self, tree, query, k, radius=None):
        q = np.ascontiguousarray(query)
        if q.dtype != POINT_DTYPE:
            raise TypeError("query must be a Point record")
        idx, d2 = tree.knn(q.reshape(1), k, radius=radius)
        keep = idx[0] >= 0
        self._idx, self._d2 = idx[0][keep], d2[0][keep]

    def __iter__(self):
        return iter(zip(self._idx.tolist(), self._d2.tolist()))

    def __len__(self):
        return int(self._idx.shape[0])


# ---- device-buffer API (torch tensors as HBM handles; torch is plumbing only) ----------------

def _tptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return ctypes.c_void_p(s.cuda_stream)


class DeviceTree(Tree):
    """Index built from coordinates already resident in HBM (bench `value`, slabs)."""

    def __init__(self, pos, attrs=None, ids=None):
        import torch
        assert pos.is_cuda and pos.is_contiguous() and pos.dim() == 2 and pos.shape[1] == 4
        assert pos.dtype in (torch.float32, torch.float64)
        n = pos.shape[0]
        if attrs is not None:
            assert attrs.is_cuda and attrs.is_contiguous() and attrs.dtype == torch.uint8
            assert attrs.numel() == 16 * n
        if ids is not None:
            assert ids.is_cuda and ids.is_contiguous() and ids.dtype == torch.int32
            assert ids.numel() == n
        self._h = ctypes.c_void_p()
        self._ids = None
        self.torch_device = pos.device
        torch.cuda.current_stream(pos.device).synchronize()
        _check(lib().pt_index_build_device(_tptr(pos), 1 if pos.dtype == torch.float64 else 0,
                                           _tptr(attrs), _tptr(ids), n, pos.device.index,
                                           ctypes.byref(self._h)), "pt_index_build_device")

    def query(self, queries, k, radius=None, radius2_per_query=None, idx=None, d2=None,
              rgba=None, normal=None, cand=None, stream=None):
        """Asynchronous on ``stream`` (default: torch's current stream).  ``queries`` is a
        float64 ``[m,3]`` CUDA tensor; outputs are pre-allocated CUDA tensors or None."""
        import torch
        assert queries.is_cuda and queries.dtype == torch.float64 and queries.is_contiguous()
        m = queries.shape[0]
        for t, dt, cnt in ((idx, torch.int32, m * k), (d2, torch.float64, m * k),
                           (rgba, torch.uint8, m * 4), (normal, torch.float32, m * 3),
                           (cand, torch.uint8, m * k * 32),
                           (radius2_per_query, torch.float64, m)):
            if t is not None:
                assert t.is_cuda and t.is_contiguous() and t.dtype == dt and t.numel() == cnt
        with torch.cuda.device(queries.device):
            _check(lib().pt_query_device(self._h, _tptr(queries), m, int(k), _radius(radius),
                                         _tptr(radius2_per_query), _tptr(idx), _tptr(d2),
                                         _tptr(rgba), _tptr(normal), _tptr(cand),
                                         _stream_ptr(stream)), "pt_query_device")


    def estimate_normals(self, k=16, radius=None, viewpoint=None, store=False, normal=None, variation=None,
                         stream=None):
        """``Tree.estimate_normals`` into pre-allocated CUDA tensors (``normal`` float32 [n,3],
        ``variation`` float32 [n], either may be None; both None needs ``store``), asynchronous on
        ``stream`` (default: torch's current stream)."""
        import torch
        n = self.size()
        for t, cnt in ((normal, 3 * n), (variation, n)):
            if t is not None:
                assert t.is_cuda and t.is_contiguous() and t.dtype == torch.float32 and t.numel() == cnt
        with torch.cuda.device(self.torch_device):
            _check(lib().pt_estimate_normals_device(self._h, int(k), _radius(radius), _viewpoint(viewpoint),
                                                    1 if store else 0, _tptr(normal), _tptr(variation),
                                                    _stream_ptr(stream)), "pt_estimate_normals_device")


def merge_device(lists, n_lists, m, k, idx=None, d2=None, rgba=None, normal=None, cand=None,
                 stream=None):
    """K5: merge ``n_lists`` per-slab candidate lists (uint8 tensor of n_lists*m*k*32 bytes)."""
    import torch
    assert lists.is_cuda and lists.is_contiguous() and lists.dtype == torch.uint8
    assert lists.numel() == n_lists * m * k * 32
    with torch.cuda.device(lists.device):
        _check(lib().pt_merge_device(_tptr(lists), int(n_lists), int(m), int(k), _tptr(idx),
                                     _tptr(d2), _tptr(rgba), _tptr(normal), _tptr(cand),
                                     lists.device.index, _stream_ptr(stream)), "pt_merge_device")


def bake_texels_device(vertices_xyzuv, faces, resolution, texels=None, xyz=None, stream=None):
    """``pt_bake_texels_device``: the covered texels of the mesh's UV atlas as samples.
    vertices_xyzuv: float64 [n,5] CUDA tensor (x, y, z, u, v), faces: int32 [F,3] CUDA tensor.
    Returns (texel ids [m], positions float64 [m,3]) as views into ``texels`` / ``xyz``, which are
    allocated with room for resolution^2 samples unless given.  Texel ids are row * resolution +
    col in ascending order, held in an int32 tensor (torch has no uint32 arithmetic; they are
    < 2^28).  Synchronises ``stream``."""
    import torch
    assert vertices_xyzuv.is_cuda and vertices_xyzuv.dtype == torch.float64 and vertices_xyzuv.is_contiguous()
    assert vertices_xyzuv.dim() == 2 and vertices_xyzuv.shape[1] == 5
    assert faces.is_cuda and faces.dtype == torch.int32 and faces.is_contiguous() and faces.numel() % 3 == 0
    dev = vertices_xyzuv.device
    cap = int(resolution) * int(resolution)
    if texels is None:
        texels = torch.empty(cap, dtype=torch.int32, device=dev)
    if xyz is None:
        xyz = torch.empty((cap, 3), dtype=torch.float64, device=dev)
    assert texels.is_cuda and texels.dtype == torch.int32 and texels.is_contiguous() and texels.numel() >= cap
    assert xyz.is_cuda and xyz.dtype == torch.float64 and xyz.is_contiguous() and xyz.numel() >= 3 * cap
    count = ctypes.c_size_t(0)
    with torch.cuda.device(dev):
        _check(lib().pt_bake_texels_device(_tptr(vertices_xyzuv), vertices_xyzuv.shape[0], _tptr(faces),
                                           faces.numel() // 3, int(resolution), _tptr(texels), _tptr(xyz),
                                           ctypes.byref(count), dev.index, _stream_ptr(stream)),
               "pt_bake_texels_device")
    m = count.value
    return texels[:m], xyz.view(-1)[:3 * m].view(m, 3)


def bake_compose_device(texels, rgba, normal, resolution, pad=True, bgra=None, normal_bgra=None,
                        normal_out=None, stream=None):
    """``pt_bake_compose_device``: the bake's maps from the samples' blend results (``rgba`` uint8
    [m,4], ``normal`` float32 [m,3] as ``DeviceTree.query`` returns them).  Outputs are
    pre-allocated CUDA tensors (uint8 [res,res,4], uint8 [res,res,4], float32 [res,res,3]) or
    None; at least one must be given.  Asynchronous on ``stream``."""
    import torch
    m = texels.numel()
    assert texels.is_cuda and texels.dtype == torch.int32 and texels.is_contiguous()
    assert rgba.is_cuda and rgba.dtype == torch.uint8 and rgba.is_contiguous() and rgba.numel() == 4 * m
    assert normal.is_cuda and normal.dtype == torch.float32 and normal.is_contiguous() and normal.numel() == 3 * m
    n_pix = int(resolution) * int(resolution)
    for t, dt, cnt in ((bgra, torch.uint8, 4 * n_pix), (normal_bgra, torch.uint8, 4 * n_pix),
                       (normal_out, torch.float32, 3 * n_pix)):
        if t is not None:
            assert t.is_cuda and t.is_contiguous() and t.dtype == dt and t.numel() == cnt
    with torch.cuda.device(texels.device):
        _check(lib().pt_bake_compose_device(_tptr(texels), m, _tptr(rgba), _tptr(normal), int(resolution),
                                            1 if pad else 0, _tptr(bgra), _tptr(normal_bgra), _tptr(normal_out),
                                            texels.device.index, _stream_ptr(stream)), "pt_bake_compose_device")


def bake_samples_device(vertices_xyzuv, faces, resolution, stream=None):
    """``pt_bake_samples_device``: ``bake_texels_device`` plus the owner face of every sample.
    Returns (texel ids int32 [m], positions float64 [m,3], faces int32 [m]).  Synchronises
    ``stream``."""
    import torch
    assert vertices_xyzuv.is_cuda and vertices_xyzuv.dtype == torch.float64 and vertices_xyzuv.is_contiguous()
    assert vertices_xyzuv.dim() == 2 and vertices_xyzuv.shape[1] == 5
    assert faces.is_cuda and faces.dtype == torch.int32 and faces.is_contiguous() and faces.numel() % 3 == 0
    dev = vertices_xyzuv.device
    cap = int(resolution) * int(resolution)
    texels = torch.empty(cap, dtype=torch.int32, device=dev)
    xyz = torch.empty((cap, 3), dtype=torch.float64, device=dev)
    owner = torch.empty(cap, dtype=torch.int32, device=dev)
    count = ctypes.c_size_t(0)
    with torch.cuda.device(dev):
        _check(lib().pt_bake_samples_device(_tptr(vertices_xyzuv), vertices_xyzuv.shape[0], _tptr(faces),
                                            faces.numel() // 3, int(resolution), _tptr(texels), _tptr(xyz),
                                            _tptr(owner), ctypes.byref(count), dev.index, _stream_ptr(stream)),
               "pt_bake_samples_device")
    m = count.value
    return texels[:m], xyz.view(-1)[:3 * m].view(m, 3), owner[:m]


def bake_frames_device(vertices_xyzuvn, faces, tangents=True, stream=None):
    """``pt_bake_frames_device``: the tangent bake's vertex frames.  vertices_xyzuvn: float64
    [n,8] CUDA tensor (x, y, z, u, v, nx, ny, nz), faces: int32 [F,3].  Returns (frames float64
    [n,8] = N xyz, T xyz, w, 0; tangents float32 [n,4] or None).  Asynchronous on ``stream``."""
    import torch
    assert vertices_xyzuvn.is_cuda and vertices_xyzuvn.dtype == torch.float64 and vertices_xyzuvn.is_contiguous()
    assert vertices_xyzuvn.dim() == 2 and vertices_xyzuvn.shape[1] == 8
    assert faces.is_cuda and faces.dtype == torch.int32 and faces.is_contiguous() and faces.numel() % 3 == 0
    dev, n = vertices_xyzuvn.device, vertices_xyzuvn.shape[0]
    frames = torch.empty((n, 8), dtype=torch.float64, device=dev)
    tg = torch.empty((n, 4), dtype=torch.float32, device=dev) if tangents else None
    with torch.cuda.device(dev):
        _check(lib().pt_bake_frames_device(_tptr(vertices_xyzuvn), n, _tptr(faces), faces.numel() // 3, _tptr(frames),
                                           _tptr(tg), dev.index, _stream_ptr(stream)), "pt_bake_frames_device")
    return frames, tg


def bake_compose_tangent_device(vertices_xyzuvn, frames, faces, texels, sample_faces, rgba, normal, resolution,
                                pad=True, tangent_bgra=None, tangent_normal=None, stream=None):
    """``pt_bake_compose_tangent_device``: the tangent maps from the samples (``texels`` and
    ``sample_faces`` of ``bake_samples_device``, ``rgba`` / ``normal`` of ``DeviceTree.query``)
    and the frames of ``bake_frames_device``.  Outputs are pre-allocated CUDA tensors (uint8
    [res,res,4], float32 [res,res,3]) or None; at least one must be given.  Asynchronous on
    ``stream``."""
    import torch
    m, n = texels.numel(), vertices_xyzuvn.shape[0]
    assert vertices_xyzuvn.is_cuda and vertices_xyzuvn.dtype == torch.float64 and vertices_xyzuvn.is_contiguous()
    assert vertices_xyzuvn.dim() == 2 and vertices_xyzuvn.shape[1] == 8
    assert frames.is_cuda and frames.dtype == torch.float64 and frames.is_contiguous() and frames.numel() == 8 * n
    assert faces.is_cuda and faces.dtype == torch.int32 and faces.is_contiguous() and faces.numel() % 3 == 0
    for t, dt, cnt in ((texels, torch.int32, m), (sample_faces, torch.int32, m), (rgba, torch.uint8, 4 * m),
                       (normal, torch.float32, 3 * m)):
        assert t.is_cuda and t.is_contiguous() and t.dtype == dt and t.numel() == cnt
    n_pix = int(resolution) * int(resolution)
    for t, dt, cnt in ((tangent_bgra, torch.uint8, 4 * n_pix), (tangent_normal, torch.float32, 3 * n_pix)):
        if t is not None:
            assert t.is_cuda and t.is_contiguous() and t.dtype == dt and t.numel() == cnt
    with torch.cuda.device(texels.device):
        _check(lib().pt_bake_compose_tangent_device(_tptr(vertices_xyzuvn), _tptr(frames), n, _tptr(faces),
                                                    faces.numel() // 3, _tptr(texels), _tptr(sample_faces), m,
                                                    _tptr(rgba), _tptr(normal), int(resolution), 1 if pad else 0,
                                                    _tptr(tangent_bgra), _tptr(tangent_normal), texels.device.index,
                                                    _stream_ptr(stream)), "pt_bake_compose_tangent_device")


def bake_compose_height_device(vertices_xyzuvn, frames, faces, texels, sample_faces, sample_xyz, idx, k, cloud_xyz,
                               resolution, pad=True, height_range=None, height=None, height_u16=None, range_out=None,
                               stream=None):
    """``pt_bake_compose_height_device``: the height maps from the samples (``texels``,
    ``sample_faces`` and ``sample_xyz`` of ``bake_samples_device``), their neighbour lists ``idx``
    (int32 [m,k] of ``DeviceTree.query``), the frames of ``bake_frames_device`` and the cloud's
    positions ``cloud_xyz`` (float64 [n,3], original order).  Outputs are pre-allocated CUDA tensors
    (float32 [res,res], uint16 [res,res], float64 [2] for the range used) or None; at least one map
    must be given.  ``height_range`` = (lo, hi) fixes the code range when finite with lo < hi.
    Asynchronous on ``stream``."""
    import torch
    m, n = texels.numel(), vertices_xyzuvn.shape[0]
    assert vertices_xyzuvn.is_cuda and vertices_xyzuvn.dtype == torch.float64 and vertices_xyzuvn.is_contiguous()
    assert vertices_xyzuvn.dim() == 2 and vertices_xyzuvn.shape[1] == 8
    assert frames.is_cuda and frames.dtype == torch.float64 and frames.is_contiguous() and frames.numel() == 8 * n
    assert faces.is_cuda and faces.dtype == torch.int32 and faces.is_contiguous() and faces.numel() % 3 == 0
    for t, dt, cnt in ((texels, torch.int32, m), (sample_faces, torch.int32, m), (sample_xyz, torch.float64, 3 * m),
                       (idx, torch.int32, m * int(k))):
        assert t.is_cuda and t.is_contiguous() and t.dtype == dt and t.numel() == cnt
    assert cloud_xyz.is_cuda and cloud_xyz.dtype == torch.float64 and cloud_xyz.is_contiguous()
    assert cloud_xyz.numel() % 3 == 0
    n_pix = int(resolution) * int(resolution)
    for t, dt, cnt in ((height, torch.float32, n_pix), (height_u16, torch.uint16, n_pix), (range_out, torch.float64, 2)):
        if t is not None:
            assert t.is_cuda and t.is_contiguous() and t.dtype == dt and t.numel() == cnt
    rng = None if height_range is None else (ctypes.c_double * 2)(*map(float, height_range))
    with torch.cuda.device(texels.device):
        _check(lib().pt_bake_compose_height_device(_tptr(vertices_xyzuvn), _tptr(frames), n, _tptr(faces),
                                                   faces.numel() // 3, _tptr(texels), _tptr(sample_faces),
                                                   _tptr(sample_xyz), m, _tptr(idx), int(k), _tptr(cloud_xyz),
                                                   cloud_xyz.numel() // 3, int(resolution), 1 if pad else 0,
                                                   None if rng is None else ctypes.cast(rng, ctypes.c_void_p),
                                                   _tptr(height), _tptr(height_u16), _tptr(range_out),
                                                   texels.device.index, _stream_ptr(stream)),
               "pt_bake_compose_height_device")
