"""ctypes binding of the CPU oracle (oracle/libpt_oracle.so, every C statement under oracle/).

TEST INFRASTRUCTURE ONLY -- see oracle/pt_oracle.h.  Imported by tests/,
``__graft_entry__.smoke()`` and bench.py's cpu_baseline / ``--impl reference``
legs; never by the product package.  The neighbour SEARCH is parity-unpinned (no reference
goldens, CGAL absent); the metric, the box bound and the record layout are pinned on the
reference's own headers through ``ref_metric()`` (oracle/ref_shim.cpp -> oracle/_ref/).
This module loads the one library; pto_bake, pto_normals and pto_orient declare their own entry
points on it through ``bind()``.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

# Byte-for-byte mirror of the reference ``struct Point`` (src/Point.h:1-6).
POINT_DTYPE = np.dtype(
    [("ver", "<f8", 3), ("normal", "<f8", 3), ("color", "<i4", 3), ("pad_", "<i4"),
     ("U", "<f8"), ("V", "<f8")]
)
assert POINT_DTYPE.itemsize == 80


def build(force=False):
    """Compile the C oracle (gcc, oracle/Makefile) unless the library is up to date; returns its
    path.  Where make cannot update oracle/ (a read-only tree), the library is built in a per-user
    temporary directory instead."""
    make = ["make", "-C", _HERE, "-s"] + (["-B"] if force else [])
    try:
        subprocess.run(make, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        return os.path.join(_HERE, "libpt_oracle.so")
    except subprocess.CalledProcessError:
        out = os.path.join(tempfile.gettempdir(), f"pt_oracle_{os.getuid()}")
    os.makedirs(out, exist_ok=True)
    subprocess.run(make + ["OUT=" + out], check=True, stdout=subprocess.DEVNULL)
    return os.path.join(out, "libpt_oracle.so")


_REF_PATH = os.path.join(_HERE, "_ref", "libref_metric.so")
_ref = None


def reference_src():
    """The original project's src/ directory, named by the PT_REFERENCE_SRC environment variable
    (it is not part of this repository), or None where it is not set or holds no Distance.h."""
    src = os.environ.get("PT_REFERENCE_SRC")
    return src if src and os.path.exists(os.path.join(src, "Distance.h")) else None


def ref_metric():
    """The reference's OWN src/Point.h + src/Distance.h compiled by `make -C oracle ref REF=<src>`
    (oracle/ref_shim.cpp), or None where it was never built and no reference_src() is given."""
    global _ref
    if _ref is None:
        if not os.path.exists(_REF_PATH):
            src = reference_src()
            if src is None:
                return None
            subprocess.run(["make", "-C", _HERE, "-s", "ref", "REF=" + src], check=True,
                           stdout=subprocess.DEVNULL)
        R = ctypes.CDLL(_REF_PATH)
        vp, dbl = ctypes.c_void_p, ctypes.c_double
        R.ref_point_layout.argtypes = [vp]
        R.ref_transformed_distance.restype = dbl
        R.ref_transformed_distance.argtypes = [vp, vp]
        R.ref_min_distance_to_rectangle.restype = dbl
        R.ref_min_distance_to_rectangle.argtypes = [vp, vp, vp, vp]
        R.ref_new_distance.restype = dbl
        R.ref_new_distance.argtypes = [dbl, dbl, dbl]
        R.ref_transformed_radius.restype = dbl
        R.ref_transformed_radius.argtypes = [dbl]
        R.ref_inverse_of_transformed_distance.restype = dbl
        R.ref_inverse_of_transformed_distance.argtypes = [dbl]
        _ref = R
    return _ref


_vp, _i64, _i32, _dbl, _u64 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_double, ctypes.c_uint64
# (name, restype, argtypes) of this module's entry points; bind() adds the other modules' tables
_PROTOS = [
    ("pto_transformed_distance", _dbl, [_vp, _vp]),
    ("pto_min_distance_to_rectangle", _dbl, [_vp, _vp, _vp, _vp]),
    ("pto_new_distance", _dbl, [_dbl, _dbl, _dbl]),
    ("pto_transformed_radius", _dbl, [_dbl]),
    ("pto_knn_bruteforce", _i32, [_vp, _i64, _vp, _i64, _i32, _dbl, _vp, _vp, _i32]),
    ("pto_blend", _i32, [_vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp]),
    ("pto_kdtree_build", _vp, [_vp, _i64, _i32]),
    ("pto_kdtree_free", None, [_vp]),
    ("pto_kdtree_node_count", _i64, [_vp]),
    ("pto_kdtree_knn", _i32, [_vp, _vp, _i64, _i32, _dbl, _i32, _vp, _vp, _i32]),
    ("pto_reference_face_loop", _i64, [_vp, _vp, _vp, _i64, _i32, _i32]),
    ("pto_max_threads", _i32, []),
    ("pto_synth_cloud", _i32, [_vp, _i64, _i32, _u64, _u64, _dbl, _dbl, _dbl, _dbl, _dbl, _i32]),
    ("pto_synth_samples", _i32, [_vp, _i64, _i64, _dbl, _dbl, _dbl, _dbl, _i32]),
    ("pto_texture_faces", _i32, [_vp, _vp, _vp, _i32, _vp, _i64, _i32, _vp, _vp]),
    ("pto_texture_pad", _i32, [_vp, _i32, _vp]),
]
_lib = None


def _declare(L, protos):
    for name, res, args in protos:
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args


def bind(protos):
    """Declare more entry points of lib() from (name, restype, argtypes) rows, now if the library
    is loaded, else when it is."""
    protos = list(protos)
    _PROTOS.extend(protos)
    if _lib is not None:
        _declare(_lib, protos)


def lib():
    """The oracle library, built by build() if needed, with every bound prototype declared."""
    global _lib
    if _lib is None:
        L = ctypes.CDLL(build())
        _declare(L, _PROTOS)
        _lib = L
    return _lib


def make_points(xyz, normal=None, color=None, uv=None):
    """Pack arrays into the 80-byte AoS ``Point`` records."""
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


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _chk_points(a):
    a = np.ascontiguousarray(a)
    assert a.dtype == POINT_DTYPE, a.dtype
    return a


def transformed_distance(p1, p2):
    a, b = _chk_points(p1.reshape(1)), _chk_points(p2.reshape(1))
    return lib().pto_transformed_distance(_ptr(a), _ptr(b))


def min_distance_to_rectangle(p, lo, hi, dists=None):
    a = _chk_points(p.reshape(1))
    lo = np.ascontiguousarray(lo, dtype=np.float64)
    hi = np.ascontiguousarray(hi, dtype=np.float64)
    d = np.zeros(3) if dists is None else dists
    return lib().pto_min_distance_to_rectangle(_ptr(a), _ptr(lo), _ptr(hi), _ptr(d)), d


def knn_bruteforce(points, queries, k, radius=-1.0, nthreads=0, want_d2=True):
    points, queries = _chk_points(points), _chk_points(queries)
    m = queries.shape[0]
    idx = np.empty((m, k), dtype=np.int32)
    d2 = np.empty((m, k), dtype=np.float64) if want_d2 else None
    rc = lib().pto_knn_bruteforce(_ptr(points), points.shape[0], _ptr(queries), m, k,
                                  float(radius), _ptr(idx), _ptr(d2) if want_d2 else None,
                                  nthreads)
    assert rc == 0, rc
    return idx, d2


def blend(points, idx, d2):
    points = _chk_points(points)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    d2 = np.ascontiguousarray(d2, dtype=np.float64)
    m, k = idx.shape
    rgba = np.empty((m, 4), dtype=np.uint8)
    nrm = np.empty((m, 3), dtype=np.float32)
    rc = lib().pto_blend(_ptr(points), points.shape[0], m, k, _ptr(idx), _ptr(d2),
                         _ptr(rgba), _ptr(nrm))
    assert rc == 0, rc
    return rgba, nrm


class KdTree:
    """The reference's CPU path restated: ``Tree tree(points.begin(), points.end())``
    (src/pointsTransfer.cpp:259) + ``K_neighbor_search`` (:474)."""

    def __init__(self, points, bucket_size=10):
        self._points = _chk_points(points)
        self._h = lib().pto_kdtree_build(_ptr(self._points), self._points.shape[0], bucket_size)
        assert self._h

    def close(self):
        if self._h:
            lib().pto_kdtree_free(self._h)
            self._h = None

    __del__ = close

    @property
    def node_count(self):
        return lib().pto_kdtree_node_count(self._h)

    def knn(self, queries, k, radius=-1.0, exact_ties=True, nthreads=0, want_d2=True):
        queries = _chk_points(queries)
        m = queries.shape[0]
        idx = np.empty((m, k), dtype=np.int32)
        d2 = np.empty((m, k), dtype=np.float64) if want_d2 else None
        rc = lib().pto_kdtree_knn(self._h, _ptr(queries), m, k, float(radius),
                                  1 if exact_ties else 0, _ptr(idx),
                                  _ptr(d2) if want_d2 else None, nthreads)
        assert rc == 0, rc
        return idx, d2

    def reference_face_loop(self, vertices, faces, k, nthreads=0):
        vertices = _chk_points(vertices)
        faces = np.ascontiguousarray(faces, dtype=np.int32)
        return lib().pto_reference_face_loop(self._h, _ptr(vertices), _ptr(faces),
                                             faces.shape[0], k, nthreads)


def max_threads():
    return lib().pto_max_threads()


def synth_cloud(n, seed, kind=0, u0=0.0, u1=1000.0, v0=0.0, v1=1000.0, sigma=0.01, first_index=0,
                nthreads=0):
    """Host restatement of the device cloud generator (pt_synth_host.c): ``n`` Point records."""
    out = np.empty(int(n), dtype=POINT_DTYPE)
    rc = lib().pto_synth_cloud(_ptr(out), int(n), int(kind), int(seed), int(first_index), u0, u1,
                               v0, v1, sigma, nthreads)
    assert rc == 0, rc
    return out


def synth_samples(gu, gv, u0=0.0, u1=1000.0, v0=0.0, v1=1000.0, center=False):
    """gu x gv mesh samples on the noise-free surface (row-major, v outer) as Point records."""
    out = np.empty(int(gu) * int(gv), dtype=POINT_DTYPE)
    rc = lib().pto_synth_samples(_ptr(out), int(gu), int(gv), u0, u1, v0, v1, 1 if center else 0)
    assert rc == 0, rc
    return out


def texture(points, vertices, idx, faces, resolution, pad=True):
    """The reference's face loop + texture post-process (pt_texture_oracle.c).  idx: int32
    [n_vertices, k] neighbour lists.  Returns (bgra uint8 [res,res,4], (triangles, inside))."""
    points, vertices = _chk_points(points), _chk_points(vertices)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    faces = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    img = np.zeros((resolution, resolution, 4), dtype=np.uint8)
    stats = np.zeros(2, dtype=np.int64)
    rc = lib().pto_texture_faces(_ptr(points), _ptr(vertices), _ptr(idx), idx.shape[1], _ptr(faces),
                                 faces.shape[0], resolution, _ptr(img), _ptr(stats))
    assert rc == 0, rc
    if pad:
        out = np.empty_like(img)
        assert lib().pto_texture_pad(_ptr(img), resolution, _ptr(out)) == 0
        img = out
    return img, (int(stats[0]), int(stats[1]))


def texture_pad(img):
    img = np.ascontiguousarray(img, dtype=np.uint8)
    out = np.empty_like(img)
    assert lib().pto_texture_pad(_ptr(img), img.shape[0], _ptr(out)) == 0
    return out
