"""ctypes binding of the per-texel bake oracle (oracle/pt_bake_oracle.c).

TEST INFRASTRUCTURE ONLY, like oracle/pto.py, whose k-NN, blend and padding it uses.  The C file
is compiled on first use with the flags of oracle/Makefile (-ffp-contract=off: no FMA) into
oracle/libpt_bake_oracle.so, or into a per-user temporary directory where oracle/ is read-only.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from . import pto

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "pt_bake_oracle.c")
_DEPS = (_SRC, os.path.join(_HERE, "pt_oracle.h"))
_CFLAGS = ["-O3", "-std=c11", "-fPIC", "-ffp-contract=off", "-Wall", "-Wextra"]
_lib_handle = None


def build(force=False):
    """Compile pt_bake_oracle.c (gcc) unless an up-to-date library exists; returns its path."""
    newest = max(os.path.getmtime(f) for f in _DEPS)
    for d in (_HERE, os.path.join(tempfile.gettempdir(), f"pto_bake_{os.getuid()}")):
        path = os.path.join(d, "libpt_bake_oracle.so")
        if not force and os.path.exists(path) and os.path.getmtime(path) >= newest:
            return path
        tmp = f"{path}.{os.getpid()}.tmp"
        try:
            os.makedirs(d, exist_ok=True)
            subprocess.run(["/usr/bin/gcc", *_CFLAGS, "-I" + _HERE, "-shared", "-o", tmp, _SRC, "-lm"],
                           check=True, stdout=subprocess.DEVNULL,
                           stderr=subprocess.DEVNULL if d == _HERE else None)
            os.replace(tmp, path)
            return path
        except (OSError, subprocess.CalledProcessError):
            if os.path.exists(tmp):
                os.remove(tmp)
            if d != _HERE:
                raise
    raise RuntimeError("unreachable")


def _lib():
    global _lib_handle
    if _lib_handle is None:
        L = ctypes.CDLL(build())
        vp, i64, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
        L.pto_bake_texels.restype = i64
        L.pto_bake_texels.argtypes = [vp, i64, vp, i64, i32, vp, vp]
        L.pto_bake_encode.restype = i32
        L.pto_bake_encode.argtypes = [ctypes.c_float]
        L.pto_bake_compose.restype = i32
        L.pto_bake_compose.argtypes = [vp, i64, vp, vp, i32, vp, vp, vp]
        _lib_handle = L
    return _lib_handle


def bake_texels(vertices, faces, resolution):
    """Per-texel bake, texel stage (pt_bake_oracle.c): (texel ids uint32 [m], positions float64
    [m,3]) of the covered texels in ascending texel order."""
    vertices = pto._chk_points(vertices)
    faces = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    texels = np.empty(resolution * resolution, dtype=np.uint32)
    xyz = np.empty((resolution * resolution, 3), dtype=np.float64)
    m = _lib().pto_bake_texels(pto._ptr(vertices), vertices.shape[0], pto._ptr(faces), faces.shape[0],
                               resolution, pto._ptr(texels), pto._ptr(xyz))
    assert m >= 0, m
    return texels[:m].copy(), xyz[:m].copy()


def bake_encode(n):
    """The normal-map byte of one fp32 normal component."""
    return _lib().pto_bake_encode(float(n))


def bake_compose(texels, rgba, normal, resolution, pad=True):
    """Per-texel bake, composition: (bgra uint8 [res,res,4], normal_bgra uint8 [res,res,4], normal
    float32 [res,res,3]) from the samples' blend results; the 8-bit maps padded like pto.texture()."""
    texels = np.ascontiguousarray(texels, dtype=np.uint32)
    rgba = np.ascontiguousarray(rgba, dtype=np.uint8).reshape(-1, 4)
    normal = np.ascontiguousarray(normal, dtype=np.float32).reshape(-1, 3)
    assert rgba.shape[0] == normal.shape[0] == texels.shape[0]
    bgra = np.empty((resolution, resolution, 4), dtype=np.uint8)
    nbgra = np.empty((resolution, resolution, 4), dtype=np.uint8)
    nf = np.empty((resolution, resolution, 3), dtype=np.float32)
    rc = _lib().pto_bake_compose(pto._ptr(texels), texels.shape[0], pto._ptr(rgba), pto._ptr(normal),
                                 resolution, pto._ptr(bgra), pto._ptr(nbgra), pto._ptr(nf))
    assert rc == 0, rc
    if pad:
        bgra, nbgra = pto.texture_pad(bgra), pto.texture_pad(nbgra)
    return bgra, nbgra, nf


def bake(points, vertices, faces, k, resolution, radius=-1.0, pad=True):
    """The whole per-texel bake on the CPU: texels, exact k-NN (lowest index on ties) + pto.blend,
    composition.  A sample position with a NaN coordinate gets an empty neighbour list, as the
    device query kernels answer NaN rows.  Returns (bgra, normal_bgra, normal, (texels, empty))."""
    texels, xyz = bake_texels(vertices, faces, resolution)
    q = pto.make_points(xyz)
    idx, d2 = pto.KdTree(points).knn(q, k, radius=radius, exact_ties=True)
    nan_rows = np.isnan(xyz).any(axis=1)
    idx[nan_rows], d2[nan_rows] = -1, np.inf
    rgba, nrm = pto.blend(points, idx, d2)
    bgra, nbgra, nf = bake_compose(texels, rgba, nrm, resolution, pad=pad)
    return bgra, nbgra, nf, (int(texels.shape[0]), int((idx[:, 0] < 0).sum()))
