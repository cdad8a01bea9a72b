"""ctypes binding of the tangent-space bake oracle (tests/bake_tangent_oracle.c).

TEST INFRASTRUCTURE ONLY.  The C file is compiled on first use with the flags of oracle/Makefile
(-ffp-contract=off: no FMA) into a per-user temporary directory, so the tree is never written.  The
texel list, sample positions, k-NN, blend, object-space maps and padding come from the existing
oracle (oracle/pto.py, oracle/pto_bake.py); this file adds the owner faces, the vertex frames and the
composition of the tangent maps.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from oracle import pto, pto_bake

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_SRC = os.path.join(_HERE, "bake_tangent_oracle.c")
_DEPS = (_SRC, os.path.join(_ORACLE, "pt_oracle.h"))
_CFLAGS = ["-O3", "-std=c11", "-fPIC", "-ffp-contract=off", "-Wall", "-Wextra"]
_lib_handle = None


def build(force=False):
    """Compile bake_tangent_oracle.c (gcc) unless an up-to-date library exists; returns its path."""
    d = os.path.join(tempfile.gettempdir(), f"pto_bake_tangent_{os.getuid()}")
    path = os.path.join(d, "libbake_tangent_oracle.so")
    if not force and os.path.exists(path) and os.path.getmtime(path) >= max(os.path.getmtime(f) for f in _DEPS):
        return path
    os.makedirs(d, exist_ok=True)
    tmp = f"{path}.{os.getpid()}.tmp"
    try:
        subprocess.run(["/usr/bin/gcc", *_CFLAGS, "-I" + _ORACLE, "-shared", "-o", tmp, _SRC, "-lm"], check=True)
        os.replace(tmp, path)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)
    return path


def _lib():
    global _lib_handle
    if _lib_handle is None:
        L = ctypes.CDLL(build())
        vp, i64, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
        L.ptt_bake_owners.restype = i64
        L.ptt_bake_owners.argtypes = [vp, i64, vp, i64, i32, vp, vp]
        L.ptt_bake_frames.restype = i32
        L.ptt_bake_frames.argtypes = [vp, i64, vp, i64, vp, vp]
        L.ptt_bake_compose_tangent.restype = i32
        L.ptt_bake_compose_tangent.argtypes = [vp, i64, vp, vp, i64, vp, vp, i64, vp, vp, i32, vp, vp]
        _lib_handle = L
    return _lib_handle


def bake_samples(vertices, faces, resolution):
    """bake_texels plus the owner face of every sample: (texels uint32 [m], positions float64
    [m,3], faces int32 [m])."""
    vertices = pto._chk_points(vertices)
    faces = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    n = resolution * resolution
    texels, owner = np.empty(n, np.uint32), np.empty(n, np.int32)
    m = _lib().ptt_bake_owners(pto._ptr(vertices), vertices.shape[0], pto._ptr(faces), faces.shape[0],
                               resolution, pto._ptr(texels), pto._ptr(owner))
    assert m >= 0, m
    ref_t, xyz = pto_bake.bake_texels(vertices, faces, resolution)
    assert np.array_equal(texels[:m], ref_t), "owner pass and texel stage disagree on the covered texels"
    return ref_t, xyz, owner[:m].copy()


def bake_frames(vertices, faces):
    """Tangent-space bake, vertex frames: (frames float64 [n,8] = N xyz, T xyz, w, 0, tangents
    float32 [n,4] = T xyz, w), zero for a vertex without a frame."""
    vertices = pto._chk_points(vertices)
    faces = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    n = vertices.shape[0]
    frames, tangents = np.empty((n, 8), np.float64), np.empty((n, 4), np.float32)
    rc = _lib().ptt_bake_frames(pto._ptr(vertices), n, pto._ptr(faces), faces.shape[0], pto._ptr(frames),
                                pto._ptr(tangents))
    assert rc == 0, rc
    return frames, tangents


def bake_compose_tangent(vertices, frames, faces, texels, sample_faces, rgba, normal, resolution, pad=True):
    """Tangent-space bake, composition: (tangent_bgra uint8 [res,res,4], tangent_normal float32
    [res,res,3]); the 8-bit map padded like pto.texture()."""
    vertices = pto._chk_points(vertices)
    frames = np.ascontiguousarray(frames, dtype=np.float64).reshape(-1, 8)
    faces = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    texels = np.ascontiguousarray(texels, dtype=np.uint32)
    sample_faces = np.ascontiguousarray(sample_faces, dtype=np.int32)
    rgba = np.ascontiguousarray(rgba, dtype=np.uint8).reshape(-1, 4)
    normal = np.ascontiguousarray(normal, dtype=np.float32).reshape(-1, 3)
    assert frames.shape[0] == vertices.shape[0]
    assert texels.shape[0] == sample_faces.shape[0] == rgba.shape[0] == normal.shape[0]
    tb = np.empty((resolution, resolution, 4), np.uint8)
    tn = np.empty((resolution, resolution, 3), np.float32)
    rc = _lib().ptt_bake_compose_tangent(pto._ptr(vertices), vertices.shape[0], pto._ptr(frames), pto._ptr(faces),
                                         faces.shape[0], pto._ptr(texels), pto._ptr(sample_faces), texels.shape[0],
                                         pto._ptr(rgba), pto._ptr(normal), resolution, pto._ptr(tb), pto._ptr(tn))
    assert rc == 0, rc
    if pad:
        tb = pto.texture_pad(tb)
    return tb, tn


def bake_tangent(points, vertices, faces, k, resolution, radius=-1.0, pad=True):
    """The whole bake with every output on the CPU, one k-NN pass as pt_texture_bake_ex.  Returns a
    dict: bgra, normal_bgra, normal, tangent_bgra, tangent_normal, tangents, frames, and
    texels / empty (counts), m (blended normal per sample), samples (texels, faces)."""
    texels, xyz, owner = bake_samples(vertices, faces, resolution)
    q = pto.make_points(xyz)
    idx, d2 = pto.KdTree(points).knn(q, k, radius=radius, exact_ties=True)
    nan_rows = np.isnan(xyz).any(axis=1)
    idx[nan_rows], d2[nan_rows] = -1, np.inf
    rgba, nrm = pto.blend(points, idx, d2)
    bgra, nbgra, nf = pto_bake.bake_compose(texels, rgba, nrm, resolution, pad=pad)
    frames, tangents = bake_frames(vertices, faces)
    tb, tn = bake_compose_tangent(vertices, frames, faces, texels, owner, rgba, nrm, resolution, pad=pad)
    return {"bgra": bgra, "normal_bgra": nbgra, "normal": nf, "tangent_bgra": tb, "tangent_normal": tn,
            "tangents": tangents, "frames": frames, "texels": int(texels.shape[0]),
            "empty": int((idx[:, 0] < 0).sum()), "m": nrm, "rgba": rgba, "samples": (texels, owner)}
