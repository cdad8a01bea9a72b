"""ctypes binding of the height bake oracle (tests/bake_height_oracle.c).

TEST INFRASTRUCTURE ONLY.  The C file is compiled on first use with the flags of oracle/Makefile
(-ffp-contract=off: no FMA) into a per-user temporary directory, so the tree is never written.  The
texel list, sample positions, owner faces and vertex frames come from tests/bake_tangent_oracle.py,
the neighbour lists from the existing oracle (oracle/pto.py); this file adds the heights, their
16-bit codes and the padding of the codes.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

import bake_tangent_oracle as tgo
from oracle import pto

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_SRC = os.path.join(_HERE, "bake_height_oracle.c")
_DEPS = (_SRC, os.path.join(_ORACLE, "pt_oracle.h"))
_CFLAGS = ["-O3", "-std=c11", "-fPIC", "-ffp-contract=off", "-Wall", "-Wextra"]
_lib_handle = None


def build(force=False):
    """Compile bake_height_oracle.c (gcc) unless an up-to-date library exists; returns its path."""
    d = os.path.join(tempfile.gettempdir(), f"pto_bake_height_{os.getuid()}")
    path = os.path.join(d, "libbake_height_oracle.so")
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
        L.pth_bake_height.restype = i32
        L.pth_bake_height.argtypes = [vp, i64, vp, vp, i64, vp, vp, vp, i64, vp, i64, vp, vp, i32, i32, vp]
        L.pth_bake_height_encode.restype = i64
        L.pth_bake_height_encode.argtypes = [vp, i64, vp, vp, vp]
        L.pth_bake_height_pad.restype = i32
        L.pth_bake_height_pad.argtypes = [vp, vp, i32, vp]
        _lib_handle = L
    return _lib_handle


def bake_height(vertices, frames, faces, texels, sample_faces, xyz, points, idx, d2, resolution):
    """Steps 1-4: the float height map [res,res], NaN (0x7fc00000) without a value."""
    vertices, points = pto._chk_points(vertices), pto._chk_points(points)
    frames = np.ascontiguousarray(frames, dtype=np.float64).reshape(-1, 8)
    faces = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    texels = np.ascontiguousarray(texels, dtype=np.uint32)
    sample_faces = np.ascontiguousarray(sample_faces, dtype=np.int32)
    xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    d2 = np.ascontiguousarray(d2, dtype=np.float64)
    m, k = idx.shape
    assert texels.shape[0] == sample_faces.shape[0] == xyz.shape[0] == m == d2.shape[0]
    h = np.empty((resolution, resolution), np.float32)
    rc = _lib().pth_bake_height(pto._ptr(vertices), vertices.shape[0], pto._ptr(frames), pto._ptr(faces),
                                faces.shape[0], pto._ptr(texels), pto._ptr(sample_faces), pto._ptr(xyz), m,
                                pto._ptr(points), points.shape[0], pto._ptr(idx), pto._ptr(d2), k, resolution,
                                pto._ptr(h))
    assert rc == 0, rc
    return h


def encode(height, height_range=None):
    """(unpadded codes uint16 [res,res], range used (lo, hi), texels with a value)."""
    height = np.ascontiguousarray(height, dtype=np.float32)
    codes = np.empty(height.shape, np.uint16)
    used = np.empty(2, np.float64)
    rin = None if height_range is None else np.ascontiguousarray(height_range, dtype=np.float64)
    valued = _lib().pth_bake_height_encode(pto._ptr(height), height.size, None if rin is None else pto._ptr(rin),
                                           pto._ptr(codes), pto._ptr(used))
    return codes, (float(used[0]), float(used[1])), int(valued)


def pad(height, codes):
    """The 16-bit padding of the codes."""
    height = np.ascontiguousarray(height, dtype=np.float32)
    codes = np.ascontiguousarray(codes, dtype=np.uint16)
    res = height.shape[0]
    out = np.empty_like(codes)
    assert _lib().pth_bake_height_pad(pto._ptr(height), pto._ptr(codes), res, pto._ptr(out)) == 0
    return out


def neighbours(points, xyz, k, radius=-1.0):
    """The bake's exact k-NN of the sample positions (lowest index on ties); a position with a NaN
    coordinate gets an empty list, as the device query kernels answer NaN rows."""
    idx, d2 = pto.KdTree(points).knn(pto.make_points(xyz), k, radius=radius, exact_ties=True)
    nan_rows = np.isnan(xyz).any(axis=1)
    idx[nan_rows], d2[nan_rows] = -1, np.inf
    return idx, d2


def bake(points, vertices, faces, k, resolution, radius=-1.0, pad_codes=True, height_range=None):
    """The whole height bake on the CPU.  Returns a dict: height, height_u16, height_range, texels
    (with a value), samples (texels, faces, positions), lists (idx, d2), frames."""
    texels, xyz, owner = tgo.bake_samples(vertices, faces, resolution)
    frames, _ = tgo.bake_frames(vertices, faces)
    idx, d2 = neighbours(points, xyz, k, radius)
    h = bake_height(vertices, frames, faces, texels, owner, xyz, points, idx, d2, resolution)
    codes, used, valued = encode(h, height_range)
    if pad_codes:
        codes = pad(h, codes)
    return {"height": h, "height_u16": codes, "height_range": used, "texels": valued,
            "samples": (texels, owner, xyz), "lists": (idx, d2), "frames": frames}
