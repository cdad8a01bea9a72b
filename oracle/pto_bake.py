"""ctypes binding of the per-texel bake oracle (oracle/pt_bake_oracle.c): the object-space,
tangent-space and height bakes.

TEST INFRASTRUCTURE ONLY, like oracle/pto.py, whose library holds it and whose k-NN, blend and
padding it uses.
"""
import ctypes

import numpy as np

from . import pto

_vp, _i64, _i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
pto.bind([
    ("pto_bake_texels", _i64, [_vp, _i64, _vp, _i64, _i32, _vp, _vp, _vp]),
    ("pto_bake_encode", _i32, [ctypes.c_float]),
    ("pto_bake_compose", _i32, [_vp, _i64, _vp, _vp, _i32, _vp, _vp, _vp]),
    ("pto_bake_frames", _i32, [_vp, _i64, _vp, _i64, _vp, _vp]),
    ("pto_bake_compose_tangent", _i32, [_vp, _i64, _vp, _vp, _i64, _vp, _vp, _i64, _vp, _vp, _i32, _vp, _vp]),
    ("pto_bake_height", _i32, [_vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _i32, _i32, _vp]),
    ("pto_bake_height_encode", _i64, [_vp, _i64, _vp, _vp, _vp]),
    ("pto_bake_height_pad", _i32, [_vp, _vp, _i32, _vp]),
])


# ---- texels and the object-space maps ------------------------------------------------------------
def bake_samples(vertices, faces, resolution):
    """Per-texel bake, texel stage: (texel ids uint32 [m], positions float64 [m,3], owner faces
    int32 [m]) of the covered texels in ascending texel order."""
    vertices = pto._chk_points(vertices)
    faces = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    n = resolution * resolution
    texels, xyz, owner = np.empty(n, np.uint32), np.empty((n, 3), np.float64), np.empty(n, np.int32)
    m = pto.lib().pto_bake_texels(pto._ptr(vertices), vertices.shape[0], pto._ptr(faces), faces.shape[0],
                                  resolution, pto._ptr(texels), pto._ptr(xyz), pto._ptr(owner))
    assert m >= 0, m
    return texels[:m].copy(), xyz[:m].copy(), owner[:m].copy()


def bake_texels(vertices, faces, resolution):
    """bake_samples without the owner faces: (texel ids uint32 [m], positions float64 [m,3])."""
    texels, xyz, _ = bake_samples(vertices, faces, resolution)
    return texels, xyz


def bake_encode(n):
    """The normal-map byte of one fp32 normal component."""
    return pto.lib().pto_bake_encode(float(n))


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
    rc = pto.lib().pto_bake_compose(pto._ptr(texels), texels.shape[0], pto._ptr(rgba), pto._ptr(normal),
                                    resolution, pto._ptr(bgra), pto._ptr(nbgra), pto._ptr(nf))
    assert rc == 0, rc
    if pad:
        bgra, nbgra = pto.texture_pad(bgra), pto.texture_pad(nbgra)
    return bgra, nbgra, nf


def neighbours(points, xyz, k, radius=-1.0):
    """The bake's exact k-NN of the sample positions (lowest index on ties); a position with a NaN
    coordinate gets an empty list, as the device query kernels answer NaN rows."""
    idx, d2 = pto.KdTree(points).knn(pto.make_points(xyz), k, radius=radius, exact_ties=True)
    nan_rows = np.isnan(xyz).any(axis=1)
    idx[nan_rows], d2[nan_rows] = -1, np.inf
    return idx, d2


def bake(points, vertices, faces, k, resolution, radius=-1.0, pad=True):
    """The whole per-texel bake on the CPU: texels, neighbours() + pto.blend, composition.  Returns
    (bgra, normal_bgra, normal, (texels, empty))."""
    texels, xyz = bake_texels(vertices, faces, resolution)
    idx, d2 = neighbours(points, xyz, k, radius)
    rgba, nrm = pto.blend(points, idx, d2)
    bgra, nbgra, nf = bake_compose(texels, rgba, nrm, resolution, pad=pad)
    return bgra, nbgra, nf, (int(texels.shape[0]), int((idx[:, 0] < 0).sum()))


# ---- tangent-space bake -------------------------------------------------------------------------
def bake_frames(vertices, faces):
    """Tangent-space bake, vertex frames: (frames float64 [n,8] = N xyz, T xyz, w, 0, tangents
    float32 [n,4] = T xyz, w), zero for a vertex without a frame."""
    vertices = pto._chk_points(vertices)
    faces = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    n = vertices.shape[0]
    frames, tangents = np.empty((n, 8), np.float64), np.empty((n, 4), np.float32)
    rc = pto.lib().pto_bake_frames(pto._ptr(vertices), n, pto._ptr(faces), faces.shape[0], pto._ptr(frames),
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
    rc = pto.lib().pto_bake_compose_tangent(pto._ptr(vertices), vertices.shape[0], pto._ptr(frames), pto._ptr(faces),
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
    idx, d2 = neighbours(points, xyz, k, radius)
    rgba, nrm = pto.blend(points, idx, d2)
    bgra, nbgra, nf = bake_compose(texels, rgba, nrm, resolution, pad=pad)
    frames, tangents = bake_frames(vertices, faces)
    tb, tn = bake_compose_tangent(vertices, frames, faces, texels, owner, rgba, nrm, resolution, pad=pad)
    return {"bgra": bgra, "normal_bgra": nbgra, "normal": nf, "tangent_bgra": tb, "tangent_normal": tn,
            "tangents": tangents, "frames": frames, "texels": int(texels.shape[0]),
            "empty": int((idx[:, 0] < 0).sum()), "m": nrm, "rgba": rgba, "samples": (texels, owner)}


# ---- height bake --------------------------------------------------------------------------------
def bake_height(vertices, frames, faces, texels, sample_faces, xyz, points, idx, d2, resolution):
    """Height bake steps 1-4: the float height map [res,res], NaN (0x7fc00000) without a value."""
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
    rc = pto.lib().pto_bake_height(pto._ptr(vertices), vertices.shape[0], pto._ptr(frames), pto._ptr(faces),
                                   faces.shape[0], pto._ptr(texels), pto._ptr(sample_faces), pto._ptr(xyz), m,
                                   pto._ptr(points), points.shape[0], pto._ptr(idx), pto._ptr(d2), k, resolution,
                                   pto._ptr(h))
    assert rc == 0, rc
    return h


def bake_height_encode(height, height_range=None):
    """(unpadded codes uint16 [res,res], range used (lo, hi), texels with a value)."""
    height = np.ascontiguousarray(height, dtype=np.float32)
    codes = np.empty(height.shape, np.uint16)
    used = np.empty(2, np.float64)
    rin = None if height_range is None else np.ascontiguousarray(height_range, dtype=np.float64)
    valued = pto.lib().pto_bake_height_encode(pto._ptr(height), height.size, None if rin is None else pto._ptr(rin),
                                              pto._ptr(codes), pto._ptr(used))
    return codes, (float(used[0]), float(used[1])), int(valued)


def bake_height_pad(height, codes):
    """The 16-bit padding of the codes."""
    height = np.ascontiguousarray(height, dtype=np.float32)
    codes = np.ascontiguousarray(codes, dtype=np.uint16)
    res = height.shape[0]
    out = np.empty_like(codes)
    assert pto.lib().pto_bake_height_pad(pto._ptr(height), pto._ptr(codes), res, pto._ptr(out)) == 0
    return out


def bake_heights(points, vertices, faces, k, resolution, radius=-1.0, pad_codes=True, height_range=None):
    """The whole height bake on the CPU.  Returns a dict: height, height_u16, height_range, texels
    (with a value), samples (texels, faces, positions), lists (idx, d2), frames."""
    texels, xyz, owner = bake_samples(vertices, faces, resolution)
    frames, _ = bake_frames(vertices, faces)
    idx, d2 = neighbours(points, xyz, k, radius)
    h = bake_height(vertices, frames, faces, texels, owner, xyz, points, idx, d2, resolution)
    codes, used, valued = bake_height_encode(h, height_range)
    if pad_codes:
        codes = bake_height_pad(h, codes)
    return {"height": h, "height_u16": codes, "height_range": used, "texels": valued,
            "samples": (texels, owner, xyz), "lists": (idx, d2), "frames": frames}
