"""ctypes binding of the normal-estimation oracle (oracle/pt_normals_oracle.c).

TEST INFRASTRUCTURE ONLY, like oracle/pto.py, whose library holds it and whose exact k-NN it uses
for the neighbour lists.
"""
import ctypes

import numpy as np

from . import pto

_vp, _i64 = ctypes.c_void_p, ctypes.c_int64
pto.bind([("pto_estimate_normals", _i64, [_vp, _vp, _i64, _vp, _i64, _vp, ctypes.c_int, _vp, _vp, _vp, _vp])])


def estimate(xyz, normal, idx, viewpoint=None, rows=None, fp64=False):
    """The definition on given neighbour lists.  xyz float64 [n,3] (the cloud), normal [n,3] (the
    input normals, rounded to float32 as the index stores them) or None, idx int32 [m,k] (the list of
    point rows[r], or of point r when rows is None).  Returns (normal float32 [m,3], variation
    float32 [m], number estimated), and with ``fp64`` also the values before the rounding to fp32
    (float64 [m,4]: n xyz, variation)."""
    xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
    nrm = None if normal is None else np.ascontiguousarray(normal, dtype=np.float32).reshape(-1, 3)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    m, k = idx.shape
    rws = None if rows is None else np.ascontiguousarray(rows, dtype=np.int32)
    assert rws is None or rws.shape == (m,)
    assert nrm is None or nrm.shape == xyz.shape
    view = None if viewpoint is None else np.ascontiguousarray(viewpoint, dtype=np.float64).reshape(3)
    out_n, out_v = np.empty((m, 3), np.float32), np.empty(m, np.float32)
    out64 = np.empty((m, 4), np.float64) if fp64 else None
    est = pto.lib().pto_estimate_normals(pto._ptr(xyz), None if nrm is None else pto._ptr(nrm), xyz.shape[0],
                                         None if rws is None else pto._ptr(rws), m, pto._ptr(idx), k,
                                         None if view is None else pto._ptr(view), pto._ptr(out_n), pto._ptr(out_v),
                                         None if out64 is None else pto._ptr(out64))
    assert est >= 0, est
    return (out_n, out_v, int(est)) + ((out64,) if fp64 else ())


def neighbours(xyz, k, radius=-1.0, rows=None, nthreads=0):
    """The exact k-NN self-query lists (ascending (d2, id), -1 padded) of every point, or of the
    points ``rows``."""
    xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
    q = xyz if rows is None else xyz[np.asarray(rows)]
    idx, _ = pto.KdTree(pto.make_points(xyz)).knn(pto.make_points(q), k, radius=radius, exact_ties=True,
                                                  nthreads=nthreads, want_d2=False)
    return idx


def estimate_normals(xyz, normal, k, radius=-1.0, viewpoint=None, rows=None, nthreads=0):
    """neighbours() + estimate(): (normal, variation, number estimated)."""
    idx = neighbours(xyz, k, radius, rows, nthreads)
    return estimate(xyz, normal, idx, viewpoint, rows)
