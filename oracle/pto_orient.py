"""ctypes binding of the normal-orientation oracle (oracle/pt_orient_oracle.c).

TEST INFRASTRUCTURE ONLY, like oracle/pto.py, whose library holds it.  The neighbour lists come from
pto_normals.neighbours, the exact k-NN self-query the estimation oracle uses.
"""
import ctypes

import numpy as np

from . import pto, pto_normals

_vp, _i64 = ctypes.c_void_p, ctypes.c_int64
pto.bind([("pto_orient_normals", ctypes.c_int, [_vp, _vp, _i64, _vp, ctypes.c_int, _vp, _vp, _vp, _vp, _vp])])


def orient(xyz, normal, idx, viewpoint=None):
    """The definition on given neighbour lists.  xyz float64 [n,3] (the stored positions), normal
    [n,3] (rounded to float32 as the index stores them), idx int32 [n,k] (point i's list).  Returns a
    dict: ``normal`` float32 [n,3], ``root`` int32 [n], ``parent`` int32 [n] (the forest, -1 at roots
    and at points that do not take part) and the counts ``oriented``, ``flipped``, ``components``,
    ``edges``."""
    xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
    nrm = np.ascontiguousarray(normal, dtype=np.float32).reshape(-1, 3)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    n, k = idx.shape
    assert nrm.shape == xyz.shape and n == xyz.shape[0]
    view = None if viewpoint is None else np.ascontiguousarray(viewpoint, dtype=np.float64).reshape(3)
    out = {"normal": np.empty((n, 3), np.float32), "root": np.empty(n, np.int32), "parent": np.empty(n, np.int32)}
    counts = np.zeros(4, np.int64)
    rc = pto.lib().pto_orient_normals(pto._ptr(xyz), pto._ptr(nrm), n, pto._ptr(idx), k,
                                      None if view is None else pto._ptr(view), pto._ptr(out["normal"]),
                                      pto._ptr(out["root"]), pto._ptr(out["parent"]), pto._ptr(counts))
    assert rc == 0, rc
    out.update(zip(("oriented", "flipped", "components", "edges"), map(int, counts)))
    return out


def orient_normals(xyz, normal, k, radius=-1.0, viewpoint=None):
    """pto_normals.neighbours() + orient()."""
    return orient(xyz, normal, pto_normals.neighbours(xyz, k, radius), viewpoint)
