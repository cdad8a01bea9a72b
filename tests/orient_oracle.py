"""ctypes binding of the normal-orientation oracle (tests/orient_oracle.c).

TEST INFRASTRUCTURE ONLY.  The C file is compiled on first use with -ffp-contract=off (no FMA) into a
per-user temporary directory, so the source tree is never written to.  The neighbour lists come from
oracle.pto_normals.neighbours, the exact k-NN self-query the estimation oracle uses.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from oracle import pto, pto_normals

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "orient_oracle.c")
_CFLAGS = ["-O2", "-std=c11", "-fPIC", "-ffp-contract=off", "-Wall", "-Wextra"]
_lib_handle = None


def build():
    """Compile orient_oracle.c (gcc) unless an up-to-date library exists; returns its path."""
    d = os.path.join(tempfile.gettempdir(), f"pt_orient_oracle_{os.getuid()}")
    path = os.path.join(d, "liborient_oracle.so")
    if os.path.exists(path) and os.path.getmtime(path) >= os.path.getmtime(_SRC):
        return path
    os.makedirs(d, exist_ok=True)
    tmp = f"{path}.{os.getpid()}.tmp"
    subprocess.run(["/usr/bin/gcc", *_CFLAGS, "-shared", "-o", tmp, _SRC, "-lm"], check=True)
    os.replace(tmp, path)
    return path


def _lib():
    global _lib_handle
    if _lib_handle is None:
        L = ctypes.CDLL(build())
        vp, i64 = ctypes.c_void_p, ctypes.c_int64
        L.pto_orient_normals.restype = ctypes.c_int
        L.pto_orient_normals.argtypes = [vp, vp, i64, vp, ctypes.c_int, vp, vp, vp, vp, vp]
        _lib_handle = L
    return _lib_handle


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
    rc = _lib().pto_orient_normals(pto._ptr(xyz), pto._ptr(nrm), n, pto._ptr(idx), k,
                                   None if view is None else pto._ptr(view), pto._ptr(out["normal"]),
                                   pto._ptr(out["root"]), pto._ptr(out["parent"]), pto._ptr(counts))
    assert rc == 0, rc
    out.update(zip(("oriented", "flipped", "components", "edges"), map(int, counts)))
    return out


def orient_normals(xyz, normal, k, radius=-1.0, viewpoint=None):
    """pto_normals.neighbours() + orient()."""
    return orient(xyz, normal, pto_normals.neighbours(xyz, k, radius), viewpoint)
