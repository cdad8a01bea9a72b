"""Normal estimation on a sharded cloud (pt_sharded_estimate_normals, ShardedTree.estimate_normals):
normal and variation equal, bit for bit, Tree.estimate_normals on one index of the same cloud, and so
does stats.estimated.  Devices may repeat in the device list, so one GPU runs 1-4 slabs on device 0;
with >= 2 GPUs the slabs also sit on different devices.  With store, later sharded transfers and
bakes equal the single index's after its own store, also once the slabs have been rebuilt."""
import glob
import os

import numpy as np
import pytest

from oracle import pto_normals
from test_bake import grid_mesh
from test_bake_tangent import ALL_OUTPUTS

pytestmark = pytest.mark.gpu

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "*.npz")))
INVALID_ARG = 1                                        # PT_ERR_INVALID_ARG
KS = (3, 8, 16, 20, 32)
VIEW = (0.3, -2.0, 5.0)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def assert_same(got, ref, what=""):
    assert np.array_equal(got["normal"].view(np.uint32), ref["normal"].view(np.uint32)), what
    assert np.array_equal(got["variation"].view(np.uint32), ref["variation"].view(np.uint32)), what
    assert got["stats"]["estimated"] == ref["stats"]["estimated"], what


def compare(pkg, P, devices, calls, coord_mode=0, halo=0.0, k_hint=20):
    """Tree.estimate_normals and ShardedTree.estimate_normals for every (k, radius, viewpoint) of
    calls; returns the sharded info."""
    with pkg.Tree(P, coord_mode=coord_mode) as tree:
        refs = [tree.estimate_normals(k, radius=radius, viewpoint=view) for k, radius, view in calls]
    with pkg.ShardedTree(P, devices, halo=halo, k_hint=k_hint, coord_mode=coord_mode) as st:
        for (k, radius, view), ref in zip(calls, refs):
            got = st.estimate_normals(k, radius=radius, viewpoint=view)
            assert_same(got, ref, (devices, k, radius, view))
        return st.info()


def every_call(radius):
    return [(k, r, v) for k in KS for r in (None, radius) for v in (None, VIEW)]


def cloud(pkg, kind, n=40_000, seed=5):
    P = pkg.synth.cloud_host(n, seed=seed, side=30.0)
    if kind == "none":
        P["normal"] = 0.0
    elif kind == "half":
        P["normal"][::2] = 0.0
    return P


@pytest.mark.parametrize("n_slabs", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["normals", "none", "half"])
def test_equals_single_index(n_slabs, kind, pkg, torch_cuda):
    P = cloud(pkg, kind, seed=50 + n_slabs)
    info = compare(pkg, P, [0] * n_slabs, every_call(0.3))
    assert info["n_slabs"] == n_slabs
    assert sum(info["slab_points"]) == len(P)


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_golden_clouds(path, pkg, torch_cuda):
    """Ties, lattice points on the cuts, duplicates, collinear and coplanar clouds, k > n."""
    g = np.load(path)
    f64 = "f64" in os.path.basename(path)
    mode = pkg.COORD_F64 if f64 else pkg.COORD_AUTO
    P = pkg.make_points(g["xyz"], normal=g["normal"], color=g["color"])
    zero = pkg.make_points(g["xyz"], color=g["color"])
    calls = every_call(float(g["radius"]))
    for devices in ([0, 0], [0, 0, 0]):
        for c in (P, zero):
            compare(pkg, c, devices, calls, coord_mode=mode)


def test_cut_on_lattice_points(pkg, torch_cuda):
    """A lattice: the cuts are sampled x values, so whole columns of points sit exactly on them."""
    x, y, z = np.meshgrid(np.arange(40.0), np.arange(30.0), np.arange(3.0) * 0.5, indexing="ij")
    xyz = np.c_[x.ravel(), y.ravel(), z.ravel()]
    P = pkg.make_points(xyz, color=np.full((len(xyz), 3), 7))
    compare(pkg, P, [0, 0, 0], [(k, None, None) for k in (8, 20)] + [(16, 1.2, VIEW)])


def test_fp64_and_mixed_storage(pkg, torch_cuda):
    rng = np.random.default_rng(12)
    P = pkg.synth.cloud_host(60_000, seed=12, side=30.0)
    calls = [(8, None, None), (16, 0.3, VIEW), (32, None, None)]
    # not fp32-exact anywhere: fp64 storage everywhere
    P64 = pkg.make_points(P["ver"] + 1e-9 * rng.random(P["ver"].shape), normal=P["normal"], color=P["color"])
    compare(pkg, P64, [0, 0, 0], calls, coord_mode=pkg.COORD_F64)
    compare(pkg, P64, [0, 0], calls)
    # fp32-exact on the left half only: the single index and the right slabs store fp64, the left fp32
    mixed = P["ver"].astype(np.float32).astype(np.float64)
    right = mixed[:, 0] > 15.0
    mixed[right] += 1e-9 * rng.random((int(right.sum()), 3))
    Pm = pkg.make_points(mixed, normal=P["normal"], color=P["color"])
    compare(pkg, Pm, [0, 0, 0, 0], calls)


def test_narrow_halo_rebuilds(pkg, torch_cuda):
    P = cloud(pkg, "half", 60_000, seed=21)
    info = compare(pkg, P, [0, 0, 0], [(16, None, None), (20, 0.3, VIEW)], halo=1e-4)
    assert info["rebuilds"] > 0 and info["halo"] > 1e-4


def test_two_chunks_per_slab(pkg, torch_cuda):
    """2 slabs of 4.5 M points each: every slab self-queries its own points in two chunks of 2^22."""
    n = 9_000_000
    pos, attrs = pkg.synth.cloud_device(n, seed=20261018 + 7, u1=600.0, v1=600.0)
    P = pkg.synth.points_to_host(pos, attrs)
    del pos, attrs
    info = compare(pkg, P, [0, 0], [(8, None, None)])
    assert min(info["slab_points"]) > 1 << 22


def test_cloud_smaller_than_k(pkg, torch_cuda):
    rng = np.random.default_rng(24)
    P = pkg.make_points(rng.random((12, 3)) * 30.0, normal=rng.standard_normal((12, 3)),
                        color=rng.integers(0, 256, (12, 3)))
    for devices in ([0, 0], [0, 0, 0]):
        info = compare(pkg, P, devices, [(20, None, None), (32, None, VIEW), (16, 8.0, None)])
        assert info["n_slabs"] == len(devices)


def test_equals_oracle(pkg, pto, torch_cuda):
    """Against the CPU oracle on a seeded sample of points, independent of Tree."""
    P = cloud(pkg, "half", 40_000, seed=31)
    rows = np.sort(np.random.default_rng(31).choice(len(P), 2_000, replace=False))
    with pkg.ShardedTree(P, [0, 0, 0]) as st:
        for k, view in ((12, None), (20, VIEW)):
            got = st.estimate_normals(k, viewpoint=view)
            ref_n, ref_v, _ = pto_normals.estimate_normals(P["ver"], P["normal"], k, viewpoint=view, rows=rows)
            assert np.array_equal(got["normal"][rows].view(np.uint32), ref_n.view(np.uint32)), k
            assert np.array_equal(got["variation"][rows].view(np.uint32), ref_v.view(np.uint32)), k


def test_store_feeds_sharded_transfer_and_bake(pkg, torch_cuda):
    side = 30.0
    P = pkg.synth.cloud_host(60_000, seed=9, side=side)
    P["normal"][::2] = 0.0                                     # half the cloud arrives without normals
    P["ver"][:5] = P["ver"][5]                                  # a duplicates-only neighbourhood at k = 3
    V, F = grid_mesh(pkg, 12, side)
    q = pkg.make_points(V["ver"] + 0.01)
    # one sample far above slab 0: its ball reaches every slab, so the transfer widens the halo
    far = pkg.make_points(np.r_[V["ver"] + 0.01, [[2.0, 15.0, 200.0]]])
    want = ALL_OUTPUTS + ("height",)
    for k in (3, 16):
        with pkg.Tree(P) as tree:
            before = tree.transfer(q, 8)
            est = tree.estimate_normals(k, store=True)
            ref_t = tree.transfer(q, 8)
            ref_far = tree.transfer(far, 8)
            ref_b = tree.bake(V, F, k=16, resolution=200, want=want)
            again = tree.estimate_normals(k)                       # rule (a) now reads the stored normals
        with pkg.ShardedTree(P, [0, 0, 0]) as st:
            got = st.estimate_normals(k, store=False)
            assert_same(got, est)
            t = st.transfer(q, 8)
            for key in ("rgba", "normal", "idx"):
                assert t[key].tobytes() == before[key].tobytes(), key
            got = st.estimate_normals(k, store=True)
            assert_same(got, est)
            r0 = st.info()["rebuilds"]
            t = st.transfer(q, 8)
            for key in ("rgba", "normal", "idx"):
                assert t[key].tobytes() == ref_t[key].tobytes(), key
            b = st.bake(V, F, k=16, resolution=200, want=want)
            for key in want:
                assert b[key].tobytes() == ref_b[key].tobytes(), key
            assert_same(st.estimate_normals(k), again)
            # rebuilt slabs take their records from the caller's points: the stored normals must
            # reach them too
            t = st.transfer(far, 8)
            assert st.info()["rebuilds"] > r0
            for key in ("rgba", "normal", "idx"):
                assert t[key].tobytes() == ref_far[key].tobytes(), key
            b = st.bake(V, F, k=16, resolution=200, want=want)
            for key in want:
                assert b[key].tobytes() == ref_b[key].tobytes(), key
            assert_same(st.estimate_normals(k), again)


def empty_slab_clouds(pkg):
    """Clouds whose sampled cuts leave slabs without a point: a planar scan at one x on 3 slabs (all
    cuts at that x), and a lattice of 2 x columns on 4 slabs."""
    rng = np.random.default_rng(44)
    yz = rng.random((3_000, 2)) * 20.0
    plane = np.c_[np.full(len(yz), 7.25), yz]
    x, y, z = np.meshgrid(np.arange(2.0), np.arange(40.0), np.arange(30.0) * 0.5, indexing="ij")
    lattice = np.c_[x.ravel(), y.ravel(), z.ravel()]
    for xyz, devices in ((plane, [0, 0, 0]), (lattice, [0, 0, 0, 0])):
        normal = rng.standard_normal(xyz.shape)
        normal[::2] = 0.0
        yield pkg.make_points(xyz, normal=normal, color=rng.integers(0, 256, xyz.shape)), devices


def test_store_with_empty_slabs(pkg, torch_cuda):
    for P, devices in empty_slab_clouds(pkg):
        q = pkg.make_points(P["ver"][::7] + 0.01)
        with pkg.Tree(P) as tree:
            est = tree.estimate_normals(12, store=True)
            ref_t = tree.transfer(q, 8)
            again = tree.estimate_normals(12)
        with pkg.ShardedTree(P, devices) as st:
            assert 0 in st.info()["slab_points"]
            assert_same(st.estimate_normals(12, store=True), est)
            t = st.transfer(q, 8)
            for key in ("rgba", "normal", "idx"):
                assert t[key].tobytes() == ref_t[key].tobytes(), key
            assert_same(st.estimate_normals(12), again)


def test_error_codes(pkg, torch_cuda):
    P = pkg.synth.cloud_host(2_000, seed=1, side=10.0)
    L, ptr = pkg.lib(), pkg.api._np_ptr
    n = len(P)
    nrm, var = np.empty((n, 3), np.float32), np.empty(n, np.float32)
    bad_view = np.array([0.0, np.inf, 1.0])
    good_view = np.array([0.0, 1.0, 2.0])
    cases = [(2, None, 0, True), (1, None, 0, True), (33, None, 0, True), (8, bad_view, 0, True),
             (33, bad_view, 0, True), (8, None, 0, False), (8, good_view, 0, True), (8, None, 1, False)]

    def codes(fn, h):
        return [fn(h, k, -1.0, None if v is None else ptr(v), store, ptr(nrm) if out else None,
                   ptr(var) if out else None, None) for k, v, store, out in cases]
    with pkg.Tree(P) as tree:
        ref = codes(L.pt_index_estimate_normals, tree.handle)
    with pkg.ShardedTree(P, [0, 0]) as st:
        got = codes(L.pt_sharded_estimate_normals, st._h)
    assert got == ref
    assert ref[:6] == [INVALID_ARG, INVALID_ARG, pkg.api.PT_ERR_UNSUPPORTED, INVALID_ARG, INVALID_ARG, INVALID_ARG]
    assert ref[6:] == [0, 0]
    assert L.pt_sharded_estimate_normals(None, 8, -1.0, None, 0, ptr(nrm), None, None) == INVALID_ARG


def test_distinct_devices(pkg, torch_cuda):
    if torch_cuda.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    P = cloud(pkg, "half", 60_000, seed=41)
    for devices in ([0, 1], [0, 1, 0, 1]):
        compare(pkg, P, devices, [(8, None, None), (16, 0.3, VIEW), (32, None, None)])
    info = compare(pkg, P, [1, 0], [(20, None, None)], halo=1e-4)
    assert info["rebuilds"] > 0
