"""Normal orientation on a sharded cloud (pt_sharded_orient_normals, ShardedTree.orient_normals):
normal (bit for bit), root and the counts oriented, flipped, components and edges equal
Tree.orient_normals on one index of the same cloud.  Devices may repeat in the device list, so one GPU
runs 1-4 slabs on device 0; with >= 2 GPUs the slabs also sit on different devices.  With store,
later sharded transfers and bakes equal the single index's after its own store, also once the slabs
have been rebuilt."""
import glob
import os

import numpy as np
import pytest

from oracle import pto_normals, pto_orient
from test_bake import grid_mesh
from test_bake_tangent import ALL_OUTPUTS
from test_orient import TIE_CLOUDS, expected_roots, scramble, sphere, torus

pytestmark = pytest.mark.gpu

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "*.npz")))
INVALID_ARG, UNSUPPORTED = 1, 5
KS = (2, 3, 8, 18, 32)
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
    assert np.array_equal(got["root"], ref["root"]), what
    for key in ("oriented", "flipped", "components", "edges"):
        assert got["stats"][key] == ref["stats"][key], (key, what)


def compare(pkg, P, devices, calls, coord_mode=0, halo=0.0, k_hint=20):
    """Tree.orient_normals and ShardedTree.orient_normals for every (k, radius, viewpoint) of calls;
    returns the single index's results and the sharded info."""
    with pkg.Tree(P, coord_mode=coord_mode) as tree:
        refs = [tree.orient_normals(k, radius=radius, viewpoint=view) for k, radius, view in calls]
    with pkg.ShardedTree(P, devices, halo=halo, k_hint=k_hint, coord_mode=coord_mode) as st:
        for (k, radius, view), ref in zip(calls, refs):
            got = st.orient_normals(k, radius=radius, viewpoint=view)
            assert_same(got, ref, (devices, k, radius, view))
        return refs, st.info()


def every_call(radius, ks=KS):
    return [(k, r, v) for k in ks for r in (None, radius) for v in (None, VIEW)]


def signed_cloud(pkg, n=40_000, seed=5, zero_every=0):
    """A synthetic scan with its analytic normals under seeded random signs."""
    P = pkg.synth.cloud_host(n, seed=seed, side=30.0)
    P["normal"] *= np.where(np.random.default_rng(seed).random(n) < 0.5, -1.0, 1.0)[:, None]
    if zero_every:
        P["normal"][::zero_every] = 0.0
    return P


@pytest.mark.parametrize("n_slabs", [1, 2, 3, 4])
def test_equals_single_index(n_slabs, pkg, torch_cuda):
    P = signed_cloud(pkg, seed=50 + n_slabs, zero_every=7)
    refs, info = compare(pkg, P, [0] * n_slabs, every_call(0.3))
    assert info["n_slabs"] == n_slabs
    assert refs[2]["stats"]["components"] > 1                       # k = 2 and the radius split the graph


@pytest.mark.parametrize("shape", ["sphere", "torus", "two_spheres"])
def test_closed_surfaces_come_out_outward(shape, pkg, torch_cuda):
    rng = np.random.default_rng(2026)
    if shape == "sphere":
        xyz, d = sphere(20_000, rng)
        comp_of = np.zeros(20_000, int)
    elif shape == "torus":
        xyz, d = torus(30_000, rng)
        comp_of = np.zeros(30_000, int)
    else:
        a, da = sphere(20_000, rng)
        b, db = sphere(20_000, rng, centre=(5.0, 0.0, 0.5))
        xyz, d = np.r_[a, b], np.r_[da, db]
        comp_of = np.r_[np.zeros(20_000, int), np.ones(20_000, int)]
    P = pkg.make_points(xyz, normal=scramble(d, rng))
    for devices in ([0, 0], [0, 0, 0, 0]):
        refs, _ = compare(pkg, P, devices, [(18, None, None), (8, None, None)])
        got = refs[0]
        assert (np.einsum("ij,ij->i", got["normal"].astype(np.float64), d) > 0).all()
        assert np.array_equal(got["root"], expected_roots(xyz, comp_of))


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_golden_clouds(path, pkg, torch_cuda):
    """Ties, lattice points on the cuts, duplicates, collinear and coplanar clouds, k > n."""
    g = np.load(path)
    mode = pkg.COORD_F64 if "f64" in os.path.basename(path) else pkg.COORD_AUTO
    rng = np.random.default_rng(1)
    flipped = g["normal"] * np.where(rng.random(len(g["xyz"])) < 0.5, -1.0, 1.0)[:, None]
    P = pkg.make_points(g["xyz"], normal=flipped, color=g["color"])
    for devices in ([0, 0], [0, 0, 0]):
        compare(pkg, P, devices, every_call(float(g["radius"])), coord_mode=mode)


@pytest.mark.parametrize("name", sorted(TIE_CLOUDS))
def test_tie_clouds(name, pkg, torch_cuda):
    """All-zero weights with ids in lattice order and shuffled, a plateau of top-z ties with -0 / +0,
    frustrated triangles: the cuts run through them, so (lo, hi) decides between slabs."""
    xyz, m, radius = TIE_CLOUDS[name]()
    P = pkg.make_points(xyz, normal=m)
    calls = [(k, radius, None) for k in (2, 8, 32)] + [(18, radius, VIEW)]
    for devices in ([0, 0], [0, 0, 0, 0]):
        compare(pkg, P, devices, calls)


def test_filter_drops_a_cycle_through_another_slab(pkg, torch_cuda):
    """A ring of points around x = 0 on 2 slabs: the heaviest edge of the ring lies inside slab 1,
    and the ring closes through slab 0.  Slab 1's own forest keeps it (it is a bridge there); the
    whole cloud's forest must not."""
    t = np.linspace(0.0, 2 * np.pi, 64, endpoint=False)
    xyz = np.c_[np.cos(t) * 10.0, np.sin(t) * 10.0, np.zeros_like(t)]
    nrm = np.c_[np.zeros_like(t), np.zeros_like(t), np.ones_like(t)]
    heavy = int(np.argmin(np.abs(t - np.pi / 2)))                # top of the ring, x ~ 0: move it into slab 1
    xyz[heavy, 0] = 0.5
    nrm[heavy] = (0.0, 0.6, -0.8)                               # its two ring edges are the heaviest
    nrm[heavy + 1] = (0.0, 0.4, -0.9)
    P = pkg.make_points(xyz, normal=nrm.astype(np.float32))
    refs, info = compare(pkg, P, [0, 0], [(3, None, None), (3, 2.0, None), (3, None, VIEW)])
    assert info["slab_points"][0] > 0 and info["slab_points"][1] > 0
    assert refs[0]["stats"]["components"] == 1


def test_cut_on_lattice_points(pkg, torch_cuda):
    x, y, z = np.meshgrid(np.arange(40.0), np.arange(30.0), np.arange(3.0) * 0.5, indexing="ij")
    xyz = np.c_[x.ravel(), y.ravel(), z.ravel()]
    rng = np.random.default_rng(3)
    nrm = rng.standard_normal(xyz.shape)
    compare(pkg, pkg.make_points(xyz, normal=nrm), [0, 0, 0], [(k, None, None) for k in (8, 18)] + [(18, 1.2, VIEW)])


def test_fp64_and_mixed_storage(pkg, torch_cuda):
    rng = np.random.default_rng(12)
    P = signed_cloud(pkg, 60_000, seed=12)
    calls = [(8, None, None), (18, 0.3, VIEW), (32, None, None)]
    P64 = pkg.make_points(P["ver"] + 1e-9 * rng.random(P["ver"].shape), normal=P["normal"], color=P["color"])
    compare(pkg, P64, [0, 0, 0], calls, coord_mode=pkg.COORD_F64)
    compare(pkg, P64, [0, 0], calls)
    mixed = P["ver"].astype(np.float32).astype(np.float64)
    right = mixed[:, 0] > 15.0
    mixed[right] += 1e-9 * rng.random((int(right.sum()), 3))
    compare(pkg, pkg.make_points(mixed, normal=P["normal"], color=P["color"]), [0, 0, 0, 0], calls)


def test_narrow_halo_rebuilds(pkg, torch_cuda):
    P = signed_cloud(pkg, 60_000, seed=21, zero_every=5)
    _, info = compare(pkg, P, [0, 0, 0], [(18, None, None), (32, 0.3, VIEW)], halo=1e-4)
    assert info["rebuilds"] > 0 and info["halo"] > 1e-4


def test_two_chunks_per_slab(pkg, torch_cuda):
    """2 slabs of 4.5 M points each: every slab self-queries its own points in two chunks of 2^22."""
    n = 9_000_000
    pos, attrs = pkg.synth.cloud_device(n, seed=20261018 + 7, u1=600.0, v1=600.0)
    P = pkg.synth.points_to_host(pos, attrs)
    del pos, attrs
    P["normal"] *= np.where(np.random.default_rng(8).random(n) < 0.5, -1.0, 1.0)[:, None]
    _, info = compare(pkg, P, [0, 0], [(18, None, None)])
    assert min(info["slab_points"]) > 1 << 22


def test_zero_normals_isolated_points_and_no_part(pkg, torch_cuda):
    rng = np.random.default_rng(3)
    xyz = np.r_[np.c_[rng.random((400, 2)) * 4.0, np.zeros(400)], [[50.0, 50.0, -3.0], [-40.0, 2.0, 1.0]]]
    m = np.r_[np.tile([[0.0, 0.0, -1.0]], (400, 1)), [[0.0, 0.0, -2.0], [0.0, 1.0, 0.0]]].astype(np.float32)
    m[17] = 0.0
    m[18] = np.nan
    m[200:210] = np.inf
    P = pkg.make_points(xyz, normal=m)
    refs, _ = compare(pkg, P, [0, 0, 0], [(2, 0.5, None), (8, 0.5, None), (8, None, VIEW)])
    assert (refs[0]["root"][[17, 18, 200]] == -1).all() and refs[0]["root"][400] == 400
    none = pkg.make_points(xyz)                                        # no point takes part
    refs, _ = compare(pkg, none, [0, 0], [(8, None, None)])
    assert refs[0]["stats"]["oriented"] == 0 and (refs[0]["root"] == -1).all()


def test_equals_oracle(pkg, pto, torch_cuda):
    """Against the CPU oracle on a seeded cloud, independent of Tree."""
    P = signed_cloud(pkg, 20_000, seed=31, zero_every=9)
    xyz = P["ver"]
    m = P["normal"].astype(np.float32)
    with pkg.ShardedTree(P, [0, 0, 0]) as st:
        for k, view in ((12, None), (18, VIEW)):
            got = st.orient_normals(k, viewpoint=view)
            ref = pto_orient.orient(xyz, m, pto_normals.neighbours(xyz, k), view)
            rows = np.sort(np.random.default_rng(k).choice(len(P), 2_000, replace=False))
            assert np.array_equal(got["normal"][rows].view(np.uint32), ref["normal"][rows].view(np.uint32)), k
            assert np.array_equal(got["root"], ref["root"]), k
            for key in ("oriented", "flipped", "components", "edges"):
                assert got["stats"][key] == ref[key], (key, k)


def test_store_feeds_sharded_transfer_and_bake(pkg, torch_cuda):
    """estimate (store) then orient (store) on the sharded cloud, then transfer and bake: the same
    bytes as the chain on one index, also after a rebuild that follows the store."""
    side = 30.0
    P = pkg.synth.cloud_host(60_000, seed=9, side=side)
    P["normal"][::2] = 0.0
    V, F = grid_mesh(pkg, 12, side)
    q = pkg.make_points(V["ver"] + 0.01)
    far = pkg.make_points(np.r_[V["ver"] + 0.01, [[2.0, 15.0, 200.0]]])
    want = ALL_OUTPUTS + ("height",)
    with pkg.Tree(P) as tree:
        tree.estimate_normals(16, store=True)
        ori = tree.orient_normals(18, store=True)
        ref_t = tree.transfer(q, 8)
        ref_far = tree.transfer(far, 8)
        ref_b = tree.bake(V, F, k=16, resolution=200, want=want)
        again = tree.orient_normals(18)
    assert ori["stats"]["flipped"] > 0
    with pkg.ShardedTree(P, [0, 0, 0]) as st:
        st.estimate_normals(16, store=True)
        assert_same(st.orient_normals(18, store=True), ori)
        r0 = st.info()["rebuilds"]
        t = st.transfer(q, 8)
        for key in ("rgba", "normal", "idx"):
            assert t[key].tobytes() == ref_t[key].tobytes(), key
        b = st.bake(V, F, k=16, resolution=200, want=want)
        for key in want:
            assert b[key].tobytes() == ref_b[key].tobytes(), key
        assert_same(st.orient_normals(18), again)
        t = st.transfer(far, 8)                                    # widens the halo: rebuilt slabs
        assert st.info()["rebuilds"] > r0
        for key in ("rgba", "normal", "idx"):
            assert t[key].tobytes() == ref_far[key].tobytes(), key
        b = st.bake(V, F, k=16, resolution=200, want=want)
        for key in want:
            assert b[key].tobytes() == ref_b[key].tobytes(), key
        assert_same(st.orient_normals(18), again)


def test_empty_slabs(pkg, torch_cuda):
    """A planar scan at one x on 3 slabs (all cuts at that x) and a lattice of 2 x columns on 4."""
    rng = np.random.default_rng(44)
    yz = rng.random((3_000, 2)) * 20.0
    plane = np.c_[np.full(len(yz), 7.25), yz]
    x, y, z = np.meshgrid(np.arange(2.0), np.arange(40.0), np.arange(30.0) * 0.5, indexing="ij")
    lattice = np.c_[x.ravel(), y.ravel(), z.ravel()]
    for xyz, devices in ((plane, [0, 0, 0]), (lattice, [0, 0, 0, 0])):
        normal = rng.standard_normal(xyz.shape)
        normal[::5] = 0.0
        P = pkg.make_points(xyz, normal=normal, color=rng.integers(0, 256, xyz.shape))
        q = pkg.make_points(xyz[::7] + 0.01)
        with pkg.Tree(P) as tree:
            ori = tree.orient_normals(12, store=True)
            ref_t = tree.transfer(q, 8)
        with pkg.ShardedTree(P, devices) as st:
            assert 0 in st.info()["slab_points"]
            assert_same(st.orient_normals(12, store=True), ori)
            t = st.transfer(q, 8)
            for key in ("rgba", "normal", "idx"):
                assert t[key].tobytes() == ref_t[key].tobytes(), key


def test_error_codes(pkg, torch_cuda):
    P = pkg.synth.cloud_host(2_000, seed=1, side=10.0)
    L, ptr = pkg.lib(), pkg.api._np_ptr
    n = len(P)
    nrm, root = np.empty((n, 3), np.float32), np.empty(n, np.int32)
    bad_view = np.array([0.0, np.inf, 1.0])
    good_view = np.array([0.0, 1.0, 2.0])
    cases = [(1, None, 0, True), (0, None, 0, True), (33, None, 0, True), (8, bad_view, 0, True),
             (33, bad_view, 0, True), (8, None, 0, False), (2, None, 0, True), (8, good_view, 0, True),
             (8, None, 1, False)]

    def codes(fn, h):
        return [fn(h, k, -1.0, None if v is None else ptr(v), store, ptr(nrm) if out else None,
                   ptr(root) if out else None, None) for k, v, store, out in cases]
    with pkg.Tree(P) as tree:
        ref = codes(L.pt_index_orient_normals, tree.handle)
    with pkg.ShardedTree(P, [0, 0]) as st:
        got = codes(L.pt_sharded_orient_normals, st._h)
    assert got == ref
    assert ref == [INVALID_ARG, INVALID_ARG, UNSUPPORTED, INVALID_ARG, INVALID_ARG, INVALID_ARG, 0, 0, 0]
    assert L.pt_sharded_orient_normals(None, 8, -1.0, None, 0, ptr(nrm), None, None) == INVALID_ARG


def test_distinct_devices(pkg, torch_cuda):
    if torch_cuda.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    P = signed_cloud(pkg, 60_000, seed=41, zero_every=6)
    for devices in ([0, 1], [0, 1, 0, 1], [1, 0]):
        compare(pkg, P, devices, [(8, None, None), (18, 0.3, VIEW), (32, None, None)])
    _, info = compare(pkg, P, [1, 0], [(18, None, None)], halo=1e-4)
    assert info["rebuilds"] > 0
