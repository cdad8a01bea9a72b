"""The per-texel bake of a sharded cloud (pt_sharded_bake, ShardedTree.bake): every output equals,
byte for byte, Tree.bake on one index of the same cloud.  Devices may repeat in the device list, so
one GPU runs 1-4 slabs on device 0; the option "sharded_copy" makes slabs on the home device work on
copies of their rows, as slabs on another device do.  With >= 2 GPUs the slabs also sit on
different devices and the rows travel by peer copies."""
import ctypes

import numpy as np
import pytest

from oracle import pto_bake
from test_bake import grid_mesh, lattice_case
from test_bake_tangent import ALL_OUTPUTS, tilted_normals

pytestmark = pytest.mark.gpu

HEIGHTS = ("height", "height_u16")
INVALID_ARG = 1                                        # PT_ERR_INVALID_ARG
EVERYTHING = ALL_OUTPUTS + HEIGHTS


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def assert_same(got, ref):
    assert set(got) == set(ref)
    for key in ref:
        if key == "stats":
            for s in ("texels", "empty", "height_texels"):
                assert got["stats"].get(s) == ref["stats"].get(s), s
        elif key == "height_range":
            assert np.array(got[key]).tobytes() == np.array(ref[key]).tobytes()
        else:
            assert got[key].dtype == ref[key].dtype and got[key].shape == ref[key].shape, key
            assert got[key].tobytes() == ref[key].tobytes(), key


def compare(pkg, P, V, F, devices, coord_mode=0, halo=0.0, **kw):
    """Tree.bake and ShardedTree.bake of the same call; returns (result, sharded info)."""
    with pkg.Tree(P, coord_mode=coord_mode) as tree:
        ref = tree.bake(V, F, **kw)
    with pkg.ShardedTree(P, devices, halo=halo, k_hint=kw.get("k", 20), coord_mode=coord_mode) as st:
        got = st.bake(V, F, **kw)
        info = st.info()
    assert_same(got, ref)
    return got, info


def mesh_case(pkg, seed, side=30.0, g=20):
    V, F = grid_mesh(pkg, g, side)
    V["normal"] = tilted_normals(np.random.default_rng(seed), len(V))
    return V, F


@pytest.mark.parametrize("n_slabs,k,pad", [(1, 20, 1), (2, 1, 1), (2, 32, 0), (3, 8, 0), (3, 16, 1), (4, 20, 0),
                                           (4, 32, 1), (4, 1, 0)])
def test_all_outputs_equal_single_index(n_slabs, k, pad, pkg, torch_cuda):
    P = pkg.synth.cloud_host(90_000, seed=60 + k, side=30.0)
    V, F = mesh_case(pkg, k)
    got, info = compare(pkg, P, V, F, [0] * n_slabs, k=k, resolution=300, pad=bool(pad), want=EVERYTHING)
    assert info["n_slabs"] == n_slabs and info["rebuilds"] == 0
    assert got["stats"]["texels"] > 300 * 300 // 2 and got["stats"]["height_texels"] > 0


def test_copy_path_equals_single_index(pkg, torch_cuda):
    P = pkg.synth.cloud_host(90_000, seed=3, side=30.0)
    V, F = mesh_case(pkg, 3)
    pkg.set_option("sharded_copy", 1)
    try:
        for devices, k in (([0, 0, 0], 16), ([0], 20)):
            compare(pkg, P, V, F, devices, k=k, resolution=257, want=EVERYTHING)
        _, info = compare(pkg, P, V, F, [0, 0], halo=1e-4, k=8, resolution=200, want=EVERYTHING)
        assert info["rebuilds"] > 0
    finally:
        pkg.set_option("sharded_copy", 0)


def test_bounded_radius_and_height_ranges(pkg, torch_cuda):
    P, V, F, _ = lattice_case(pkg)
    V = V.copy()
    V["normal"] = tilted_normals(np.random.default_rng(5), len(V))
    got, _ = compare(pkg, P, V, F, [0, 0, 0], k=8, resolution=200, radius=0.2, pad=False, want=EVERYTHING)
    assert 0 < got["stats"]["empty"] < got["stats"]["texels"]
    P = pkg.synth.cloud_host(60_000, seed=8, side=30.0)
    V, F = mesh_case(pkg, 8)
    for height_range in (None, (-0.5, 0.5), (3.0, 3.0)):
        compare(pkg, P, V, F, [0, 0], k=16, resolution=256, want=HEIGHTS, height_range=height_range)


def test_fp64_clouds(pkg, torch_cuda):
    rng = np.random.default_rng(12)
    P = pkg.synth.cloud_host(60_000, seed=12, side=30.0)
    V, F = mesh_case(pkg, 12)
    # not fp32-exact anywhere: fp64 storage everywhere
    P64 = pkg.make_points(P["ver"] + 1e-9 * rng.random(P["ver"].shape), normal=P["normal"], color=P["color"])
    compare(pkg, P64, V, F, [0, 0, 0], coord_mode=pkg.COORD_F64, k=20, resolution=256, want=EVERYTHING)
    compare(pkg, P64, V, F, [0, 0], k=20, resolution=256, want=EVERYTHING)
    # fp32-exact on the left half only: the single index and the right slabs store fp64, the left fp32
    mixed = P["ver"].astype(np.float32).astype(np.float64)
    right = mixed[:, 0] > 15.0
    mixed[right] += 1e-9 * rng.random((int(right.sum()), 3))
    Pm = pkg.make_points(mixed, normal=P["normal"], color=P["color"])
    compare(pkg, Pm, V, F, [0, 0, 0, 0], k=16, resolution=256, want=EVERYTHING)


def test_narrow_halo_rebuilds(pkg, torch_cuda):
    P = pkg.synth.cloud_host(60_000, seed=21, side=30.0)
    V, F = mesh_case(pkg, 21)
    _, info = compare(pkg, P, V, F, [0, 0, 0], halo=1e-4, k=20, resolution=256, want=EVERYTHING)
    assert info["rebuilds"] > 0 and info["halo"] > 1e-4


def test_nan_vertices_do_not_rebuild(pkg, torch_cuda):
    P = pkg.synth.cloud_host(60_000, seed=22, side=30.0)
    V, F = mesh_case(pkg, 22)
    V["ver"][[30, 31, 200]] = np.nan                   # every component
    V["ver"][[100, 150, 300], 1] = np.nan              # y only: x still routes these samples somewhere
    got, info = compare(pkg, P, V, F, [0, 0, 0], k=16, resolution=256, want=EVERYTHING)
    assert info["rebuilds"] == 0
    assert 0 < got["stats"]["empty"] < got["stats"]["texels"]


def test_mesh_inside_one_slab(pkg, torch_cuda):
    P = pkg.synth.cloud_host(60_000, seed=23, side=30.0)
    V, F = mesh_case(pkg, 23)
    V["ver"][:, 0] = V["ver"][:, 0] * 0.1 + 1.0        # x in [1, 4]: the leftmost of 4 slabs (cuts near 7.5, 15, 22.5)
    compare(pkg, P, V, F, [0, 0, 0, 0], k=20, resolution=256, want=EVERYTHING)


def test_cloud_smaller_than_k(pkg, torch_cuda):
    rng = np.random.default_rng(24)
    P = pkg.make_points(rng.random((12, 3)) * 30.0, normal=rng.standard_normal((12, 3)),
                        color=rng.integers(0, 256, (12, 3)))
    V, F = mesh_case(pkg, 24, g=8)
    for devices in ([0, 0], [0, 0, 0]):
        got, _ = compare(pkg, P, V, F, devices, k=20, resolution=128, want=EVERYTHING)
        assert got["stats"]["empty"] == 0


def test_tangents_only(pkg, torch_cuda):
    P = pkg.synth.cloud_host(20_000, seed=25, side=30.0)
    V, F = mesh_case(pkg, 25)
    got, _ = compare(pkg, P, V, F, [0, 0], k=8, resolution=128, want=("tangents",))
    assert got["stats"]["texels"] == 0 and got["stats"]["empty"] == 0


def test_error_codes(pkg, torch_cuda):
    P = pkg.synth.cloud_host(2_000, seed=1, side=10.0)
    V, F = grid_mesh(pkg, 4, 10.0)
    L, ptr, api = pkg.lib(), pkg.api._np_ptr, pkg.api
    h = np.empty(64 * 64, np.float32)
    with pkg.ShardedTree(P, [0, 0]) as st:
        def call(o, hb, n_faces=len(F), res=64, k=8, faces=F):
            return L.pt_sharded_bake(st._h, ptr(V), len(V), ptr(faces), n_faces, k, -1.0, res, 1,
                                     None if o is None else ctypes.byref(o),
                                     None if hb is None else ctypes.byref(hb), None)
        assert call(None, None) == INVALID_ARG
        assert call(api.BakeOutputs(), None) == INVALID_ARG
        assert call(None, api.BakeHeight()) == INVALID_ARG
        hb = api.BakeHeight(height=h.ctypes.data)
        # the 3 n_faces limit is refused before the faces are read (there are only len(F) of them)
        assert call(None, hb, n_faces=(2**31 - 1) // 3 + 1) == api.PT_ERR_UNSUPPORTED
        for res in (0, 16385):
            assert call(None, hb, res=res) == INVALID_ARG
        for k in (0, 33):
            assert call(None, hb, k=k) == api.PT_ERR_UNSUPPORTED
        assert call(None, hb) == 0 and hb.texels > 0
        with pytest.raises(ValueError):
            st.bake(V, F, k=8, resolution=64, want=("displacement",))
    assert L.pt_sharded_bake(None, ptr(V), len(V), ptr(F), len(F), 8, -1.0, 64, 1, None, ctypes.byref(hb),
                             None) == INVALID_ARG
    with pkg.Tree(P) as tree:                                    # the single index answers the same codes
        for k in (0, 33):
            assert L.pt_texture_bake_height(tree.handle, ptr(V), len(V), ptr(F), len(F), k, -1.0, 64, 1, None,
                                            ctypes.byref(hb), None) == api.PT_ERR_UNSUPPORTED


def test_4096_heights_cross_chunks(pkg, torch_cuda):
    """A 4096^2 atlas on 2 slabs: each slab answers more than 2^22 samples, in two chunks."""
    rng = np.random.default_rng(10)
    n = 40_000
    P = pkg.make_points(np.c_[rng.random((n, 2)) * 10.0, rng.normal(0, 0.05, n)], normal=rng.standard_normal((n, 3)),
                        color=rng.integers(0, 256, (n, 3)))
    V = pkg.make_points([[0, 0, 0], [10, 0, 0], [10, 10, 0], [0, 10, 0.0]], normal=np.tile([0.1, -0.2, 1.0], (4, 1)),
                        uv=[[0, 0], [1, 0], [1, 1], [0, 1.0]])
    F = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    got, _ = compare(pkg, P, V, F, [0, 0], k=3, resolution=4096, pad=True, want=("bgra", "tangent_bgra") + HEIGHTS)
    assert got["stats"]["texels"] == 4096 * 4096          # about 2^23 per slab


def test_equals_oracle(pkg, pto, torch_cuda):
    side, k, res = 30.0, 12, 160
    P = pkg.synth.cloud_host(20_000, seed=31, side=side)
    V, F = mesh_case(pkg, 31, g=10)
    with pkg.ShardedTree(P, [0, 0, 0]) as st:
        got = st.bake(V, F, k=k, resolution=res, want=("bgra", "normal_bgra", "normal") + HEIGHTS)
    bgra, nbgra, nf, (n, empty) = pto_bake.bake(P, V, F, k, res, pad=True)
    assert (got["stats"]["texels"], got["stats"]["empty"]) == (n, empty)
    assert np.array_equal(got["bgra"], bgra) and np.array_equal(got["normal_bgra"], nbgra)
    assert np.array_equal(got["normal"].view(np.uint32), nf.view(np.uint32))
    ref = pto_bake.bake_heights(P, V, F, k, res, pad_codes=True)
    assert np.array_equal(got["height"].view(np.uint32), ref["height"].view(np.uint32))
    assert np.array_equal(got["height_u16"], ref["height_u16"])
    assert got["stats"]["height_texels"] == ref["texels"]


def test_distinct_devices(pkg, torch_cuda):
    if torch_cuda.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    P = pkg.synth.cloud_host(90_000, seed=41, side=30.0)
    V, F = mesh_case(pkg, 41)
    for devices in ([0, 1], [0, 1, 0, 1]):
        compare(pkg, P, V, F, devices, k=16, resolution=300, want=EVERYTHING)
    _, info = compare(pkg, P, V, F, [1, 0], halo=1e-4, k=20, resolution=256, want=EVERYTHING)
    assert info["rebuilds"] > 0
