"""knn_grid_block_kernel (option "grid_block", default 1) against knn_grid_span_kernel ("grid_block"
0), knn_grid_pair_kernel ("grid_span" 0) and the CPU oracle, bit for bit.

The block kernel stages a sample's candidates from the one block run the build wrote for its cell
-- the span kernel's records and span heads in the span kernel's slot order -- so it must give
exactly the answers of both other kernels.  Samples whose cell is empty, or whose block is too
dense to stage, are redone by the whole warp and must stay exact too."""
import glob
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = (("block", 1, 1), ("span", 0, 1), ("pair", 1, 0))   # name, grid_block, grid_span


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


@pytest.fixture(autouse=True)
def _default_options(pkg):
    yield
    for name, value in (("knn_variant", -1), ("grid_pair", 1), ("grid_span", 1), ("grid_block", 1)):
        pkg.set_option(name, value)


def _run_modes(pkg, P, V, k, radius, expect_block=None):
    """One index, the three kernels in turn: their outputs (equal to each other) and whether the
    block kernel ran."""
    outs = {}
    with pkg.Tree(P) as t:
        for name, block, span in MODES:
            pkg.set_option("grid_block", block)
            pkg.set_option("grid_span", span)
            pkg.set_option("grid_pair", 2)       # two samples per warp whatever the expected count
            pkg.set_option("knn_variant", 6)
            outs[name] = t.transfer(V, k, radius=radius, want_idx=True, want_d2=True)
            used = pkg.get_option("grid_block_used")
            if name != "block":
                assert used == 0, name
            elif expect_block is not None:
                assert used == expect_block
    for name in ("span", "pair"):
        for key in ("idx", "d2", "rgba", "normal"):
            assert np.array_equal(outs["block"][key], outs[name][key]), (name, key)
    return outs["block"]


def _check_oracle(pto, P, V, k, radius, out):
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, radius=-1.0 if radius is None else radius, exact_ties=True)
    ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
    assert np.array_equal(out["idx"], ref_idx)
    assert np.array_equal(out["d2"], ref_d2)
    assert np.array_equal(out["rgba"], ref_rgba)
    assert np.allclose(out["normal"], ref_nrm, rtol=1e-5, atol=1e-7)


def _awkward_samples(pkg, P, rng):
    """Samples on the surface, above it in empty cells, exactly on cell faces of every level from
    4 to 14 (lattice origin + multiples of extent / 2^l), and outside the cloud's box."""
    xyz = P["ver"]
    lo, hi = xyz.min(0), xyz.max(0)
    ext = float((hi - lo).max())
    surf = xyz[rng.choice(len(xyz), 600, replace=False)]
    above = surf[:200] + np.array([0.0, 0.0, 0.05 * ext])
    faces = []
    for lvl in range(4, 15):
        step = ext / 2.0 ** lvl
        j = rng.integers(1, 2 ** lvl, (40, 3)).astype(np.float64)
        f = surf[200:240].copy()
        ax = lvl % 3
        f[:, ax] = lo[ax] + j[:, ax] * step        # on a face along one axis
        f[:4] = lo + j[:4] * step                  # on a corner of the lattice
        faces.append(f)
    outside = np.concatenate([lo - 0.3 * ext + rng.random((40, 3)), hi + 0.2 * ext * rng.random((40, 3)),
                              surf[:40] + np.array([2.0 * ext, 0.0, 0.0])])
    return pkg.api.make_points(np.concatenate([surf, above] + faces + [outside]))


@pytest.mark.parametrize("k", [1, 4, 8, 16])
@pytest.mark.parametrize("radius", [None, 0.3])
def test_block_kernel_equals_span_pair_and_oracle(k, radius, pkg, pto, torch_cuda):
    """A scanned surface with an odd sample count and awkward samples; a dense blob whose blocks
    hold more than a half-warp stages and a pile of duplicates whose parent is too dense for the
    cell tables' counts (both redone by the whole warp)."""
    rng = np.random.default_rng(11)
    surf = pkg.synth.cloud_host(150_001, seed=31, side=50.0)
    V = pkg.api.make_points(np.concatenate([pkg.synth.samples_host(41, side=50.0)["ver"],
                                            _awkward_samples(pkg, surf, rng)["ver"]]))
    out = _run_modes(pkg, surf, V, k, radius, expect_block=1 if (k == 16 and radius is None) else None)
    _check_oracle(pto, surf, V, k, radius, out)

    blob = np.float32(25.0 + 0.4 * rng.standard_normal((40_000, 3))).astype(np.float64)
    # 70 000 points in a 1e-3 cube: one parent cell over the tables' 16-bit counts (distinct
    # points: the oracle's kd-tree does not take that many identical ones)
    pile = np.array([10.0, 10.0, pkg.synth.surface_np(10.0, 10.0)]) + 1e-3 * rng.random((70_000, 3))
    pile = pile.astype(np.float32).astype(np.float64)
    dense = pkg.api.make_points(np.concatenate([surf["ver"][::3], blob, pile]))
    near = np.concatenate([25.0 + 0.5 * rng.standard_normal((300, 3)), pile[:50] + rng.normal(0, 0.2, (50, 3)),
                           pkg.synth.samples_host(17, side=50.0)["ver"]])
    Vd = pkg.api.make_points(near.astype(np.float32).astype(np.float64))
    out = _run_modes(pkg, dense, Vd, k, radius)
    _check_oracle(pto, dense, Vd, k, radius, out)


@pytest.mark.parametrize("name", sorted(os.path.basename(p)[:-4] for p in glob.glob(
    os.path.join(os.path.dirname(__file__), "golden", "*.npz"))))
def test_block_kernel_golden_fixtures(name, pkg, pto, golden_dir, torch_cuda):
    z = np.load(os.path.join(golden_dir, name + ".npz"))
    if "xyz" not in z:
        pytest.skip("not a k-NN fixture")
    P = pkg.make_points(z["xyz"], normal=z["normal"], color=z["color"])
    Q = pkg.make_points(z["queries"])
    radius = float(z["radius"])
    for k in (1, 4, 8, 16):
        for r in (None, radius if radius > 0 else None):
            _check_oracle(pto, P, Q, k, r, _run_modes(pkg, P, Q, k, r))


@pytest.mark.parametrize("k", [1, 8, 16])
def test_block_kernel_slab_entry_with_per_sample_bounds(k, pkg, pto, torch_cuda):
    """The device entry as the sharded path calls it: per-sample squared bounds, some rows NaN or
    negative (empty answers), candidate records out."""
    torch = torch_cuda
    n, g = 200_000, 45
    pos, attrs = pkg.synth.cloud_device(n, seed=7, u1=60.0, v1=60.0)
    q = pkg.synth.samples_device(g, g, u1=60.0, v1=60.0)
    m = q.shape[0]
    r2 = torch.full((m,), float("inf"), dtype=torch.float64, device="cuda")
    r2[5::11] = float("nan")
    r2[7::13] = -1.0
    r2[3::17] = 0.09
    r2[2::19] = 0.0
    outs = {}
    tree = pkg.DeviceTree(pos, attrs)
    try:
        for name, block, span in MODES:
            pkg.set_option("grid_block", block)
            pkg.set_option("grid_span", span)
            pkg.set_option("grid_pair", 2)
            o = {"idx": torch.empty((m, k), dtype=torch.int32, device="cuda"),
                 "d2": torch.empty((m, k), dtype=torch.float64, device="cuda"),
                 "rgba": torch.empty((m, 4), dtype=torch.uint8, device="cuda"),
                 "normal": torch.empty((m, 3), dtype=torch.float32, device="cuda"),
                 "cand": torch.empty((m * k * 32,), dtype=torch.uint8, device="cuda")}
            tree.query(q, k, radius2_per_query=r2, **o)
            torch.cuda.synchronize()
            if name == "block" and k == 16:
                assert pkg.get_option("grid_block_used") == 1
            outs[name] = {key: v.cpu().numpy() for key, v in o.items()}
    finally:
        tree.close()
    for name in ("span", "pair"):
        for key in ("idx", "d2", "rgba", "normal", "cand"):
            assert np.array_equal(outs["block"][key], outs[name][key]), (name, key)
    P = pkg.synth.points_to_host(pos, attrs)
    V = pkg.synth.queries_to_host(q)
    r2h = r2.cpu().numpy()
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, exact_ties=True)
    free = np.isinf(r2h)
    assert np.array_equal(outs["block"]["idx"][free], ref_idx[free])
    assert np.array_equal(outs["block"]["d2"][free], ref_d2[free])
    bad = ~(r2h >= 0.0)
    assert (outs["block"]["idx"][bad] == -1).all() and (outs["block"]["rgba"][bad] == 0).all()


def test_index_over_the_memory_budget_has_no_block_runs(pkg, pto, torch_cuda):
    """With the device nearly full the build leaves the runs out (they may take a quarter of the
    free memory): the default launch then runs the span kernel, with the same answers, and the
    index's device bytes are those of the index without runs."""
    torch = torch_cuda
    P = pkg.synth.cloud_host(1_000_003, seed=41, side=100.0)
    V = pkg.synth.samples_host(61, side=100.0)
    ref = {}
    with pkg.Tree(P) as t:
        ref = t.transfer(V, 16, want_idx=True, want_d2=True)
        assert pkg.get_option("grid_block_used") == 1
        full_bytes = t.info().device_bytes
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    # leave 320 MB: the build's sort and tables fit (the library's pool keeps what the first build
    # used), a quarter of it does not hold the runs (about nine records per point, 16 bytes each)
    ballast = torch.empty(max(free - (320 << 20), 0), dtype=torch.uint8, device="cuda")
    try:
        with pkg.Tree(P) as t:
            out = t.transfer(V, 16, want_idx=True, want_d2=True)
            assert pkg.get_option("grid_span_used") == 1
            assert pkg.get_option("grid_block_used") == 0
            assert t.info().device_bytes < full_bytes
    finally:
        del ballast
        torch.cuda.empty_cache()
    for key in ("idx", "d2", "rgba", "normal"):
        assert np.array_equal(out[key], ref[key]), key
