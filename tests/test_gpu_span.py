"""knn_grid_span_kernel (option "grid_span", default 1) against knn_grid_pair_kernel ("grid_span" 0)
and the CPU oracle, bit for bit.

The span kernel looks up each parent cell once, stages whole spans of the sorted cloud and reads
the winners' attributes from the sorted-order copy; it must stage exactly the pair kernel's
candidates and give exactly its answers."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


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
    pkg.set_option("knn_variant", -1)
    pkg.set_option("grid_pair", 1)
    pkg.set_option("grid_span", 1)
    pkg.set_option("pool_guard", 0)


def _clouds(pkg):
    rng = np.random.default_rng(5)
    surf = pkg.synth.cloud_host(120_001, seed=19, side=50.0)
    g = np.arange(40, dtype=np.float64) * 0.25
    lat = pkg.api.make_points(np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3))
    dup = pkg.synth.cloud_host(40_000, seed=29, side=30.0)
    dup = np.concatenate([dup, dup[::3], dup[::7]])
    dense = pkg.synth.cloud_host(60_000, seed=23, side=50.0)
    blob = np.float32(25.0 + 0.4 * rng.standard_normal((40_000, 3))).astype(np.float64)
    dense = np.concatenate([dense, pkg.api.make_points(blob)])
    samples = pkg.synth.samples_host(41, side=50.0)
    return (("surface", surf, samples),                                   # 1 681 samples: odd
            ("one", surf, samples[777:778]),
            ("lattice", lat, pkg.api.make_points(lat["ver"][::37] + 0.125)),
            ("duplicates", dup, pkg.synth.samples_host(33, side=30.0)),
            ("blob", dense, pkg.api.make_points(np.float32(25.0 + 0.5 * rng.standard_normal((999, 3))).astype(np.float64))))


@pytest.mark.parametrize("k,radius", [(1, None), (7, None), (16, None), (1, 0.3), (7, 0.05), (16, 0.35)])
def test_span_kernel_equals_pair_kernel_and_oracle(k, radius, pkg, pto, torch_cuda):
    """A scanned surface with an odd sample count, a single sample, a lattice (exact re-selection
    in both halves), duplicated points and a dense blob (redo by the whole warp and hand-over)."""
    for name, P, V in _clouds(pkg):
        ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, radius=-1.0 if radius is None else radius, exact_ties=True)
        ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
        outs = {}
        for span in (1, 0):
            pkg.set_option("grid_span", span)
            pkg.set_option("grid_pair", 2)       # two samples per warp whatever the expected count
            pkg.set_option("knn_variant", 6)
            with pkg.Tree(P) as t:
                outs[span] = t.transfer(V, k, radius=radius, want_idx=True, want_d2=True)
            if name == "surface":
                assert pkg.get_option("grid_span_used") == span, (name, span)
            assert np.array_equal(outs[span]["idx"], ref_idx), (name, span)
            assert np.array_equal(outs[span]["d2"], ref_d2), (name, span)
            assert np.array_equal(outs[span]["rgba"], ref_rgba), (name, span)
        for key in ("idx", "d2", "rgba", "normal"):
            assert np.array_equal(outs[1][key], outs[0][key]), (name, key)
        assert np.allclose(outs[1]["normal"], ref_nrm, rtol=1e-5, atol=1e-7), name


@pytest.mark.parametrize("k", [1, 7, 16])
def test_span_kernel_slab_entry_with_bad_bounds(k, pkg, pto, torch_cuda):
    """The device entry as the sharded path calls it: per-sample squared bounds, some rows NaN or
    negative (unused rows of a routing block: empty answers), candidate records out."""
    torch = torch_cuda
    n, g = 200_000, 45
    pos, attrs = pkg.synth.cloud_device(n, seed=7, u1=60.0, v1=60.0)
    q = pkg.synth.samples_device(g, g, u1=60.0, v1=60.0)
    m = q.shape[0]
    r2 = torch.full((m,), float("inf"), dtype=torch.float64, device="cuda")
    r2[5::11] = float("nan")
    r2[7::13] = -1.0
    r2[3::17] = 0.09
    outs = {}
    tree = pkg.DeviceTree(pos, attrs)
    try:
        for span in (1, 0):
            pkg.set_option("grid_span", span)
            pkg.set_option("grid_pair", 2)
            o = {"idx": torch.empty((m, k), dtype=torch.int32, device="cuda"),
                 "d2": torch.empty((m, k), dtype=torch.float64, device="cuda"),
                 "rgba": torch.empty((m, 4), dtype=torch.uint8, device="cuda"),
                 "normal": torch.empty((m, 3), dtype=torch.float32, device="cuda"),
                 "cand": torch.empty((m * k * 32,), dtype=torch.uint8, device="cuda")}
            tree.query(q, k, radius2_per_query=r2, **o)
            torch.cuda.synchronize()
            assert pkg.get_option("grid_span_used") == span
            outs[span] = {key: v.cpu().numpy() for key, v in o.items()}
    finally:
        tree.close()
    for key in ("idx", "d2", "rgba", "normal", "cand"):
        assert np.array_equal(outs[1][key], outs[0][key]), key
    # the unbounded rows against the oracle; the NaN / negative rows are empty
    P = pkg.synth.points_to_host(pos, attrs)
    V = pkg.synth.queries_to_host(q)
    r2h = r2.cpu().numpy()
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, exact_ties=True)
    free = np.isinf(r2h)
    assert np.array_equal(outs[1]["idx"][free], ref_idx[free])
    assert np.array_equal(outs[1]["d2"][free], ref_d2[free])
    bad = ~(r2h >= 0.0)
    assert (outs[1]["idx"][bad] == -1).all() and (outs[1]["rgba"][bad] == 0).all()


def test_span_kernel_is_the_default_and_keeps_the_guard_words(pkg, pto, torch_cuda):
    """A cfg-like launch (k = 16, unbounded, float4 cloud with attributes) runs the span kernel by
    default; with "pool_guard" on, the fences around the sorted-order attribute copy and every
    other allocation stay intact."""
    pkg.set_option("pool_guard", 1)
    before = pkg.get_option("pool_guard_hits")
    P = pkg.synth.cloud_host(150_001, seed=31, side=50.0)
    V = pkg.synth.samples_host(57, side=50.0)
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, 16, exact_ties=True)
    ref_rgba, _ = pto.blend(P, ref_idx, ref_d2)
    with pkg.Tree(P) as t:
        out = t.transfer(V, 16, want_idx=True, want_d2=True)
        assert pkg.get_option("grid_span_used") == 1
        assert pkg.get_option("grid_pair_used") == 0
    assert np.array_equal(out["idx"], ref_idx)
    assert np.array_equal(out["d2"], ref_d2)
    assert np.array_equal(out["rgba"], ref_rgba)
    assert pkg.get_option("pool_guard_hits") == before
