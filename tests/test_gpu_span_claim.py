"""knn_grid_span_kernel with warps claiming their pairs (option "grid_claim", default 1: used when
the launch has more than two pairs per resident warp) against the static stride ("grid_claim" 0),
against knn_grid_pair_kernel ("grid_span" 0) and against the CPU oracle, bit for bit.

Claiming changes only which warp answers which pair; no count, decision or output may change.  The
sample counts are above 2 samples x 2 pairs x the resident warps of a B200 (148 SMs x 7 blocks x
4 warps), so the launches below do claim."""
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
    pkg.set_option("grid_claim", 1)


def _clouds(pkg):
    rng = np.random.default_rng(7)
    surf = pkg.synth.cloud_host(200_001, seed=19, side=50.0)
    g = np.arange(40, dtype=np.float64) * 0.25
    lat = pkg.api.make_points(np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3))
    lat_s = pkg.api.make_points(np.float32(rng.uniform(0.0, 9.75, (20_001, 3))).astype(np.float64))
    dup = pkg.synth.cloud_host(40_000, seed=29, side=30.0)
    dup = np.concatenate([dup, dup[::3], dup[::7]])
    dense = pkg.synth.cloud_host(60_000, seed=23, side=50.0)
    blob = np.float32(25.0 + 0.4 * rng.standard_normal((40_000, 3))).astype(np.float64)
    dense = np.concatenate([dense, pkg.api.make_points(blob)])
    inner = pkg.api.make_points(np.float32(25.0 + 0.5 * rng.standard_normal((3_001, 3))).astype(np.float64))
    return (("surface", surf, pkg.synth.samples_host(151, side=50.0)),        # 22 801 samples: odd
            ("lattice", lat, lat_s),
            ("duplicates", dup, pkg.synth.samples_host(149, side=30.0)),
            ("blob", dense, np.concatenate([pkg.synth.samples_host(141, side=50.0), inner])))


@pytest.mark.parametrize("k,radius", [(1, None), (7, None), (16, None), (1, 0.3), (7, 0.05), (16, 0.35)])
def test_claimed_pairs_equal_static_stride_pair_kernel_and_oracle(k, radius, pkg, pto, torch_cuda):
    for name, P, V in _clouds(pkg):
        assert len(V) > 2 * 2 * 148 * 7 * 4, name
        ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, radius=-1.0 if radius is None else radius, exact_ties=True)
        ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
        pkg.set_option("grid_pair", 2)
        pkg.set_option("knn_variant", 6)
        outs = {}
        for span, claim in ((1, 1), (1, 0), (0, 0)):
            pkg.set_option("grid_span", span)
            pkg.set_option("grid_claim", claim)
            with pkg.Tree(P) as t:
                outs[span, claim] = t.transfer(V, k, radius=radius, want_idx=True, want_d2=True)
            if name == "surface":
                assert pkg.get_option("grid_span_used") == span, name
            o = outs[span, claim]
            assert np.array_equal(o["idx"], ref_idx), (name, span, claim)
            assert np.array_equal(o["d2"], ref_d2), (name, span, claim)
            assert np.array_equal(o["rgba"], ref_rgba), (name, span, claim)
        for arm in outs:
            for key in ("idx", "d2", "rgba", "normal"):
                assert np.array_equal(outs[arm][key], outs[1, 1][key]), (name, arm, key)
        assert np.allclose(outs[1, 1]["normal"], ref_nrm, rtol=1e-5, atol=1e-7), name
