"""The hand-over chain behind the grid kernel launched as programmatic dependents (option
"chain_pdl", default 1) against plain stream order ("chain_pdl" 0) and the CPU oracle, bit for bit.

With "chain_pdl" on, the kernels that answer the samples a grid launch hands over start while the
kernel ahead of them still runs and wait for it on the device; the list-mode scan and thread
launches get a grid of the resident blocks and walk the list grid-stride.  Neither may change a
result, on short hand-over lists (the warp kernel) or long ones (the scan / thread kernel)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHORT_LIST = 2048       # hand-over lists up to this size go to the warp kernel (pt_knn.cu)


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
    pkg.set_option("chain_pdl", 1)
    pkg.set_option("queue_cap", 1 << 20)
    pkg.set_option("pool_guard", 0)
    pkg.set_option("smem_pad", 0)


def _blob_cloud(pkg, n_blob_samples):
    """A scanned surface with a dense blob on it: every block around a sample inside the blob
    holds far more candidates than a half-warp stages, so the grid kernel hands those samples
    over (skewed clusters, as cfg5)."""
    rng = np.random.default_rng(11)
    surf = pkg.synth.cloud_host(100_000, seed=43, side=50.0)
    blob = np.float32(25.0 + 0.2 * rng.standard_normal((100_000, 3))).astype(np.float64)
    P = np.concatenate([surf, pkg.api.make_points(blob)])
    inner = np.float32(25.0 + 0.2 * rng.standard_normal((n_blob_samples, 3))).astype(np.float64)
    V = np.concatenate([pkg.synth.samples_host(41, side=50.0), pkg.api.make_points(inner)])
    return P, V


@pytest.mark.parametrize("n_blob,long_list", [(700, False), (6001, True)])
@pytest.mark.parametrize("k,radius", [(16, None), (7, 0.3)])
def test_hand_over_chain_equals_plain_order_and_oracle(n_blob, long_list, k, radius, pkg, pto, torch_cuda):
    P, V = _blob_cloud(pkg, n_blob)
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, radius=-1.0 if radius is None else radius, exact_ties=True)
    ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
    outs = {}
    pkg.set_option("knn_variant", 6)
    for pdl in (1, 0):
        pkg.set_option("chain_pdl", pdl)
        with pkg.Tree(P) as t:
            outs[pdl] = t.transfer(V, k, radius=radius, want_idx=True, want_d2=True)
            handed = t.fallback_counts()[1]
        assert (handed > SHORT_LIST) if long_list else (0 < handed <= SHORT_LIST), (pdl, handed)
        assert np.array_equal(outs[pdl]["idx"], ref_idx), pdl
        assert np.array_equal(outs[pdl]["d2"], ref_d2), pdl
        assert np.array_equal(outs[pdl]["rgba"], ref_rgba), pdl
    for key in ("idx", "d2", "rgba", "normal"):
        assert np.array_equal(outs[1][key], outs[0][key]), key
    assert np.allclose(outs[1]["normal"], ref_nrm, rtol=1e-5, atol=1e-7)


def test_all_three_lists_nonempty(pkg, pto, torch_cuda):
    """A long grid hand-over list whose samples then overflow the scan / thread kernel's tiny
    queue: every kernel of the chain has work, and the result is still the oracle's."""
    P, V = _blob_cloud(pkg, 6001)
    k = 16
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, exact_ties=True)
    pkg.set_option("knn_variant", 6)
    pkg.set_option("queue_cap", 2)
    for pdl in (1, 0):
        pkg.set_option("chain_pdl", pdl)
        with pkg.Tree(P) as t:
            out = t.transfer(V, k, want_idx=True, want_d2=True)
            rerun, handed = t.fallback_counts()
        assert handed > SHORT_LIST and rerun > 0, (pdl, handed, rerun)
        assert np.array_equal(out["idx"], ref_idx), pdl
        assert np.array_equal(out["d2"], ref_d2), pdl


@pytest.mark.parametrize("k,radius", [(16, None), (7, 0.3)])
def test_list_mode_grid_takes_several_turns(k, radius, pkg, pto, torch_cuda):
    """With the scan / thread kernel's shared memory padded to one resident block per SM, the
    list-mode grid is one block of 32 list entries per SM, and a list of > 9 472 samples takes
    several grid-stride turns per block: the result must not depend on the grid size."""
    P, V = _blob_cloud(pkg, 12001)
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, radius=-1.0 if radius is None else radius, exact_ties=True)
    pkg.set_option("knn_variant", 6)
    for pad in (150_000, 0):
        pkg.set_option("smem_pad", pad)
        with pkg.Tree(P) as t:
            out = t.transfer(V, k, radius=radius, want_idx=True, want_d2=True)
            handed = t.fallback_counts()[1]
        assert handed > 2 * 148 * 32, handed
        assert np.array_equal(out["idx"], ref_idx), pad
        assert np.array_equal(out["d2"], ref_d2), pad


def test_concurrent_chains_on_two_streams(pkg, pto, torch_cuda):
    """Two launches of one index in flight on different streams, each with a long hand-over list
    and a tiny traversal queue: each chain waits on its own stream only and owns its lists."""
    torch = torch_cuda
    pkg.set_option("knn_variant", 6)
    pkg.set_option("queue_cap", 2)
    P, V = _blob_cloud(pkg, 6001)
    k = 16
    ref_idx, _ = pto.KdTree(P).knn(V, k, exact_ties=True)
    pos = torch.zeros((len(P), 4), dtype=torch.float32, device="cuda")
    pos[:, :3] = torch.from_numpy(P["ver"].astype(np.float32)).cuda()
    tree = pkg.DeviceTree(pos)
    q = torch.from_numpy(np.ascontiguousarray(V["ver"])).cuda()
    perm = np.random.default_rng(3).permutation(len(V))       # blob samples in both halves
    half = len(V) // 2
    parts = [(q[torch.from_numpy(perm[:half]).cuda()].contiguous(), ref_idx[perm[:half]]),
             (q[torch.from_numpy(perm[half:]).cuda()].contiguous(), ref_idx[perm[half:]])]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = [torch.empty((p[0].shape[0], k), dtype=torch.int32, device="cuda") for p in parts]
    torch.cuda.synchronize()
    try:
        for rep in range(5):
            for (qq, _), st, o in zip(parts, streams, outs):
                tree.query(qq, k, idx=o, stream=st)
            torch.cuda.synchronize()
            for (_, ref), o in zip(parts, outs):
                assert np.array_equal(o.cpu().numpy(), ref), rep
    finally:
        tree.close()


def test_guard_words_with_chain_pdl(pkg, pto, torch_cuda):
    """With "pool_guard" on, no fence around the hand-over workspace or any other allocation is
    touched by the chain, on ragged sample counts with short and long hand-over lists."""
    pkg.set_option("pool_guard", 1)
    before = pkg.get_option("pool_guard_hits")
    P, V = _blob_cloud(pkg, 6001)
    kd = pto.KdTree(P)
    with pkg.Tree(P) as t:
        for m, k, radius in ((1, 1, None), (33, 16, None), (1681 + 700, 16, None), (len(V), 16, None),
                             (len(V) - 1, 7, 0.3)):
            W = V[-m:]
            ref_idx, ref_d2 = kd.knn(W, k, radius=-1.0 if radius is None else radius)
            out = t.transfer(W, k, radius=radius, want_idx=True, want_d2=True)
            assert np.array_equal(out["idx"], ref_idx), (m, k)
            assert np.array_equal(out["d2"], ref_d2), (m, k)
    assert pkg.get_option("pool_guard_hits") == before
