"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle.

Bars (BASELINE.json north_star): neighbour indices and squared distances bit-exact (ties ->
lowest point index); blended colours exact, normals within 1e-5 relative.
"""
import glob
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLDEN = sorted(os.path.basename(p)[:-4] for p in glob.glob(
    os.path.join(os.path.dirname(__file__), "golden", "*.npz")))
NORMAL_RTOL = 1e-5   # tolerance stated by north_star for transferred normals


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def _check_blend(got_rgba, got_nrm, ref_rgba, ref_nrm):
    assert np.array_equal(got_rgba, ref_rgba)
    assert np.allclose(got_nrm, ref_nrm, rtol=NORMAL_RTOL, atol=1e-7)


@pytest.fixture(autouse=True)
def _default_options(pkg):
    yield
    pkg.set_option("knn_variant", -1)     # auto (the default)
    pkg.set_option("queue_cap", 1 << 20)  # the compiled capacity
    pkg.set_option("order", 1)            # Hilbert order + cell tables (the default)
    pkg.set_option("grid_tma", 1)
    pkg.set_option("pool_guard", 0)
    pkg.set_option("sort_bits", 0)
    pkg.set_option("grid_pair", 1)
    pkg.set_option("grid_admit100", 100)
    pkg.set_option("grid_lookup_cost", 8)
    pkg.set_option("grid_min_occ10", 40)


# (knn_variant, order): grid / thread / warp / scan kernel x Morton, Hilbert, Hilbert + kd
# refinement (order 2 has no cell tables: variant 6 then falls through to the auto rule)
MODES = [(6, 1), (6, 0), (-1, 1), (2, 1), (0, 1), (5, 1), (2, 0), (2, 2), (0, 2), (5, 2), (5, 0), (6, 2)]


@pytest.mark.parametrize("mode", MODES, ids=lambda m: f"variant{m[0]}-order{m[1]}")
@pytest.mark.parametrize("name", GOLDEN)
def test_golden_fixtures(name, mode, pkg, golden_dir, torch_cuda):
    pkg.set_option("knn_variant", mode[0])
    pkg.set_option("order", mode[1])
    z = np.load(os.path.join(golden_dir, name + ".npz"))
    P = pkg.make_points(z["xyz"], normal=z["normal"], color=z["color"])
    Q = pkg.make_points(z["queries"])
    radius = float(z["radius"])
    with pkg.Tree(P) as tree:
        expect_f64 = not np.array_equal(z["xyz"].astype(np.float32).astype(np.float64), z["xyz"])
        assert tree.info().coord_mode == (pkg.COORD_F64 if expect_f64 else pkg.COORD_F32)
        for k in z["ks"]:
            k = int(k)
            idx, d2 = tree.knn(Q, k, radius=radius)
            assert np.array_equal(idx, z[f"idx_k{k}"]), f"{name} k={k}: indices"
            assert np.array_equal(d2, z[f"d2_k{k}"]), f"{name} k={k}: d2"
            out = tree.transfer(Q, k, radius=radius, want_idx=True, want_d2=True)
            assert np.array_equal(out["idx"], idx) and np.array_equal(out["d2"], d2)
            _check_blend(out["rgba"], out["normal"], z[f"rgba_k{k}"], z[f"normal_k{k}"])


def test_f64_storage_forced_and_f32_rejected(pkg, pto, torch_cuda):
    rng = np.random.default_rng(5)
    xyz = rng.random((3000, 3))          # not fp32-representable
    P, Q = pkg.make_points(xyz), pkg.make_points(rng.random((100, 3)))
    with pytest.raises(pkg.PointsTransferError) as e:
        pkg.Tree(P, coord_mode=pkg.COORD_F32)
    assert e.value.status == 6
    ref_idx, ref_d2 = pto.knn_bruteforce(P, Q, 20)
    for mode in (pkg.COORD_AUTO, pkg.COORD_F64):
        with pkg.Tree(P, coord_mode=mode) as t:
            idx, d2 = t.knn(Q, 20)
        assert np.array_equal(idx, ref_idx) and np.array_equal(d2, ref_d2)
    # representable data stored as fp64 on request gives the same answer
    P32 = pkg.make_points(xyz.astype(np.float32))
    ref_idx, ref_d2 = pto.knn_bruteforce(P32, Q, 8)
    for mode in (pkg.COORD_F32, pkg.COORD_F64):
        with pkg.Tree(P32, coord_mode=mode) as t:
            idx, d2 = t.knn(Q, 8)
        assert np.array_equal(idx, ref_idx) and np.array_equal(d2, ref_d2)


@pytest.mark.parametrize("variant", [6, 5, 2, 0])
@pytest.mark.parametrize("k", [1, 8, 16, 20, 32])
def test_surface_cloud_vs_kdtree_oracle(k, variant, pkg, pto, torch_cuda):
    pkg.set_option("knn_variant", variant)
    # config-1 shaped (SURVEY 8 M1), sized so the oracle finishes in seconds
    P = pkg.synth.cloud_host(300_000, seed=100 + k, side=80.0)
    V = pkg.synth.samples_host(70, side=80.0)
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, exact_ties=True)
    ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
    with pkg.Tree(P) as tree:
        out = tree.transfer(V, k, want_idx=True, want_d2=True)
    assert np.array_equal(out["idx"], ref_idx)
    assert np.array_equal(out["d2"], ref_d2)
    _check_blend(out["rgba"], out["normal"], ref_rgba, ref_nrm)


def test_gpu_d2_is_the_reference_metric(pkg, pto, torch_cuda):
    """Every squared distance the CUDA path returns equals, bit for bit, what the reference's own
    Distance::transformed_distance (src/Distance.h:6-11, compiled into oracle/_ref from the
    reference's header) computes for that (sample, neighbour) pair."""
    R = pto.ref_metric()
    if R is None:
        pytest.skip("needs the reference's own headers: set PT_REFERENCE_SRC to its src/ directory")
    P = pkg.synth.cloud_host(100_000, seed=3, side=50.0)
    V = pkg.synth.samples_host(40, side=50.0)
    for variant in (6, 5, 2, 0):
        pkg.set_option("knn_variant", variant)
        with pkg.Tree(P) as tree:
            idx, d2 = tree.knn(V, 16)
        assert (idx >= 0).all()
        for qi in range(0, len(V), 7):
            for j in range(16):
                ref = R.ref_transformed_distance(V[qi:qi + 1].ctypes.data,
                                                 P[idx[qi, j]:idx[qi, j] + 1].ctypes.data)
                assert d2[qi, j] == ref, (variant, qi, j)


def test_reference_call_site_shape(pkg, pto, torch_cuda):
    # src/pointsTransfer.cpp:470-479: per face, per corner, K=20 search; iterate (point, d2)
    P = pkg.synth.cloud_host(20_000, seed=9, side=20.0)
    V = pkg.synth.samples_host(6, side=20.0)
    F = pkg.synth.grid_faces(6, 6)
    K = 20
    ref_idx, ref_d2 = pto.knn_bruteforce(P, V, K)
    with pkg.Tree(P) as tree:
        for j in (0, 7, F.shape[0] - 1):
            for i in range(3):
                v = int(F[j, i])
                search = pkg.K_neighbor_search(tree, V[v], K)
                got = list(search)
                assert len(search) == K
                assert [g[0] for g in got] == ref_idx[v].tolist()
                assert [g[1] for g in got] == ref_d2[v].tolist()


@pytest.mark.parametrize("variant", [6, 5, 2])
def test_device_api_ids_and_radius_per_query(variant, pkg, pto, torch_cuda):
    pkg.set_option("knn_variant", variant)
    torch = torch_cuda
    rng = np.random.default_rng(21)
    n, m, k = 50_000, 2_000, 16
    xyz = (rng.random((n, 3)) * 30).astype(np.float32)
    P = pkg.make_points(xyz, normal=rng.standard_normal((n, 3)).astype(np.float32),
                        color=rng.integers(0, 256, (n, 3)))
    qxyz = (rng.random((m, 3)) * 30).astype(np.float32).astype(np.float64)
    Q = pkg.make_points(qxyz)
    ids = np.cumsum(rng.integers(1, 4, n)).astype(np.int32)   # strictly increasing global ids
    pos = torch.zeros((n, 4), dtype=torch.float32, device="cuda")
    pos[:, :3] = torch.from_numpy(xyz).cuda()
    attrs = np.zeros(n, dtype=pkg.ATTR_DTYPE)
    attrs["nx"], attrs["ny"], attrs["nz"] = P["normal"][:, 0], P["normal"][:, 1], P["normal"][:, 2]
    attrs["rgba"][:, :3] = P["color"]
    attrs["rgba"][:, 3] = 255
    t_attrs = torch.from_numpy(attrs.view(np.uint8).reshape(n, 16)).cuda()
    tree = pkg.DeviceTree(pos, t_attrs, torch.from_numpy(ids).cuda())
    tq = torch.from_numpy(qxyz).cuda()
    idx = torch.empty((m, k), dtype=torch.int32, device="cuda")
    d2 = torch.empty((m, k), dtype=torch.float64, device="cuda")
    rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
    nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
    tree.query(tq, k, idx=idx, d2=d2, rgba=rgba, normal=nrm)
    torch.cuda.synchronize()
    ref_idx, ref_d2 = pto.knn_bruteforce(P, Q, k)
    assert np.array_equal(idx.cpu().numpy(), np.where(ref_idx >= 0, ids[ref_idx], -1))
    assert np.array_equal(d2.cpu().numpy(), ref_d2)
    ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
    _check_blend(rgba.cpu().numpy(), nrm.cpu().numpy(), ref_rgba, ref_nrm)
    # per-query squared bound: bound = the 5th neighbour's d2 -> exactly 5 results (no ties here)
    r2 = torch.from_numpy(ref_d2[:, 4].copy()).cuda()
    tree.query(tq, k, radius2_per_query=r2, idx=idx, d2=d2)
    torch.cuda.synchronize()
    got = idx.cpu().numpy()
    assert np.array_equal(got[:, :5], ids[ref_idx[:, :5]]) and np.all(got[:, 5:] == -1)
    tree.close()


@pytest.mark.parametrize("variant", [6, 5, 2])
@pytest.mark.parametrize("n_slabs,k", [(2, 8), (3, 16), (8, 32)])
def test_slab_merge_equals_single_index(n_slabs, k, variant, pkg, pto, torch_cuda):
    pkg.set_option("knn_variant", variant)
    """SURVEY 8(e): R slabs on one GPU, per-slab top-k, merged by the K5 kernel, must be
    bit-identical to the single-index result."""
    torch = torch_cuda
    P = pkg.synth.cloud_host(120_000, seed=33, side=60.0)
    V = pkg.synth.samples_host(40, side=60.0)
    m = V.shape[0]
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k)
    ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
    order = np.argsort(P["ver"][:, 0], kind="stable")
    bounds = np.linspace(0, len(P), n_slabs + 1).astype(int)
    tq = torch.from_numpy(np.ascontiguousarray(V["ver"])).cuda()
    lists = torch.empty((n_slabs, m, k, 32), dtype=torch.uint8, device="cuda")
    trees = []
    for s in range(n_slabs):
        ids = np.sort(order[bounds[s]:bounds[s + 1]]).astype(np.int32)   # increasing global ids
        sub = P[ids]
        pos = torch.zeros((len(ids), 4), dtype=torch.float32, device="cuda")
        pos[:, :3] = torch.from_numpy(sub["ver"].astype(np.float32)).cuda()
        attrs = np.zeros(len(ids), dtype=pkg.ATTR_DTYPE)
        attrs["nx"], attrs["ny"], attrs["nz"] = sub["normal"][:, 0], sub["normal"][:, 1], sub["normal"][:, 2]
        attrs["rgba"][:, :3] = sub["color"]
        attrs["rgba"][:, 3] = 255
        t = pkg.DeviceTree(pos, torch.from_numpy(attrs.view(np.uint8).reshape(-1, 16)).cuda(),
                           torch.from_numpy(ids).cuda())
        t.query(tq, k, cand=lists[s].view(-1))
        trees.append(t)
    idx = torch.empty((m, k), dtype=torch.int32, device="cuda")
    d2 = torch.empty((m, k), dtype=torch.float64, device="cuda")
    rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
    nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
    pkg.merge_device(lists.view(-1), n_slabs, m, k, idx=idx, d2=d2, rgba=rgba, normal=nrm)
    torch.cuda.synchronize()
    assert np.array_equal(idx.cpu().numpy(), ref_idx)
    assert np.array_equal(d2.cpu().numpy(), ref_d2)
    _check_blend(rgba.cpu().numpy(), nrm.cpu().numpy(), ref_rgba, ref_nrm)
    for t in trees:
        t.close()


def test_queue_overflow_falls_back_exactly(pkg, pto, torch_cuda):
    """Thousands of exact duplicates make every box bound 0, so the per-thread best-first
    queue overflows; those samples are re-run by the warp kernel and must stay index-exact
    (ties -> lowest index)."""
    rng = np.random.default_rng(77)
    dup = np.tile(np.array([[0.5, 0.25, 0.125]]), (30_000, 1))
    rest = rng.random((10_000, 3)).astype(np.float32).astype(np.float64)
    xyz = np.concatenate([dup, rest])[rng.permutation(40_000)]
    P = pkg.make_points(xyz, normal=rng.standard_normal((40_000, 3)).astype(np.float32),
                        color=rng.integers(0, 256, (40_000, 3)))
    Q = pkg.make_points(np.concatenate([np.array([[0.5, 0.25, 0.125], [0.5, 0.25, 0.2]]),
                                        rng.random((200, 3))]))
    for k in (8, 32):
        ref_idx, ref_d2 = pto.knn_bruteforce(P, Q, k)
        ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
        with pkg.Tree(P) as tree:
            out = tree.transfer(Q, k, want_idx=True, want_d2=True)
        assert np.array_equal(out["idx"], ref_idx) and np.array_equal(out["d2"], ref_d2)
        _check_blend(out["rgba"], out["normal"], ref_rgba, ref_nrm)


@pytest.mark.parametrize("variant", [2, 5])
@pytest.mark.parametrize("cap", [2, 3, 5, 8])
def test_tiny_queue_stays_exact(cap, variant, pkg, pto, golden_dir, torch_cuda):
    """A full traversal queue gives up its least promising entry and remembers the smallest key
    it dropped; the sample is final only if the final bound stays below that key, otherwise it is
    re-run by the exact warp kernel.  Results must therefore be exact for ANY capacity."""
    pkg.set_option("knn_variant", variant)
    pkg.set_option("queue_cap", cap)
    P = pkg.synth.cloud_host(200_000, seed=31 + cap, side=70.0)
    V = pkg.synth.samples_host(64, side=70.0)
    for k in (8, 20):
        ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, exact_ties=True)
        ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
        with pkg.Tree(P) as tree:
            out = tree.transfer(V, k, want_idx=True, want_d2=True)
            fallbacks = tree.info().last_fallback_samples
        assert np.array_equal(out["idx"], ref_idx) and np.array_equal(out["d2"], ref_d2)
        _check_blend(out["rgba"], out["normal"], ref_rgba, ref_nrm)
        if cap <= 3:
            assert fallbacks > 0        # the give-up path and its fallback were exercised
    for name in ("skewed", "lattice_ties", "duplicates", "radius_bounded"):
        z = np.load(os.path.join(golden_dir, name + ".npz"))
        Pg = pkg.make_points(z["xyz"], normal=z["normal"], color=z["color"])
        Qg = pkg.make_points(z["queries"])
        with pkg.Tree(Pg) as tree:
            for k in z["ks"]:
                k = int(k)
                idx, d2 = tree.knn(Qg, k, radius=float(z["radius"]))
                assert np.array_equal(idx, z[f"idx_k{k}"]), (name, k)
                assert np.array_equal(d2, z[f"d2_k{k}"]), (name, k)


@pytest.mark.parametrize("variant", [-1, 6, 5, 2, 0])
def test_edge_cases(variant, pkg, torch_cuda):
    pkg.set_option("knn_variant", variant)
    empty = np.zeros(0, dtype=pkg.POINT_DTYPE)
    Q = pkg.make_points(np.zeros((3, 3)))
    with pkg.Tree(empty) as t:                       # empty cloud
        idx, d2 = t.knn(Q, 4)
        assert np.all(idx == -1) and np.all(np.isinf(d2))
        out = t.transfer(Q, 4)
        assert not out["rgba"].any() and not out["normal"].any()
    one = pkg.make_points(np.array([[1.0, 2.0, 3.0]]), color=[[7, 8, 9]], normal=[[0, 0, 2.0]])
    with pkg.Tree(one) as t:                         # single point, zero queries, k limits
        idx, d2 = t.knn(Q, 3)
        assert idx.tolist() == [[0, -1, -1]] * 3 and np.all(d2[:, 0] == 14.0)
        out = t.transfer(Q, 3)
        assert out["rgba"].tolist() == [[7, 8, 9, 255]] * 3
        assert np.allclose(out["normal"], [[0, 0, 1.0]] * 3)
        i0, _ = t.knn(empty, 3)
        assert i0.shape == (0, 3)
        for bad_k in (0, 33):
            with pytest.raises(pkg.PointsTransferError) as e:
                t.knn(Q, bad_k)
            assert e.value.status == 5
    bad = pkg.make_points(np.array([[0.0, np.nan, 0.0], [1.0, 1.0, 1.0]]))
    with pytest.raises(pkg.PointsTransferError) as e:
        pkg.Tree(bad)
    assert e.value.status == 7


def test_full_size_properties(pkg, pto, torch_cuda):
    """BASELINE config 2 at full size (50M points, 200k samples, k=16): size-independent
    properties + exact verification of sampled queries by restriction (every true neighbour of
    a sample lies within its reported k-th distance, so the oracle on that ball must agree)."""
    torch = torch_cuda
    w = pkg.synth.CONFIGS["cfg2"]
    free, _ = torch.cuda.mem_get_info()
    n = w.n_points if free > 24e9 else 5_000_000
    pos, attrs = pkg.synth.cloud_device(n, w.seed)
    q = pkg.synth.samples_device(w.gu, w.gv)
    m, k = q.shape[0], w.k
    tree = pkg.DeviceTree(pos, attrs)
    idx = torch.empty((m, k), dtype=torch.int32, device="cuda")
    d2 = torch.empty((m, k), dtype=torch.float64, device="cuda")
    rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
    nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
    tree.query(q, k, idx=idx, d2=d2, rgba=rgba, normal=nrm)
    torch.cuda.synchronize()
    # sortedness, uniqueness, full lists
    assert bool((d2[:, 1:] >= d2[:, :-1]).all())
    assert bool((idx >= 0).all()) and bool((idx < n).all())
    srt = idx.sort(dim=1).values
    assert bool((srt[:, 1:] != srt[:, :-1]).all())
    # reported d2 equals the metric recomputed from the coordinates (torch fp64, same op order)
    p = pos[idx.long().view(-1), :3].double().view(m, k, 3)
    diff = q.view(m, 1, 3) - p
    sq = diff * diff
    assert bool((((sq[..., 0] + sq[..., 1]) + sq[..., 2]) == d2).all())
    # idempotence: a second pass gives identical bits
    idx2 = torch.empty_like(idx)
    tree.query(q, k, idx=idx2)
    torch.cuda.synchronize()
    assert bool((idx2 == idx).all())
    # unit normals, opaque alpha
    nn = nrm.double().norm(dim=1)
    assert bool(((nn - 1).abs() < 1e-5).all()) and bool((rgba[:, 3] == 255).all())
    # exact check of sampled queries by restriction to the k-th-distance ball
    sel = np.linspace(0, m - 1, 48).astype(int)
    pos64 = pos[:, :3].double()
    for s in sel:
        r2 = float(d2[s, k - 1])
        dd = ((pos64 - q[s]) ** 2).sum(1)
        cand = torch.nonzero(dd <= r2 * (1 + 1e-9)).view(-1)
        ids = cand.cpu().numpy().astype(np.int32)          # ascending
        sub = pkg.make_points(pos[cand, :3].cpu().numpy().astype(np.float64))
        ridx, rd2 = pto.knn_bruteforce(sub, pkg.make_points(q[s].cpu().numpy()[None]), k)
        assert np.array_equal(ids[ridx[0]], idx[s].cpu().numpy())
        assert np.array_equal(rd2[0], d2[s].cpu().numpy())
    tree.close()


@pytest.mark.parametrize("cfg,n,g,k", [("cfg5", 1_500_000, 120, 16), ("cfg4", 1_000_000, 128, 32),
                                       ("cfg1", 1_000_000, 100, 8)])
def test_baseline_config_shapes_vs_oracle(cfg, n, g, k, pkg, pto, torch_cuda):
    """BASELINE.json configs at oracle-checkable sizes, generated by the same device generators
    the bench uses: cfg5 = skewed clusters + radius-bounded (short / empty lists expected),
    cfg4 = texel-centre samples with k = 32, cfg1 = the reference's CPU-runnable case in full."""
    torch = torch_cuda
    w = pkg.synth.CONFIGS[cfg]
    side = 1000.0 if cfg == "cfg1" else 150.0
    pos, attrs = pkg.synth.cloud_device(n, w.seed, u1=side, v1=side, kind=w.kind, sigma=w.sigma
                                        if cfg != "cfg5" else side / 2000.0)
    q = pkg.synth.samples_device(g, g, u1=side, v1=side, center=w.center)
    radius = None if w.radius is None else w.radius * (side / 1000.0) * 4
    P = pkg.synth.points_to_host(pos, attrs)
    Q = pkg.synth.queries_to_host(q)
    ref_idx, ref_d2 = pto.KdTree(P).knn(Q, k, radius=-1.0 if radius is None else radius)
    ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
    for variant in (6, 5, 2, 0):
        pkg.set_option("knn_variant", variant)
        tree = pkg.DeviceTree(pos, attrs)
        m = q.shape[0]
        idx = torch.empty((m, k), dtype=torch.int32, device="cuda")
        d2 = torch.empty((m, k), dtype=torch.float64, device="cuda")
        rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
        nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
        tree.query(q, k, radius=radius, idx=idx, d2=d2, rgba=rgba, normal=nrm)
        torch.cuda.synchronize()
        tree.close()
        assert np.array_equal(idx.cpu().numpy(), ref_idx), (cfg, variant)
        assert np.array_equal(d2.cpu().numpy(), ref_d2), (cfg, variant)
        _check_blend(rgba.cpu().numpy(), nrm.cpu().numpy(), ref_rgba, ref_nrm)
    if cfg == "cfg5":
        short = (ref_idx < 0).any(axis=1).mean()
        assert 0.05 < short < 1.0      # the radius bound really bites on the sparse part


def test_host_generator_matches_device(pkg, pto, torch_cuda):
    """oracle/pt_synth_host.c restates the device generators (csrc/pt_synth.cu) for the CPU arm of
    bench.py: same Philox streams and formulas; only the libm differs, so after the rounding to
    fp32 at most a few coordinates per million may be one fp32 ulp apart."""
    for cfg in ("cfg2", "cfg5"):
        w = pkg.synth.CONFIGS[cfg]
        n = 400_000
        pos, attrs = pkg.synth.cloud_device(n, w.seed, kind=w.kind, sigma=w.sigma, first_index=12345)
        D = pkg.synth.points_to_host(pos, attrs)
        H = pto.synth_cloud(n, w.seed, kind=w.kind, sigma=w.sigma, first_index=12345)
        diff = np.abs(D["ver"] - H["ver"])
        ulp = np.spacing(np.abs(D["ver"]).astype(np.float32)).astype(np.float64)
        assert np.all(diff <= ulp)
        assert (diff > 0).mean() < 1e-4
        assert (np.abs(D["normal"] - H["normal"]) > 1e-6).mean() < 1e-4
        assert (D["color"] != H["color"]).mean() < 1e-4
    q = pkg.synth.samples_device(300, 200, center=True)
    Qd = pkg.synth.queries_to_host(q)
    Qh = pto.synth_samples(300, 200, center=True)
    assert (np.abs(Qd["ver"] - Qh["ver"]) > 0).mean() < 1e-4


@pytest.mark.parametrize("variant", [5, 2, 6])
def test_concurrent_launches_on_two_streams(variant, pkg, pto, torch_cuda):
    """Launches of one index that are in flight on different streams own their hand-over lists
    (round 1 shared slot 0: one launch's reset could erase samples another had queued for the
    fallback).  A tiny traversal queue forces hand-overs; both results must stay exact."""
    torch = torch_cuda
    pkg.set_option("knn_variant", variant)
    pkg.set_option("queue_cap", 2)
    P = pkg.synth.cloud_host(200_000, seed=41, side=70.0)
    V = pkg.synth.samples_host(90, side=70.0)
    k = 20
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, exact_ties=True)
    pos = torch.zeros((len(P), 4), dtype=torch.float32, device="cuda")
    pos[:, :3] = torch.from_numpy(P["ver"].astype(np.float32)).cuda()
    tree = pkg.DeviceTree(pos)
    q = torch.from_numpy(np.ascontiguousarray(V["ver"])).cuda()
    half = len(V) // 2
    parts = [(q[:half].contiguous(), ref_idx[:half]), (q[half:].contiguous(), ref_idx[half:])]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = [torch.empty((p[0].shape[0], k), dtype=torch.int32, device="cuda") for p in parts]
    torch.cuda.synchronize()
    for rep in range(5):
        for (qq, _), st, o in zip(parts, streams, outs):
            tree.query(qq, k, idx=o, stream=st)
        torch.cuda.synchronize()
        for (_, ref), o in zip(parts, outs):
            assert np.array_equal(o.cpu().numpy(), ref), (variant, rep)
    tree.close()


@pytest.mark.parametrize("k,radius", [(8, None), (16, 0.5)])
def test_large_host_call_equals_oracle(k, radius, pkg, pto, torch_cuda):
    """A host-buffer call large enough for the chunk pipeline (8 chunks on 8 streams): same
    results as the oracle from pageable and from pinned caller buffers, repeatedly."""
    torch = torch_cuda
    P = pkg.synth.cloud_host(400_000, seed=51, side=90.0)
    V = pkg.synth.samples_host(270, side=90.0)           # 72 900 samples
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, radius=-1.0 if radius is None else radius)
    ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
    with pkg.Tree(P) as tree:
        for chunks in (8, 1, 3):
            pkg.set_option("host_chunks", chunks)
            out = tree.transfer(V, k, radius=radius, want_idx=True, want_d2=True)
            assert np.array_equal(out["idx"], ref_idx), chunks
            assert np.array_equal(out["d2"], ref_d2), chunks
            _check_blend(out["rgba"], out["normal"], ref_rgba, ref_nrm)
        pkg.set_option("host_chunks", 8)
        m = len(V)
        qpin = torch.from_numpy(V.view(np.uint8).reshape(m, 80)).pin_memory()
        o = {"idx": torch.empty((m, k), dtype=torch.int32).pin_memory().numpy(),
             "rgba": torch.empty((m, 4), dtype=torch.uint8).pin_memory().numpy(),
             "normal": torch.empty((m, 3), dtype=torch.float32).pin_memory().numpy()}
        for _ in range(3):
            tree.transfer(qpin.numpy().view(pkg.POINT_DTYPE).reshape(-1), k, radius=radius, out=o)
            assert np.array_equal(o["idx"], ref_idx)
            _check_blend(o["rgba"], o["normal"], ref_rgba, ref_nrm)


def test_guard_words_stay_intact(pkg, pto, torch_cuda):
    """The library's own bounds check (compute-sanitizer is not available on the GPU pool): with
    option "pool_guard" every device allocation is fenced by 256 bytes of 0xA5 on both sides and
    the fences are compared when the allocation is released.  Ragged sample counts, every kernel
    family, the texture stage and the single-process slabs: no fence may be touched, and the
    results stay those of the oracle."""
    pkg.set_option("pool_guard", 1)
    before = pkg.get_option("pool_guard_hits")
    side = 25.0
    P = pkg.synth.cloud_host(60_001, seed=77, side=side)
    Vall = pkg.synth.samples_host(67, side=side)        # 4 489 samples
    kd = pto.KdTree(P)
    for order in (1, 0, 2):
        pkg.set_option("order", order)
        for variant in (-1, 6, 5, 2, 0):
            pkg.set_option("knn_variant", variant)
            with pkg.Tree(P) as t:
                for m, k, radius in ((1, 1, None), (31, 8, None), (33, 20, 0.4), (1000, 32, None),
                                     (4489, 20, None), (257, 32, 0.3)):
                    V = Vall[:m]
                    ref_idx, ref_d2 = kd.knn(V, k, radius=-1.0 if radius is None else radius)
                    out = t.transfer(V, k, radius=radius, want_idx=True, want_d2=True)
                    assert np.array_equal(out["idx"], ref_idx), (order, variant, m, k)
                    assert np.array_equal(out["d2"], ref_d2)
    pkg.set_option("order", 1)
    pkg.set_option("knn_variant", -1)
    V = Vall.copy()
    V["U"] = V["ver"][:, 0] / side * 0.9 + 0.05
    V["V"] = V["ver"][:, 1] / side * 0.9 + 0.05
    F = pkg.synth.grid_faces(67, 67)
    with pkg.Tree(P) as t:
        t.texture(V, F, k=20, resolution=300)
    with pkg.ShardedTree(P, [0, 0, 0]) as s:
        o = s.transfer(Vall, 20, want_idx=True)
        assert np.array_equal(o["idx"], kd.knn(Vall, 20)[0])
    assert pkg.get_option("pool_guard_hits") == before


@pytest.mark.parametrize("bits", [16, 24, 40, 48, 63])
def test_any_number_of_ordered_key_bits_is_exact(bits, pkg, pto, torch_cuda):
    """The radix sort orders only the top `sort_bits` key bits (auto: 40 or 48).  Cell tables
    are built down to the finest level those bits keep contiguous, so every setting -- also one
    that leaves only 5 levels -- answers exactly, on every kernel."""
    pkg.set_option("sort_bits", bits)
    P = pkg.synth.cloud_host(150_000, seed=91, side=60.0)
    V = pkg.synth.samples_host(50, side=60.0)
    k = 20
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k)
    for variant in (-1, 6, 5):
        pkg.set_option("knn_variant", variant)
        with pkg.Tree(P) as t:
            out = t.transfer(V, k, want_idx=True, want_d2=True)
        assert np.array_equal(out["idx"], ref_idx), (bits, variant)
        assert np.array_equal(out["d2"], ref_d2)


@pytest.mark.parametrize("k,radius", [(1, None), (7, None), (16, None), (16, 0.35), (12, 0.05), (17, None),
                                      (20, None), (32, None), (32, 0.5), (31, 0.08)])
def test_two_samples_per_warp_equals_one_sample_per_warp(k, radius, pkg, pto, torch_cuda):
    """The grid kernel answers two samples per warp (16 lanes each; two neighbours per lane when
    k > 16) when the first attempt is expected to fit (option "grid_pair", default on) and one per
    warp otherwise.  Both forms against the oracle on: an odd number of samples (the
    last pair is half empty), a single sample, a scanned surface, a lattice (every selection is
    ambiguous after truncation: the exact (d2, index) selection runs in both halves), and a cloud
    with a cluster far denser than the rest (more candidates than a half-warp stages: those
    samples are redone by the whole warp)."""
    rng = np.random.default_rng(5)
    surf = pkg.synth.cloud_host(120_001, seed=19, side=50.0)
    g = np.arange(40, dtype=np.float64) * 0.25
    lat = pkg.api.make_points(np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3))
    dense = pkg.synth.cloud_host(60_000, seed=23, side=50.0)
    blob = np.float32(25.0 + 0.4 * rng.standard_normal((40_000, 3))).astype(np.float64)
    dense = np.concatenate([dense, pkg.api.make_points(blob)])
    for name, P, V in (("surface", surf, pkg.synth.samples_host(41, side=50.0)),          # 1 681 samples: odd
                       ("one", surf, pkg.synth.samples_host(41, side=50.0)[777:778]),
                       ("lattice", lat, pkg.api.make_points(lat["ver"][::37] + 0.125)),
                       ("blob", dense, pkg.api.make_points(np.float32(25.0 + 0.5 * rng.standard_normal((999, 3))).astype(np.float64)))):
        ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, radius=-1.0 if radius is None else radius, exact_ties=True)
        ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
        for pair in (2, 1, 0):            # 2: two per warp whatever the expected candidate count
            pkg.set_option("grid_pair", pair)
            pkg.set_option("knn_variant", 6)
            with pkg.Tree(P) as t:
                out = t.transfer(V, k, radius=radius, want_idx=True, want_d2=True)
            assert np.array_equal(out["idx"], ref_idx), (name, pair)
            assert np.array_equal(out["d2"], ref_d2), (name, pair)
            _check_blend(out["rgba"], out["normal"], ref_rgba, ref_nrm)


@pytest.mark.parametrize("min_occ10,admit100,lookup_cost", [(5, 10, 0), (5, 100, 8), (40, 30, 50), (400, 100, 8),
                                                            (40, 300, 0), (2000, 10, 0)])
def test_any_search_schedule_is_exact(min_occ10, admit100, lookup_cost, pkg, pto, torch_cuda):
    """The constants behind the cell tables and the attempt schedule (finest level by points per
    cell, how far a block must reach to be tried first, what a look-up costs) only decide how
    much work an answer takes: tables down to 0.5 points per cell, schedules that start with
    blocks far too small (every sample needs a second attempt or the hand-over) or far too large
    -- all answer exactly, with one and with two samples per warp."""
    pkg.set_option("grid_min_occ10", min_occ10)
    pkg.set_option("grid_admit100", admit100)
    pkg.set_option("grid_lookup_cost", lookup_cost)
    P = pkg.synth.cloud_host(200_000, seed=61, side=80.0)
    V = pkg.synth.samples_host(45, side=80.0)
    kd = pto.KdTree(P)
    for k, radius in ((16, None), (32, None), (5, 0.6)):
        ref_idx, ref_d2 = kd.knn(V, k, radius=-1.0 if radius is None else radius)
        ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
        for pair in (2, 0):
            pkg.set_option("grid_pair", pair)
            with pkg.Tree(P) as t:
                out = t.transfer(V, k, radius=radius, want_idx=True, want_d2=True)
            assert np.array_equal(out["idx"], ref_idx), (k, radius, pair)
            assert np.array_equal(out["d2"], ref_d2)
            _check_blend(out["rgba"], out["normal"], ref_rgba, ref_nrm)


@pytest.mark.parametrize("k", [4, 16, 24])
def test_overflowing_weights_in_one_half_of_a_pair(k, pkg, pto, torch_cuda):
    """Frozen blend, overflow rule: a sample 1e-160 away from a point has d2 = 1e-320 and a weight
    of +inf, so its blend falls back to the nearest neighbour alone.  Here that sample shares a
    warp with an ordinary one (and with another of its kind): each half takes its own branch."""
    rng = np.random.default_rng(11)
    xyz = np.float32(rng.uniform(-1.0, 1.0, (20_000, 3))).astype(np.float64)
    xyz[0] = 0.0
    P = pkg.api.make_points(xyz, normal=rng.standard_normal((len(xyz), 3)),
                            color=rng.integers(0, 256, (len(xyz), 3)))
    q = np.float32(rng.uniform(-0.9, 0.9, (64, 3))).astype(np.float64)
    q[0] = (1e-160, 0.0, 0.0)           # half A overflows, half B ordinary
    q[3] = (0.0, -1e-160, 0.0)          # half B overflows
    q[6] = (1e-160, 1e-160, 0.0)        # both halves
    q[7] = (0.0, 0.0, 1e-161)
    q[10] = (0.0, 0.0, 0.0)             # exact hit next to an overflowing one
    q[11] = (1e-162, 0.0, 0.0)
    V = pkg.api.make_points(q)
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k)
    ref_rgba, ref_nrm = pto.blend(P, ref_idx, ref_d2)
    assert ref_d2[0, 0] > 0.0 and 1.0 / ref_d2[0, 0] == np.inf
    for pair in (2, 0):
        pkg.set_option("grid_pair", pair)
        pkg.set_option("knn_variant", 6)
        with pkg.Tree(P) as t:
            out = t.transfer(V, k, want_idx=True, want_d2=True)
        assert np.array_equal(out["idx"], ref_idx), pair
        assert np.array_equal(out["d2"], ref_d2), pair
        _check_blend(out["rgba"], out["normal"], ref_rgba, ref_nrm)
