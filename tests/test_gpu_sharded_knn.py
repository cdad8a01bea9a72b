"""k-NN and transfer on a sharded cloud (pt_sharded_knn / pt_sharded_transfer, ShardedTree.knn and
.transfer): idx and d2 equal, bit for bit, Tree.knn / Tree.transfer on one index of the same cloud,
and rgba and normal byte for byte, since both paths run the same blend.  Some cases are also checked
against the CPU oracle, so the file does not rest on Tree alone.  Samples always arrive shuffled.
Devices may repeat in the device list, so one GPU runs 1-4 slabs on device 0; with >= 2 GPUs the
slabs also sit on different devices.

Every sharded call must also finish within its attempt budget (DESIGN.md section 6): at most 8
rebuilds, and a halo no wider than the diagonal of the cloud's bounding box.  The clouds that test
this are the ones whose x-cuts leave slabs without a point (a facade at one x, a lattice of two x
columns, one point on two slabs), samples 10^3 and 10^12 extents away from the cloud, and clouds on a
line, whose surface and volume estimates of the k-th-neighbour distance are zero.  The bake and the
normal estimation of a sharded cloud meet the same clouds here."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import test_frames as tf
from test_gpu_parity import GOLDEN, _check_blend
from test_gpu_sharded_bake import EVERYTHING
from test_gpu_sharded_bake import compare as compare_bake
from test_gpu_sharded_normals import VIEW, empty_slab_clouds
from test_gpu_sharded_normals import compare as compare_normals

pytestmark = pytest.mark.gpu

INVALID_ARG = 1                                        # PT_ERR_INVALID_ARG
UNSUPPORTED = 5                                        # PT_ERR_UNSUPPORTED
MAX_REBUILDS = 8                                       # one per widening, 8 answers per call at most
LINE_SPACING = 3.0


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def points(pkg, xyz, seed):
    """Point records with random colours and unit normals, so that every blend depends on which
    neighbours it got."""
    xyz = np.asarray(xyz, np.float64).reshape(-1, 3)
    rng = np.random.default_rng(seed)
    nrm = rng.standard_normal((len(xyz), 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    return pkg.make_points(xyz, normal=nrm.astype(np.float32), color=rng.integers(0, 256, (len(xyz), 3)))


def samples(pkg, xyz, seed=0):
    """Sample records in shuffled order."""
    xyz = np.asarray(xyz, np.float64).reshape(-1, 3)
    return pkg.make_points(xyz[np.random.default_rng(seed).permutation(len(xyz))])


def diagonal(P):
    if len(P) == 0:
        return 0.0
    e = P["ver"].max(0) - P["ver"].min(0)
    return float(np.sqrt((e * e).sum()))


def assert_bounded(info, P):
    """The rebuild loop's termination bound: at most 8 widenings, never past the bounding-box
    diagonal, where every slab that owns a point holds the whole cloud."""
    assert info["rebuilds"] <= MAX_REBUILDS, info
    assert info["halo"] <= diagonal(P) * (1 + 1e-9), (info["halo"], diagonal(P))


def assert_same(got, ref, what=""):
    assert set(got) == set(ref), what
    for key in ref:
        assert got[key].dtype == ref[key].dtype and got[key].shape == ref[key].shape, (key, what)
        assert got[key].tobytes() == ref[key].tobytes(), (key, what)


def compare(pkg, P, Q, devices, calls, coord_mode=0, halo=0.0, k_hint=20):
    """Tree and ShardedTree on the same cloud and samples: knn (idx, d2) and transfer (idx, d2,
    rgba, normal) for every (k, radius) of calls, equal bit for bit.  Returns the single index's
    transfers (one dict per call) and the sharded info."""
    with pkg.Tree(P, coord_mode=coord_mode) as tree:
        refs = [tree.transfer(Q, k, radius=radius, want_idx=True, want_d2=True) for k, radius in calls]
        knns = [tree.knn(Q, k, radius=radius) for k, radius in calls]
    with pkg.ShardedTree(P, devices, halo=halo, k_hint=k_hint, coord_mode=coord_mode) as st:
        for (k, radius), ref, (idx, d2) in zip(calls, refs, knns):
            what = (devices, k, radius)
            assert idx.tobytes() == ref["idx"].tobytes() and d2.tobytes() == ref["d2"].tobytes(), what
            got_idx, got_d2 = st.knn(Q, k, radius=radius)
            assert got_idx.tobytes() == idx.tobytes(), what
            assert got_d2.tobytes() == d2.tobytes(), what
            assert_same(st.transfer(Q, k, radius=radius, want_idx=True, want_d2=True), ref, what)
        info = st.info()
    assert_bounded(info, P)
    return refs, info


def check_oracle(pto, P, Q, ref, k, radius=None):
    """One transfer of compare() against the oracle's exact-tie k-NN and blend on the whole cloud."""
    idx, d2 = pto.KdTree(P).knn(Q, k, radius=-1.0 if radius is None else radius, exact_ties=True)
    assert np.array_equal(ref["idx"], idx), (k, radius)
    assert np.array_equal(ref["d2"], d2), (k, radius)
    rgba, nrm = pto.blend(P, idx, d2)
    _check_blend(ref["rgba"], ref["normal"], rgba, nrm)


# ---- ordinary clouds ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_slabs", [1, 2, 3, 4])
def test_equals_single_index(n_slabs, pkg, pto, torch_cuda):
    P = pkg.synth.cloud_host(60_000, seed=70 + n_slabs, side=40.0)
    Q = samples(pkg, pkg.synth.samples_host(50, side=40.0)["ver"], seed=n_slabs)
    calls = [(1, None), (8, None), (16, 0.5), (20, None), (32, None)]
    refs, info = compare(pkg, P, Q, [0] * n_slabs, calls)
    assert info["n_slabs"] == n_slabs and sum(info["slab_points"]) == len(P)
    assert info["rebuilds"] == 0
    check_oracle(pto, P, Q, refs[2], 16, 0.5)


@pytest.mark.parametrize("path", GOLDEN)
def test_golden_clouds(path, pkg, golden_dir, torch_cuda):
    """Ties, duplicates, exact hits, collinear and coplanar clouds, k > n: the lowest global id wins
    a tie across a cut, whichever slab holds the point as own or ghost.  The fixture's stored answers
    pin the sharded results independently of Tree."""
    g = np.load(os.path.join(golden_dir, path + ".npz"))
    mode = pkg.COORD_F64 if "f64" in path else pkg.COORD_AUTO
    P = pkg.make_points(g["xyz"], normal=g["normal"], color=g["color"])
    radius = float(g["radius"])
    ks = [int(k) for k in g["ks"]]
    # the fixture's samples, then the cloud's own points (exact hits on both sides of every cut)
    rng = np.random.default_rng(3)
    order = rng.permutation(len(g["queries"]))
    own = g["xyz"][::5]
    Q = pkg.make_points(np.r_[g["queries"][order], own[rng.permutation(len(own))]])
    nq = len(order)
    calls = [(k, None) for k in ks] + ([(k, radius) for k in ks] if radius > 0 else [])
    for devices in ([0, 0], [0, 0, 0]):
        refs, _ = compare(pkg, P, Q, devices, calls, coord_mode=mode)
        for k in ks:
            ref = refs[calls.index((k, radius if radius > 0 else None))]
            assert np.array_equal(ref["idx"][:nq], g[f"idx_k{k}"][order]), (path, k)
            assert np.array_equal(ref["d2"][:nq], g[f"d2_k{k}"][order]), (path, k)
            assert np.array_equal(ref["rgba"][:nq], g[f"rgba_k{k}"][order]), (path, k)


def lattice_cloud(pkg):
    x, y, z = np.meshgrid(np.arange(40.0), np.arange(30.0), np.arange(3.0) * 0.5, indexing="ij")
    return points(pkg, np.c_[x.ravel(), y.ravel(), z.ravel()], 9)


def test_cut_on_lattice_points(pkg, pto, torch_cuda):
    """The cuts are sampled x values, so whole columns of lattice points, and of samples placed on
    them, sit exactly on a cut; samples halfway between columns tie across it."""
    P = lattice_cloud(pkg)
    xyz = P["ver"]
    Q = samples(pkg, np.r_[xyz[::3], xyz[::7] + [0.5, 0.0, 0.0], xyz[::11] + [0.5, 0.5, 0.25]], seed=4)
    calls = [(1, None), (8, None), (20, None), (32, None), (16, 1.2)]
    refs, info = compare(pkg, P, Q, [0, 0, 0], calls)
    assert info["rebuilds"] == 0
    check_oracle(pto, P, Q, refs[2], 20)
    check_oracle(pto, P, Q, refs[4], 16, 1.2)


def test_fp64_and_mixed_storage(pkg, torch_cuda):
    rng = np.random.default_rng(12)
    P = pkg.synth.cloud_host(60_000, seed=12, side=30.0)
    Q = samples(pkg, np.r_[pkg.synth.samples_host(40, side=30.0)["ver"], P["ver"][::50]], seed=12)
    calls = [(8, None), (16, 0.3), (32, None)]
    # not fp32-exact anywhere: fp64 storage everywhere
    P64 = pkg.make_points(P["ver"] + 1e-9 * rng.random(P["ver"].shape), normal=P["normal"], color=P["color"])
    compare(pkg, P64, Q, [0, 0, 0], calls, coord_mode=pkg.COORD_F64)
    compare(pkg, P64, Q, [0, 0], calls)
    # fp32-exact on the left half only: the single index and the right slabs store fp64, the left fp32
    mixed = P["ver"].astype(np.float32).astype(np.float64)
    right = mixed[:, 0] > 15.0
    mixed[right] += 1e-9 * rng.random((int(right.sum()), 3))
    Pm = pkg.make_points(mixed, normal=P["normal"], color=P["color"])
    compare(pkg, Pm, Q, [0, 0, 0, 0], calls)


def test_output_combinations(pkg, torch_cuda):
    """Every combination of outputs the C entry points take, including k-NN without a blend output
    (the sharded host then blends into scratch): the same bytes as pt_knn / pt_transfer, and the
    outputs not asked for stay untouched."""
    L, ptr = pkg.lib(), pkg.api._np_ptr
    P = pkg.synth.cloud_host(30_000, seed=14, side=30.0)
    Q = samples(pkg, np.r_[pkg.synth.samples_host(40, side=30.0)["ver"], P["ver"][::40]], seed=14)
    m = len(Q)
    combos = [("knn", i, d, False, False) for i, d in ((1, 0), (1, 1))]
    combos += [("transfer", i, d, c, n) for i in (0, 1) for d in (0, 1) for c, n in ((1, 0), (0, 1), (1, 1))]

    def run(fn_knn, fn_transfer, h, k, radius):
        out = []
        for kind, i, d, c, n in combos:
            o = {"idx": np.full((m, k), 0x5A5A5A5A, np.int32), "d2": np.full((m, k), -7.0),
                 "rgba": np.full((m, 4), 0xA5, np.uint8), "normal": np.full((m, 3), -3.0, np.float32)}
            args = [ptr(o["idx"]) if i else None, ptr(o["d2"]) if d else None]
            if kind == "knn":
                rc = fn_knn(h, ptr(Q), m, k, radius, *args)
            else:
                rc = fn_transfer(h, ptr(Q), m, k, radius, *args, ptr(o["rgba"]) if c else None,
                                 ptr(o["normal"]) if n else None)
            assert rc == 0, (kind, i, d, c, n)
            out.append(o)
        return out

    with pkg.Tree(P) as tree, pkg.ShardedTree(P, [0, 0, 0]) as st:
        for k, radius in ((1, -1.0), (32, -1.0), (16, 0.4)):
            ref = run(L.pt_knn, L.pt_transfer, tree.handle, k, radius)
            got = run(L.pt_sharded_knn, L.pt_sharded_transfer, st._h, k, radius)
            for combo, r, g in zip(combos, ref, got):
                for key in r:
                    assert g[key].tobytes() == r[key].tobytes(), (k, radius, combo, key)
            untouched = ref[0]                                 # idx only: d2, rgba, normal keep the fill
            assert np.all(untouched["d2"] == -7.0) and np.all(untouched["rgba"] == 0xA5)
        assert_bounded(st.info(), P)


# ---- slabs that own no point -------------------------------------------------------------------------------
def around(x_values, yz_lo, yz_hi, per_x, rng):
    """Samples on both sides of, on, and between the given x values, spread over a y-z box."""
    x = np.unique(x_values)
    xs = np.r_[x.min() - 5.0, x.min() - 1.0, x.min() - 0.01, x, 0.5 * (x[:-1] + x[1:]), x.max() + 0.01,
               x.max() + 1.0, x.max() + 5.0]
    yz = yz_lo + rng.random((len(xs) * per_x, 2)) * (np.asarray(yz_hi) - yz_lo)
    return np.c_[np.repeat(xs, per_x), yz]


def case_empty_slabs(pkg, pto, devices=None):
    """The facade at one x (3 slabs, two empty) and the lattice of two x columns (4 slabs, two empty),
    queried on both sides of the populated x values; one point on 2 slabs; an empty cloud on 3."""
    rng = np.random.default_rng(45)
    for c, (P, devs) in enumerate(empty_slab_clouds(pkg)):
        yz = P["ver"][:, 1:]
        Q = samples(pkg, around(P["ver"][:, 0], yz.min(0) - 2.0, yz.max(0) + 2.0, 60, rng), seed=c)
        calls = [(1, None), (8, None), (16, 2.0), (32, None)]
        refs, info = compare(pkg, P, Q, devices or devs, calls)
        if devices is None:
            assert 0 in info["slab_points"]
        if c == 0:
            check_oracle(pto, P, Q, refs[1], 8)
            check_oracle(pto, P, Q, refs[2], 16, 2.0)
    one = points(pkg, [[2.0, 3.0, 4.0]], 1)
    Q = samples(pkg, around([2.0], [0.0, 0.0], [6.0, 8.0], 20, rng), seed=7)
    refs, info = compare(pkg, one, Q, devices or [0, 0], [(1, None), (8, None), (32, 3.0)])
    check_oracle(pto, one, Q, refs[1], 8)
    empty = points(pkg, np.zeros((0, 3)), 2)
    Q = samples(pkg, rng.random((200, 3)) * 10.0 - 5.0, seed=8)
    refs, _ = compare(pkg, empty, Q, devices or [0, 0, 0], [(1, None), (8, 0.5), (32, None)])
    for ref in refs:
        assert np.all(ref["idx"] == -1) and np.all(np.isinf(ref["d2"]))


def test_empty_slabs(pkg, pto, torch_cuda):
    case_empty_slabs(pkg, pto)


# ---- samples far outside the cloud -------------------------------------------------------------------------
def case_far_samples(pkg, devices_list=([0, 0], [0, 0, 0])):
    """The far_samples frame of test_frames.py (a 128 x 100 x 6 cloud, samples 10^3 and 10^12 extents
    out in 14 directions), with samples inside the cloud mixed in."""
    P0, far, _, radius = tf.frame_clouds()["far_samples"]
    P = points(pkg, P0, 5)
    rng = np.random.default_rng(6)
    inner = P0.min(0) + rng.random((200, 3)) * (P0.max(0) - P0.min(0))
    Q = samples(pkg, np.r_[far, inner], seed=6)
    calls = [(16, None), (7, None), (16, radius), (7, radius)]
    for devices in devices_list:
        refs, _ = compare(pkg, P, Q, devices, calls)
    for (k, r), ref in zip(calls, refs):
        idx, d2 = tf.ref_knn(P0, Q["ver"], k, radius=r)
        assert np.array_equal(ref["idx"], idx), (k, r)
        assert np.array_equal(ref["d2"], d2), (k, r)


def test_far_samples(pkg, torch_cuda):
    case_far_samples(pkg)


# ---- clouds on a line ----------------------------------------------------------------------------------------
def line_cloud(pkg, n=1_000, scale=1.0):
    """n points spaced LINE_SPACING along x (times scale, a power of two)."""
    return points(pkg, np.c_[np.arange(n) * LINE_SPACING, np.zeros((n, 2))] * scale, 11)


def line_samples(n=1_000, seed=12):
    """On the line, off it, halfway between points (ties) and beyond both ends; dyadic, so that
    scaling by a power of two is exact."""
    rng = np.random.default_rng(seed)
    x = np.round(rng.uniform(-30.0, n * LINE_SPACING + 30.0, 300) * 16) / 16
    off = np.round(rng.normal(0.0, 2.0, (300, 2)) * 16) / 16
    off[::3] = 0.0
    mid = np.c_[(np.arange(0, n - 1, 7) + 0.5) * LINE_SPACING, np.zeros((len(range(0, n - 1, 7)), 2))]
    return np.r_[np.c_[x, off], mid]


def case_line_clouds(pkg, pto, devices_list=([0, 0], [0, 0, 0])):
    """k up to 32 on 2 and 3 slabs, at three scales: identical idx, d2 scaled by exactly 4^s."""
    xyz = line_samples()
    calls = [(16, None), (32, None), (16, 10.0)]
    base = {}
    for s in (0, -8, 8):
        scale = 2.0 ** s
        P = line_cloud(pkg, scale=scale)
        Q = samples(pkg, xyz * scale, seed=13)
        for devices in devices_list:
            cs = [(k, None if r is None else r * scale) for k, r in calls]
            refs, _ = compare(pkg, P, Q, devices, cs)
            _, info = compare(pkg, P, Q, devices, cs[:2], halo=1e-4 * scale)
            assert info["rebuilds"] > 0
            for c, ref in enumerate(refs):
                if s == 0:
                    base[devices[0], len(devices), c] = ref
                    continue
                b = base[devices[0], len(devices), c]
                assert np.array_equal(ref["idx"], b["idx"]), (s, devices, calls[c])
                assert np.array_equal(ref["d2"], b["d2"] * 4.0 ** s), (s, devices, calls[c])
        if s == 0:
            check_oracle(pto, P, Q, refs[1], 32)


def test_line_clouds(pkg, pto, torch_cuda):
    case_line_clouds(pkg, pto)


# ---- the rebuild loop across the host pipeline's chunks ---------------------------------------------------
def case_rebuild_across_chunks(pkg, chunk_options=(1, 8, 16), devices=(0, 0)):
    """About 100 000 samples, so host_query cuts each slab's rows into chunks (option host_chunks);
    a halo of 1e-4; only the samples at the end of the batch sit next to a cut, so only the last
    chunk of each slab flags its step."""
    rng = np.random.default_rng(8)
    n, R = 120_000, len(devices)
    xyz = np.c_[rng.random((n, 2)) * 60.0, rng.random(n) * 0.5]
    P = points(pkg, xyz, 8)
    cuts = np.sort(xyz[:, 0])[[n * r // R for r in range(1, R)]]          # the build's quantile cuts
    bulk = np.c_[rng.random((130_000, 2)) * 60.0, rng.random(130_000) * 0.5]
    bulk = bulk[np.abs(bulk[:, :1] - cuts[None, :]).min(1) > 3.0][:100_000]
    edge = np.c_[np.repeat(cuts, 64) + rng.uniform(-0.05, 0.05, 64 * (R - 1)),
                 rng.random((64 * (R - 1), 2)) * [60.0, 0.5]]
    Q = np.concatenate([samples(pkg, bulk, seed=9), samples(pkg, edge, seed=10)])
    old = pkg.get_option("host_chunks")
    try:
        for chunks in chunk_options:
            pkg.set_option("host_chunks", chunks)
            _, info = compare(pkg, P, Q, list(devices), [(16, None), (8, 0.3)], halo=1e-4)
            assert info["rebuilds"] > 0 and min(info["slab_points"]) > 0, chunks
    finally:
        pkg.set_option("host_chunks", old)
    assert pkg.get_option("host_chunks") == old


def test_rebuild_across_host_chunks(pkg, torch_cuda):
    case_rebuild_across_chunks(pkg)


# ---- error codes and guard words ---------------------------------------------------------------------------
def test_error_codes(pkg, torch_cuda):
    """The same status as pt_knn / pt_transfer on a Tree of the same cloud."""
    L, ptr = pkg.lib(), pkg.api._np_ptr
    P = pkg.synth.cloud_host(2_000, seed=1, side=10.0)
    Q = samples(pkg, pkg.synth.samples_host(10, side=10.0)["ver"])
    m = len(Q)
    idx, d2 = np.empty((m, 33), np.int32), np.empty((m, 33))
    rgba, nrm = np.empty((m, 4), np.uint8), np.empty((m, 3), np.float32)
    # (k, m, queries, idx, d2) for knn, then (k, m, queries, idx, d2, rgba, normal) for transfer
    knn_cases = [(0, m, Q, idx, d2), (33, m, Q, idx, d2), (8, m, Q, None, d2), (8, m, None, idx, d2),
                 (8, 0, Q, None, None), (0, 0, Q, idx, None), (8, m, Q, idx, None), (32, m, Q, idx, d2)]
    transfer_cases = [(0, m, Q, idx, d2, rgba, nrm), (33, m, Q, None, None, rgba, None),
                      (8, m, Q, idx, d2, None, None), (8, m, None, None, None, rgba, nrm),
                      (8, 0, Q, None, None, None, None), (33, 0, Q, None, None, None, None),
                      (8, m, Q, None, None, None, nrm), (1, m, Q, idx, d2, rgba, nrm)]

    def codes(knn, transfer, h):
        return ([knn(h, ptr(q), mm, k, -1.0, ptr(i), ptr(d)) for k, mm, q, i, d in knn_cases],
                [transfer(h, ptr(q), mm, k, -1.0, ptr(i), ptr(d), ptr(c), ptr(n))
                 for k, mm, q, i, d, c, n in transfer_cases])
    with pkg.Tree(P) as tree:
        ref = codes(L.pt_knn, L.pt_transfer, tree.handle)
    with pkg.ShardedTree(P, [0, 0]) as st:
        got = codes(L.pt_sharded_knn, L.pt_sharded_transfer, st._h)
    assert got == ref
    assert ref[0] == [UNSUPPORTED, UNSUPPORTED, INVALID_ARG, INVALID_ARG, 0, UNSUPPORTED, 0, 0]
    assert ref[1] == [UNSUPPORTED, UNSUPPORTED, INVALID_ARG, INVALID_ARG, 0, UNSUPPORTED, 0, 0]
    null = ctypes.c_void_p()
    assert L.pt_sharded_knn(null, ptr(Q), m, 8, -1.0, ptr(idx), None) == L.pt_knn(null, ptr(Q), m, 8, -1.0, ptr(idx),
                                                                                 None) == INVALID_ARG
    assert (L.pt_sharded_transfer(null, ptr(Q), m, 8, -1.0, None, None, ptr(rgba), None)
            == L.pt_transfer(null, ptr(Q), m, 8, -1.0, None, None, ptr(rgba), None) == INVALID_ARG)


def test_guard_words_through_rebuilds(pkg, pto, torch_cuda):
    """Option "pool_guard" fences every device allocation; the rebuild path frees and reallocates every
    slab, and no fence may be touched over the empty-slab, far-sample, line and chunk cases."""
    old = pkg.get_option("pool_guard")
    pkg.set_option("pool_guard", 1)
    try:
        before = pkg.get_option("pool_guard_hits")
        case_empty_slabs(pkg, pto)
        case_far_samples(pkg, devices_list=([0, 0, 0],))
        case_line_clouds(pkg, pto, devices_list=([0, 0, 0],))
        case_rebuild_across_chunks(pkg, chunk_options=(8,))
        assert pkg.get_option("pool_guard_hits") == before
    finally:
        pkg.set_option("pool_guard", old)


# ---- the same clouds through the sharded bake and normal estimation ---------------------------------------
def strip_mesh(pkg, x0, x1, y, z, g=24):
    """A strip of 2 (g - 1) triangles along x at height z over the line y, normals tilted towards +z."""
    x = np.linspace(x0, x1, g)
    xyz = np.r_[np.c_[x, np.full(g, y - 1.0), np.full(g, z)], np.c_[x, np.full(g, y + 1.0), np.full(g, z)]]
    uv = np.r_[np.c_[np.linspace(0.05, 0.95, g), np.full(g, 0.3)], np.c_[np.linspace(0.05, 0.95, g), np.full(g, 0.7)]]
    V = pkg.make_points(xyz, normal=np.tile([0.1, -0.2, 1.0], (2 * g, 1)), uv=uv)
    F = np.array([f for i in range(g - 1) for f in ([i, i + 1, g + i + 1], [i, g + i + 1, g + i])], np.int32)
    return V, F


def wall_mesh(pkg, x, y0, y1, z0, z1, g=12):
    """A g x g grid in the plane at x, normals towards -x."""
    u, v = np.meshgrid(np.linspace(0.0, 1.0, g), np.linspace(0.0, 1.0, g))
    u, v = u.ravel(), v.ravel()
    xyz = np.c_[np.full(g * g, x), y0 + u * (y1 - y0), z0 + v * (z1 - z0)]
    V = pkg.make_points(xyz, normal=np.tile([-1.0, 0.2, 0.1], (g * g, 1)), uv=np.c_[u * 0.9 + 0.05, v * 0.9 + 0.05])
    return V, pkg.synth.grid_faces(g, g)


def test_bake_on_empty_side_far_and_line(pkg, torch_cuda):
    # the facade at x = 7.25 on 3 slabs, a wall mesh on its empty side (x < every cut)
    P, devices = next(empty_slab_clouds(pkg))
    V, F = wall_mesh(pkg, 3.0, -1.0, 21.0, -1.0, 21.0)
    _, info = compare_bake(pkg, P, V, F, devices, k=16, resolution=200, want=EVERYTHING)
    assert 0 in info["slab_points"]
    assert_bounded(info, P)
    # a mesh 10^3 extents above the far_samples cloud, across every cut
    P0, _, _, _ = tf.frame_clouds()["far_samples"]
    P = points(pkg, P0, 5)
    V, F = strip_mesh(pkg, -10.0, 138.0, 50.0, 1.28e5)
    for devices in ([0, 0], [0, 0, 0]):
        _, info = compare_bake(pkg, P, V, F, devices, k=16, resolution=128, want=EVERYTHING)
        assert_bounded(info, P)
    # the line cloud with a strip along it
    P = line_cloud(pkg)
    V, F = strip_mesh(pkg, -20.0, 3020.0, 0.0, 0.5)
    for devices, k in (([0, 0], 16), ([0, 0, 0], 32)):
        _, info = compare_bake(pkg, P, V, F, devices, k=k, resolution=256, want=EVERYTHING)
        assert_bounded(info, P)


def test_normals_on_line_cloud(pkg, torch_cuda):
    for s in (0, -8, 8):
        P = line_cloud(pkg, scale=2.0 ** s)
        for devices in ([0, 0], [0, 0, 0]):
            info = compare_normals(pkg, P, devices, [(16, None, None), (32, None, VIEW), (8, 10.0 * 2.0 ** s, None)])
            assert_bounded(info, P)


def test_cli_with_mesh_on_empty_side(pkg, torch_cuda, tmp_path):
    """`pointsTransfer -g 2` on the facade, its mesh on the side of the slab that owns no point: the
    same texture.png as `pointsTransfer` on one index."""
    from test_cli import CLI, write_cloud, write_mesh
    if not os.path.exists(CLI):
        subprocess.run(["make", "-C", os.path.dirname(CLI)], check=True, stdout=subprocess.DEVNULL)
    P, _ = next(empty_slab_clouds(pkg))
    V, F = wall_mesh(pkg, 3.0, -1.0, 21.0, -1.0, 21.0)
    write_cloud(tmp_path / "c.ply", P)
    write_mesh(tmp_path / "m.ply", V, F)
    pngs = []
    for g in ([], ["-g", "2"]):
        d = tmp_path / ("g" if g else "one")
        d.mkdir()
        r = subprocess.run([CLI, *g, "-R", "256", str(tmp_path / "c.ply"), str(tmp_path / "m.ply")],
                           capture_output=True, text=True, cwd=d)
        assert r.returncode == 0 and "failed" not in r.stderr, r.stderr
        pngs.append((d / "texture.png").read_bytes())
    assert pngs[0] == pngs[1]


# ---- distinct devices ----------------------------------------------------------------------------------------
def test_distinct_devices(pkg, pto, golden_dir, torch_cuda):
    if torch_cuda.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    g = np.load(os.path.join(golden_dir, "lattice_ties.npz"))
    P = pkg.make_points(g["xyz"], normal=g["normal"], color=g["color"])
    Q = samples(pkg, np.r_[g["queries"], g["xyz"][::5]])
    for devices in ([0, 1], [0, 1, 0, 1], [1, 0]):
        compare(pkg, P, Q, devices, [(1, None), (8, None), (32, None)])
    case_empty_slabs(pkg, pto, devices=[0, 1])
    case_far_samples(pkg, devices_list=([0, 1], [1, 0, 1]))
    case_line_clouds(pkg, pto, devices_list=([0, 1],))
    case_rebuild_across_chunks(pkg, chunk_options=(8,), devices=(1, 0))
