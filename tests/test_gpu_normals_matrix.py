"""Normal estimation and orientation under every k-NN kernel a self-query can take, and at the edges
of the PCA and Boruvka kernels, bit for bit against the CPU oracles.

Both features get their lists from launch_query (self_query_chunks): every sample lies on a cloud
point (the first neighbour has d2 = 0, duplicates tie at 0) and samples arrive in curve order, 32
sorted rows per warp.  Here each option that picks a kernel (knn_variant, order, grid_pair,
grid_span, queue_cap, sort_bits) is run on a scanned surface, a lattice with duplicated points and a
dense blob in a sparse cloud, on F32 and F64 indexes; then every lane-group width of
normals_pca_kernel with short and full lists mixed in one warp, chunk edges at 2^22 rows, degenerate
spectra (also with subnormal scatter) and the tie-breaking of the orientation forest.  Where normals
or orientation differ from the oracle, the message says whether the index's own k-NN of the
differing points equals pto.knn_bruteforce, which tells a k-NN fault from a PCA or forest fault."""
import numpy as np
import pytest

import test_normals as tn
import test_orient as to
from oracle import pto_normals, pto_orient
from test_gpu_parity import MODES

pytestmark = pytest.mark.gpu

CHUNK = 1 << 22                       # HEIGHT_CHUNK: sorted rows per self-query chunk


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
    pkg.set_option("knn_variant", -1)     # auto (the default)
    pkg.set_option("queue_cap", 1 << 20)  # the compiled capacity
    pkg.set_option("order", 1)            # Hilbert order + cell tables (the default)
    pkg.set_option("grid_tma", 1)
    pkg.set_option("pool_guard", 0)
    pkg.set_option("sort_bits", 0)
    pkg.set_option("grid_pair", 1)
    pkg.set_option("grid_span", 1)
    pkg.set_option("grid_admit100", 100)
    pkg.set_option("grid_lookup_cost", 8)
    pkg.set_option("grid_min_occ10", 40)


# every kernel and hand-over path of launch_query: the (knn_variant, order) pairs of the parity
# suite, then the grid kernel with one sample per warp, the pair and span kernels, a traversal queue
# of 2 (the give-up path and the warp kernel behind it), and a 16-bit sort
MATRIX = [{"knn_variant": v, "order": o} for v, o in MODES] + [
    {"knn_variant": 6, "grid_pair": 0},
    {"knn_variant": 6, "grid_pair": 2, "grid_span": 0},
    {"knn_variant": 6, "grid_pair": 2, "grid_span": 1},
    {"knn_variant": 2, "queue_cap": 2},
    {"knn_variant": 5, "queue_cap": 2},
    {"knn_variant": 6, "queue_cap": 2},
    {"sort_bits": 16},
    {"knn_variant": 6, "grid_pair": 2, "sort_bits": 16},
]
RUNS = ((7, None), (18, None), (18, 0.3))      # a short k, a long k, and a radius-bounded run


def mode_id(mode):
    return "-".join(f"{key}{v}" for key, v in mode.items())


def set_mode(pkg, mode):
    for key, v in mode.items():
        pkg.set_option(key, v)


def knn_report(pto, tree, P, ref_idx, rows, k, radius):
    """The index's own k-NN of the points `rows` (at most 64) against brute force and the oracle's
    self-query lists: equal lists put the fault in the PCA or orientation kernels."""
    rows = np.asarray(rows)[:64]
    Q = P[rows]
    got, _ = tree.knn(Q, k, radius=radius)
    bf, _ = pto.knn_bruteforce(P, Q, k, radius=-1.0 if radius is None else radius)
    return (f"tree.knn of {len(rows)} of those points {'equals' if np.array_equal(got, bf) else 'DIFFERS from'} "
            f"brute force, which {'equals' if np.array_equal(bf, ref_idx[rows]) else 'DIFFERS from'} the oracle's lists")


def check_normals(pto, tree, P, got, ref, idx, radius, what):
    ref_n, ref_v, ref_e = ref
    bad = np.flatnonzero((got["normal"].view(np.uint32) != ref_n.view(np.uint32)).any(1) |
                         (got["variation"].view(np.uint32) != ref_v.view(np.uint32)))
    if len(bad):
        pytest.fail(f"{what}: {len(bad)} normals differ from the oracle (rows {bad[:8].tolist()}); "
                    + knn_report(pto, tree, P, idx, bad, idx.shape[1], radius))
    if "stats" in got:
        assert got["stats"]["estimated"] == ref_e, what


def check_orient(pto, tree, P, got, ref, idx, radius, what):
    bad = np.flatnonzero((got["normal"].view(np.uint32) != ref["normal"].view(np.uint32)).any(1) |
                         (got["root"] != ref["root"]))
    counts = {key: (got["stats"][key], ref[key]) for key in ("oriented", "flipped", "components", "edges")}
    if len(bad) or any(a != b for a, b in counts.values()):
        pytest.fail(f"{what}: {len(bad)} points differ from the oracle (rows {bad[:8].tolist()}), counts "
                    f"(got, oracle) {counts}; " + knn_report(pto, tree, P, idx, bad if len(bad) else np.arange(64),
                                                              idx.shape[1], radius))


# ---- 1. the kernel matrix ----------------------------------------------------------------------------
def matrix_clouds(pkg):
    """Point records: a scanned surface, a lattice with every third and seventh point duplicated, and
    a dense blob inside a sparse cloud (more candidates than a half-warp stages: redone by the whole
    warp or handed over).  fp32-representable; every fifth normal is zero (rule (c) in estimation,
    left out of orientation), the others have random signs."""
    rng = np.random.default_rng(20261021)
    surf = pkg.synth.cloud_host(120_001, seed=19, side=50.0)
    g = np.arange(28, dtype=np.float64) * 0.25
    lat = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    lat = np.r_[lat, lat[::3], lat[::7]]
    lat = pkg.make_points(lat, normal=rng.standard_normal(lat.shape))
    blob = np.float32(25.0 + 0.4 * rng.standard_normal((40_000, 3))).astype(np.float64)
    dense = np.concatenate([pkg.synth.cloud_host(60_000, seed=23, side=50.0),
                            pkg.make_points(blob, normal=rng.standard_normal(blob.shape))])
    out = {}
    for name, P in (("surface", surf), ("lattice", lat), ("blob", dense)):
        P = P.copy()
        P["normal"] *= np.where(rng.random(len(P)) < 0.5, -1.0, 1.0)[:, None]
        P["normal"][::5] = 0.0
        out[name] = P
    return out


@pytest.fixture(scope="module")
def matrix_refs(pkg, pto, torch_cuda):
    """cloud -> (P, {(k, radius): (lists, normals oracle, orientation oracle)})."""
    out = {}
    for name, P in matrix_clouds(pkg).items():
        xyz, m = P["ver"], P["normal"].astype(np.float32)
        refs = {}
        for k, radius in RUNS:
            idx = pto_normals.neighbours(xyz, k, -1.0 if radius is None else radius)
            refs[k, radius] = (idx, pto_normals.estimate(xyz, m, idx), pto_orient.orient(xyz, m, idx))
        out[name] = (P, refs)
    return out


@pytest.mark.parametrize("mode", MATRIX, ids=mode_id)
def test_kernel_matrix(mode, pkg, pto, matrix_refs, torch_cuda):
    variant = mode.get("knn_variant", -1)
    for name, (P, refs) in matrix_refs.items():
        for coord in (pkg.COORD_F32, pkg.COORD_F64):
            set_mode(pkg, mode)
            fallbacks = []
            with pkg.Tree(P, coord_mode=coord) as tree:
                assert tree.info().coord_mode == coord
                for (k, radius), (idx, ref_n, ref_o) in refs.items():
                    what = (name, coord, k, radius)
                    got = tree.estimate_normals(k, radius=radius)
                    if (name == "surface" and coord == pkg.COORD_F32 and k <= 16 and radius is None and variant == 6
                            and "sort_bits" not in mode):
                        # the span and pair kernels are reached where they are meant to be
                        pair, span = mode.get("grid_pair", 1), mode.get("grid_span", 1)
                        if pair == 2:
                            assert pkg.get_option("grid_span_used") == span, what
                            assert pkg.get_option("grid_pair_used") == 1 - span, what
                        if pair == 0:
                            assert pkg.get_option("grid_span_used") == 0, what
                            assert pkg.get_option("grid_pair_used") == 0, what
                    fallbacks.append(tree.info().last_fallback_samples)
                    check_normals(pto, tree, P, got, ref_n, idx, radius, what)
                    check_orient(pto, tree, P, tree.orient_normals(k, radius=radius), ref_o, idx, radius, what)
            if mode.get("queue_cap") == 2 and variant in (2, 5):
                assert max(fallbacks) > 0, (name, coord, fallbacks)      # the give-up path was taken


# ---- 2. every lane-group width ------------------------------------------------------------------------
WIDTH_KS = (3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32)      # groups of 4, 8, 16, 32 lanes, full and partial


def molecules(sizes, count, seed):
    """xyz of `count` molecules 4 apart, each made of groups 3 apart whose sizes are `sizes` (one
    array per molecule, or one for all), every group inside a ball of radius 0.3: with a radius of 1
    a point's list holds exactly the points of its group, at most k of them."""
    rng = np.random.default_rng(seed)
    pts = []
    for c in range(count):
        s = sizes[c] if isinstance(sizes[0], (list, tuple, np.ndarray)) else sizes
        for gi, size in enumerate(s):
            centre = np.array([c * 4.0, gi * 3.0, 0.0])
            d = rng.standard_normal((size, 3))
            d *= (0.3 * rng.random(size) ** (1 / 3) / np.linalg.norm(d, axis=1))[:, None]
            pts.append(centre + d)
    return np.concatenate(pts).astype(np.float32).astype(np.float64)


def list_kinds(idx):
    """(full, short with >= 3 entries, fewer than 3) rows of the lists."""
    cnt = (idx >= 0).sum(1)
    k = idx.shape[1]
    return cnt == k, (cnt >= 3) & (cnt < k), cnt < 3


def test_every_lane_group_width(pkg, pto, torch_cuda):
    """Every k of each group width on a scanned surface, with the input-normal rule and with a
    viewpoint."""
    P = pkg.synth.cloud_host(50_000, seed=29, side=40.0)
    P["normal"][::4] = 0.0
    xyz, m = P["ver"], P["normal"].astype(np.float32)
    bare = pkg.make_points(xyz)
    for cloud, nrm, view in ((P, m, None), (bare, None, (20.0, 20.0, 60.0))):
        with pkg.Tree(cloud) as tree:
            for k in WIDTH_KS:
                idx = pto_normals.neighbours(xyz, k)
                got = tree.estimate_normals(k, viewpoint=view)
                check_normals(pto, tree, cloud, got, pto_normals.estimate(xyz, nrm, idx, view), idx, None, (k, view))


def test_short_lists_next_to_full_ones_in_one_warp(pkg, pto, torch_cuda):
    """A radius that cuts lists short inside the lane groups: full lists, short ones with at least 3
    entries and ones with fewer than 3 (no estimate) side by side.  First a cloud of at most 32
    points for every k up to 17 -- one warp holds all its rows, whatever the curve order, so the
    three kinds provably share a warp (and the warp is partly empty) -- then, for every k, 1 500
    molecules whose groups have 40 points (full), 3..30 (short or full) and 1 and 2 (fewer than 3)."""
    rng = np.random.default_rng(31)
    for k in WIDTH_KS:
        if k + 6 <= 32:
            xyz = molecules([k, 3, 1, 2] if k > 3 else [3, 1, 2], 1, seed=k)
            idx = pto_normals.neighbours(xyz, k, 1.0)
            full, short, few = list_kinds(idx)
            assert len(xyz) <= 32 and full.any() and few.any() and (short.any() or k == 3), k
            with pkg.Tree(pkg.make_points(xyz)) as tree:
                got = tree.estimate_normals(k, radius=1.0)
                check_normals(pto, tree, pkg.make_points(xyz), got, pto_normals.estimate(xyz, None, idx), idx, 1.0,
                              ("one warp", k))
    sizes = [[40, int(s), 1, 2] for s in rng.integers(3, 31, 1500)]
    xyz = molecules(sizes, 1500, seed=32)
    m = rng.standard_normal(xyz.shape).astype(np.float32)
    P = pkg.make_points(xyz, normal=m)
    with pkg.Tree(P) as tree:
        for k in WIDTH_KS:
            idx = pto_normals.neighbours(xyz, k, 1.0)
            full, short, few = list_kinds(idx)
            assert full.any() and few.any() and (short.any() or k == 3), k
            check_normals(pto, tree, P, tree.estimate_normals(k, radius=1.0), pto_normals.estimate(xyz, m, idx), idx,
                          1.0, ("molecules", k))


# ---- 3. chunk edges ------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [CHUNK - 1, CHUNK, CHUNK + 1, CHUNK + 33])
def test_chunk_edges(n, pkg, pto, torch_cuda):
    """n at and around one chunk of 2^22 sorted rows; 2^22 + 33 leaves a last chunk of one full warp
    and one warp with a single row.  Every row is compared, so the last two warps of each chunk are;
    at 2^22 + 1 orientation too, with random signs, over the whole cloud."""
    torch = torch_cuda
    pos, attrs = pkg.synth.cloud_device(n, seed=20261018 + 2, u1=410.0, v1=410.0)   # ~0.2 apart
    if n == CHUNK + 1:
        flip = torch.from_numpy(np.where(np.random.default_rng(8).random(n) < 0.5, -1.0, 1.0).astype(np.float32))
        attrs.view(torch.float32).view(n, 4)[:, :3] *= flip.cuda()[:, None]
    P = pkg.synth.points_to_host(pos, attrs)
    xyz, m = P["ver"], P["normal"].astype(np.float32)
    tree = pkg.DeviceTree(pos, attrs)
    normal = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    variation = torch.empty(n, dtype=torch.float32, device="cuda")
    try:
        for k in (9, 31) if n == CHUNK + 33 else (9,):
            tree.estimate_normals(k, normal=normal, variation=variation)
            torch.cuda.synchronize()
            idx = pto_normals.neighbours(xyz, k)
            got = {"normal": normal.cpu().numpy(), "variation": variation.cpu().numpy()}
            check_normals(pto, tree, P, got, pto_normals.estimate(xyz, m, idx), idx, None, (n, k))
        if n == CHUNK + 1:
            idx = pto_normals.neighbours(xyz, 18)
            ref = pto_orient.orient(xyz, m, idx)
            assert ref["flipped"] > n // 4
            check_orient(pto, tree, P, tree.orient_normals(18), ref, idx, None, n)
    finally:
        tree.close()


# ---- 4. degenerate spectra -----------------------------------------------------------------------------
@pytest.mark.parametrize("kind", sorted(tn.DEGENERATE))
def test_degenerate_spectra(kind, pkg, pto, torch_cuda):
    """Isotropic neighbourhoods (three equal eigenvalues), collinear runs (two equal smallest) and
    exact planes (a zero smallest), each with the input-normal rule, a viewpoint and the
    largest-component rule, on F32 and F64 indexes; then the same cloud scaled by 2^-530 (subnormal
    scatter products) on an F64 index."""
    xyz, k, aligned = tn.degenerate_cloud(kind)
    nrm = tn.degenerate_normals(len(xyz))
    idx = pto_normals.neighbours(xyz, k)
    tiny = np.ldexp(xyz, tn.TINY)
    idx_tiny = pto_normals.neighbours(tiny, k)
    rules = ((nrm, None), (None, (100.0, -30.0, 70.0)), (None, None))
    for pts, lists, coords in ((xyz, idx, (pkg.COORD_F32, pkg.COORD_F64)), (tiny, idx_tiny, (pkg.COORD_F64,))):
        for coord in coords:
            for normal, view in rules:
                P = pkg.make_points(pts, normal=normal)
                ref = pto_normals.estimate(pts, normal, lists, view)
                assert ref[2] == len(pts)
                with pkg.Tree(P, coord_mode=coord) as tree:
                    assert tree.info().coord_mode == coord
                    got = tree.estimate_normals(k, viewpoint=view)
                    check_normals(pto, tree, P, got, ref, lists, None, (kind, pts is tiny, coord, view))
                if normal is None and view is None:
                    tn.check_exact_scatter(kind, aligned, got["normal"], got["variation"])


# ---- 5. orientation ties -------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(to.TIE_CLOUDS))
def test_orientation_ties(name, pkg, pto, torch_cuda):
    """All weights 0 on a flat lattice (ids in lattice order and shuffled), many points sharing the
    top z (-0.0 with +0.0), and 3 000 components whose tied weights close frustrated triangles."""
    xyz, m, radius = to.TIE_CLOUDS[name]()
    lists = {k: pto_normals.neighbours(xyz, k, -1.0 if radius is None else radius) for k in (2, 8, 32)}
    refs = {k: pto_orient.orient(xyz, m, idx) for k, idx in lists.items()}
    for k, idx in lists.items():
        to.check_tie_cloud(name, xyz, m, idx, refs[k])
    P = pkg.make_points(xyz, normal=m)
    for coord in (pkg.COORD_F32, pkg.COORD_F64):
        with pkg.Tree(P, coord_mode=coord) as tree:
            for k, idx in lists.items():
                check_orient(pto, tree, P, tree.orient_normals(k, radius=radius), refs[k], idx, radius, (name, coord, k))


# ---- 6. bakes under the kernel matrix ------------------------------------------------------------------
@pytest.fixture(scope="module")
def bake_case(pkg, torch_cuda):
    """A modest bake and its outputs under the default options (which the bake suites pin to the
    oracle)."""
    from test_bake import grid_mesh
    from test_bake_tangent import ALL_OUTPUTS
    side = 30.0
    P = pkg.synth.cloud_host(60_000, seed=9, side=side)
    V, F = grid_mesh(pkg, 12, side)
    want = ALL_OUTPUTS + ("height",)
    with pkg.Tree(P) as tree:
        ref = tree.bake(V, F, k=16, resolution=200, want=want)
    return P, V, F, want, ref


@pytest.mark.parametrize("mode", MATRIX, ids=mode_id)
def test_bake_under_kernel_matrix(mode, pkg, bake_case):
    P, V, F, want, ref = bake_case
    set_mode(pkg, mode)
    with pkg.Tree(P) as tree:
        got = tree.bake(V, F, k=16, resolution=200, want=want)
    for key in want:
        assert got[key].tobytes() == ref[key].tobytes(), key
    assert got["stats"]["texels"] == ref["stats"]["texels"] and got["height_range"] == ref["height_range"]
