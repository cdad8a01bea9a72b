"""k-NN exactness in real-world coordinate frames and at saturated cell counts, on the GPU, under every
kernel a query can take (MATRIX of test_gpu_normals_matrix).

a. Frames against the oracle (pinned on numpy in each frame by test_frames.py): UTM easting /
   northing with mm quantisation (F64 storage), an offset below 2^19 on the 2^-4 lattice (F32 storage
   where fp32 boxes are coarse), a 1e-3-wide patch at a UTM offset, a plane at z = 312 and samples
   1e3 and 1e12 extents outside the cloud; idx and d2 bit for bit, the blend at the suite's bars.
b. Identities without an oracle on a 300 000-point dyadic cloud: the same idx and d2 under dyadic
   translations (F32 and F64 storage), and the same idx with d2 times exactly 4^s under 2^s scaling,
   with d2 below the fp32 normal range (s = -70), above FLT_MAX (s = 70) and in range (+-10, +-40).
c. Which path answered: the cloud's x extent is 128, so every cell boundary, every sample and every
   d2 lies on a dyadic grid, and fmin(k-th d2, r^2) differs from the squared distance to any block
   face by at least 2^-12 unless equal -- far more than the termination slack at a UTM offset
   (64 eps |x| + 1.8e-15 |q| ~ 1e-7).  The lattice coordinates, the level choice and the candidate
   caps are the same in every translated frame, so the grid hands over exactly as many samples as
   at the origin; under 2^s scaling everything the grid and the box pyramid compute scales exactly.
   The counts are asserted equal, and the grid is asserted to answer most samples itself.
d. Saturated cell counts: a parent cell of 65 533 .. 200 000 duplicates, or a jittered blob of 70 000
   points in one child next to sparse siblings, whose 16-bit cumulative counts saturate; the build's
   level choice is restated in numpy to assert the count each case names.
e. Consumers in one UTM frame: the bake (colour, tangent, height), normal estimation and
   orientation, the sharded bake and the slab-sharded transfer with cuts at UTM x values."""
import numpy as np
import pytest

import orient_oracle
import test_frames as tf
from oracle import pto_normals
from test_bake import grid_mesh
from test_bake_height import check_height
from test_bake_tangent import check_bake_ex, tilted_normals
from test_gpu_normals_matrix import MATRIX, check_normals, check_orient, mode_id, set_mode
from test_gpu_parity import _check_blend
from test_gpu_sharded_bake import EVERYTHING, compare
from test_gpu_slab_emulated import Slabs, _check, _exchange_step

pytestmark = pytest.mark.gpu

# the MATRIX entries that build cell tables and query them (order 2 has none)
GRID_MODES = [m for m in MATRIX if m.get("knn_variant", -1) in (-1, 6) and m.get("order", 1) != 2]
HANDOVER_LOG = []       # (what, counts): printed at the end of the module


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    yield torch
    for what, counts in HANDOVER_LOG:
        print("fallback_counts", what, counts)


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


def storage(pkg, name):
    return pkg.COORD_F32 if name == "f32" else pkg.COORD_F64


def with_attrs(pkg, xyz, seed):
    rng = np.random.default_rng(seed)
    return pkg.make_points(xyz, normal=rng.standard_normal(xyz.shape), color=rng.integers(0, 256, xyz.shape))


# ---- a. frames against the oracle ----------------------------------------------------------------------
@pytest.fixture(scope="module")
def frame_refs(pkg, pto):
    out = {}
    for i, (name, (P, Q, kind, radius)) in enumerate(tf.frame_clouds().items()):
        pts, qs = with_attrs(pkg, P, 70 + i), pkg.make_points(Q)
        tree = pto.KdTree(pts)
        runs = {}
        for k, r in ((16, None), (7, None), (16, radius)):
            idx, d2 = tree.knn(qs, k, radius=-1.0 if r is None else r, exact_ties=True)
            runs[k, r] = (idx, d2) + pto.blend(pts, idx, d2)
        out[name] = (pts, qs, kind, runs)
    return out


@pytest.mark.parametrize("mode", MATRIX, ids=mode_id)
def test_frames_against_oracle(mode, pkg, frame_refs, torch_cuda):
    set_mode(pkg, mode)
    for name, (pts, qs, kind, runs) in frame_refs.items():
        with pkg.Tree(pts) as tree:
            assert tree.info().coord_mode == storage(pkg, kind), name
            for (k, r), (idx, d2, rgba, nrm) in runs.items():
                out = tree.transfer(qs, k, radius=r, want_idx=True, want_d2=True)
                what = (name, k, r)
                bad = np.flatnonzero((out["idx"] != idx).any(1) | (out["d2"].view(np.uint64) != d2.view(np.uint64)).any(1))
                assert len(bad) == 0, (what, f"{len(bad)} samples differ, rows {bad[:8].tolist()}")
                _check_blend(out["rgba"], out["normal"], rgba, nrm)


# ---- b, c. identities and the path that answered --------------------------------------------------------
IDENT_RUNS = ((16, None), (9, tf.DYADIC_RADIUS), (32, None))
PINNED = 2000                                           # origin samples checked against the oracle


@pytest.fixture(scope="module")
def ident_cloud(pkg, pto):
    P0, Q0 = tf.dyadic_cloud(300_000, 8192, 11)
    tree = pto.KdTree(pkg.make_points(P0))
    ref = {(k, r): tree.knn(pkg.make_points(Q0[:PINNED]), k, radius=-1.0 if r is None else r, exact_ties=True)
           for k, r in IDENT_RUNS}
    return P0, Q0, ref


def run_frame(pkg, P, Q, coord, scale=0):
    """{(k, r): (idx, d2, fallback_counts)} of one frame; r is the origin's radius (scaled here)."""
    out = {}
    with pkg.Tree(pkg.make_points(P), coord_mode=coord) as tree:
        assert tree.info().coord_mode == coord
        qs = pkg.make_points(Q)
        for k, r in IDENT_RUNS:
            idx, d2 = tree.knn(qs, k, radius=None if r is None else np.ldexp(r, scale))
            out[k, r] = (idx, d2, tree.fallback_counts())
    return out


@pytest.mark.parametrize("mode", MATRIX, ids=mode_id)
def test_translation_and_scaling_identities(mode, pkg, ident_cloud, torch_cuda):
    P0, Q0, ref = ident_cloud
    set_mode(pkg, mode)
    grid = mode in GRID_MODES
    m = len(Q0)
    for coord in (pkg.COORD_F32, pkg.COORD_F64):
        base = run_frame(pkg, P0, Q0, coord)
        for key, (idx, d2, counts) in base.items():
            assert np.array_equal(idx[:PINNED], ref[key][0]) and np.array_equal(d2[:PINNED], ref[key][1]), (coord, key)
            HANDOVER_LOG.append(((mode_id(mode), coord, "origin", key), counts))
        if mode.get("knn_variant") == 6 and mode.get("order", 1) != 2 and "sort_bits" not in mode:
            # the grid answers the samples itself: a frame cannot pass by handing everything over
            # (a 16-bit sort orders cells down to level 5 only: ~190 points a cell here, over the caps)
            assert base[16, None][2][1] < m // 4, (coord, base[16, None][2])
        offsets = tf.F32_OFFSETS + (tf.F64_OFFSETS if coord == pkg.COORD_F64 else ())
        for off in offsets:
            got = run_frame(pkg, P0 + np.array(off), Q0 + np.array(off), coord)
            for key, (idx, d2, counts) in got.items():
                what = (coord, off, key)
                assert np.array_equal(idx, base[key][0]), what
                assert np.array_equal(d2.view(np.uint64), base[key][1].view(np.uint64)), what
                HANDOVER_LOG.append(((mode_id(mode), coord, off, key), counts))
                if max(map(abs, off)) < 1e7:
                    # slack ~1e-7 against a 2^-12 gap between d2 and any squared face distance
                    assert counts[1] == base[key][2][1], (what, counts, base[key][2])
        for s in tf.SCALES:
            got = run_frame(pkg, np.ldexp(P0, s), np.ldexp(Q0, s), coord, scale=s)
            for key, (idx, d2, counts) in got.items():
                what = (coord, s, key)
                assert np.array_equal(idx, base[key][0]), what
                assert np.array_equal(d2, np.ldexp(base[key][1], 2 * s)), what
                HANDOVER_LOG.append(((mode_id(mode), coord, s, key), counts))
                assert counts[1] == base[key][2][1], (what, counts, base[key][2])
                if grid and abs(s) <= 40:
                    assert counts == base[key][2], (what, counts, base[key][2])


# ---- d. saturated 16-bit cell counts ---------------------------------------------------------------------
def cell_keys(c21, sh):
    c = c21 >> sh
    return c[:, 0] | (c[:, 1] << 21) | (c[:, 2] << 42)


def grid_tables(xyz, sort_bits=40, min_occ10=40):
    """(lattice coordinates, table levels finest first) as build_grid_impl chooses them (pt_grid.cu):
    lo = bbox min, inv = 2^21 / max extent, the finest level averaging >= min_occ10 / 10 points per
    occupied cell among the levels the sorted key bits order, and up to 4 tables."""
    lo = xyz.min(0)
    inv = 2097152.0 / float((xyz.max(0) - lo).max())
    c21 = np.floor(np.clip((xyz - lo) * inv, 0.0, 2097151.0)).astype(np.int64)
    passes = (sort_bits + 7) // 8
    low_shift = 0 if passes >= 8 else 63 - 8 * passes
    lf = 1
    for level in range(1, min(16, (63 - low_shift) // 3) + 1):
        if len(xyz) / len(np.unique(cell_keys(c21, 21 - level))) >= 0.1 * min_occ10:
            lf = level
    return c21, [lf - t for t in range(4) if lf - t >= 1]


STAR = 64.0 + 0.5 / 64            # inside the lowest child (octant 0) of its parent at every level >= 2
BLOB = 70_000
SAT_CASES = (65_533, 65_534, 65_535, 65_536, 200_000, "blob")


def saturation_cloud(case, seed=90):
    """(xyz, samples, parent count at the finest table, tables): 60 000 points on the 2^-4 lattice in
    [0, 128]^3, then D duplicates at STAR (case D) or a jittered blob in STAR's level-13 cell plus one
    point in each of the 7 sibling children of its parent at the finest table ("blob"); the base
    points inside that parent are removed, so the parent holds exactly the points the case names."""
    rng = np.random.default_rng(seed)
    base = np.round(rng.random((60_000, 3)) * 128.0 * 16) / 16
    base[0], base[1] = (0.0, 0.0, 0.0), (128.0, 128.0, 128.0)
    if case == "blob":
        extra = np.float32(64.0 + (0.05 + 0.9 * rng.random((BLOB, 3))) / 64).astype(np.float64)
    else:
        extra = np.full((case, 3), STAR)
    sib = np.empty((0, 3))
    for _ in range(4):                       # removing points may change the level choice: iterate
        _, tables = grid_tables(np.r_[base, extra, sib])
        L = tables[0]
        cell = 128.0 / (1 << L)
        plo, phi = 64.0, 64.0 + 2 * cell     # STAR's parent at level L - 1
        base = base[~((base >= plo) & (base < phi)).all(1)]
        if case == "blob":
            octs = np.array([[(o >> a) & 1 for a in range(3)] for o in range(1, 8)], np.float64)
            sib = 64.0 + (octs + 0.5) * cell
        P = np.r_[base, extra, sib]
        c21, again = grid_tables(P)
        if again == tables:
            break
    assert again == tables
    keys = cell_keys(c21, 22 - L)
    count = int((keys == keys[len(base)]).sum())
    nb = len(base)
    near = STAR + np.concatenate([np.eye(3) * f * cell for f in (-1.5, -0.5, 1.0, 1.5, 2.5)])
    Q = np.r_[[[STAR] * 3], P[nb:nb + len(extra)][rng.choice(len(extra), 20)], near, sib,
              base[rng.choice(nb, 100)]]
    return P, Q, count, tables


@pytest.fixture(scope="module")
def saturation_refs(pkg, pto):
    out = {}
    for case in SAT_CASES:
        P, Q, count, tables = saturation_cloud(case)
        if case == "blob":
            c21, _ = grid_tables(P)
            L = tables[0]
            pk, ck = cell_keys(c21, 22 - L), cell_keys(c21, 21 - L)
            inparent = pk == pk[-1]
            assert count == BLOB + 7 and len(np.unique(ck[inparent])) == 8
            assert (ck == ck[len(P) - 8]).sum() == BLOB          # the blob fills one child
        else:
            assert count == case, (case, count, tables)
        pts, qs = with_attrs(pkg, P, 5), pkg.make_points(Q)
        refs = {k: pto.knn_bruteforce(pts, qs, k) for k in (16, 32)}
        out[case] = (pts, qs, count, refs)
    return out


@pytest.mark.parametrize("mode", GRID_MODES, ids=mode_id)
def test_saturated_cell_counts(mode, pkg, saturation_refs, torch_cuda):
    set_mode(pkg, mode)
    for case, (pts, qs, count, refs) in saturation_refs.items():
        for coord in (pkg.COORD_F32, pkg.COORD_F64):
            with pkg.Tree(pts, coord_mode=coord) as tree:
                assert tree.info().coord_mode == coord
                for k, (idx, d2) in refs.items():
                    got_i, got_d = tree.knn(qs, k)
                    what = (case, coord, k)
                    bad = np.flatnonzero((got_i != idx).any(1) | (got_d != d2).any(1))
                    assert len(bad) == 0, (what, f"{len(bad)} samples differ, rows {bad[:8].tolist()}")
                    counts = tree.fallback_counts()
                    HANDOVER_LOG.append(((mode_id(mode), "saturation", case, coord, k), counts))
                    if count >= 65_535 and mode.get("knn_variant") == 6:
                        # the sample at STAR meets an occupied child of a saturated parent in every table
                        assert counts[1] > 0, (what, counts)


# ---- e. consumers in one UTM frame ------------------------------------------------------------------------
def to_utm(xyz, step=1e-3):
    return (np.round(xyz / step) + np.array(tf.UTM) / step) * step


@pytest.fixture(scope="module")
def utm_case(pkg):
    side = 30.0
    P = pkg.synth.cloud_host(60_000, seed=33, side=side)
    P["ver"] = to_utm(P["ver"])
    V, F = grid_mesh(pkg, 12, side)
    V["ver"] = to_utm(V["ver"])
    V["normal"] = tilted_normals(np.random.default_rng(33), len(V))
    return P, V, F


def test_bake_in_utm_frame(pkg, pto, utm_case, torch_cuda):
    P, V, F = utm_case
    with pkg.Tree(P) as tree:
        assert tree.info().coord_mode == pkg.COORD_F64
    got, ref = check_bake_ex(pkg, pto, P, V, F, 16, 200)
    assert ref["texels"] > 200 * 200 // 2
    got, ref = check_height(pkg, pto, P, V, F, 16, 200)
    assert ref["texels"] > 200 * 200 // 2


def test_normals_in_utm_frame(pkg, pto, utm_case, torch_cuda):
    P, _, _ = utm_case
    P = P.copy()
    rng = np.random.default_rng(34)
    P["normal"] *= np.where(rng.random(len(P)) < 0.5, -1.0, 1.0)[:, None]
    P["normal"][::5] = 0.0
    xyz, m = P["ver"], P["normal"].astype(np.float32)
    with pkg.Tree(P) as tree:
        assert tree.info().coord_mode == pkg.COORD_F64
        for k, radius in ((16, None), (18, 0.3)):
            idx = pto_normals.neighbours(xyz, k, -1.0 if radius is None else radius)
            what = ("utm", k, radius)
            check_normals(pto, tree, P, tree.estimate_normals(k, radius=radius), pto_normals.estimate(xyz, m, idx),
                          idx, radius, what)
            ref_o = orient_oracle.orient(xyz, m, idx)
            assert ref_o["flipped"] > 0
            check_orient(pto, tree, P, tree.orient_normals(k, radius=radius), ref_o, idx, radius, what)


def test_sharded_bake_in_utm_frame(pkg, utm_case, torch_cuda):
    P, V, F = utm_case
    for devices in ([0, 0], [0, 0, 0]):
        got, info = compare(pkg, P, V, F, devices, k=16, resolution=200, want=EVERYTHING)
        assert info["n_slabs"] == len(devices) and got["stats"]["texels"] > 200 * 200 // 2


@pytest.mark.parametrize("R,k,radius", [(2, 16, None), (3, 8, 0.6)])
def test_slab_transfer_in_utm_frame(R, k, radius, pkg, pto, torch_cuda):
    """The slab helper stores float32 positions: the cloud sits at the easting on the 2^-5 lattice."""
    torch = torch_cuda
    side, off = 60.0, np.array([452_304.0, 0.0, 312.0])
    P = pkg.synth.cloud_host(150_000, seed=35, side=side)
    P["ver"] = np.round(P["ver"] * 32) / 32 + off
    assert tf.f32_exact(P["ver"])
    V = pkg.synth.samples_host(60, side=side)
    V["ver"] += off
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, radius=-1.0 if radius is None else radius)
    ref = (ref_idx, ref_d2) + pto.blend(P, ref_idx, ref_d2)
    S = Slabs(pkg, torch, P, R)
    try:
        assert (S.x_cut[1:-1] > off[0]).all()
        owner = S.owner_of(V)
        sels = [np.nonzero(owner == r)[0] for r in range(R)]
        queries = [torch.from_numpy(np.ascontiguousarray(V["ver"][s])).cuda() for s in sels]
        out, crossing = _exchange_step(S, queries, k, radius, cap=2048)
        assert 0 < crossing < len(V)
        for r in range(R):
            _check(out[r], ref, sels[r])
    finally:
        S.close()
