"""Normal estimation (DESIGN.md section 8, "Normal estimation"): PCA over each point's k nearest
neighbours, cyclic Jacobi, orientation by the input normal, a viewpoint or the largest component.

CPU part: the oracle (oracle/pt_normals_oracle.c via oracle/pto_normals.py) against an independent
numpy statement (sequential ufunc sums, np.linalg.eigh), known answers, accuracy against the analytic
normals of a synthetic scan, and the CLI's refusals.  GPU part: pt_index_estimate_normals, the device
piece and the CLI must equal the oracle bit for bit; `store` must feed transfers and bakes."""
import ctypes
import glob
import os
import subprocess

import numpy as np
import pytest

from oracle import pto_normals

NAN_BITS = 0x7FC00000
GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "*.npz")))


# ---- the definition restated in numpy (sequential sums, eigh for the eigenvectors) ----------------
def numpy_normals(xyz, normal, idx, viewpoint=None, rows=None):
    """(n float64 [m,3], variation float64 [m], eigenvalues [m,3] ascending, estimated [m], decided [m]:
    the orientation rule is not a near-tie, so rounding cannot change the sign)."""
    rows = np.arange(len(idx)) if rows is None else np.asarray(rows)
    m, k = idx.shape
    valid = (idx >= 0) & (idx < len(xyz))
    cnt = np.where(valid.all(1), k, np.argmin(valid, 1))
    p = xyz[np.where(valid, idx, 0)]
    with np.errstate(all="ignore"):
        s = np.zeros((m, 3))
        for j in range(k):
            s = np.where((j < cnt)[:, None], np.add(s, p[:, j]), s)
        mu = np.divide(s, cnt[:, None].astype(np.float64))
        e = np.subtract(p, mu[:, None, :])
        c = np.zeros((m, 3, 3))
        for j in range(k):
            outer = np.multiply(e[:, j, :, None], e[:, j, None, :])
            c = np.where((j < cnt)[:, None, None], np.add(c, outer), c)
        trace = np.add(np.add(c[:, 0, 0], c[:, 1, 1]), c[:, 2, 2])
    est = (cnt >= 3) & (trace > 0) & np.isfinite(trace)
    lam, vec = np.linalg.eigh(np.where(est[:, None, None], c, np.eye(3)))
    n = vec[:, :, 0]
    n = n / np.linalg.norm(n, axis=1)[:, None]
    mi = None if normal is None else np.asarray(normal, np.float32)[rows].astype(np.float64)
    use_m = np.zeros(m, bool) if mi is None else (np.isfinite(mi).all(1) & ((mi * mi).sum(1) > 0))
    srt = np.sort(np.abs(n), axis=1)
    decided = srt[:, 2] - srt[:, 1] > 1e-9
    if viewpoint is not None:
        ref = np.asarray(viewpoint, np.float64) - xyz[rows]
        decided = np.ones(m, bool)
    else:
        big = np.argmax(np.abs(n), axis=1)
        ref = np.eye(3)[big]
    if mi is not None:
        ref = np.where(use_m[:, None], mi, ref)
        decided |= use_m
    dot = (n * ref).sum(1)
    decided &= np.abs(dot) > 1e-9 * np.linalg.norm(ref, axis=1)
    n = np.where((dot < 0)[:, None], -n, n)
    with np.errstate(all="ignore"):
        var = np.maximum(lam[:, 0], 0) / trace
    return n, var, lam, est, decided


def check_oracle_vs_numpy(xyz, normal, idx, viewpoint=None, rows=None):
    got_n, got_v, n_est, got64 = pto_normals.estimate(xyz, normal, idx, viewpoint, rows, fp64=True)
    n, var, lam, est, decided = numpy_normals(xyz, normal, idx, viewpoint, rows)
    assert n_est == est.sum()
    assert np.array_equal(np.isnan(got_v), ~est)
    assert (got_v.view(np.uint32)[~est] == NAN_BITS).all() and (got_n[~est] == 0).all()
    sep = est & (lam[:, 1] - lam[:, 0] >= 1e-6 * lam[:, 2])     # a well-defined smallest eigenvector
    assert ((got64[sep & decided, :3] * n[sep & decided]).sum(1) > 0).all(), "orientation differs"
    # the angle from its sine: |a x b| (arccos loses half the digits near 0)
    ang = np.arcsin(np.clip(np.linalg.norm(np.cross(got64[sep, :3], n[sep]), axis=1), 0, 1))
    assert (ang <= 1e-9).all(), ang.max()
    assert (np.abs(got64[sep, 3] - var[sep]) <= 1e-9 * np.abs(var[sep]) + 1e-15).all()
    assert np.array_equal(got_n[est], got64[est, :3].astype(np.float32))
    return est


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_equals_numpy_on_golden_clouds(path, pto):
    g = np.load(path)
    xyz, nrm = g["xyz"], g["normal"]
    for k in (3, 8, 16, 32):
        for radius in (-1.0, float(g["radius"])):
            idx = pto_normals.neighbours(xyz, k, radius)
            check_oracle_vs_numpy(xyz, nrm, idx)
            check_oracle_vs_numpy(xyz, None, idx, viewpoint=(0.3, -2.0, 5.0))
            check_oracle_vs_numpy(xyz, None, idx)


def test_oracle_equals_numpy_on_a_noisy_patch(pto):
    rng = np.random.default_rng(11)
    uv = rng.random((3000, 2)) * 4.0
    xyz = np.c_[uv, 0.3 * np.sin(uv[:, 0]) * np.cos(uv[:, 1]) + 0.01 * rng.standard_normal(3000)]
    nrm = rng.standard_normal((3000, 3))
    nrm[::3] = 0.0
    for k in (3, 8, 20, 32):
        est = check_oracle_vs_numpy(xyz, nrm, pto_normals.neighbours(xyz, k))
        assert est.all()


# ---- known answers --------------------------------------------------------------------------------
def test_plane_is_exact(pto):
    rng = np.random.default_rng(3)
    xyz = np.c_[rng.random((500, 2)) * 7.0, np.full(500, 0.75)]
    for k in (3, 16, 32):
        n, v, e = pto_normals.estimate_normals(xyz, None, k)
        assert e == 500
        assert (n == np.array([0, 0, 1], np.float32)).all() and (v == 0).all()
        n, v, e = pto_normals.estimate_normals(xyz, None, k, viewpoint=(1.0, 1.0, -3.0))
        assert (n == np.array([0, 0, -1], np.float32)).all() and (v == 0).all()


def test_collinear_gives_a_perpendicular(pto):
    t = np.linspace(-3.0, 5.0, 80)
    u = np.array([1.0, 2.0, -1.0]) / np.sqrt(6.0)
    xyz = np.c_[t, 2.0 * t + 1.0, -t + 0.5]
    for k in (3, 8, 32):
        n, v, e, n64 = pto_normals.estimate(xyz, None, pto_normals.neighbours(xyz, k), fp64=True)
        assert e == 80
        assert np.abs(n64[:, :3] @ u).max() < 1e-9
        assert np.abs(np.linalg.norm(n64[:, :3], axis=1) - 1.0).max() < 1e-15
        again = pto_normals.estimate(xyz, None, pto_normals.neighbours(xyz, k))[0]
        assert np.array_equal(n, again)
    axis = np.c_[np.arange(40) * 0.5, np.full(40, 2.0), np.full(40, 3.0)]
    n, _, _ = pto_normals.estimate_normals(axis, None, 8)
    assert (n == np.array([0, 1, 0], np.float32)).all()


def test_duplicates_only_have_no_estimate(pto):
    xyz = np.r_[np.repeat([[1.0, 2.0, 3.0]], 10, axis=0), np.random.default_rng(1).random((50, 3)) + 10.0]
    n, v, e = pto_normals.estimate_normals(xyz, None, 8)
    assert (n[:10] == 0).all() and (v[:10].view(np.uint32) == NAN_BITS).all()
    assert e == 50


def test_k_gt_n_uses_all_points(pto, golden_dir):
    g = np.load(os.path.join(golden_dir, "k_gt_n.npz"))
    xyz = g["xyz"]
    idx = pto_normals.neighbours(xyz, 8)
    assert ((idx >= 0).sum(1) == 5).all()
    n, v, e = pto_normals.estimate(xyz, None, idx)
    ref = numpy_normals(xyz, None, idx)
    assert e == 5 and ref[4].all()
    assert np.allclose(n, ref[0], atol=1e-6) and np.allclose(v, ref[1], rtol=1e-6, atol=1e-12)


def test_orientation_rules(pto):
    rng = np.random.default_rng(5)
    xyz = np.c_[rng.random((400, 2)) * 5.0, 0.5 * rng.random(400) * 1e-3]   # nearly z = 0
    idx = pto_normals.neighbours(xyz, 12)
    base = pto_normals.estimate(xyz, None, idx)[0]
    assert (base[:, 2] > 0).all()                                             # (c): largest component +
    m = np.zeros((400, 3))
    m[:200, 2] = -1.0                                                        # (a) flips these
    m[200:300, 2] = 2.0                                                      # (a) keeps these
    m[300:, :] = np.nan                                                      # not usable: (b) / (c)
    a = pto_normals.estimate(xyz, m, idx)[0]
    assert np.array_equal(a[:200], -base[:200]) and np.array_equal(a[200:], base[200:])
    b = pto_normals.estimate(xyz, m, idx, viewpoint=(2.0, 2.0, -10.0))[0]
    assert np.array_equal(b[:300], a[:300]) and np.array_equal(b[300:], -base[300:])
    b = pto_normals.estimate(xyz, m, idx, viewpoint=(2.0, 2.0, 10.0))[0]
    assert np.array_equal(b, a)


# ---- degenerate spectra: tied and zero eigenvalues ------------------------------------------------
DEGENERATE = {"cube": 9, "octahedron": 7, "collinear": 8, "plane": 8}     # kind -> k (the structure's size)
TINY = -530          # 2^-530: the scatter products (~2^-1062) are subnormal


def degenerate_cloud(kind, seed=0):
    """(xyz float64 [n,3], k, aligned bool [n]): 216 structures 8 apart on a 6^3 lattice, whose k-NN
    scatter has tied or zero eigenvalues -- cube corners or an octahedron around a centre point (three
    equal), collinear runs (two equal smallest), plane patches (a zero smallest) -- and one background
    point near every lattice cell's middle.  Every structure fits a ball of radius 0.9 and lies more
    than 4 from the background, so the lists of its points hold exactly its own points.  Every other
    structure is rotated (tilted: z = x for planes); ``aligned`` marks the points of the others, whose
    scatter is exact.  Coordinates are fp32-representable; ids are shuffled."""
    rng = np.random.default_rng(seed)
    g = np.arange(6) * 8.0
    centres = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    parts, flags = [], []
    for i, c in enumerate(centres):
        a = (0.25, 0.5, 0.375)[i % 3]
        aligned = i % 2 == 0
        if kind == "cube":
            local = a * np.r_[np.array(np.meshgrid([-1, 1], [-1, 1], [-1, 1])).reshape(3, -1).T, np.zeros((1, 3))]
        elif kind == "octahedron":
            local = a * np.r_[np.eye(3), -np.eye(3), np.zeros((1, 3))]
        elif kind == "collinear":
            local = np.outer((np.arange(12) - 5.5) * a / 4.0, [1.0, 0.0, 0.0])
        else:
            uv = rng.integers(-256, 257, (16, 2)) / 512.0
            local = np.c_[uv, np.zeros(16)] if aligned else np.c_[uv[:, 0], uv[:, 1], uv[:, 0]]
        if not aligned and kind != "plane":
            q, _ = np.linalg.qr(rng.standard_normal((3, 3)))
            local = local @ q
        parts.append(c + local)
        flags.append(np.full(len(local), aligned))
    back = centres + 4.0 + rng.uniform(-1.0, 1.0, centres.shape)
    xyz = np.r_[np.concatenate(parts), back].astype(np.float32).astype(np.float64)
    aligned = np.r_[np.concatenate(flags), np.zeros(len(back), bool)]
    p = rng.permutation(len(xyz))
    return xyz[p], DEGENERATE[kind], aligned[p]


def degenerate_normals(n, seed=1):
    """Input normals for rule (a): random directions, every fifth one zero (rule (c) there)."""
    m = np.random.default_rng(seed).standard_normal((n, 3)).astype(np.float32)
    m[::5] = 0.0
    return m


@pytest.mark.parametrize("kind", sorted(DEGENERATE))
def test_oracle_equals_numpy_on_degenerate_spectra(kind, pto):
    xyz, k, aligned = degenerate_cloud(kind)
    idx = pto_normals.neighbours(xyz, k)
    nrm = degenerate_normals(len(xyz))
    for normal, view in ((nrm, None), (None, (100.0, -30.0, 70.0)), (None, None)):
        est = check_oracle_vs_numpy(xyz, normal, idx, view)
        assert est.all()
    check_exact_scatter(kind, aligned, *pto_normals.estimate(xyz, None, idx)[:2])


def check_exact_scatter(kind, aligned, n, v):
    """Known answers (rule (c)) where the scatter is exact: ties go to the lower Jacobi column."""
    if kind in ("cube", "octahedron"):            # diag(s, s, s): no rotation at all
        assert (n[aligned] == np.array([1, 0, 0], np.float32)).all()
        assert (v[aligned] == np.float32(1.0 / 3.0)).all()
    elif kind == "collinear":                     # diag(s, 0, 0)
        assert (n[aligned] == np.array([0, 1, 0], np.float32)).all() and (v[aligned] == 0).all()
    else:                                         # z = c: the third row and column are exact zeros
        assert (n[aligned] == np.array([0, 0, 1], np.float32)).all() and (v[aligned] == 0).all()


@pytest.mark.parametrize("kind", sorted(DEGENERATE))
def test_oracle_on_subnormal_scatter(kind, pto):
    """The degenerate clouds scaled by 2^-530: exact in fp64, but every scatter product is subnormal,
    so the Jacobi sweeps round with a few significant bits and the numpy statement's eigenvectors
    (eigh scales the matrix first) are no reference for the others.  What still holds: which points
    get an estimate, the NaN bits, unit normals and the exact answers of the aligned structures, whose
    products are exact multiples of 2^-1072.  The lists are those of the scaled cloud."""
    xyz, k, aligned = degenerate_cloud(kind)
    tiny = np.ldexp(xyz, TINY)
    idx = pto_normals.neighbours(tiny, k)
    for normal, view in ((degenerate_normals(len(xyz)), None), (None, (1.0, -2.0, 3.0)), (None, None)):
        got_n, got_v, n_est = pto_normals.estimate(tiny, normal, idx, view)
        est = numpy_normals(tiny, normal, idx, view)[3]
        assert n_est == est.sum() == len(xyz)
        assert np.array_equal(np.isnan(got_v), ~est)
        assert np.abs(np.linalg.norm(got_n.astype(np.float64), axis=1) - 1.0).max() < 1e-6
        assert ((got_v >= 0) & (got_v <= np.float32(1.0 / 3.0))).all()
    check_exact_scatter(kind, aligned, *pto_normals.estimate(tiny, None, idx)[:2])


# ---- accuracy against the analytic normals of a noisy scan ----------------------------------------
ACCURACY = {8: (2.3, 7.5), 16: (1.0, 2.7), 32: (0.5, 1.3)}    # mean, p99 (degrees) bounds


def angles_deg(n, ref):
    ref = ref / np.linalg.norm(ref, axis=1)[:, None]
    return np.degrees(np.arccos(np.clip(np.abs((n.astype(np.float64) * ref).sum(1)), 0, 1)))


@pytest.fixture(scope="module")
def scan(pto):
    P = pto.synth_cloud(1_000_000, 20261018 + 2, u1=200.0, v1=200.0)
    rows = np.sort(np.random.default_rng(20261021).choice(len(P), 20_000, replace=False))
    return P, rows


@pytest.mark.parametrize("k", sorted(ACCURACY))
def test_accuracy_against_analytic_normals(k, scan):
    P, rows = scan
    n, v, e = pto_normals.estimate_normals(P["ver"], P["normal"], k, rows=rows)
    assert e == len(rows)
    ang = angles_deg(n, P["normal"][rows])
    mean_b, p99_b = ACCURACY[k]
    assert ang.mean() < mean_b and np.percentile(ang, 99) < p99_b, (ang.mean(), np.percentile(ang, 99))
    assert ((n.astype(np.float64) * P["normal"][rows]).sum(1) > 0).all()     # rule (a)
    assert np.isfinite(v).all() and (v >= 0).all() and (v <= 1.0 / 3.0).all()


# ---- CLI ------------------------------------------------------------------------------------------
def _cli():
    from test_cli import CLI
    if not os.path.exists(CLI):
        subprocess.run(["make", "-C", os.path.dirname(CLI)], check=True, stdout=subprocess.DEVNULL)
    return CLI


@pytest.mark.parametrize("args", [["-e", "2"], ["-e", "33"], ["-e", "16", "-g", "2"]])
def test_cli_refuses_bad_estimation_options(args, tmp_path):
    r = subprocess.run([_cli(), *args, "a.ply", "b.ply"], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and "-e must be 3..32" in r.stderr
    assert not (tmp_path / "texture.png").exists()


# ---- GPU ------------------------------------------------------------------------------------------
def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def assert_same(got, ref_n, ref_v, what=""):
    assert np.array_equal(got["normal"].view(np.uint32), ref_n.view(np.uint32)), what
    assert np.array_equal(got["variation"].view(np.uint32), ref_v.view(np.uint32)), what


def golden_points(pkg, g):
    return pkg.make_points(g["xyz"], normal=g["normal"], color=g["color"])


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_gpu_equals_oracle_on_golden_clouds(path, pkg, pto):
    _need_gpu()
    g = np.load(path)
    P = golden_points(pkg, g)
    mode = pkg.COORD_F64 if "f64" in os.path.basename(path) else pkg.COORD_AUTO
    zero = pkg.make_points(g["xyz"], color=g["color"])
    for cloud, nrm in ((P, g["normal"]), (zero, None)):
        with pkg.Tree(cloud, coord_mode=mode) as tree:
            if "f64" in os.path.basename(path):
                assert tree.info().coord_mode == pkg.COORD_F64
            for k in (3, 8, 16, 20, 32):
                for radius in (None, float(g["radius"])):
                    idx = pto_normals.neighbours(g["xyz"], k, -1.0 if radius is None else radius)
                    for view in (None, (0.3, -2.0, 5.0)):
                        ref_n, ref_v, e = pto_normals.estimate(g["xyz"], nrm, idx, view)
                        got = tree.estimate_normals(k, radius=radius, viewpoint=view)
                        assert_same(got, ref_n, ref_v, (k, radius, view))
                        assert got["stats"]["estimated"] == e


@pytest.mark.gpu
def test_gpu_more_than_one_chunk(pkg, pto):
    _need_gpu()
    import torch
    n = 5_000_000                       # the density of the accuracy test's scan: about 0.2 apart
    pos, attrs = pkg.synth.cloud_device(n, seed=20261018 + 2, u1=447.0, v1=447.0)
    P = pkg.synth.points_to_host(pos, attrs)
    rows = np.sort(np.random.default_rng(4).choice(n, 4096, replace=False))
    tree = pkg.DeviceTree(pos, attrs)
    normal = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    variation = torch.empty(n, dtype=torch.float32, device="cuda")
    for k in (8, 16, 32):
        tree.estimate_normals(k, normal=normal, variation=variation)
        torch.cuda.synchronize()
        got_n, got_v = normal.cpu().numpy(), variation.cpu().numpy()
        ref_n, ref_v, _ = pto_normals.estimate_normals(P["ver"], P["normal"], k, rows=rows)
        assert np.array_equal(got_n[rows].view(np.uint32), ref_n.view(np.uint32)), k
        assert np.array_equal(got_v[rows].view(np.uint32), ref_v.view(np.uint32)), k
        ang = angles_deg(got_n, P["normal"])
        mean_b, p99_b = ACCURACY[k]
        assert ang.mean() < mean_b and np.percentile(ang, 99) < p99_b, (k, ang.mean(), np.percentile(ang, 99))
    tree.close()


def bake_mesh(pkg, side, g=12):
    from test_bake import grid_mesh
    return grid_mesh(pkg, g, side)


@pytest.mark.gpu
def test_gpu_store_feeds_transfer_and_bake(pkg, pto):
    _need_gpu()
    from test_bake_tangent import ALL_OUTPUTS
    side = 30.0
    P = pkg.synth.cloud_host(60_000, seed=9, side=side)
    P["normal"][::2] = 0.0                                     # half the cloud arrives without normals
    P["ver"][:5] = P["ver"][5]                                  # a duplicates-only neighbourhood at k = 3
    V, F = bake_mesh(pkg, side)
    q = pkg.make_points(V["ver"] + 0.01)
    for k in (3, 16):
        with pkg.Tree(P) as tree:
            before = tree.transfer(q, 8)
            kept = tree.estimate_normals(k, store=False)
            assert tree.transfer(q, 8)["normal"].tobytes() == before["normal"].tobytes()
            est = tree.estimate_normals(k, store=True)
            after_t = tree.transfer(q, 8)
            after_b = tree.bake(V, F, k=16, resolution=200, want=ALL_OUTPUTS + ("height",))
        assert_same(est, kept["normal"], kept["variation"])
        has = ~np.isnan(est["variation"])
        Q = P.copy()
        Q["normal"][has] = est["normal"][has]
        with pkg.Tree(Q) as ref:
            ref_t = ref.transfer(q, 8)
            ref_b = ref.bake(V, F, k=16, resolution=200, want=ALL_OUTPUTS + ("height",))
        for key in ("rgba", "normal", "idx"):
            assert after_t[key].tobytes() == ref_t[key].tobytes(), key
        for key in ALL_OUTPUTS + ("height",):
            assert after_b[key].tobytes() == ref_b[key].tobytes(), key
        if k == 3:
            assert (~has).sum() > 0


@pytest.mark.gpu
def test_gpu_device_piece_equals_host_call_and_errors(pkg, pto):
    _need_gpu()
    import torch
    n = 300_000
    pos, attrs = pkg.synth.cloud_device(n, seed=3, u1=100.0, v1=100.0)
    P = pkg.synth.points_to_host(pos, attrs)
    normal = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    variation = torch.empty(n, dtype=torch.float32, device="cuda")
    with pkg.Tree(P) as tree:
        host = tree.estimate_normals(16, viewpoint=(50.0, 50.0, 100.0))
        L = pkg.lib()
        for k, rc in ((2, 1), (0, 1), (33, 5)):          # 1 invalid argument, 5 unsupported
            assert L.pt_index_estimate_normals(tree.handle, k, -1.0, None, 0, host["normal"].ctypes.data, None,
                                               None) == rc
        assert L.pt_index_estimate_normals(tree.handle, 8, -1.0, None, 0, None, None, None) == 1
        bad = (ctypes.c_double * 3)(0.0, float("nan"), 1.0)
        assert L.pt_index_estimate_normals(tree.handle, 8, -1.0, bad, 0, host["normal"].ctypes.data, None, None) == 1
        assert L.pt_index_estimate_normals(None, 8, -1.0, None, 1, None, None, None) == 1
    dev = pkg.DeviceTree(pos, attrs)
    dev.estimate_normals(16, viewpoint=(50.0, 50.0, 100.0), normal=normal, variation=variation)
    torch.cuda.synchronize()
    assert_same({"normal": normal.cpu().numpy(), "variation": variation.cpu().numpy()}, host["normal"],
                host["variation"])
    dev.close()
    bare = pkg.DeviceTree(pos)
    with pytest.raises(pkg.PointsTransferError) as e:
        bare.estimate_normals(16, store=True)
    assert e.value.status == 1
    bare.estimate_normals(16, viewpoint=(50.0, 50.0, 100.0), normal=normal, variation=variation)
    torch.cuda.synchronize()
    ref_n, ref_v, _ = pto_normals.estimate_normals(P["ver"], None, 16, viewpoint=(50.0, 50.0, 100.0),
                                                   rows=np.arange(0, n, 97))
    assert np.array_equal(normal.cpu().numpy()[::97].view(np.uint32), ref_n.view(np.uint32))
    assert np.array_equal(variation.cpu().numpy()[::97].view(np.uint32), ref_v.view(np.uint32))
    bare.close()


@pytest.mark.gpu
def test_gpu_cli_estimate_equals_python(pkg, pto, tmp_path):
    _need_gpu()
    from test_cli import read_png_bgra, write_cloud, write_mesh
    side = 30.0
    P = pkg.synth.cloud_host(40_000, seed=12, side=side)
    P["normal"] = 0.0
    P["ver"] = P["ver"].astype(np.float32).astype(np.float64)
    V, F = bake_mesh(pkg, side)
    write_cloud(tmp_path / "c.ply", P)
    write_mesh(tmp_path / "m.ply", V, F)
    r = subprocess.run([_cli(), "-R", "128", "-e", "16", "-n", "normal.png", str(tmp_path / "c.ply"),
                        str(tmp_path / "m.ply")], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    assert "Estimated normals: 40000 of 40000 points in" in r.stdout, r.stdout
    Vm = V.copy()
    Vm["normal"] = (0.0, 0.0, 1.0)                                # write_mesh's normal column
    with pkg.Tree(P) as tree:
        tree.estimate_normals(16, store=True)
        ref = tree.bake(Vm, F, k=20, resolution=128, want=("normal_bgra",))
    assert np.array_equal(read_png_bgra(tmp_path / "normal.png"), ref["normal_bgra"])
