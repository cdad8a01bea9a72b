"""Normal orientation (DESIGN.md section 8, "Normal orientation"): signs propagated along the minimum
spanning forest of the k-NN graph under (w = 1 - |n_i.n_j|, lo, hi), from each component's top point.

CPU part: the oracle (oracle/pt_orient_oracle.c via oracle/pto_orient.py) against an independent
statement (scipy's minimum_spanning_tree on the edge ranks, breadth_first_order), known answers on
closed surfaces, and the CLI's refusals.  GPU part: pt_index_orient_normals and the CLI must equal the
oracle bit for bit; `store` must feed transfers and bakes."""
import ctypes
import glob
import os
import subprocess

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import breadth_first_order, connected_components, minimum_spanning_tree

from oracle import pto_normals, pto_orient

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "*.npz")))
VIEW = (0.3, -2.0, 5.0)


def dot(a, b):
    return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]


# ---- the definition restated with scipy ------------------------------------------------------------
def scipy_orient(xyz, normal, idx, viewpoint=None):
    """(normal float32 [n,3], root [n], parent [n], counts) from scipy's minimum spanning tree on the
    ranks 1..E of the edges under (w, lo, hi): distinct positive weights, so scipy finds exactly the
    forest of the definition, ties included (raw weights would not do: scipy drops explicit zeros)."""
    n, k = idx.shape
    m32 = np.asarray(normal, np.float32).reshape(-1, 3)
    m = m32.astype(np.float64)
    with np.errstate(all="ignore"):
        part = np.isfinite(m).all(1) & (dot(m, m) > 0)
        nh = m / np.sqrt(dot(m, m))[:, None]
    valid = np.cumprod((idx >= 0) & (idx < n), axis=1).astype(bool)
    i = np.repeat(np.arange(n), k).reshape(n, k)
    j = np.where(valid, idx, 0)
    keep = valid & (j != i) & part[i] & part[j]
    lo, hi = np.minimum(i, j)[keep], np.maximum(i, j)[keep]
    pairs = np.unique(lo.astype(np.int64) * n + hi)
    lo, hi = pairs // n, pairs % n
    d = dot(nh[lo], nh[hi])
    w = 1.0 - np.abs(d)
    w[w < 0] = 0.0
    rank = np.empty(len(w), np.float64)
    rank[np.lexsort((hi, lo, w))] = np.arange(1, len(w) + 1)
    T = minimum_spanning_tree(coo_matrix((rank, (lo, hi)), shape=(n, n)).tocsr())
    T = (T + T.T).tocsr()
    neg = coo_matrix(((d < 0).astype(np.float64) + 1.0, (lo, hi)), shape=(n, n)).tocsr()
    neg = (neg + neg.T).tocsr()
    _, comp = connected_components(T, directed=False)
    z = xyz[:, 2].astype(np.float64)
    root = np.full(n, -1, np.int64)
    parent = np.full(n, -1, np.int64)
    sigma = np.zeros(n, np.int64)
    ids = np.arange(n)[part]
    order = ids[np.lexsort((ids, -z[ids]))]           # largest z first, lowest id on ties
    top = {}
    for v in order:
        top.setdefault(comp[v], v)
    for c, r in top.items():
        nr = nh[r]
        if viewpoint is not None:
            neg_r = dot(nr[None], (np.asarray(viewpoint, np.float64) - xyz[r])[None])[0] < 0
        elif nr[2] != 0:
            neg_r = nr[2] < 0
        else:
            a = np.abs(nr)
            ax = 0 if (a[0] >= a[1] and a[0] >= a[2]) else (1 if a[1] >= a[2] else 2)
            neg_r = nr[ax] < 0
        bfs, pred = breadth_first_order(T, r, directed=False, return_predecessors=True)
        sigma[r] = -1 if neg_r else 1
        for v in bfs[1:]:
            p = pred[v]
            parent[v] = p
            sigma[v] = -sigma[p] if neg[p, v] == 2.0 else sigma[p]
        root[bfs] = r
    out = m32.copy()
    out[sigma < 0] = -out[sigma < 0]
    counts = {"oriented": int(part.sum()), "flipped": int((sigma < 0).sum()), "components": len(top),
              "edges": len(w)}
    return out, root, parent, counts


def check_oracle_vs_scipy(xyz, normal, idx, viewpoint=None):
    got = pto_orient.orient(xyz, normal, idx, viewpoint)
    ref_n, ref_root, ref_parent, counts = scipy_orient(xyz, normal, idx, viewpoint)
    assert np.array_equal(got["normal"].view(np.uint32), ref_n.view(np.uint32))
    assert np.array_equal(got["root"], ref_root)
    assert np.array_equal(got["parent"], ref_parent)
    for key, v in counts.items():
        assert got[key] == v, key
    return got


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_equals_scipy_on_golden_clouds(path, pto):
    g = np.load(path)
    xyz, nrm = g["xyz"], g["normal"]
    rng = np.random.default_rng(1)
    flipped = nrm * np.where(rng.random(len(nrm)) < 0.5, -1.0, 1.0)[:, None]
    for k in (2, 8, 18, 32):
        for radius in (-1.0, float(g["radius"])):
            idx = pto_normals.neighbours(xyz, k, radius)
            for view in (None, VIEW):
                check_oracle_vs_scipy(xyz, nrm, idx, view)
                check_oracle_vs_scipy(xyz, flipped, idx, view)


def noisy_patch(n=3000, seed=11):
    rng = np.random.default_rng(seed)
    uv = rng.random((n, 2)) * 4.0
    xyz = np.c_[uv, 0.3 * np.sin(uv[:, 0]) * np.cos(uv[:, 1]) + 0.01 * rng.standard_normal(n)]
    nrm = np.c_[np.zeros((n, 2)), np.ones(n)] + 0.3 * rng.standard_normal((n, 3))
    nrm *= np.where(rng.random(n) < 0.5, -1.0, 1.0)[:, None]
    nrm[::7] = 0.0
    return xyz, nrm


def test_oracle_equals_scipy_on_a_noisy_patch(pto):
    xyz, nrm = noisy_patch()
    for k in (2, 8, 18, 32):
        for radius in (-1.0, 0.15):
            idx = pto_normals.neighbours(xyz, k, radius)
            for view in (None, (2.0, 2.0, 10.0)):
                got = check_oracle_vs_scipy(xyz, nrm, idx, view)
                assert got["oriented"] == len(xyz) - len(xyz[::7])


# ---- known answers ---------------------------------------------------------------------------------
def sphere(n, rng, centre=(0.0, 0.0, 0.0), r=1.0):
    d = rng.standard_normal((n, 3))
    d /= np.linalg.norm(d, axis=1)[:, None]
    return np.asarray(centre) + r * d, d


def torus(n, rng, R=2.0, r=0.6):
    u, v = rng.random(n) * 2 * np.pi, rng.random(n) * 2 * np.pi
    d = np.c_[np.cos(v) * np.cos(u), np.cos(v) * np.sin(u), np.sin(v)]
    return np.c_[(R + r * np.cos(v)) * np.cos(u), (R + r * np.cos(v)) * np.sin(u), r * np.sin(v)], d


def scramble(d, rng, noise=0.05):
    m = d + noise * rng.standard_normal(d.shape)
    return (m * np.where(rng.random(len(d)) < 0.5, -1.0, 1.0)[:, None]).astype(np.float32)


def expected_roots(xyz, comp_of):
    roots = {}
    for v in np.lexsort((np.arange(len(xyz)), -xyz[:, 2])):
        roots.setdefault(comp_of[v], v)
    return np.array([roots[c] for c in comp_of])


@pytest.mark.parametrize("shape", ["sphere", "torus", "two_spheres"])
def test_closed_surfaces_come_out_outward(shape, pto):
    rng = np.random.default_rng(2026)
    if shape == "sphere":
        xyz, d = sphere(20_000, rng)
        comp_of, n_comp = np.zeros(20_000, int), 1
    elif shape == "torus":
        xyz, d = torus(30_000, rng)
        comp_of, n_comp = np.zeros(30_000, int), 1
    else:
        a, da = sphere(20_000, rng)
        b, db = sphere(20_000, rng, centre=(5.0, 0.0, 0.5))
        xyz, d = np.r_[a, b], np.r_[da, db]
        comp_of, n_comp = np.r_[np.zeros(20_000, int), np.ones(20_000, int)], 2
    m = scramble(d, rng)
    got = pto_orient.orient_normals(xyz, m, 18)
    assert got["components"] == n_comp and got["oriented"] == len(xyz)
    assert (dot(got["normal"].astype(np.float64), d) > 0).all()
    assert np.array_equal(got["root"], expected_roots(xyz, comp_of))
    assert got["flipped"] == int((dot(m.astype(np.float64), d) < 0).sum())


def test_pca_normals_of_a_sphere_come_out_outward(pto):
    rng = np.random.default_rng(7)
    xyz, d = sphere(20_000, rng)
    est, _, e = pto_normals.estimate_normals(xyz, None, 16)           # rule (c): about half point inwards
    assert e == len(xyz)
    inward = (dot(est.astype(np.float64), d) < 0).mean()
    assert 0.3 < inward < 0.7, inward
    got = pto_orient.orient_normals(xyz, est, 18)
    assert got["components"] == 1 and (dot(got["normal"].astype(np.float64), d) > 0).all()


def test_zero_normal_and_isolated_point(pto):
    rng = np.random.default_rng(3)
    xyz = np.r_[np.c_[rng.random((200, 2)), np.zeros(200)], [[50.0, 50.0, -3.0]]]
    m = np.r_[np.tile([[0.0, 0.0, -1.0]], (200, 1)), [[0.0, 0.0, -2.0]]].astype(np.float32)
    m[17] = 0.0
    m[18] = np.nan
    for k in (2, 8):
        idx = pto_normals.neighbours(xyz, k, 0.5)
        got = check_oracle_vs_scipy(xyz, m, idx)
        assert np.array_equal(got["normal"][17:19].view(np.uint32), m[17:19].view(np.uint32))
        assert (got["root"][17:19] == -1).all() and (got["parent"][17:19] == -1).all()
        assert got["root"][200] == 200 and got["parent"][200] == -1     # isolated: its own component
        assert np.array_equal(got["normal"][200].view(np.uint32),
                              np.array([-0.0, -0.0, 2.0], np.float32).view(np.uint32))
        keep = np.ones(201, bool)
        keep[17:19] = False
        assert (got["normal"][keep, 2] > 0).all()
        assert got["oriented"] == 199 and got["flipped"] == 199


def test_k_gt_n_and_duplicates(pto, golden_dir):
    for name in ("k_gt_n", "duplicates"):
        g = np.load(os.path.join(golden_dir, f"{name}.npz"))
        xyz = g["xyz"]
        m = scramble(np.tile([[0.0, 0.0, 1.0]], (len(xyz), 1)), np.random.default_rng(5), noise=0.1)
        for k in (2, 8, 32):
            got = check_oracle_vs_scipy(xyz, m, pto_normals.neighbours(xyz, k))
            assert got["oriented"] == len(xyz)
            if got["components"] == 1:
                assert (got["normal"][:, 2] > 0).all()


def test_root_with_zero_z_uses_the_largest_component(pto):
    rng = np.random.default_rng(9)
    xyz = np.c_[np.full(300, 1.5), rng.random((300, 2)) * 3.0]            # the plane x = 1.5
    m = np.c_[np.where(rng.random(300) < 0.5, -1.0, 1.0), np.zeros((300, 2))].astype(np.float32)
    got = check_oracle_vs_scipy(xyz, m, pto_normals.neighbours(xyz, 12))
    assert got["components"] == 1 and (got["normal"][:, 0] == 1.0).all()
    m[:, 0] = -np.abs(m[:, 0])
    m[:, 1] = -1e-3                                                      # |x| still the largest
    got = check_oracle_vs_scipy(xyz, m, pto_normals.neighbours(xyz, 12))
    assert (got["normal"][:, 0] == 1.0).all() and (got["normal"][:, 1] > 0).all()


def moebius(n=6000, seed=4):
    rng = np.random.default_rng(seed)
    u, t = rng.random(n) * 2 * np.pi, rng.random(n) * 0.8 - 0.4
    c, s, c2, s2 = np.cos(u), np.sin(u), np.cos(u / 2), np.sin(u / 2)
    xyz = np.c_[(1 + t * c2) * c, (1 + t * c2) * s, t * s2]
    du = np.c_[-(1 + t * c2) * s - 0.5 * t * s2 * c, (1 + t * c2) * c - 0.5 * t * s2 * s, 0.5 * t * c2]
    dt = np.c_[c2 * c, c2 * s, s2]
    return xyz, scramble(np.cross(du, dt), rng, noise=0.0)


def test_moebius_strip(pto):
    xyz, m = moebius()
    for k in (8, 18):
        got = check_oracle_vs_scipy(xyz, m, pto_normals.neighbours(xyz, k))
        assert got["components"] == 1


# ---- ties: equal weights, equal top z, many components ---------------------------------------------
def flat_lattice(g=100, permute=False, seed=6):
    """(xyz, normal float32, radius): a g x g lattice on z = 0, every tenth point at z = -0.0, with
    normals +-z of three lengths.  Every edge weight 1 - |d| is exactly 0, so the (lo, hi) keys alone
    decide the forest, and every point shares the top z.  ``permute`` shuffles the ids, so that id
    order differs from the lattice's (and the curve's) order."""
    rng = np.random.default_rng(seed)
    i, j = np.meshgrid(np.arange(g), np.arange(g), indexing="ij")
    xyz = np.c_[i.ravel() * 0.5, j.ravel() * 0.5, np.zeros(g * g)]
    xyz[::10, 2] = -0.0
    m = np.zeros((g * g, 3), np.float32)
    m[:, 2] = np.where(rng.random(g * g) < 0.5, -1.0, 1.0) * rng.choice([0.5, 1.0, 3.0], g * g)
    if permute:
        p = rng.permutation(g * g)
        xyz, m = xyz[p], m[p]
    return xyz, m, None


def plateau(n=20_000, seed=7):
    """A noisy patch cut flat at z = 0: about half the points share the top z, some of them -0.0."""
    xyz, m = noisy_patch(n, seed)
    xyz[:, 2] = np.minimum(xyz[:, 2], 0.0)
    top = np.flatnonzero(xyz[:, 2] == 0.0)
    xyz[top[::3], 2] = -0.0
    return xyz.astype(np.float32).astype(np.float64), m.astype(np.float32), None


FRUSTRATED = np.array([[1.0, 1.0, 0.0], [0.0, 1.0, 1.0], [1.0, 0.0, -1.0]])


def clusters(count=3000, seed=8):
    """(xyz, normal float32, radius): `count` clusters of 4 points, 10 apart, each inside a ball of
    radius 0.3, and a radius of 1, so every list stays inside its cluster and every cluster is a
    component of its own.  Three normals of each cluster are +-(1, 1, 0), +-(0, 1, 1), +-(1, 0, -1):
    their unit vectors' pairwise |d| round to the same value, so the three edges tie, and the edge
    signs around the triangle multiply to -1, so the sign a point gets depends on which two of the
    three edges the (lo, hi) order puts in the forest.  The fourth normal is random; ids are shuffled."""
    rng = np.random.default_rng(seed)
    g = int(np.ceil(count ** 0.5))
    c = np.c_[np.arange(count) % g * 10.0, np.arange(count) // g * 10.0, rng.uniform(-5.0, 5.0, count)]
    xyz = (np.repeat(c, 4, axis=0) + rng.uniform(-0.17, 0.17, (4 * count, 3))).astype(np.float32).astype(np.float64)
    m = np.empty((count, 4, 3))
    m[:, :3] = FRUSTRATED[np.argsort(rng.random((count, 3)), axis=1)]
    m[:, 3] = rng.standard_normal((count, 3))
    m *= np.where(rng.random((count, 4)) < 0.5, -1.0, 1.0)[..., None]
    p = rng.permutation(4 * count)
    return xyz[p], m.reshape(-1, 3).astype(np.float32)[p], 1.0


TIE_CLOUDS = {"lattice": flat_lattice, "lattice_permuted": lambda: flat_lattice(permute=True),
              "plateau": plateau, "clusters": clusters}


def list_edges(m, idx):
    """(i, j, w) of every list entry j != i, with w = 1 - |d| as the definition computes it."""
    m = m.astype(np.float64)
    nh = m / np.sqrt(dot(m, m))[:, None]
    i = np.repeat(np.arange(len(idx)), idx.shape[1]).reshape(idx.shape)
    keep = (idx >= 0) & (idx != i)
    i, j = i[keep], idx[keep]
    return i, j, np.maximum(1.0 - np.abs(dot(nh[i], nh[j])), 0.0)


def check_tie_cloud(name, xyz, m, idx, got):
    """That each tie cloud reaches what it is built for."""
    z = xyz[:, 2]
    if name.startswith("lattice"):
        assert (list_edges(m, idx)[2] == 0.0).all()                           # every weight is 0
        assert (z == 0.0).all() and np.signbit(z).sum() == len(z) // 10
        assert (got["normal"][:, 2] > 0).all()
        if idx.shape[1] >= 8:                              # one component (k = 2 leaves pairs and chains)
            assert got["components"] == 1
            assert (got["root"] == 0).all()              # every z ties, -0.0 with +0.0: the lowest id
    elif name == "plateau":
        if idx.shape[1] >= 8:
            r = np.bincount(got["root"][got["root"] >= 0]).argmax()            # the largest component
            top = (got["root"] == r) & (z == 0.0)
            assert z[r] == 0.0 and top.sum() > 1000 and np.signbit(z[top]).any() and not np.signbit(z[top]).all()
    else:
        i, j, w = list_edges(m, idx)
        tri = (np.abs(m).sum(1) == 2.0) & (m == 0.0).any(1)                   # the +-FRUSTRATED normals
        assert tri.sum() == 3 * len(z) // 4
        if idx.shape[1] >= 4:                                                  # whole clusters in every list
            assert got["components"] == len(z) // 4
            assert len(np.unique(w[tri[i] & tri[j]])) == 1                     # one tied weight


@pytest.mark.parametrize("name", sorted(TIE_CLOUDS))
def test_oracle_equals_scipy_on_ties(name, pto):
    xyz, m, radius = TIE_CLOUDS[name]()
    for k in (2, 8, 32):
        idx = pto_normals.neighbours(xyz, k, -1.0 if radius is None else radius)
        got = check_oracle_vs_scipy(xyz, m, idx)
        check_tie_cloud(name, xyz, m, idx, got)


# ---- CLI ---------------------------------------------------------------------------------------------
def _cli():
    from test_cli import CLI
    if not os.path.exists(CLI):
        subprocess.run(["make", "-C", os.path.dirname(CLI)], check=True, stdout=subprocess.DEVNULL)
    return CLI


@pytest.mark.parametrize("args", [["-O", "1"], ["-O", "33"], ["-O", "18", "-g", "2"]])
def test_cli_refuses_bad_orientation_options(args, tmp_path):
    r = subprocess.run([_cli(), *args, "a.ply", "b.ply"], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and "-O must be 2..32" in r.stderr
    assert not (tmp_path / "texture.png").exists()


# ---- GPU ---------------------------------------------------------------------------------------------
def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def assert_same(got, ref, what=""):
    assert np.array_equal(got["normal"].view(np.uint32), ref["normal"].view(np.uint32)), what
    assert np.array_equal(got["root"], ref["root"]), what
    for key in ("oriented", "flipped", "components", "edges"):
        assert got["stats"][key] == ref[key], (key, what)


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_gpu_equals_oracle_on_golden_clouds(path, pkg, pto):
    _need_gpu()
    g = np.load(path)
    f64 = "f64" in os.path.basename(path)
    mode = pkg.COORD_F64 if f64 else pkg.COORD_AUTO
    rng = np.random.default_rng(1)
    flipped = (g["normal"] * np.where(rng.random(len(g["xyz"])) < 0.5, -1.0, 1.0)[:, None]).astype(np.float32)
    for nrm in (g["normal"].astype(np.float32), flipped):
        with pkg.Tree(pkg.make_points(g["xyz"], normal=nrm, color=g["color"]), coord_mode=mode) as tree:
            if f64:
                assert tree.info().coord_mode == pkg.COORD_F64
            for k in (2, 8, 18, 32):
                for radius in (None, float(g["radius"])):
                    idx = pto_normals.neighbours(g["xyz"], k, -1.0 if radius is None else radius)
                    for view in (None, VIEW):
                        ref = pto_orient.orient(g["xyz"], nrm, idx, view)
                        assert_same(tree.orient_normals(k, radius=radius, viewpoint=view), ref, (k, radius, view))


@pytest.mark.gpu
def test_gpu_equals_oracle_on_shapes(pkg, pto):
    _need_gpu()
    rng = np.random.default_rng(2026)
    a, da = sphere(20_000, rng)
    b, db = sphere(20_000, rng, centre=(5.0, 0.0, 0.5))
    xyz_t, dt = torus(30_000, rng)
    xyz_m, mm = moebius()
    xyz_p, mp = noisy_patch()
    for xyz, m in ((np.r_[a, b], scramble(np.r_[da, db], rng)), (xyz_t, scramble(dt, rng)), (xyz_m, mm),
                   (xyz_p, mp.astype(np.float32))):
        xyz = xyz.astype(np.float32).astype(np.float64)                  # the positions an F32 index stores
        with pkg.Tree(pkg.make_points(xyz, normal=m)) as tree:
            for k, view in ((8, None), (18, None), (18, (0.0, 0.0, 10.0))):
                ref = pto_orient.orient(xyz, m, pto_normals.neighbours(xyz, k), view)
                assert_same(tree.orient_normals(k, viewpoint=view), ref, k)


@pytest.mark.gpu
def test_gpu_more_than_one_chunk(pkg, pto):
    _need_gpu()
    n = 4_500_000                            # lists of two chunks of 2^22 rows
    pos, attrs = pkg.synth.cloud_device(n, seed=20261021, u1=425.0, v1=425.0)
    P = pkg.synth.points_to_host(pos, attrs)
    rng = np.random.default_rng(8)
    P["normal"] *= np.where(rng.random(n) < 0.5, -1.0, 1.0)[:, None]
    m = P["normal"].astype(np.float32)
    xyz = P["ver"].astype(np.float32).astype(np.float64)
    with pkg.Tree(P) as tree:
        got = tree.orient_normals(18)
    ref = pto_orient.orient(xyz, m, pto_normals.neighbours(xyz, 18))
    assert_same(got, ref)


@pytest.mark.gpu
def test_gpu_store_feeds_transfer_and_bake(pkg, pto):
    _need_gpu()
    from test_bake import grid_mesh
    from test_bake_tangent import ALL_OUTPUTS
    side = 30.0
    P = pkg.synth.cloud_host(60_000, seed=9, side=side)
    rng = np.random.default_rng(10)
    P["normal"] *= np.where(rng.random(len(P)) < 0.5, -1.0, 1.0)[:, None]
    P["normal"][::5] = 0.0                                   # some points do not take part
    V, F = grid_mesh(pkg, 12, side)
    q = pkg.make_points(V["ver"] + 0.01)
    with pkg.Tree(P) as tree:
        before = tree.transfer(q, 8)
        kept = tree.orient_normals(18, store=False)
        assert tree.transfer(q, 8)["normal"].tobytes() == before["normal"].tobytes()
        again = tree.orient_normals(18, store=False)
        assert_same(again, dict(kept, **kept["stats"]))
        ori = tree.orient_normals(18, store=True)
        after_t = tree.transfer(q, 8)
        after_b = tree.bake(V, F, k=16, resolution=200, want=ALL_OUTPUTS + ("height",))
    assert_same(ori, dict(kept, **kept["stats"]))
    assert ori["stats"]["flipped"] > 0
    Q = P.copy()
    Q["normal"] = ori["normal"]
    with pkg.Tree(Q) as ref:
        ref_t = ref.transfer(q, 8)
        ref_b = ref.bake(V, F, k=16, resolution=200, want=ALL_OUTPUTS + ("height",))
    for key in ("rgba", "normal", "idx"):
        assert after_t[key].tobytes() == ref_t[key].tobytes(), key
    for key in ALL_OUTPUTS + ("height",):
        assert after_b[key].tobytes() == ref_b[key].tobytes(), key


@pytest.mark.gpu
def test_gpu_errors(pkg, pto):
    _need_gpu()
    import torch
    P = pkg.synth.cloud_host(20_000, seed=3, side=30.0)
    L = pkg.lib()
    with pkg.Tree(P) as tree:
        out = np.empty((len(P), 3), np.float32)
        h = tree.handle
        for k, rc in ((1, 1), (0, 1), (33, 5)):                 # 1 invalid argument, 5 unsupported
            assert L.pt_index_orient_normals(h, k, -1.0, None, 0, out.ctypes.data, None, None) == rc
        assert L.pt_index_orient_normals(h, 8, -1.0, None, 0, None, None, None) == 1
        bad = (ctypes.c_double * 3)(0.0, float("inf"), 1.0)
        assert L.pt_index_orient_normals(h, 8, -1.0, bad, 0, out.ctypes.data, None, None) == 1
        assert L.pt_index_orient_normals(None, 8, -1.0, None, 1, None, None, None) == 1
        assert L.pt_index_orient_normals(h, 2, -1.0, None, 0, out.ctypes.data, None, None) == 0
    pos, _ = pkg.synth.cloud_device(1000, seed=3, u1=30.0, v1=30.0)
    bare = pkg.DeviceTree(pos)                                     # no attributes: nothing to orient
    root = np.empty(1000, np.int32)
    assert L.pt_index_orient_normals(bare.handle, 8, -1.0, None, 0, None, root.ctypes.data, None) == 1
    bare.close()
    big = pkg.DeviceTree(*pkg.synth.cloud_device(70_000_000, seed=3, u1=900.0, v1=900.0))
    root = np.empty(70_000_000, np.int32)
    assert L.pt_index_orient_normals(big.handle, 32, -1.0, None, 0, None, root.ctypes.data, None) == 5  # n k > 2^31 - 1
    big.close()
    torch.cuda.synchronize()
    with pkg.Tree(pkg.make_points(np.zeros((0, 3)))) as empty:
        assert L.pt_index_orient_normals(empty.handle, 8, -1.0, None, 1, None, None, None) == 0


@pytest.mark.gpu
def test_gpu_cli_orient_equals_python(pkg, pto, tmp_path):
    _need_gpu()
    from test_bake import grid_mesh
    from test_cli import read_png_bgra, write_cloud, write_mesh
    side = 30.0
    P = pkg.synth.cloud_host(40_000, seed=12, side=side)
    P["normal"] = 0.0
    P["ver"] = P["ver"].astype(np.float32).astype(np.float64)
    V, F = grid_mesh(pkg, 12, side)
    write_cloud(tmp_path / "c.ply", P)
    write_mesh(tmp_path / "m.ply", V, F)
    r = subprocess.run([_cli(), "-R", "128", "-e", "16", "-O", "18", "-n", "normal.png", str(tmp_path / "c.ply"),
                        str(tmp_path / "m.ply")], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    assert "Oriented normals: 40000 of 40000 points, " in r.stdout, r.stdout
    Vm = V.copy()
    Vm["normal"] = (0.0, 0.0, 1.0)                                # write_mesh's normal column
    with pkg.Tree(P) as tree:
        tree.estimate_normals(16, store=True)
        ori = tree.orient_normals(18, store=True)
        ref = tree.bake(Vm, F, k=20, resolution=128, want=("normal_bgra",))
    st = ori["stats"]
    assert f"{st['flipped']} flipped, {st['components']} components" in r.stdout, r.stdout
    assert np.array_equal(read_png_bgra(tmp_path / "normal.png"), ref["normal_bgra"])
