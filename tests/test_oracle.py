"""CPU tests: the oracle against the golden fixtures and independent implementations.

The reference has no tests of its own (SURVEY.md section 4); the oracle restates
src/Distance.h and CGAL's published k-d tree search (parity unpinned, see oracle/pt_oracle.h).
"""
import glob
import os

import ctypes

import numpy as np
import pytest
from scipy.spatial import cKDTree


def _load(path, pto):
    z = np.load(path)
    P = pto.make_points(z["xyz"], normal=z["normal"], color=z["color"])
    Q = pto.make_points(z["queries"])
    return z, P, Q


def test_point_layout(pto):
    # src/Point.h:1-6 measured layout: 80 bytes, ver@0 normal@24 color@48 U@64 V@72
    dt = pto.POINT_DTYPE
    assert dt.itemsize == 80
    assert [dt.fields[f][1] for f in ("ver", "normal", "color", "U", "V")] == [0, 24, 48, 64, 72]


def test_metric_op_order(pto):
    # src/Distance.h:6-11: (dx*dx + dy*dy) + dz*dz in fp64, separately rounded
    rng = np.random.default_rng(3)
    for _ in range(200):
        a, b = rng.standard_normal(3) * 10.0 ** rng.integers(-3, 6), rng.standard_normal(3)
        pa, pb = pto.make_points(a[None]), pto.make_points(b[None])
        d = a - b
        expect = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]
        assert pto.transformed_distance(pa[0], pb[0]) == expect
    assert pto.lib().pto_transformed_radius(3.0) == 9.0          # src/Distance.h:97
    assert pto.lib().pto_new_distance(10.0, 2.0, 3.0) == 10.0 + 9.0 - 4.0   # :92-95


def test_box_lower_bound(pto):
    # src/Distance.h:27-57: zero inside, per-axis offsets outside, dists untouched inside slab
    p = pto.make_points(np.array([[0.5, 2.0, -1.0]]))[0]
    d, dists = pto.min_distance_to_rectangle(p, [0, 0, 0], [1, 1, 1])
    assert d == 1.0 + 1.0 and list(dists) == [0.0, 1.0, 1.0]
    d, _ = pto.min_distance_to_rectangle(p, [0, 0, -2], [1, 3, 0])
    assert d == 0.0


@pytest.mark.parametrize("name", sorted(os.path.basename(p)[:-4] for p in glob.glob(
    os.path.join(os.path.dirname(__file__), "golden", "*.npz"))))
def test_golden_bruteforce_and_kdtree(name, pto, golden_dir):
    z, P, Q = _load(os.path.join(golden_dir, name + ".npz"), pto)
    radius = float(z["radius"])
    tree = pto.KdTree(P)
    for k in z["ks"]:
        k = int(k)
        idx, d2 = pto.knn_bruteforce(P, Q, k, radius=radius)
        assert np.array_equal(idx, z[f"idx_k{k}"])
        assert np.array_equal(d2, z[f"d2_k{k}"])
        kidx, kd2 = tree.knn(Q, k, radius=radius, exact_ties=True)
        assert np.array_equal(kidx, idx) and np.array_equal(kd2, d2)
        # CGAL-semantics search (strict '<'): same distances, tie order may differ
        cidx, cd2 = tree.knn(Q, k, radius=radius, exact_ties=False)
        assert np.array_equal(cd2, d2)
        rgba, nrm = pto.blend(P, idx, d2)
        assert np.array_equal(rgba, z[f"rgba_k{k}"])
        assert np.array_equal(nrm, z[f"normal_k{k}"])


def test_against_scipy_and_sklearn(pto):
    from sklearn.neighbors import NearestNeighbors
    rng = np.random.default_rng(11)
    xyz = (rng.random((50_000, 3)) * 100).astype(np.float32).astype(np.float64)
    q = (rng.random((500, 3)) * 100).astype(np.float32).astype(np.float64)
    P, Q = pto.make_points(xyz), pto.make_points(q)
    k = 20
    idx, d2 = pto.knn_bruteforce(P, Q, k)
    sd, si = cKDTree(xyz, leafsize=10, balanced_tree=False, compact_nodes=False).query(q, k)
    assert np.array_equal(si.astype(np.int32), idx)           # random data: no ties
    assert np.allclose(sd ** 2, d2, rtol=1e-12)
    nd, ni = NearestNeighbors(n_neighbors=k, algorithm="brute").fit(xyz).kneighbors(q)
    assert np.array_equal(ni.astype(np.int32), idx)
    kidx, kd2 = pto.KdTree(P).knn(Q, k)
    assert np.array_equal(kidx, idx) and np.array_equal(kd2, d2)


def test_tie_rule_lowest_index(pto):
    # 8 points at identical distance: the k lowest indices must be returned in index order
    c = np.array([[x, y, z] for x in (-1.0, 1.0) for y in (-1.0, 1.0) for z in (-1.0, 1.0)])
    P, Q = pto.make_points(c), pto.make_points(np.zeros((1, 3)))
    idx, d2 = pto.knn_bruteforce(P, Q, 5)
    assert idx.tolist() == [[0, 1, 2, 3, 4]] and np.all(d2 == 3.0)
    kidx, _ = pto.KdTree(P, bucket_size=2).knn(Q, 5)
    assert kidx.tolist() == [[0, 1, 2, 3, 4]]


def test_blend_definition(pto):
    # inverse-squared-distance weights; colour truncated (src/pointsTransfer.cpp:100-102)
    xyz = np.array([[1.0, 0, 0], [0, 2.0, 0], [5.0, 5.0, 5.0]])
    P = pto.make_points(xyz, normal=[[1, 0, 0], [0, 1, 0], [0, 0, 1]],
                        color=[[255, 0, 10], [0, 255, 10], [9, 9, 9]])
    Q = pto.make_points(np.zeros((1, 3)))
    idx, d2 = pto.knn_bruteforce(P, Q, 2)
    rgba, nrm = pto.blend(P, idx, d2)
    w = np.array([1.0, 0.25]); W = w.sum()
    assert rgba.tolist() == [[int(255 * 1.0 / W), int(255 * 0.25 / W), 10, 255]]
    n = np.array([1.0, 0.25, 0.0]); n /= np.linalg.norm(n)
    assert np.allclose(nrm[0], n, rtol=1e-6)
    # exact hit: copy that point; empty list: zeros with alpha 0
    idx, d2 = pto.knn_bruteforce(P, P[:1], 3)
    rgba, nrm = pto.blend(P, idx, d2)
    assert rgba.tolist() == [[255, 0, 10, 255]] and nrm.tolist() == [[1.0, 0.0, 0.0]]
    idx, d2 = pto.knn_bruteforce(P, Q, 2, radius=0.5)
    rgba, nrm = pto.blend(P, idx, d2)
    assert idx.tolist() == [[-1, -1]] and rgba.tolist() == [[0, 0, 0, 0]] and not nrm.any()


def test_reference_face_loop(pkg, pto):
    # src/pointsTransfer.cpp:465-479: 3 K-NN searches per face
    P = pkg.synth.cloud_host(20_000, 5, side=30.0)
    V = pkg.synth.samples_host(12, side=30.0)
    F = pkg.synth.grid_faces(12, 12)
    tree = pto.KdTree(P)
    assert tree.reference_face_loop(V, F, 20) == 3 * 20 * F.shape[0]


# ---- pinned on the reference's own headers (oracle/_ref, built by `make -C oracle ref`) ----------
def _ref_or_skip(pto):
    R = pto.ref_metric()
    if R is None:
        pytest.skip("needs the reference's own headers: set PT_REFERENCE_SRC to its src/ directory")
    return R


def _rand_points(pto, n, rng, scale):
    P = np.zeros(n, dtype=pto.POINT_DTYPE)
    P["ver"] = (rng.standard_normal((n, 3)) * scale)
    return P


def test_record_layout_matches_reference_struct(pto):
    """sizeof(Point) and the field offsets of the reference's src/Point.h, as its compiler lays
    them out, are what the C ABI (PT_POINT_STRIDE), the oracle and the Python dtypes assume."""
    R = _ref_or_skip(pto)
    out = (ctypes.c_int * 6)()
    R.ref_point_layout(out)
    f = pto.POINT_DTYPE.fields
    assert list(out) == [pto.POINT_DTYPE.itemsize, f["ver"][1], f["normal"][1], f["color"][1],
                         f["U"][1], f["V"][1]] == [80, 0, 24, 48, 64, 72]


def test_metric_is_bit_identical_to_reference_distance_h(pto):
    """Distance::transformed_distance (src/Distance.h:6-11) compiled from the reference's header
    against the oracle's restatement: bit-identical on fp32-representable and on arbitrary fp64
    coordinates, at several magnitudes (no FMA contraction on either side)."""
    R = _ref_or_skip(pto)
    rng = np.random.default_rng(7)
    for scale, as_f32 in ((1.0, True), (1000.0, True), (1.0, False), (1e6, False), (1e-6, False)):
        A, B = _rand_points(pto, 20000, rng, scale), _rand_points(pto, 20000, rng, scale)
        if as_f32:
            A["ver"] = A["ver"].astype(np.float32); B["ver"] = B["ver"].astype(np.float32)
        for i in range(len(A)):
            a, b = A[i:i + 1], B[i:i + 1]
            ref = R.ref_transformed_distance(a.ctypes.data, b.ctypes.data)
            got = pto.transformed_distance(A[i], B[i])
            assert ref == got and np.float64(ref).tobytes() == np.float64(got).tobytes()
    # brute-force k-NN distances are this metric too
    P, Q = _rand_points(pto, 500, rng, 10.0), _rand_points(pto, 20, rng, 10.0)
    idx, d2 = pto.knn_bruteforce(P, Q, 5)
    for qi in range(len(Q)):
        for j in range(5):
            assert d2[qi, j] == R.ref_transformed_distance(Q[qi:qi + 1].ctypes.data,
                                                           P[idx[qi, j]:idx[qi, j] + 1].ctypes.data)


def test_box_bound_and_helpers_match_reference_distance_h(pto):
    """min_distance_to_rectangle (3-argument form, src/Distance.h:27-57), new_distance (:92-95),
    transformed_distance(d) (:97): the oracle's restatements against the reference's code."""
    R = _ref_or_skip(pto)
    rng = np.random.default_rng(11)
    for _ in range(5000):
        p = _rand_points(pto, 1, rng, 3.0)
        c = rng.standard_normal(3) * 3.0
        h = np.abs(rng.standard_normal(3))
        lo, hi = np.ascontiguousarray(c - h), np.ascontiguousarray(c + h)
        d_ref, d_got = np.zeros(3), np.zeros(3)
        ref = R.ref_min_distance_to_rectangle(p.ctypes.data, lo.ctypes.data, hi.ctypes.data,
                                              d_ref.ctypes.data)
        got, d_got = pto.min_distance_to_rectangle(p[0], lo, hi, d_got)
        assert ref == got and np.array_equal(d_ref, d_got)
        a, b, cc = rng.standard_normal(3)
        assert R.ref_new_distance(abs(a), b, cc) == pto.lib().pto_new_distance(abs(a), b, cc)
        assert R.ref_transformed_radius(a) == pto.lib().pto_transformed_radius(a)
    assert R.ref_inverse_of_transformed_distance(9.0) == 3.0


def test_golden_fixture_distances_are_the_reference_metric(pto, golden_dir):
    """The committed fixtures' squared distances, recomputed pair by pair with the reference's
    compiled Distance::transformed_distance, are bit-identical -- and ascending."""
    R = _ref_or_skip(pto)
    for path in sorted(glob.glob(os.path.join(golden_dir, "*.npz"))):
        z, P, Q = _load(path, pto)
        for k in z["ks"]:
            idx, d2 = z[f"idx_k{int(k)}"], z[f"d2_k{int(k)}"]
            for qi in range(0, len(Q), 5):
                for j in range(int(k)):
                    if idx[qi, j] < 0:
                        assert np.isinf(d2[qi, j])
                        continue
                    ref = R.ref_transformed_distance(Q[qi:qi + 1].ctypes.data,
                                                     P[idx[qi, j]:idx[qi, j] + 1].ctypes.data)
                    assert d2[qi, j] == ref, (os.path.basename(path), int(k), qi, j)
                    assert j == 0 or d2[qi, j - 1] <= d2[qi, j]
