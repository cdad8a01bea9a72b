"""k-NN exactness in real-world coordinate frames, on the CPU.

Real scans arrive georeferenced (a UTM easting is ~4.5e5, a northing ~5.4e6), and the numeric devices
of the exactness argument (DESIGN.md section 2) change behaviour with the coordinates' magnitude: the
grid's termination slack grows with the distance from the origin, fp32 box bounds coarsen, selection
keys go subnormal or saturate.  Here the oracle (pto.knn_bruteforce, pto.KdTree with exact ties) is
pinned on a plain numpy brute force in every frame tests/test_gpu_frames.py uses, and on two exact
identities that the GPU file then checks without an oracle:

- dyadic translation: a cloud on a 2^-4 lattice shifted by a multiple of 2^-4 keeps every q - p
  exact, so indices and d2 are unchanged bit for bit;
- power-of-two scaling by 2^s keeps the indices and multiplies every d2 by exactly 4^s, also where
  d2 lies below the fp32 normal range (s = -70) or above FLT_MAX (s = 70).

Out of scope (behaviour the project does not define): d2 overflowing fp64, and coordinates at or
above FLT_MAX in F32 storage."""
import numpy as np
import pytest

LATTICE = 2.0 ** -4
EXTENT = 128.0                                     # x extent of every dyadic cloud: a power of two
UTM = (452_311.0, 5_411_873.0, 312.0)              # easting, northing, height
F32_OFFSETS = ((452_304.0, 0.0, 0.0), (524_160.0, -300_000.0, 1000.0))    # 2^-4 multiples below 2^19
F64_OFFSETS = ((5_411_873.0, 452_311.0, 312.0), (2.0 ** 40, -2.0 ** 40, 2.0 ** 30))
SCALES = (-70, -40, -10, 10, 40, 70)               # F32-representable; d2 subnormal in fp32 at -70, > FLT_MAX at 70
DYADIC_RADIUS = 0.75                               # r^2 = 144 / 256: on the grid of the lattice's d2
FAR = (1e3, 1e12)                                  # far samples, in units of the extent


def ref_knn(P, Q, k, radius=None):
    """numpy fp64 brute force in the metric's operation order ((dx dx + dy dy) + dz dz), ascending
    (d2, index), radius inclusive (d2 <= r^2); padded with -1 / +inf."""
    P, Q = np.asarray(P, np.float64), np.asarray(Q, np.float64)
    idx = np.full((len(Q), k), -1, np.int32)
    d2 = np.full((len(Q), k), np.inf)
    r2 = np.inf if radius is None else radius * radius
    ids = np.arange(len(P))
    for s, q in enumerate(Q):
        dx, dy, dz = q[0] - P[:, 0], q[1] - P[:, 1], q[2] - P[:, 2]
        d = (dx * dx + dy * dy) + dz * dz
        keep = np.flatnonzero(d <= r2)
        o = keep[np.lexsort((ids[keep], d[keep]))][:k]
        idx[s, :len(o)] = o
        d2[s, :len(o)] = d[o]
    return idx, d2


def f32_exact(xyz):
    with np.errstate(over="ignore"):
        return bool(np.array_equal(np.asarray(xyz, np.float32).astype(np.float64), xyz))


def dyadic_cloud(n, m, seed):
    """(P, Q): n points and m samples on the 2^-4 lattice in [0, 128] x [0, 100] x [0, 6]; the first
    two points pin the x extent to exactly 128, so every cell boundary of the grid lies on the
    lattice's dyadic grid too."""
    rng = np.random.default_rng(seed)
    box = np.array([EXTENT, 100.0, 6.0])
    P = np.round(rng.random((n, 3)) * box / LATTICE) * LATTICE
    P[0], P[1] = (0.0, 50.0, 3.0), (EXTENT, 50.0, 3.0)
    Q = np.round(rng.random((m, 3)) * box / LATTICE) * LATTICE
    return P, Q


def far_samples(P, scales=FAR):
    """Samples 10^3 and 10^12 extents away from the cloud's centre, in the 6 axis directions and
    the 8 diagonals."""
    c = 0.5 * (P.min(0) + P.max(0))
    ext = float((P.max(0) - P.min(0)).max())
    dirs = np.r_[np.eye(3), -np.eye(3), np.array(np.meshgrid([-1, 1], [-1, 1], [-1, 1])).reshape(3, -1).T]
    return np.concatenate([c + ext * f * dirs for f in scales])


def frame_clouds(n=20_000, m=400, seed=5):
    """name -> (P, Q, storage 'f32' / 'f64', radius of the bounded run): the frames of the GPU file."""
    rng = np.random.default_rng(seed)
    box = np.array([100.0, 100.0, 5.0])
    out = {}
    # UTM easting / northing, mm quantisation: fp64 storage
    P = (np.round(rng.random((n, 3)) * box * 1000) + np.array(UTM) * 1000) / 1000
    Q = (np.round(rng.random((m, 3)) * box * 1000) + np.array(UTM) * 1000) / 1000
    out["utm_mm"] = (P, Q, "f64", 0.8)
    # below 2^19 on the 2^-4 lattice: fp32 storage far from the origin (one fp32 ulp is 2^-5 there)
    P0, Q0 = dyadic_cloud(n, m, seed + 1)
    off = np.array(F32_OFFSETS[1])
    out["f32_far"] = (P0 + off, Q0 + off, "f32", DYADIC_RADIUS)
    # a 1e-3-wide patch at the UTM offset: the slack exceeds the fine cells
    P = np.array(UTM) + rng.random((n, 3)) * np.array([1e-3, 1e-3, 1e-4])
    Q = np.array(UTM) + rng.random((m, 3)) * np.array([1e-3, 1e-3, 1e-4])
    out["thin_utm"] = (P, Q, "f64", 2e-5)
    # a plane at z = 312 (a flat roof / floor) at the easting, on the 2^-5 lattice
    xy = np.round(rng.random((n, 2)) * 100.0 * 32) / 32 + np.array([452_304.0, 0.0])
    P = np.c_[xy, np.full(n, 312.0)]
    qxy = np.round(rng.random((m, 2)) * 100.0 * 32) / 32 + np.array([452_304.0, 0.0])
    Q = np.c_[qxy, 312.0 + np.round(rng.standard_normal(m) * 32) / 32]
    out["planar"] = (P, Q, "f32", 0.7)
    # samples far outside the bounding box of a cloud at the origin
    P0, _ = dyadic_cloud(n, 1, seed + 2)
    out["far_samples"] = (P0, far_samples(P0), "f32", 2e3 * EXTENT)
    return out


# ---- the oracle against numpy in every frame ----------------------------------------------------------
@pytest.fixture(scope="module")
def frames():
    return frame_clouds()


@pytest.mark.parametrize("name", ["utm_mm", "f32_far", "thin_utm", "planar", "far_samples"])
def test_oracle_equals_numpy_in_frame(name, frames, pto):
    P, Q, storage, radius = frames[name]
    assert ("f32" if f32_exact(P) else "f64") == storage, name
    pts, qs = pto.make_points(P), pto.make_points(Q)
    tree = pto.KdTree(pts)
    for k, r in ((16, None), (7, None), (16, radius)):
        ref_i, ref_d = ref_knn(P, Q, k, r)
        rr = -1.0 if r is None else r
        if r is not None:
            assert 0 < (ref_i >= 0).sum() < ref_i.size, (name, k, r)    # the radius cuts some lists short
        bi, bd = pto.knn_bruteforce(pts, qs, k, radius=rr)
        ki, kd = tree.knn(qs, k, radius=rr, exact_ties=True)
        for what, (i, d) in (("brute force", (bi, bd)), ("kd-tree", (ki, kd))):
            assert np.array_equal(i, ref_i), (name, what, k, r)
            assert np.array_equal(d.view(np.uint64), ref_d.view(np.uint64)), (name, what, k, r)


def test_lattice_frames_have_ties():
    """The dyadic clouds tie adjacent d2 often enough that the exact tie paths run."""
    P, Q = dyadic_cloud(20_000, 400, 2)
    _, d = ref_knn(P, Q, 16)
    assert np.mean(d[:, 1:] == d[:, :-1]) > 0.002


# ---- the identities on the oracle ---------------------------------------------------------------------
@pytest.fixture(scope="module")
def dyadic(pto):
    P0, Q0 = dyadic_cloud(20_000, 400, 2)
    base = {}
    for k, r in ((16, None), (16, DYADIC_RADIUS)):
        base[k, r] = pto.KdTree(pto.make_points(P0)).knn(pto.make_points(Q0), k, radius=-1.0 if r is None else r)
    ref_i, ref_d = ref_knn(P0, Q0, 16)
    assert np.array_equal(base[16, None][0], ref_i) and np.array_equal(base[16, None][1], ref_d)
    return P0, Q0, base


@pytest.mark.parametrize("off", F32_OFFSETS + F64_OFFSETS, ids=lambda o: "%g,%g,%g" % o)
def test_dyadic_translation_on_oracle(off, dyadic, pto):
    P0, Q0, base = dyadic
    P, Q = P0 + np.array(off), Q0 + np.array(off)
    assert np.array_equal(P - np.array(off), P0)                    # the shift is exact
    assert f32_exact(P) == (off in F32_OFFSETS)
    tree = pto.KdTree(pto.make_points(P))
    for (k, r), (i0, d0) in base.items():
        rr = -1.0 if r is None else r
        for i, d in (tree.knn(pto.make_points(Q), k, radius=rr, exact_ties=True),
                     pto.knn_bruteforce(pto.make_points(P), pto.make_points(Q), k, radius=rr)):
            assert np.array_equal(i, i0), (off, k, r)
            assert np.array_equal(d.view(np.uint64), d0.view(np.uint64)), (off, k, r)


@pytest.mark.parametrize("s", SCALES + (200,))
def test_power_of_two_scaling_on_oracle(s, dyadic, pto):
    P0, Q0, base = dyadic
    P, Q = np.ldexp(P0, s), np.ldexp(Q0, s)
    assert f32_exact(P) == (s != 200)
    tree = pto.KdTree(pto.make_points(P))
    for (k, r), (i0, d0) in base.items():
        rr = -1.0 if r is None else np.ldexp(r, s)
        for i, d in (tree.knn(pto.make_points(Q), k, radius=rr, exact_ties=True),
                     pto.knn_bruteforce(pto.make_points(P), pto.make_points(Q), k, radius=rr)):
            assert np.array_equal(i, i0), (s, k, r)
            assert np.array_equal(d, np.ldexp(d0, 2 * s)), (s, k, r)
    d = np.ldexp(base[16, None][1], 2 * s)
    if s == -70:
        assert 0 < d[d > 0].min() and d.max() < np.finfo(np.float32).tiny      # every nonzero d2 subnormal in fp32
    if s == 70:
        assert d[d > 0].min() > np.finfo(np.float32).max                         # every nonzero d2 above FLT_MAX
