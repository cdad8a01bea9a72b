"""Tangent-space bake (DESIGN.md section 8, "Tangent-space bake"): tangent-space normal maps and the
per-vertex tangents they are expressed in.

CPU part: the oracle (oracle/pt_bake_oracle.c via oracle/pto_bake.py) against an independent numpy
statement of the frozen definition, known answers on a flat quad, the exact invariance under a
quarter turn about z, and the CLI's refusals.  GPU part: pt_texture_bake_ex, the device pieces and
the CLI must equal the oracle bit for bit."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import pto_bake
from test_bake import awkward_mesh, grid_mesh, lattice_case
from test_cli import read_png_bgra, write_cloud, write_mesh

ALL_OUTPUTS = ("bgra", "normal_bgra", "normal", "tangent_bgra", "tangent_normal", "tangents")


# ---- the frozen definition restated in numpy (elementwise ufuncs: every operation rounded) -------
def _dot(a, b):
    return np.add(np.add(np.multiply(a[..., 0], b[..., 0]), np.multiply(a[..., 1], b[..., 1])),
                  np.multiply(a[..., 2], b[..., 2]))


def _cross(a, b):
    return np.stack([np.subtract(np.multiply(a[..., 1], b[..., 2]), np.multiply(a[..., 2], b[..., 1])),
                     np.subtract(np.multiply(a[..., 2], b[..., 0]), np.multiply(a[..., 0], b[..., 2])),
                     np.subtract(np.multiply(a[..., 0], b[..., 1]), np.multiply(a[..., 1], b[..., 0]))], -1)


def _usable(a):
    return np.isfinite(a).all(-1) & (_dot(a, a) > 0)


def _normalise(a):
    return np.divide(a, np.sqrt(_dot(a, a))[..., None])


def _scale(s, a):
    return np.multiply(s[..., None], a)


def _tangent_dir(n, t):
    r = np.subtract(t, _scale(_dot(n, t), n))
    ax = np.abs(n)
    i = np.where((ax[..., 0] <= ax[..., 1]) & (ax[..., 0] <= ax[..., 2]), 0, np.where(ax[..., 1] <= ax[..., 2], 1, 2))
    e = np.zeros_like(n)
    e[np.arange(len(n)), i] = 1.0
    fb = _normalise(np.subtract(e, _scale(n[np.arange(len(n)), i], n)))
    return np.where(_usable(r)[:, None], _normalise(r), fb)


def numpy_face_frames(V, F):
    """(T_f, B_f, G_f, valid) per face."""
    ok = ((F >= 0) & (F < len(V))).all(1)
    Fi = np.where(ok[:, None], F, 0)
    X, U, W = V["ver"], V["U"], V["V"]
    xa = X[Fi[:, 0]]
    e1, e2 = np.subtract(X[Fi[:, 1]], xa), np.subtract(X[Fi[:, 2]], xa)
    du1, dv1 = np.subtract(U[Fi[:, 1]], U[Fi[:, 0]]), np.subtract(W[Fi[:, 1]], W[Fi[:, 0]])
    du2, dv2 = np.subtract(U[Fi[:, 2]], U[Fi[:, 0]]), np.subtract(W[Fi[:, 2]], W[Fi[:, 0]])
    with np.errstate(all="ignore"):
        det = np.subtract(np.multiply(du1, dv2), np.multiply(du2, dv1))
        r = np.divide(1.0, det)
        T = _scale(r, np.subtract(_scale(dv2, e1), _scale(dv1, e2)))
        B = _scale(r, np.subtract(_scale(du1, e2), _scale(du2, e1)))
        bad = (det == 0) | ~np.isfinite(T).all(1) | ~np.isfinite(B).all(1)
        T[bad], B[bad] = 0.0, 0.0
        G = _cross(e1, e2)
    return T, B, G, ok


def numpy_frames(V, F):
    """(frames [n,8], tangents float32 [n,4]) by the definition: sums over corner occurrences in
    face order from +0.0, then N, T and w per vertex."""
    T_f, B_f, G_f, ok = numpy_face_frames(V, F)
    n = len(V)
    T, B, G = np.zeros((n, 3)), np.zeros((n, 3)), np.zeros((n, 3))
    for f in np.flatnonzero(ok):
        for v in F[f]:
            T[v], B[v], G[v] = np.add(T[v], T_f[f]), np.add(B[v], B_f[f]), np.add(G[v], G_f[f])
    frames = np.zeros((n, 8))
    with np.errstate(all="ignore"):
        nv = V["normal"].astype(np.float64)
        has = _usable(nv) | _usable(G)
        N = _normalise(np.where(_usable(nv)[:, None], nv, G))
        Th = _tangent_dir(np.where(has[:, None], N, [0, 0, 1.0]), T)
        w = np.where(_dot(_cross(N, Th), B) < 0, -1.0, 1.0)
    frames[has, 0:3], frames[has, 3:6], frames[has, 6] = N[has], Th[has], w[has]
    return frames, frames[:, 3:7].astype(np.float32)


def numpy_owner(V, F, res):
    """Owner face per covered texel (ascending texel order), highest face index wins."""
    row, col = np.divmod(np.arange(res * res), res)
    xa, xb = col + 0.5, (res - row) - 0.5
    owner = np.full(res * res, -1, np.int64)
    uv = np.stack([V["U"] * res, V["V"] * res], 1)
    with np.errstate(all="ignore"):
        for f, tri in enumerate(F):
            if (tri < 0).any() or (tri >= len(V)).any():
                continue
            bc = _bary(uv[tri], xa, xb)
            owner[(bc >= 0).all(1)] = f
    t = np.flatnonzero(owner >= 0)
    return t.astype(np.uint32), owner[t].astype(np.int32)


def _area2(p, q, r):
    return np.subtract(np.multiply(np.subtract(q[0], p[0]), np.subtract(r[1], p[1])),
                       np.multiply(np.subtract(q[1], p[1]), np.subtract(r[0], p[0])))


def _bary(t, xa, xb):
    x = (xa, xb)
    inv = np.divide(1.0, _area2(t[0], t[1], t[2]))
    b0 = np.multiply(_area2(t[1], t[2], x), inv)
    b1 = np.multiply(_area2(t[2], t[0], x), inv)
    return np.stack([b0, b1, np.subtract(np.subtract(1.0, b0), b1)], -1)


def numpy_compose_tangent(V, frames, F, texels, owner, rgba, m, res):
    """The two unpadded tangent maps (uint8 [res,res,4], float32 [res,res,3])."""
    tb = np.zeros((res * res, 4), np.uint8)
    tn = np.zeros((res * res, 3), np.float32)
    T_f, B_f, _, _ = numpy_face_frames(V, F)
    keep = rgba[:, 3] != 0
    texels, owner, m = texels[keep], owner[keep], m[keep].astype(np.float64)
    tri = F[owner]
    uv = np.stack([V["U"] * res, V["V"] * res], 1)
    row, col = np.divmod(texels.astype(np.int64), res)
    with np.errstate(all="ignore"):
        bc = _bary([uv[tri[:, j]].T for j in range(3)], col + 0.5, (res - row) - 0.5)

        def mix(c0):
            a, b, c = (frames[tri[:, j], c0:c0 + 3] for j in range(3))
            return np.add(np.add(_scale(bc[:, 0], a), _scale(bc[:, 1], b)), _scale(bc[:, 2], c))
        n, t = mix(0), mix(3)
        ok = _usable(n)
        n, t, m, texels, Bf = n[ok], t[ok], m[ok], texels[ok], B_f[owner[ok]]
        N = _normalise(n)
        T = _tangent_dir(N, t)
        x = _cross(N, T)
        w = np.where(_dot(x, Bf) < 0, -1.0, 1.0)
        B = _scale(w, x)
        ts = np.stack([_dot(m, T), _dot(m, B), _dot(m, N)], 1).astype(np.float32)
        enc = np.clip(np.floor(np.add(np.multiply(np.add(ts.astype(np.float64), 1.0), 127.5), 0.5)), 0, 255)
    tn[texels] = ts
    tb[texels, 0], tb[texels, 1], tb[texels, 2], tb[texels, 3] = enc[:, 2], enc[:, 1], enc[:, 0], 255
    return tb.reshape(res, res, 4), tn.reshape(res, res, 3)


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64 if a.dtype == np.float64 else np.uint32)


def assert_same(a, b, what):
    assert a.shape == b.shape and a.dtype == b.dtype, what
    if a.dtype.kind == "f":
        assert np.array_equal(_bits(a), _bits(b)), what
    else:
        assert np.array_equal(a, b), what


# ---- meshes -------------------------------------------------------------------------------------
def variant_mesh(pto, seed, variant):
    """awkward_mesh with one of the definition's special cases."""
    V, F = awkward_mesh(pto, seed)
    rng = np.random.default_rng(100 + seed)
    V = V.copy()
    if variant in ("random", "nan", "mirrored", "coincident"):
        V["normal"] = rng.standard_normal((len(V), 3)) * rng.uniform(0.2, 5.0, (len(V), 1))
    if variant == "nan":
        V["normal"][7] = [np.nan, 0.0, 1.0]
    if variant == "mirrored":                                  # chart 2 with U mirrored: w = -1 there
        half = len(V) // 2
        V["U"][half:] = 1.2 - V["U"][half:]
    if variant == "coincident":                                # T_f = 0: the F(N) fallback
        extra = pto.make_points(np.tile([3.0, 4.0, 5.0], (3, 1)), normal=[[0, 0.3, 1.0], [0.2, 0, 1], [0, 0, 1]],
                                uv=[[0.2, 0.2], [0.6, 0.25], [0.3, 0.7]])
        n = len(V)
        V = np.r_[V, extra]
        F = np.r_[F, [[n, n + 1, n + 2]]].astype(np.int32)
    return V, F


def sample_blend(rng, m):
    """Synthetic blend results: some empty lists (alpha 0), non-unit normals of either sign."""
    rgba = rng.integers(0, 256, (m, 4)).astype(np.uint8)
    rgba[:, 3] = np.where(rng.random(m) < 0.1, 0, 255)
    return rgba, rng.standard_normal((m, 3)).astype(np.float32)


VARIANTS = ("zero", "random", "nan", "mirrored", "coincident")


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("seed,res", [(1, 40), (2, 57), (3, 64)])
def test_oracle_equals_numpy_definition(pto, variant, seed, res):
    V, F = variant_mesh(pto, seed, variant)
    frames, tangents = pto_bake.bake_frames(V, F)
    ref_frames, ref_tangents = numpy_frames(V, F)
    assert_same(frames, ref_frames, "frames")
    assert_same(tangents, ref_tangents, "tangents")
    texels, _, owner = pto_bake.bake_samples(V, F, res)
    ref_t, ref_owner = numpy_owner(V, F, res)
    assert np.array_equal(texels, ref_t) and np.array_equal(owner, ref_owner)
    rgba, m = sample_blend(np.random.default_rng(seed), len(texels))
    tb, tn = pto_bake.bake_compose_tangent(V, frames, F, texels, owner, rgba, m, res, pad=False)
    ref_tb, ref_tn = numpy_compose_tangent(V, ref_frames, F, texels, owner, rgba, m, res)
    assert_same(tb, ref_tb, "tangent_bgra")
    assert_same(tn, ref_tn, "tangent_normal")
    assert tb[..., 3].any() and not tb.reshape(-1, 4)[texels[rgba[:, 3] == 0]].any()
    if variant == "zero":                                      # every frame from the face normals
        assert (np.abs(frames[:, 6]) == 1).sum() > len(V) // 2
    if variant == "nan":
        assert np.isfinite(frames).all()
    if variant == "mirrored":
        assert (frames[:, 6] == -1).any() and (frames[:, 6] == 1).any()
    if variant == "coincident":                                # the fallback tangent F(N) of n = (0,0,1)
        assert np.array_equal(tangents[-1], np.float32([1, 0, 0, 1]))


def flat_quad_case(pto, uv_map):
    """Flat quad at z = 0 with vertex normals (0, 0, 2); a lattice cloud with normals (0.48, 0.36, 0.8)."""
    L = 4.0
    X = np.array([[0, 0, 0], [L, 0, 0], [L, L, 0], [0, L, 0.0]])
    V = pto.make_points(X, normal=np.tile([0, 0, 2.0], (4, 1)), uv=uv_map(X[:, 0] / L, X[:, 1] / L))
    F = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    g = np.arange(-2, 19) * 0.25
    gx, gy = np.meshgrid(g, g)
    xyz = np.c_[gx.ravel(), gy.ravel(), np.zeros(gx.size)]
    rng = np.random.default_rng(12)
    P = pto.make_points(xyz, normal=np.tile([0.48, 0.36, 0.8], (len(xyz), 1)),
                        color=rng.integers(0, 256, (len(xyz), 3)))
    return P, V, F


KNOWN = {  # uv map, ts from m, exported tangent
    "identity": (lambda x, y: np.c_[x, y], lambda m: (m[:, 0], m[:, 1], m[:, 2]), [1, 0, 0, 1]),
    "mirrored": (lambda x, y: np.c_[1 - x, y], lambda m: (-m[:, 0], m[:, 1], m[:, 2]), [-1, 0, 0, -1]),
    "quarter": (lambda x, y: np.c_[y, 1 - x], lambda m: (m[:, 1], -m[:, 0], m[:, 2]), [0, 1, 0, 1]),
}


@pytest.mark.parametrize("case", sorted(KNOWN))
def test_known_answers_flat_quad(pto, case):
    uv_map, expect, tangent = KNOWN[case]
    P, V, F = flat_quad_case(pto, uv_map)
    res = 48
    out = pto_bake.bake_tangent(P, V, F, 4, res, pad=False)
    assert np.array_equal(out["tangents"], np.tile(np.float32(tangent), (4, 1)))
    texels, m = out["samples"][0], out["m"]
    assert out["texels"] == len(texels) > res * res // 2 and out["empty"] == 0
    assert (m != 0).all()
    ts = np.stack(expect(m), 1).astype(np.float32)
    assert np.array_equal(out["tangent_normal"].reshape(-1, 3)[texels], ts)
    enc = [[pto_bake.bake_encode(c) for c in ts[:, a]] for a in (2, 1, 0)]
    assert np.array_equal(out["tangent_bgra"].reshape(-1, 4)[texels][:, :3], np.array(enc).T)
    uncovered = np.ones(res * res, bool)
    uncovered[texels] = False
    assert not out["tangent_bgra"].reshape(-1, 4)[uncovered].any()
    assert not out["tangent_normal"].reshape(-1, 3)[uncovered].any()


def turn(P):
    """(x, y, z) -> (-y, x, z) of positions and normals."""
    Q = P.copy()
    for f in ("ver", "normal"):
        Q[f] = np.c_[-P[f][:, 1], P[f][:, 0], P[f][:, 2]]
    return Q


def turn_tangents(t):
    return np.ascontiguousarray(np.c_[-t[:, 1], t[:, 0], t[:, 2], t[:, 3]])


def turn_case(pto, n_points=6000, g=9):
    """A wavy grid mesh with tilted unit-ish normals (no vertex takes F) and a cloud around it."""
    rng = np.random.default_rng(31)
    t = np.linspace(0.0, 8.0, g)
    x, y = [a.ravel() for a in np.meshgrid(t, t)]
    z = 0.4 * np.sin(x) * np.cos(0.7 * y)
    nrm = np.c_[-0.3 * np.cos(x), 0.2 * np.sin(y), np.ones_like(x)] * rng.uniform(0.5, 2.0, (len(x), 1))
    V = pto.make_points(np.c_[x, y, z], normal=nrm, uv=np.c_[x / 8.0 * 0.9 + 0.05, y / 8.0 * 0.9 + 0.05])
    F = np.array([[a, a + 1, a + g] for j in range(g - 1) for a in range(j * g, j * g + g - 1)] +
                 [[a + 1, a + g + 1, a + g] for j in range(g - 1) for a in range(j * g, j * g + g - 1)], np.int32)
    px, py = rng.random(n_points) * 8.0, rng.random(n_points) * 8.0
    P = pto.make_points(np.c_[px, py, 0.4 * np.sin(px) * np.cos(0.7 * py) + rng.normal(0, 0.05, n_points)],
                        normal=rng.standard_normal((n_points, 3)), color=rng.integers(0, 256, (n_points, 3)))
    return P, V, F


def test_quarter_turn_invariance(pto):
    P, V, F = turn_case(pto)
    a = pto_bake.bake_tangent(P, V, F, 8, 96)
    b = pto_bake.bake_tangent(turn(P), turn(V), F, 8, 96)
    # no vertex and no texel took the fallback: every T is the projection of the summed T_f
    T_f, _, _, _ = numpy_face_frames(V, F)
    assert _usable(T_f).all()
    for key in ("tangent_bgra", "tangent_normal"):
        assert_same(a[key], b[key], key)
    # object-space vectors turn with the mesh (exactly, up to the sign of zero: x - x is +0)
    assert np.array_equal(turn_tangents(a["tangents"]), b["tangents"])
    assert not np.array_equal(a["normal_bgra"], b["normal_bgra"])
    assert not np.array_equal(a["normal"], b["normal"])
    assert a["tangent_bgra"][..., 3].any()


def _cli():
    from test_cli import CLI
    if not os.path.exists(CLI):
        subprocess.run(["make", "-C", os.path.dirname(CLI)], check=True, stdout=subprocess.DEVNULL)
    return CLI


@pytest.mark.parametrize("flag", ["-t", "-T"])
def test_cli_refuses_multi_gpu_tangent_bake(tmp_path, flag):
    r = subprocess.run([_cli(), "-g", "2", flag, "x.out", "a.ply", "b.ply"], capture_output=True, text=True,
                       cwd=tmp_path)
    assert r.returncode == 0 and "-t / -T" in r.stderr and not (tmp_path / "x.out").exists()


def test_cli_tangent_bake_without_gpu(pkg, tmp_path):
    if pkg.device_count() > 0:
        pytest.skip("a GPU is present")
    P = pkg.synth.cloud_host(50, 1)
    write_cloud(tmp_path / "c.ply", P)
    write_mesh(tmp_path / "m.ply", pkg.synth.samples_host(3), pkg.synth.grid_faces(3, 3))
    r = subprocess.run([_cli(), "-t", "tangent.png", "-T", "tangents.ply", str(tmp_path / "c.ply"),
                        str(tmp_path / "m.ply")], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and "no CUDA device" in r.stderr
    assert not (tmp_path / "tangent.png").exists() and not (tmp_path / "tangents.ply").exists()


# ---- GPU ------------------------------------------------------------------------------------------
def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def check_bake_ex(pkg, pto, P, V, F, k, res, pad=True, radius=None, coord_mode=0):
    with pkg.Tree(P, coord_mode=coord_mode) as tree:
        got = tree.bake(V, F, k=k, resolution=res, radius=radius, pad=pad, want=ALL_OUTPUTS)
    ref = pto_bake.bake_tangent(P, V, F, k, res, radius=-1.0 if radius is None else radius, pad=pad)
    assert (got["stats"]["texels"], got["stats"]["empty"]) == (ref["texels"], ref["empty"])
    for key in ALL_OUTPUTS:
        assert_same(got[key], ref[key], key)
    return got, ref


def tilted_normals(rng, n):
    return np.c_[rng.normal(0, 0.3, (n, 2)), np.ones(n)] * rng.uniform(0.5, 3.0, (n, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("k,res,pad", [(20, 512, 1), (8, 257, 0), (32, 128, 1), (1, 257, 1), (20, 512, 0)])
def test_gpu_bake_ex_equals_oracle(k, res, pad, pkg, pto):
    _need_gpu()
    side = 30.0
    P = pkg.synth.cloud_host(90_000, seed=41 + k, side=side)
    V, F = grid_mesh(pkg, 20, side)
    V["normal"] = tilted_normals(np.random.default_rng(k), len(V))
    got, _ = check_bake_ex(pkg, pto, P, V, F, k, res, pad=bool(pad))
    assert got["stats"]["texels"] > res * res // 2 and got["tangent_bgra"][..., 3].any()


@pytest.mark.gpu
def test_gpu_bake_ex_awkward_meshes(pkg, pto):
    _need_gpu()
    rng = np.random.default_rng(6)
    for seed, variant in ((5, "nan"), (6, "mirrored"), (7, "zero"), (8, "coincident")):
        V, F = variant_mesh(pto, seed, variant)
        lo, hi = V["ver"].min(0), V["ver"].max(0)
        P = pkg.make_points(lo + rng.random((30_000, 3)) * (hi - lo), normal=rng.standard_normal((30_000, 3)),
                            color=rng.integers(0, 256, (30_000, 3)))
        for res in (96, 200):
            check_bake_ex(pkg, pto, P, V, F, 12, res)


@pytest.mark.gpu
def test_gpu_bake_ex_fp64_lattice_empty_nan(pkg, pto):
    _need_gpu()
    P, V, F, res = lattice_case(pto, res=300)
    V = V.copy()
    V["normal"] = tilted_normals(np.random.default_rng(3), len(V))
    check_bake_ex(pkg, pto, P, V, F, 20, res)
    rng = np.random.default_rng(8)
    P64 = pkg.make_points(P["ver"] + 1e-9 * rng.random(P["ver"].shape), normal=P["normal"], color=P["color"])
    check_bake_ex(pkg, pto, P64, V, F, 20, res, coord_mode=pkg.COORD_F64)
    got, _ = check_bake_ex(pkg, pto, P, V, F, 8, 200, pad=False, radius=0.2)
    assert got["stats"]["empty"] > 0
    V["ver"][3] = np.nan
    got, _ = check_bake_ex(pkg, pto, P, V, F, 8, 200, pad=False)
    assert got["stats"]["empty"] > 0


@pytest.mark.gpu
def test_gpu_bake_ex_object_maps_equal_bake(pkg, pto):
    _need_gpu()
    side = 30.0
    P = pkg.synth.cloud_host(60_000, seed=5, side=side)
    V, F = grid_mesh(pkg, 16, side)
    V["normal"] = tilted_normals(np.random.default_rng(2), len(V))
    res = 300
    L, ptr = pkg.lib(), pkg.api._np_ptr
    with pkg.Tree(P) as tree:
        ex = tree.bake(V, F, k=16, resolution=res, want=ALL_OUTPUTS)
        maps = [np.empty((res, res, 4), np.uint8), np.empty((res, res, 4), np.uint8),
                np.empty((res, res, 3), np.float32)]
        st = pkg.api.BakeStats()
        assert L.pt_texture_bake(tree.handle, ptr(V), len(V), ptr(F), len(F), 16, -1.0, res, 1, ptr(maps[0]),
                                 ptr(maps[1]), ptr(maps[2]), ctypes.byref(st)) == 0
    assert ex["bgra"].tobytes() == maps[0].tobytes()
    assert ex["normal_bgra"].tobytes() == maps[1].tobytes()
    assert ex["normal"].tobytes() == maps[2].tobytes()
    assert (ex["stats"]["texels"], ex["stats"]["empty"]) == (st.texels, st.empty)


@pytest.mark.gpu
def test_gpu_bake_ex_tangent_outputs_alone(pkg, pto):
    """Tangent maps without the object-space ones, and tangents without any map."""
    _need_gpu()
    P, V, F, res = lattice_case(pto, res=128)
    V = V.copy()
    V["normal"] = tilted_normals(np.random.default_rng(4), len(V))
    ref = pto_bake.bake_tangent(P, V, F, 8, res, radius=0.3)
    with pkg.Tree(P) as tree:
        got = tree.bake(V, F, k=8, resolution=res, radius=0.3, want=("tangent_bgra", "tangent_normal"))
        only = tree.bake(V, F, k=8, resolution=res, want=("tangents",))
    assert set(got) == {"tangent_bgra", "tangent_normal", "stats"}
    assert_same(got["tangent_bgra"], ref["tangent_bgra"], "tangent_bgra")
    assert_same(got["tangent_normal"], ref["tangent_normal"], "tangent_normal")
    assert (got["stats"]["texels"], got["stats"]["empty"]) == (ref["texels"], ref["empty"]) and ref["empty"] > 0
    assert_same(only["tangents"], ref["tangents"], "tangents")
    assert only["stats"]["texels"] == 0


@pytest.mark.gpu
def test_gpu_bake_tangent_device_pieces(pkg, pto):
    _need_gpu()
    import torch
    side, k, res = 30.0, 16, 256
    P = pkg.synth.cloud_host(60_000, seed=9, side=side)
    V, F = grid_mesh(pkg, 12, side)
    V["normal"] = tilted_normals(np.random.default_rng(9), len(V))
    xyzuv = torch.from_numpy(np.c_[V["ver"], V["U"], V["V"]]).cuda()
    xyzuvn = torch.from_numpy(np.c_[V["ver"], V["U"], V["V"], V["normal"]]).cuda()
    faces = torch.from_numpy(F).cuda()
    texels, xyz, owner = pkg.bake_samples_device(xyzuv, faces, res)
    texels0, xyz0 = pkg.bake_texels_device(xyzuv, faces, res)
    assert torch.equal(texels, texels0) and torch.equal(xyz.view(torch.int64), xyz0.view(torch.int64))
    ref_t, ref_xyz, ref_owner = pto_bake.bake_samples(V, F, res)
    assert np.array_equal(texels.cpu().numpy().astype(np.uint32), ref_t)
    assert np.array_equal(owner.cpu().numpy(), ref_owner)
    frames, tangents = pkg.bake_frames_device(xyzuvn, faces)
    ref_frames, ref_tangents = pto_bake.bake_frames(V, F)
    assert_same(frames.cpu().numpy(), ref_frames, "frames")
    assert_same(tangents.cpu().numpy(), ref_tangents, "tangents")
    pos = torch.from_numpy(np.c_[P["ver"], np.zeros(len(P))].astype(np.float32)).cuda()
    attrs = np.zeros(len(P), pkg.ATTR_DTYPE)
    attrs["nx"], attrs["ny"], attrs["nz"] = P["normal"].astype(np.float32).T
    attrs["rgba"][:, :3], attrs["rgba"][:, 3] = P["color"], 255
    dtree = pkg.DeviceTree(pos, torch.from_numpy(attrs.view(np.uint8).reshape(-1, 16)).cuda())
    m = texels.numel()
    rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
    nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
    dtree.query(xyz.contiguous(), k, rgba=rgba, normal=nrm)
    tb = torch.empty((res, res, 4), dtype=torch.uint8, device="cuda")
    tn = torch.empty((res, res, 3), dtype=torch.float32, device="cuda")
    pkg.bake_compose_tangent_device(xyzuvn, frames, faces, texels, owner, rgba, nrm, res, pad=True,
                                    tangent_bgra=tb, tangent_normal=tn)
    torch.cuda.synchronize()
    dtree.close()
    with pkg.Tree(P) as tree:
        got = tree.bake(V, F, k=k, resolution=res, want=ALL_OUTPUTS)
    assert np.array_equal(tb.cpu().numpy(), got["tangent_bgra"])
    assert_same(tn.cpu().numpy(), got["tangent_normal"], "tangent_normal")
    assert_same(tangents.cpu().numpy(), got["tangents"], "tangents")


@pytest.mark.gpu
def test_gpu_quarter_turn_invariance(pkg, pto):
    _need_gpu()
    P, V, F = turn_case(pto, n_points=40_000, g=17)
    with pkg.Tree(P) as t0, pkg.Tree(turn(P)) as t1:
        a = t0.bake(V, F, k=12, resolution=512, want=ALL_OUTPUTS)
        b = t1.bake(turn(V), F, k=12, resolution=512, want=ALL_OUTPUTS)
    for key in ("tangent_bgra", "tangent_normal"):
        assert_same(a[key], b[key], key)
    assert np.array_equal(turn_tangents(a["tangents"]), b["tangents"])
    assert not np.array_equal(a["normal_bgra"], b["normal_bgra"])
    assert a["stats"]["texels"] > 512 * 512 // 2


@pytest.mark.gpu
def test_gpu_bake_ex_error_codes(pkg):
    _need_gpu()
    P = pkg.synth.cloud_host(2_000, seed=1, side=10.0)
    V, F = grid_mesh(pkg, 4, 10.0)
    L, ptr = pkg.lib(), pkg.api._np_ptr
    api = pkg.api
    img = np.empty(64 * 64 * 4, np.uint8)
    tg = np.empty((len(V), 4), np.float32)
    with pkg.Tree(P) as tree:
        def call(o, n_faces=len(F), res=64, faces=F):
            return L.pt_texture_bake_ex(tree.handle, ptr(V), len(V), ptr(faces), n_faces, 8, -1.0, res, 1,
                                        ctypes.byref(o), None)
        none = api.BakeOutputs()
        assert call(none) == 1
        assert L.pt_texture_bake_ex(tree.handle, ptr(V), len(V), ptr(F), len(F), 8, -1.0, 64, 1, None, None) == 1
        # 3 * n_faces above INT32_MAX: refused before the (far too short) face array is read
        tangent_map = api.BakeOutputs(tangent_bgra=img.ctypes.data)
        assert call(tangent_map, n_faces=(2**31 - 1) // 3 + 1) == api.PT_ERR_UNSUPPORTED
        assert call(api.BakeOutputs(vertex_tangents=tg.ctypes.data), n_faces=(2**31 - 1) // 3 + 1) == \
            api.PT_ERR_UNSUPPORTED
        for res in (0, 16385):
            assert call(tangent_map, res=res) == 1
        for kw, status in (({"resolution": 0}, 1), ({"resolution": 16385}, 1), ({"k": 33}, api.PT_ERR_UNSUPPORTED)):
            with pytest.raises(pkg.PointsTransferError) as e:
                tree.bake(V, F, **{"k": 8, "resolution": 64, "want": ("tangent_bgra",), **kw})
            assert e.value.status == status, kw
        with pytest.raises(ValueError):
            tree.bake(V, F, k=8, resolution=64, want=("bitangents",))
        assert call(tangent_map) == 0
    with pkg.Tree(P, ids=np.arange(len(P), dtype=np.int32)) as slab:
        with pytest.raises(pkg.PointsTransferError) as e:
            slab.bake(V, F, k=8, resolution=64, want=("tangent_normal", "tangents"))
        assert e.value.status == api.PT_ERR_UNSUPPORTED
    assert L.pt_bake_frames_device(None, 0, ptr(F), (2**31 - 1) // 3 + 1, None, None, 0, None) == api.PT_ERR_UNSUPPORTED


def read_tangent_ply(path):
    lines = open(path).read().splitlines()
    end = lines.index("end_header")
    assert "property float tw" in lines[:end]
    n = int(next(ln.split()[2] for ln in lines if ln.startswith("element vertex")))
    rows = [ln.split() for ln in lines[end + 1:end + 1 + n]]
    assert all(len(r) == 15 for r in rows)
    return np.array([[float(x) for x in r[:8]] for r in rows]), np.array([[float(x) for x in r[11:]] for r in rows],
                                                                          np.float32)


@pytest.mark.gpu
def test_gpu_cli_tangent_bake(pkg, pto, tmp_path):
    _need_gpu()
    cli = _cli()
    side = 20.0
    P = pkg.synth.cloud_host(20_000, 3, side=side)
    V, F = grid_mesh(pkg, 12, side)
    write_cloud(tmp_path / "c.ply", P)
    write_mesh(tmp_path / "m.ply", V, F)
    args = [str(tmp_path / "c.ply"), str(tmp_path / "m.ply")]
    r = subprocess.run([cli, "-R", "256", "-b", "bake.png", "-n", "normal.png", "-t", "tangent.png", "-T",
                        "tangents.ply", "-o", "tex_t.png", *args], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    assert "Bake total time:" in r.stdout
    Vm = V.copy()
    Vm["normal"] = [0, 0, 1]
    Vm["color"] = np.array([10, 20, 30])                  # what write_mesh put in the file
    ref = pto_bake.bake_tangent(P, Vm, F, 20, 256)
    assert np.array_equal(read_png_bgra(tmp_path / "tangent.png"), ref["tangent_bgra"])
    rows, tangents = read_tangent_ply(tmp_path / "tangents.ply")
    assert np.array_equal(tangents, ref["tangents"])
    assert np.array_equal(rows[:, :3], Vm["ver"]) and np.array_equal(rows[:, 6], Vm["U"])
    assert np.array_equal(read_png_bgra(tmp_path / "bake.png"), ref["bgra"])
    assert np.array_equal(read_png_bgra(tmp_path / "normal.png"), ref["normal_bgra"])
    # the other outputs are those of a run without -t / -T
    r = subprocess.run([cli, "-R", "256", "-b", "bake0.png", "-n", "normal0.png", "-o", "tex0.png", *args],
                       capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    for a, b in (("bake.png", "bake0.png"), ("normal.png", "normal0.png"), ("tex_t.png", "tex0.png")):
        assert (tmp_path / a).read_bytes() == (tmp_path / b).read_bytes(), a
