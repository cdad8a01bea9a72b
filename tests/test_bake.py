"""Per-texel bake (DESIGN.md section 8, "Per-texel bake"): colour and normal maps of the cloud on a
mesh's UV atlas.

CPU part: the oracle's texel stage (oracle/pt_bake_oracle.c via oracle/pto_bake.py) against an independent numpy
statement of the frozen definition, a known answer on a lattice cloud, the normal-map encoding and
the CLI's refusals.  GPU part: pt_texture_bake, the device pieces and the CLI must equal the
oracle bit for bit."""
import subprocess

import numpy as np
import pytest

from oracle import pto_bake
from test_cli import read_png_bgra, write_cloud, write_mesh


# ---- the frozen definition restated in numpy ---------------------------------------------------
def _area2(pa, pb, qa, qb, ra, rb):
    return np.subtract(np.multiply(np.subtract(qa, pa), np.subtract(rb, pb)),
                       np.multiply(np.subtract(qb, pb), np.subtract(ra, pa)))


def numpy_texels(V, F, res):
    """Owner face per texel by brute force over the whole image, highest face index wins."""
    row, col = np.divmod(np.arange(res * res), res)
    xa = col + 0.5
    xb = (res - row) - 0.5
    owner = np.full(res * res, -1, np.int64)
    uv = np.stack([V["U"] * res, V["V"] * res], 1)
    with np.errstate(all="ignore"):
        for f, tri in enumerate(F):
            if (tri < 0).any() or (tri >= len(V)).any():
                continue
            (pa, pb), (qa, qb), (ra, rb) = uv[tri[0]], uv[tri[1]], uv[tri[2]]
            inv = np.divide(1.0, _area2(pa, pb, qa, qb, ra, rb))
            b0 = np.multiply(_area2(qa, qb, ra, rb, xa, xb), inv)
            b1 = np.multiply(_area2(ra, rb, pa, pb, xa, xb), inv)
            b2 = np.subtract(np.subtract(1.0, b0), b1)
            owner[(b0 >= 0) & (b1 >= 0) & (b2 >= 0)] = f
    texels = np.flatnonzero(owner >= 0)
    xyz = np.empty((len(texels), 3))
    with np.errstate(all="ignore"):
        for i, t in enumerate(texels):
            tri = F[owner[t]]
            (pa, pb), (qa, qb), (ra, rb) = uv[tri[0]], uv[tri[1]], uv[tri[2]]
            inv = np.divide(1.0, _area2(pa, pb, qa, qb, ra, rb))
            b0 = np.multiply(_area2(qa, qb, ra, rb, xa[t], xb[t]), inv)
            b1 = np.multiply(_area2(ra, rb, pa, pb, xa[t], xb[t]), inv)
            b2 = np.subtract(np.subtract(1.0, b0), b1)
            X = V["ver"][tri]
            xyz[i] = np.add(np.add(np.multiply(b0, X[0]), np.multiply(b1, X[1])), np.multiply(b2, X[2]))
    return texels.astype(np.uint32), xyz


def awkward_mesh(pto, seed):
    """Shared edges (a grid chart), a second chart overlapping the first in UV space, a zero-area
    UV face, UVs partly outside [0, 1] and a face with an out-of-range vertex index."""
    rng = np.random.default_rng(seed)
    g = 5
    t = np.linspace(0.0, 1.0, g)
    u, v = [a.ravel() for a in np.meshgrid(t, t)]
    uv1 = np.c_[u * 0.7 - 0.1, v * 0.8 + 0.05] + rng.normal(0, 0.01, (g * g, 2))
    uv2 = np.c_[u * 0.5 + 0.35, v * 0.6 + 0.3]                       # overlaps chart 1 and leaves [0, 1]
    xyz = np.r_[np.c_[u, v, rng.random(g * g)], np.c_[u + 2.0, v, rng.random(g * g)]] * 10.0
    j, i = np.meshgrid(np.arange(g - 1), np.arange(g - 1), indexing="ij")
    a = (j * g + i).ravel()
    grid = np.stack([np.stack([a, a + 1, a + g], 1), np.stack([a + 1, a + g + 1, a + g], 1)], 1).reshape(-1, 3)
    F = np.r_[grid, grid + g * g, [[0, 1, 1]], [[3, 7, 2 * g * g + 5]], [[0, 6, 12]]].astype(np.int32)
    rng.shuffle(F[: len(F) - 3])
    V = pto.make_points(xyz, uv=np.r_[uv1, uv2 * 1.3 - 0.1])
    return V, F


@pytest.mark.parametrize("seed,res", [(1, 40), (2, 57), (3, 64)])
def test_oracle_texels_equal_numpy_definition(pto, seed, res):
    V, F = awkward_mesh(pto, seed)
    texels, xyz = pto_bake.bake_texels(V, F, res)
    ref_t, ref_xyz = numpy_texels(V, F, res)
    assert len(texels) > res * res // 4
    assert np.array_equal(texels, ref_t)
    assert np.array_equal(xyz.view(np.uint64), ref_xyz.view(np.uint64))


def test_oracle_overlap_highest_face_wins(pto):
    # two faces with the same UV triangle but different 3-D corners: the later one owns every texel
    V = pto.make_points([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 5], [1, 0, 5], [0, 1, 5.0]],
                        uv=[[0.1, 0.1], [0.9, 0.1], [0.1, 0.9]] * 2)
    texels, xyz = pto_bake.bake_texels(V, np.array([[0, 1, 2], [3, 4, 5]]), 32)
    assert len(texels) > 0 and np.allclose(xyz[:, 2], 5.0)
    texels2, xyz2 = pto_bake.bake_texels(V, np.array([[3, 4, 5], [0, 1, 2]]), 32)
    assert np.array_equal(texels, texels2) and np.allclose(xyz2[:, 2], 0.0)


def lattice_case(pto, res=64):
    """Lattice cloud on z = 0 with per-point colours and normal (0, 0, 1), one quad of 2 triangles."""
    rng = np.random.default_rng(4)
    gx, gy = np.meshgrid(np.arange(21) * 0.5, np.arange(21) * 0.5)
    xyz = np.c_[gx.ravel(), gy.ravel(), np.zeros(gx.size)]
    P = pto.make_points(xyz, normal=np.tile([0, 0, 1.0], (len(xyz), 1)), color=rng.integers(0, 256, (len(xyz), 3)))
    Vx = np.array([[0.3, 0.2, 0], [9.7, 0.2, 0], [9.7, 9.9, 0], [0.3, 9.9, 0.0]])
    V = pto.make_points(Vx, uv=[[0.05, 0.1], [0.9, 0.1], [0.9, 0.95], [0.05, 0.95]])
    F = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    return P, V, F, res


def test_known_answer_lattice_k1(pto):
    P, V, F, res = lattice_case(pto)
    bgra, nbgra, nf, (n_texels, empty) = pto_bake.bake(P, V, F, 1, res, pad=False)
    ref_t, ref_xyz = numpy_texels(V, F, res)
    assert n_texels == len(ref_t) > 0 and empty == 0
    # nearest lattice point per texel, lowest index on ties
    d = ref_xyz[:, None, :] - P["ver"][None, :, :]
    d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    nearest = np.argmin(d2, axis=1)                           # first minimum = lowest index
    # the frozen blend with one neighbour: trunc((w * c) / w), w = 1 / d2 (w = 1 on an exact hit),
    # which is the neighbour's colour or, after rounding, one below it
    dn = d2[np.arange(len(nearest)), nearest]
    w = np.where(dn == 0.0, 1.0, np.divide(1.0, dn))
    colour = P["color"][nearest]
    expect = np.trunc(np.divide(np.multiply(w[:, None], colour), w[:, None])).astype(np.int64)
    assert set(np.unique(colour - expect).tolist()) <= {0, 1}
    flat = bgra.reshape(-1, 4)
    assert np.array_equal(flat[ref_t, :3], expect[:, ::-1])
    assert (flat[ref_t, 3] == 255).all()
    covered = np.zeros(res * res, bool)
    covered[ref_t] = True
    assert not flat[~covered].any() and not nbgra.reshape(-1, 4)[~covered].any()
    assert (nbgra.reshape(-1, 4)[covered] == [255, 128, 128, 255]).all()
    assert (nf.reshape(-1, 3)[covered] == [0, 0, 1]).all()


def test_normal_encoding(pto):
    assert [pto_bake.bake_encode(x) for x in (-1.0, 0.0, 1.0)] == [0, 128, 255]
    assert pto_bake.bake_encode(-2.0) == 0 and pto_bake.bake_encode(2.0) == 255


def test_oracle_empty_lists_are_zero(pto):
    """A radius-bounded search and NaN sample positions (a vertex with NaN coordinates) leave
    covered texels at 0 in all three maps, and count as empty."""
    P, V, F, res = lattice_case(pto, res=48)
    V = V.copy()
    bgra, nbgra, nf, (n, empty) = pto_bake.bake(P, V, F, 4, res, radius=0.2, pad=False)
    assert 0 < empty < n
    V["ver"][3] = np.nan                                     # every texel of face 1 has a NaN position
    texels, xyz = pto_bake.bake_texels(V, F, res)
    nan_rows = np.isnan(xyz).any(1)
    assert nan_rows.any() and not nan_rows.all()
    bgra, nbgra, nf, (n, empty) = pto_bake.bake(P, V, F, 4, res, pad=False)
    assert empty == nan_rows.sum()
    for img, w in ((bgra, 4), (nbgra, 4), (nf, 3)):
        assert not img.reshape(-1, w)[texels[nan_rows]].any()
        assert img.reshape(-1, w)[texels[~nan_rows]].any()


def test_cli_refuses_multi_gpu_bake(tmp_path):
    from test_cli import CLI
    if not __import__("os").path.exists(CLI):
        subprocess.run(["make", "-C", __import__("os").path.dirname(CLI)], check=True, stdout=subprocess.DEVNULL)
    r = subprocess.run([CLI, "-g", "2", "-b", "x.png", "a.ply", "b.ply"], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and "-b / -n" in r.stderr and not (tmp_path / "x.png").exists()


def test_cli_bake_without_gpu(pkg, tmp_path):
    from test_cli import CLI
    if pkg.device_count() > 0:
        pytest.skip("a GPU is present")
    P = pkg.synth.cloud_host(50, 1)
    write_cloud(tmp_path / "c.ply", P)
    write_mesh(tmp_path / "m.ply", pkg.synth.samples_host(3), pkg.synth.grid_faces(3, 3))
    r = subprocess.run([CLI, "-b", "bake.png", "-n", "normal.png", str(tmp_path / "c.ply"), str(tmp_path / "m.ply")],
                       capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and "no CUDA device" in r.stderr
    assert not (tmp_path / "bake.png").exists() and not (tmp_path / "normal.png").exists()


# ---- GPU ------------------------------------------------------------------------------------------
def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def grid_mesh(pkg, g, side):
    V = pkg.synth.samples_host(g, side=side)
    V["U"] = V["ver"][:, 0] / side * 0.9 + 0.05
    V["V"] = V["ver"][:, 1] / side * 0.9 + 0.05
    return V, pkg.synth.grid_faces(g, g)


def check_bake(pkg, pto, P, V, F, k, res, pad=True, radius=None, coord_mode=0):
    with pkg.Tree(P, coord_mode=coord_mode) as tree:
        got = tree.bake(V, F, k=k, resolution=res, radius=radius, pad=pad)
    bgra, nbgra, nf, (n, empty) = pto_bake.bake(P, V, F, k, res, radius=-1.0 if radius is None else radius, pad=pad)
    st = got["stats"]
    assert (st["texels"], st["empty"]) == (n, empty)
    assert np.array_equal(got["bgra"], bgra)
    assert np.array_equal(got["normal_bgra"], nbgra)
    assert np.array_equal(got["normal"].view(np.uint32), nf.view(np.uint32))
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("k,res,pad", [(20, 512, 1), (8, 257, 0), (32, 300, 1), (1, 128, 1)])
def test_gpu_bake_equals_oracle(k, res, pad, pkg, pto):
    _need_gpu()
    side = 30.0
    P = pkg.synth.cloud_host(90_000, seed=21 + k, side=side)
    V, F = grid_mesh(pkg, 20, side)
    got = check_bake(pkg, pto, P, V, F, k, res, pad=bool(pad))
    assert got["stats"]["texels"] > res * res // 2 and got["stats"]["empty"] == 0


@pytest.mark.gpu
def test_gpu_bake_overlapping_charts(pkg, pto):
    _need_gpu()
    V, F = awkward_mesh(pto, 5)
    rng = np.random.default_rng(6)
    lo, hi = V["ver"].min(0), V["ver"].max(0)
    P = pkg.make_points(lo + rng.random((30_000, 3)) * (hi - lo), normal=rng.standard_normal((30_000, 3)),
                        color=rng.integers(0, 256, (30_000, 3)))
    for res in (96, 200):
        check_bake(pkg, pto, P, V, F, 12, res)


@pytest.mark.gpu
def test_gpu_bake_fp64_and_lattice(pkg, pto):
    _need_gpu()
    P, V, F, res = lattice_case(pto, res=300)
    check_bake(pkg, pto, P, V, F, 20, res)
    check_bake(pkg, pto, P, V, F, 1, res)
    rng = np.random.default_rng(8)
    P64 = pkg.make_points(P["ver"] + 1e-9 * rng.random(P["ver"].shape), normal=P["normal"], color=P["color"])
    check_bake(pkg, pto, P64, V, F, 20, res, coord_mode=pkg.COORD_F64)


@pytest.mark.gpu
def test_gpu_bake_empty_lists(pkg, pto):
    _need_gpu()
    P, V, F, res = lattice_case(pto, res=200)
    got = check_bake(pkg, pto, P, V, F, 8, res, pad=False, radius=0.2)
    assert got["stats"]["empty"] > 0
    V = V.copy()
    V["ver"][3] = np.nan
    got = check_bake(pkg, pto, P, V, F, 8, res, pad=False)
    assert got["stats"]["empty"] > 0


@pytest.mark.gpu
def test_gpu_bake_device_pieces(pkg, pto):
    _need_gpu()
    import torch
    side, k, res = 30.0, 16, 256
    P = pkg.synth.cloud_host(60_000, seed=9, side=side)
    V, F = grid_mesh(pkg, 12, side)
    xyzuv = torch.from_numpy(np.c_[V["ver"], V["U"], V["V"]]).cuda()
    texels, xyz = pkg.bake_texels_device(xyzuv, torch.from_numpy(F).cuda(), res)
    ref_t, ref_xyz = pto_bake.bake_texels(V, F, res)
    assert np.array_equal(texels.cpu().numpy().astype(np.uint32), ref_t)
    assert np.array_equal(xyz.cpu().numpy().view(np.uint64), ref_xyz.view(np.uint64))
    pos = torch.from_numpy(np.c_[P["ver"], np.zeros(len(P))].astype(np.float32)).cuda()
    attrs = np.zeros(len(P), pkg.ATTR_DTYPE)
    attrs["nx"], attrs["ny"], attrs["nz"] = P["normal"].astype(np.float32).T
    attrs["rgba"][:, :3], attrs["rgba"][:, 3] = P["color"], 255
    dtree = pkg.DeviceTree(pos, torch.from_numpy(attrs.view(np.uint8).reshape(-1, 16)).cuda())
    m = texels.numel()
    rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
    nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
    dtree.query(xyz.contiguous(), k, rgba=rgba, normal=nrm)
    maps = [torch.empty((res, res, 4), dtype=torch.uint8, device="cuda"),
            torch.empty((res, res, 4), dtype=torch.uint8, device="cuda"),
            torch.empty((res, res, 3), dtype=torch.float32, device="cuda")]
    pkg.bake_compose_device(texels, rgba, nrm, res, pad=True, bgra=maps[0], normal_bgra=maps[1], normal_out=maps[2])
    torch.cuda.synchronize()
    dtree.close()
    with pkg.Tree(P) as tree:
        got = tree.bake(V, F, k=k, resolution=res)
    assert np.array_equal(maps[0].cpu().numpy(), got["bgra"])
    assert np.array_equal(maps[1].cpu().numpy(), got["normal_bgra"])
    assert np.array_equal(maps[2].cpu().numpy().view(np.uint32), got["normal"].view(np.uint32))


@pytest.mark.gpu
def test_gpu_bake_full_atlas_quad(pkg, pto):
    """Two faces covering a 2048^2 atlas: the work is split over many warps per face."""
    _need_gpu()
    rng = np.random.default_rng(10)
    P = pkg.make_points(np.c_[rng.random((20_000, 2)) * 10.0, rng.normal(0, 0.01, 20_000)],
                        normal=rng.standard_normal((20_000, 3)), color=rng.integers(0, 256, (20_000, 3)))
    V = pkg.make_points([[0, 0, 0], [10, 0, 0], [10, 10, 0], [0, 10, 0.0]],
                        uv=[[0, 0], [1, 0], [1, 1], [0, 1.0]])
    F = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    got = check_bake(pkg, pto, P, V, F, 1, 2048)
    assert got["stats"]["texels"] == 2048 * 2048


@pytest.mark.gpu
def test_gpu_bake_error_codes(pkg):
    _need_gpu()
    P = pkg.synth.cloud_host(2_000, seed=1, side=10.0)
    V, F = grid_mesh(pkg, 4, 10.0)
    with pkg.Tree(P) as tree:
        for kw, status in (({"k": 0}, pkg.api.PT_ERR_UNSUPPORTED), ({"k": 33}, pkg.api.PT_ERR_UNSUPPORTED),
                           ({"resolution": 0}, 1), ({"resolution": 16385}, 1)):
            with pytest.raises(pkg.PointsTransferError) as e:
                tree.bake(V, F, **{"k": 8, "resolution": 64, **kw})
            assert e.value.status == status, kw
        L, vp = pkg.lib(), None
        assert L.pt_texture_bake(tree.handle, None, 5, None, 0, 8, -1.0, 64, 1, None, None, None, None) == 1
        out = np.empty(64 * 64 * 4, np.uint8)
        assert L.pt_texture_bake(tree.handle, pkg.api._np_ptr(V), len(V), None, 3, 8, -1.0, 64, 1,
                                 pkg.api._np_ptr(out), vp, vp, None) == 1
        assert L.pt_texture_bake(tree.handle, pkg.api._np_ptr(V), len(V), pkg.api._np_ptr(F), len(F), 8, -1.0,
                                 64, 1, vp, vp, vp, None) == 1
        assert L.pt_texture_bake(tree.handle, pkg.api._np_ptr(V), len(V), pkg.api._np_ptr(F), 1 << 31, 8, -1.0,
                                 64, 1, pkg.api._np_ptr(out), vp, vp, None) == 1
    with pkg.Tree(P, ids=np.arange(len(P), dtype=np.int32)) as slab:
        with pytest.raises(pkg.PointsTransferError) as e:
            slab.bake(V, F, k=8, resolution=64)
        assert e.value.status == pkg.api.PT_ERR_UNSUPPORTED


@pytest.mark.gpu
def test_gpu_cli_bake(pkg, pto, tmp_path):
    _need_gpu()
    from test_cli import CLI
    side = 20.0
    P = pkg.synth.cloud_host(20_000, 3, side=side)
    V, F = grid_mesh(pkg, 12, side)
    write_cloud(tmp_path / "c.ply", P)
    write_mesh(tmp_path / "m.ply", V, F)
    r = subprocess.run([CLI, "-R", "256", "-b", "bake.png", "-n", "normal.png", str(tmp_path / "c.ply"),
                        str(tmp_path / "m.ply")], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    assert "Bake total time:" in r.stdout and "Output time:" in r.stdout
    Vm = V.copy()
    Vm["normal"] = [0, 0, 1]
    Vm["color"] = np.array([10, 20, 30])                  # what write_mesh put in the file
    bgra, nbgra, _, _ = pto_bake.bake(P, Vm, F, 20, 256)
    assert np.array_equal(read_png_bgra(tmp_path / "bake.png"), bgra)
    assert np.array_equal(read_png_bgra(tmp_path / "normal.png"), nbgra)
    idx, _ = pto.knn_bruteforce(P, Vm, 20)
    ref_img, _ = pto.texture(P, Vm, idx, F, 256, pad=True)
    assert np.array_equal(read_png_bgra(tmp_path / "texture.png"), ref_img)
