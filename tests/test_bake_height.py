"""Height bake (DESIGN.md section 8, "Height bake"): the cloud's signed height above the mesh along the
interpolated mesh normal, as a float map and a padded 16-bit code map.

CPU part: the oracle (tests/bake_height_oracle.c via tests/bake_height_oracle.py) against an
independent numpy statement of the frozen definition, the 16-bit padding against a direct 25 x 25
window, known answers on a flat quad, the exact symmetries, and the CLI's refusals.  GPU part:
pt_texture_bake_height, the device piece and the CLI must equal the oracle bit for bit; the other
outputs equal pt_texture_bake_ex's; a noisy heightfield is recovered within a stated bound."""
import ctypes
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

import bake_height_oracle as hgo
import bake_tangent_oracle as tgo
from test_bake import awkward_mesh, grid_mesh, lattice_case
from test_bake_tangent import (ALL_OUTPUTS, _bary, _dot, _normalise, _scale, _usable, tilted_normals, turn,
                               turn_case, variant_mesh)
from test_cli import write_cloud, write_mesh

NAN_BITS = 0x7FC00000
HEIGHTS = ("height", "height_u16")


# ---- the frozen definition restated in numpy (elementwise ufuncs: every operation rounded) -------
def numpy_height(V, frames, F, texels, owner, xyz, P, idx, d2, res):
    """Steps 1-4: float32 [res,res], NaN (0x7fc00000) without a value."""
    out = np.full(res * res, np.uint32(NAN_BITS)).view(np.float32)
    tri = F[owner]
    uv = np.stack([V["U"] * res, V["V"] * res], 1)
    row, col = np.divmod(texels.astype(np.int64), res)
    with np.errstate(all="ignore"):
        bc = _bary([uv[tri[:, j]].T for j in range(3)], col + 0.5, (res - row) - 0.5)
        a, b, c = (frames[tri[:, j], 0:3] for j in range(3))
        n = np.add(np.add(_scale(bc[:, 0], a), _scale(bc[:, 1], b)), _scale(bc[:, 2], c))
        ok = _usable(n)
        N = _normalise(np.where(ok[:, None], n, 1.0))
        m, k = idx.shape
        valid = (idx >= 0) & (idx < len(P))
        cnt = np.where(valid.all(1), k, np.argmin(valid, 1))
        p = P["ver"][np.where(valid, idx, 0)]                               # [m,k,3]
        o = _dot(np.subtract(p, xyz[:, None, :]), N[:, None, :])           # [m,k]

        def sums(w):
            W, S = np.zeros(m), np.zeros(m)
            for j in range(k):
                use = j < cnt
                W = np.where(use, np.add(W, w[:, j]), W)
                S = np.where(use, np.add(S, np.multiply(w[:, j], o[:, j])), S)
            return W, S
        w01 = np.where((d2[:, :1] == 0), np.where(d2 == 0, 1.0, 0.0), np.divide(1.0, d2))
        W, S = sums(w01)
        redo = ~((W > 0) & (W < np.inf))
        W2, S2 = sums(np.broadcast_to(np.r_[1.0, np.zeros(k - 1)], (m, k)))
        W, S = np.where(redo, W2, W), np.where(redo, S2, S)
        h = np.divide(S, W).astype(np.float32)
    has = ok & (cnt > 0)
    h = np.where(np.isnan(h), np.uint32(NAN_BITS).view(np.float32), h)
    out[texels[has]] = h[has]
    return out.reshape(res, res)


def numpy_encode(h, height_range=None):
    """(codes uint16, (lo, hi), valued) without padding."""
    v = h[~np.isnan(h)]
    if height_range is not None and np.isfinite(height_range).all() and height_range[0] < height_range[1]:
        lo, hi = float(height_range[0]), float(height_range[1])
    elif v.size:
        lo, hi = float(v.min()), float(v.max())
        if lo == 0 and np.signbit(v[v == 0]).any():
            lo = -0.0
        if hi == 0 and (~np.signbit(v[v == 0])).any():
            hi = 0.0
    else:
        lo, hi = 0.0, 0.0
    with np.errstate(all="ignore"):
        if hi == lo:
            e = np.zeros(h.shape)
        else:
            s = 65535.0 / (hi - lo)
            e = np.clip(np.floor(np.add(np.multiply(np.subtract(h.astype(np.float64), lo), s), 0.5)), 0, 65535)
        codes = np.where(np.isnan(h), 0, e).astype(np.uint16)
    return codes, (lo, hi), int(v.size)


def direct_pad(h, codes):
    """A texel without a value takes the largest code of the valued texels in its 25 x 25 window."""
    res = h.shape[0]
    word = np.where(np.isnan(h), 0, codes.astype(np.int64) + 1)
    big = np.zeros((res + 24, res + 24), np.int64)
    big[12:12 + res, 12:12 + res] = word
    m = np.lib.stride_tricks.sliding_window_view(big, (25, 25)).max(axis=(-1, -2))
    return np.where(word > 0, word - 1, np.maximum(m - 1, 0)).astype(np.uint16)


def assert_heights(a, b, what="height"):
    assert a.shape == b.shape and a.dtype == b.dtype == np.float32, what
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), what


def cloud_around(pto, V, n, seed, exact_hits=None):
    rng = np.random.default_rng(seed)
    lo, hi = V["ver"].min(0), V["ver"].max(0)
    xyz = lo - 0.5 + rng.random((n, 3)) * (hi - lo + 1.0)
    if exact_hits is not None:                                   # cloud points at sample positions
        xyz = np.r_[xyz, exact_hits]
    return pto.make_points(xyz, normal=rng.standard_normal((len(xyz), 3)), color=rng.integers(0, 256, (len(xyz), 3)))


def oracle_vs_numpy(pto, P, V, F, k, res, radius=-1.0, frames=None, ranges=((-1.0, 2.0), None, (3.0, 3.0))):
    texels, xyz, owner = tgo.bake_samples(V, F, res)
    if frames is None:
        frames, _ = tgo.bake_frames(V, F)
    idx, d2 = hgo.neighbours(P, xyz, k, radius)
    h = hgo.bake_height(V, frames, F, texels, owner, xyz, P, idx, d2, res)
    assert_heights(h, numpy_height(V, frames, F, texels, owner, xyz, P, idx, d2, res))
    for rng_in in ranges:
        codes, used, valued = hgo.encode(h, rng_in)
        ref_codes, ref_used, ref_valued = numpy_encode(h, rng_in)
        assert np.array_equal(codes, ref_codes) and valued == ref_valued
        assert np.array_equal(np.array(used).view(np.uint64), np.array(ref_used).view(np.uint64))
        assert np.array_equal(hgo.pad(h, codes), direct_pad(h, codes))
    return h, (texels, owner, xyz), (idx, d2)


# ---- CPU ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ("zero", "random", "nan", "coincident"))
@pytest.mark.parametrize("seed,res,k", [(1, 40, 6), (2, 57, 1), (3, 64, 32)])
def test_oracle_equals_numpy_definition(pto, variant, seed, res, k):
    V, F = variant_mesh(pto, seed, variant)
    texels, xyz, _ = tgo.bake_samples(V, F, res)
    P = cloud_around(pto, V, 3000, seed, exact_hits=xyz[::7])
    h, _, (idx, d2) = oracle_vs_numpy(pto, P, V, F, k, res)
    assert (d2[:, 0] == 0).any() and np.isfinite(h).sum() > len(texels) // 2
    # radius-bounded lists: some are empty, those texels have no value
    h, (texels, _, _), (idx, _) = oracle_vs_numpy(pto, P, V, F, k, res, radius=0.3)
    empty = idx[:, 0] < 0
    assert empty.any() and np.isnan(h.reshape(-1)[texels[empty]]).all()


def test_oracle_unusable_normals_and_degenerate_frames(pto):
    V, F = awkward_mesh(pto, 4)
    frames, _ = tgo.bake_frames(V, F)
    frames = frames.copy()
    frames[::3, 0:3] = 0.0                                        # zero normals
    frames[1::5, 0:3] = np.nan                                    # NaN normals
    res = 48
    texels, xyz, _ = tgo.bake_samples(V, F, res)
    P = cloud_around(pto, V, 2000, 4)
    h, _, _ = oracle_vs_numpy(pto, P, V, F, 5, res, frames=frames)
    assert np.isnan(h.reshape(-1)[texels]).any() and np.isfinite(h).any()


def test_oracle_lattice_ties(pto):
    P, V, F, res = lattice_case(pto, res=64)
    V = V.copy()
    V["normal"] = tilted_normals(np.random.default_rng(3), len(V))
    oracle_vs_numpy(pto, P, V, F, 12, res)


def test_oracle_no_value_at_all(pto):
    P, V, F, res = lattice_case(pto, res=32)
    h, _, _ = oracle_vs_numpy(pto, P, V, F, 4, res, radius=1e-6)
    assert np.isnan(h).all()
    codes, used, valued = hgo.encode(h)
    assert used == (0.0, 0.0) and valued == 0 and not codes.any()
    assert not hgo.pad(h, codes).any()


def test_pad_equals_direct_window(pto):
    rng = np.random.default_rng(5)
    res = 90
    h = rng.normal(0, 3, (res, res)).astype(np.float32)
    h[rng.random((res, res)) < 0.7] = np.nan
    h[40:75, 10:60] = np.nan                                      # a hole wider than the window
    codes, _, _ = hgo.encode(h)
    padded = hgo.pad(h, codes)
    assert np.array_equal(padded, direct_pad(h, codes))
    assert (padded[~np.isnan(h)] == codes[~np.isnan(h)]).all() and (padded[55:60, 30:40] == 0).all()


def flat_quad(pto, z, normal=(0.0, 0.0, 1.0)):
    """Quad z = 0 with vertex normals `normal`, lattice cloud (spacing 0.25) at height z."""
    L = 4.0
    X = np.array([[0, 0, 0], [L, 0, 0], [L, L, 0], [0, L, 0.0]])
    V = pto.make_points(X, normal=np.tile(normal, (4, 1)), uv=np.c_[X[:, 0] / L, X[:, 1] / L])
    F = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    g = np.arange(-2, 19) * 0.25
    gx, gy = np.meshgrid(g, g)
    P = pto.make_points(np.c_[gx.ravel(), gy.ravel(), np.full(gx.size, z)], normal=np.tile([0, 0, 1.0], (gx.size, 1)))
    return P, V, F


@pytest.mark.parametrize("z", [0.25, -2.0])
def test_known_answers_flat_quad(pto, z):
    P, V, F = flat_quad(pto, z)
    res = 40
    out = hgo.bake(P, V, F, 6, res, pad_codes=False, height_range=(-2.0, 0.25))
    texels = out["samples"][0]
    h = out["height"].reshape(-1)
    assert out["texels"] == len(texels) > res * res // 2
    assert (h[texels] == np.float32(z)).all()
    uncovered = np.ones(res * res, bool)
    uncovered[texels] = False
    assert (h[uncovered].view(np.uint32) == NAN_BITS).all()
    assert (out["height_u16"].reshape(-1)[texels] == (65535 if z > 0 else 0)).all()
    assert not out["height_u16"].reshape(-1)[uncovered].any()
    auto = hgo.bake(P, V, F, 6, res)                              # automatic range (z, z): every code 0
    assert auto["height_range"] == (z, z) and not auto["height_u16"].any()


def test_quarter_turn_invariance(pto):
    P, V, F = turn_case(pto)
    a = hgo.bake(P, V, F, 8, 96)
    b = hgo.bake(turn(P), turn(V), F, 8, 96)
    assert_heights(a["height"], b["height"])
    assert np.array_equal(a["height_u16"], b["height_u16"]) and a["height_range"] == b["height_range"]
    assert a["texels"] > 96 * 96 // 2


def test_negated_normals_negate_heights(pto):
    P, V, F = turn_case(pto)
    Vn = V.copy()
    Vn["normal"] = -V["normal"]
    assert _usable(V["normal"].astype(np.float64)).all()
    a, b = hgo.bake(P, V, F, 8, 96)["height"], hgo.bake(P, Vn, F, 8, 96)["height"]
    has = ~np.isnan(a)
    assert np.array_equal(has, ~np.isnan(b)) and has.sum() > 96 * 96 // 2
    assert np.array_equal(np.negative(a[has]).view(np.uint32), b[has].view(np.uint32))


def _cli():
    from test_cli import CLI
    if not os.path.exists(CLI):
        subprocess.run(["make", "-C", os.path.dirname(CLI)], check=True, stdout=subprocess.DEVNULL)
    return CLI


def test_cli_refuses_multi_gpu_height_bake(tmp_path):
    r = subprocess.run([_cli(), "-g", "2", "-H", "h.png", "a.ply", "b.ply"], capture_output=True, text=True,
                       cwd=tmp_path)
    assert r.returncode == 0 and "-H" in r.stderr and "-b / -n" in r.stderr and "-t / -T" in r.stderr
    assert not (tmp_path / "h.png").exists()


def test_cli_height_bake_without_gpu(pkg, tmp_path):
    if pkg.device_count() > 0:
        pytest.skip("a GPU is present")
    P = pkg.synth.cloud_host(50, 1)
    write_cloud(tmp_path / "c.ply", P)
    write_mesh(tmp_path / "m.ply", pkg.synth.samples_host(3), pkg.synth.grid_faces(3, 3))
    r = subprocess.run([_cli(), "-H", "height.png", str(tmp_path / "c.ply"), str(tmp_path / "m.ply")],
                       capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and "no CUDA device" in r.stderr
    assert not (tmp_path / "height.png").exists()


# ---- GPU ------------------------------------------------------------------------------------------
def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def check_height(pkg, pto, P, V, F, k, res, pad=True, radius=None, coord_mode=0, height_range=None):
    with pkg.Tree(P, coord_mode=coord_mode) as tree:
        got = tree.bake(V, F, k=k, resolution=res, radius=radius, pad=pad, want=HEIGHTS, height_range=height_range)
    ref = hgo.bake(P, V, F, k, res, radius=-1.0 if radius is None else radius, pad_codes=pad,
                   height_range=height_range)
    assert_heights(got["height"], ref["height"])
    assert np.array_equal(got["height_u16"], ref["height_u16"])
    assert np.array_equal(np.array(got["height_range"]).view(np.uint64), np.array(ref["height_range"]).view(np.uint64))
    assert got["stats"]["height_texels"] == ref["texels"] and got["stats"]["texels"] == len(ref["samples"][0])
    return got, ref


@pytest.mark.gpu
@pytest.mark.parametrize("k,res,pad", [(20, 512, 1), (8, 257, 0), (32, 128, 1), (1, 300, 1), (5, 256, 1)])
def test_gpu_bake_height_equals_oracle(k, res, pad, pkg, pto):
    _need_gpu()
    side = 30.0
    P = pkg.synth.cloud_host(90_000, seed=41 + k, side=side)
    V, F = grid_mesh(pkg, 20, side)
    V["normal"] = tilted_normals(np.random.default_rng(k), len(V))
    got, _ = check_height(pkg, pto, P, V, F, k, res, pad=bool(pad))
    assert got["stats"]["height_texels"] > res * res // 2
    check_height(pkg, pto, P, V, F, k, res, pad=bool(pad), height_range=(-0.5, 0.5))


@pytest.mark.gpu
def test_gpu_bake_height_fp64_lattice_radius_nan(pkg, pto):
    _need_gpu()
    P, V, F, res = lattice_case(pto, res=300)
    V = V.copy()
    V["normal"] = tilted_normals(np.random.default_rng(3), len(V))
    check_height(pkg, pto, P, V, F, 20, res)
    rng = np.random.default_rng(8)
    P64 = pkg.make_points(P["ver"] + 1e-9 * rng.random(P["ver"].shape), normal=P["normal"], color=P["color"])
    check_height(pkg, pto, P64, V, F, 20, res, coord_mode=pkg.COORD_F64)
    got, _ = check_height(pkg, pto, P, V, F, 8, 200, pad=False, radius=0.2)
    assert 0 < got["stats"]["height_texels"] < got["stats"]["texels"]
    V["ver"][3] = np.nan
    got, _ = check_height(pkg, pto, P, V, F, 8, 200)
    assert 0 < got["stats"]["height_texels"] < got["stats"]["texels"]
    for seed, variant in ((5, "nan"), (7, "zero"), (8, "coincident")):
        Vv, Fv = variant_mesh(pto, seed, variant)
        check_height(pkg, pto, cloud_around(pto, Vv, 30_000, seed), Vv, Fv, 12, 160)


@pytest.mark.gpu
def test_gpu_bake_height_other_outputs_unchanged(pkg, pto):
    _need_gpu()
    side = 30.0
    P = pkg.synth.cloud_host(60_000, seed=5, side=side)
    V, F = grid_mesh(pkg, 16, side)
    V["normal"] = tilted_normals(np.random.default_rng(2), len(V))
    with pkg.Tree(P) as tree:
        ex = tree.bake(V, F, k=16, resolution=300, want=ALL_OUTPUTS)
        both = tree.bake(V, F, k=16, resolution=300, want=ALL_OUTPUTS + HEIGHTS)
        alone = tree.bake(V, F, k=16, resolution=300, want=("height",))
    for key in ALL_OUTPUTS:
        assert ex[key].tobytes() == both[key].tobytes(), key
    assert (ex["stats"]["texels"], ex["stats"]["empty"]) == (both["stats"]["texels"], both["stats"]["empty"])
    assert set(alone) == {"height", "height_range", "stats"}
    assert_heights(alone["height"], both["height"])
    assert "height_texels" not in ex["stats"] and "height_range" not in ex


@pytest.mark.gpu
def test_gpu_bake_height_two_chunks(pkg, pto):
    """A 4096^2 atlas: 2^24 covered texels, four query + height chunks."""
    _need_gpu()
    rng = np.random.default_rng(10)
    n = 40_000
    P = pkg.make_points(np.c_[rng.random((n, 2)) * 10.0, rng.normal(0, 0.05, n)], normal=rng.standard_normal((n, 3)),
                        color=rng.integers(0, 256, (n, 3)))
    V = pkg.make_points([[0, 0, 0], [10, 0, 0], [10, 10, 0], [0, 10, 0.0]], normal=np.tile([0.1, -0.2, 1.0], (4, 1)),
                        uv=[[0, 0], [1, 0], [1, 1], [0, 1.0]])
    F = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    res, k = 4096, 3
    with pkg.Tree(P) as tree:
        got = tree.bake(V, F, k=k, resolution=res, pad=False, want=HEIGHTS)
    assert got["stats"]["texels"] == res * res > 2 * 2**22
    texels, xyz, owner = tgo.bake_samples(V, F, res)
    pick = np.sort(np.random.default_rng(11).choice(len(texels), 50_000, replace=False))
    frames, _ = tgo.bake_frames(V, F)
    idx, d2 = hgo.neighbours(P, xyz[pick], k)
    ref = hgo.bake_height(V, frames, F, texels[pick], owner[pick], xyz[pick], P, idx, d2, res)
    assert np.array_equal(got["height"].reshape(-1)[texels[pick]].view(np.uint32),
                          ref.reshape(-1)[texels[pick]].view(np.uint32))
    h = got["height"]
    codes, used, valued = hgo.encode(h)
    assert used == got["height_range"] == (float(np.nanmin(h)), float(np.nanmax(h)))
    assert valued == got["stats"]["height_texels"] == res * res
    assert np.array_equal(codes, got["height_u16"])


@pytest.mark.gpu
def test_gpu_bake_height_device_piece(pkg, pto):
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
    frames, _ = pkg.bake_frames_device(xyzuvn, faces)
    pos = torch.from_numpy(np.c_[P["ver"], np.zeros(len(P))].astype(np.float32)).cuda()
    dtree = pkg.DeviceTree(pos)
    m = texels.numel()
    idx = torch.empty((m, k), dtype=torch.int32, device="cuda")
    dtree.query(xyz.contiguous(), k, idx=idx)
    cloud = torch.from_numpy(np.ascontiguousarray(P["ver"])).cuda()
    for pad, rng_in in ((True, None), (False, (-1.0, 1.0))):
        h = torch.empty((res, res), dtype=torch.float32, device="cuda")
        h16 = torch.empty((res, res), dtype=torch.uint16, device="cuda")
        used = torch.empty(2, dtype=torch.float64, device="cuda")
        pkg.bake_compose_height_device(xyzuvn, frames, faces, texels, owner, xyz.contiguous(), idx, k, cloud, res,
                                       pad=pad, height_range=rng_in, height=h, height_u16=h16, range_out=used)
        torch.cuda.synchronize()
        with pkg.Tree(P) as tree:
            ref = tree.bake(V, F, k=k, resolution=res, pad=pad, want=HEIGHTS, height_range=rng_in)
        assert_heights(h.cpu().numpy(), ref["height"])
        assert np.array_equal(h16.cpu().numpy(), ref["height_u16"])
        assert tuple(used.cpu().numpy()) == ref["height_range"]
        h16b = torch.empty((res, res), dtype=torch.uint16, device="cuda")       # the u16 map alone
        pkg.bake_compose_height_device(xyzuvn, frames, faces, texels, owner, xyz.contiguous(), idx, k, cloud, res,
                                       pad=pad, height_range=rng_in, height_u16=h16b)
        torch.cuda.synchronize()
        assert torch.equal(h16b, h16)
    dtree.close()


@pytest.mark.gpu
def test_gpu_bake_height_error_codes(pkg):
    _need_gpu()
    P = pkg.synth.cloud_host(2_000, seed=1, side=10.0)
    V, F = grid_mesh(pkg, 4, 10.0)
    L, ptr = pkg.lib(), pkg.api._np_ptr
    api = pkg.api
    h = np.empty(64 * 64, np.float32)
    with pkg.Tree(P) as tree:
        def call(o, hb, n_faces=len(F), res=64, k=8):
            return L.pt_texture_bake_height(tree.handle, ptr(V), len(V), ptr(F), n_faces, k, -1.0, res, 1,
                                            None if o is None else ctypes.byref(o),
                                            None if hb is None else ctypes.byref(hb), None)
        assert call(None, None) == 1
        assert call(api.BakeOutputs(), None) == 1
        assert call(None, api.BakeHeight()) == 1                          # a height struct asking for nothing
        hb = api.BakeHeight(height=h.ctypes.data)
        assert call(None, hb, n_faces=(2**31 - 1) // 3 + 1) == api.PT_ERR_UNSUPPORTED
        for res in (0, 16385):
            assert call(None, hb, res=res) == 1
        assert call(None, hb, k=33) == api.PT_ERR_UNSUPPORTED
        assert call(None, hb) == 0 and hb.texels > 0
        with pytest.raises(ValueError):
            tree.bake(V, F, k=8, resolution=64, want=("displacement",))
    with pkg.Tree(P, ids=np.arange(len(P), dtype=np.int32)) as slab:
        with pytest.raises(pkg.PointsTransferError) as e:
            slab.bake(V, F, k=8, resolution=64, want=("height",))
        assert e.value.status == api.PT_ERR_UNSUPPORTED
    dev = L.pt_bake_compose_height_device
    big = (2**31 - 1) // 3 + 1
    assert dev(None, None, 0, ptr(F), big, None, None, None, 0, None, 8, None, 0, 64, 1, None, ptr(h), None, None, 0,
               None) == api.PT_ERR_UNSUPPORTED
    assert dev(None, None, 0, None, 0, None, None, None, 0, None, 33, None, 0, 64, 1, None, ptr(h), None, None, 0,
               None) == api.PT_ERR_UNSUPPORTED
    assert dev(None, None, 0, None, 0, None, None, None, 0, None, 8, None, 0, 64, 1, None, None, None, None, 0,
               None) == 1
    assert dev(None, None, 0, None, 0, None, None, None, 5, None, 8, None, 0, 64, 1, None, ptr(h), None, None, 0,
               None) == 1


def read_png_gray16(path):
    """Decode a 16-bit greyscale, non-interlaced PNG written with filter 0 on every scanline."""
    data = open(path, "rb").read()
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    pos, idat, hdr = 8, b"", None
    while pos < len(data):
        n, kind = struct.unpack(">I4s", data[pos:pos + 8])
        body = data[pos + 8:pos + 8 + n]
        assert struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])[0] == zlib.crc32(kind + body), kind
        pos += 12 + n
        if kind == b"IHDR":
            hdr = struct.unpack(">IIBBBBB", body)
        elif kind == b"IDAT":
            idat += body
    w, h, depth, ctype, _, _, interlace = hdr
    assert (depth, ctype, interlace) == (16, 0, 0), hdr
    raw = np.frombuffer(zlib.decompress(idat), np.uint8).reshape(h, 1 + 2 * w)
    assert (raw[:, 0] == 0).all()
    return raw[:, 1:].copy().view(">u2").astype(np.uint16)


@pytest.mark.gpu
def test_gpu_cli_height_bake(pkg, pto, tmp_path):
    _need_gpu()
    cli = _cli()
    side = 20.0
    P = pkg.synth.cloud_host(20_000, 3, side=side)
    V, F = grid_mesh(pkg, 12, side)
    write_cloud(tmp_path / "c.ply", P)
    write_mesh(tmp_path / "m.ply", V, F)
    args = [str(tmp_path / "c.ply"), str(tmp_path / "m.ply")]
    r = subprocess.run([cli, "-R", "256", "-b", "bake.png", "-t", "tangent.png", "-H", "height.png", "-o", "tex_h.png",
                        *args], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    Vm = V.copy()
    Vm["normal"] = [0, 0, 1]
    ref = hgo.bake(P, Vm, F, 20, 256)
    assert np.array_equal(read_png_gray16(tmp_path / "height.png"), ref["height_u16"])
    line = next(ln for ln in r.stdout.splitlines() if ln.startswith("Height range:"))
    assert line == "Height range: %.9g %.9g" % ref["height_range"]
    r = subprocess.run([cli, "-R", "256", "-b", "bake0.png", "-t", "tangent0.png", "-o", "tex0.png", *args],
                       capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    assert "Height range" not in r.stdout
    for a, b in (("bake.png", "bake0.png"), ("tangent.png", "tangent0.png"), ("tex_h.png", "tex0.png")):
        assert (tmp_path / a).read_bytes() == (tmp_path / b).read_bytes(), a


@pytest.mark.gpu
def test_gpu_heightfield_recovered_on_flat_plane(pkg):
    """Cloud z = f(x, y) + noise (|noise| <= 3 sigma) over a plane mesh z = 0 with normals +z.  The
    height is a weighted mean of neighbour heights, so |h - f(x)| <= G * r_k + 3 sigma at every
    texel, where G bounds |grad f| and r_k is the texel's k-th neighbour distance (>= the horizontal
    distance to every neighbour used)."""
    _need_gpu()
    from scipy.spatial import cKDTree
    A, lam, sigma, side, k, res = 0.5, 8.0, 0.01, 20.0, 16, 384
    G = A * 2 * np.pi / lam * np.sqrt(2.0)

    def f(x, y):
        return A * np.sin(2 * np.pi * x / lam) * np.cos(2 * np.pi * y / lam)
    rng = np.random.default_rng(21)
    n = 400_000
    x, y = rng.random(n) * (side + 2) - 1, rng.random(n) * (side + 2) - 1
    z = f(x, y) + np.clip(rng.normal(0, sigma, n), -3 * sigma, 3 * sigma)
    P = pkg.make_points(np.c_[x, y, z])
    V = pkg.make_points([[0, 0, 0], [side, 0, 0], [side, side, 0], [0, side, 0.0]],
                        normal=np.tile([0, 0, 1.0], (4, 1)), uv=[[0, 0], [1, 0], [1, 1], [0, 1.0]])
    F = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    with pkg.Tree(P) as tree:
        got = tree.bake(V, F, k=k, resolution=res, pad=False, want=("height",))
    h = got["height"].reshape(-1)
    row, col = np.divmod(np.arange(res * res), res)
    tx, ty = (col + 0.5) / res * side, (res - row - 0.5) / res * side
    rk = cKDTree(np.c_[x, y, z]).query(np.c_[tx, ty, np.zeros_like(tx)], k)[0][:, -1]
    err = np.abs(h.astype(np.float64) - f(tx, ty))
    assert np.isfinite(h).all()
    assert (err <= G * rk + 3 * sigma + 1e-6).all(), float(np.max(err - G * rk - 3 * sigma))
    assert np.mean(err) < 0.05 * A
