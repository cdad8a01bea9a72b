"""The C++ multi-GPU host behind the C ABI (csrc/pt_sharded.cu: pt_sharded_build / _knn /
_transfer, one host thread and one index per x-slab, ghost zones, automatic halo widening) and
pt_texture_render_lists.  Devices may repeat in the device list, so the single-GPU box runs 2-4
slabs on device 0; with >= 2 GPUs the slabs really sit on different devices.  Everything is
compared with the oracle on the WHOLE cloud (the reference's loop: src/pointsTransfer.cpp:465-479)."""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _check(out, ref):
    ref_idx, ref_d2, ref_rgba, ref_nrm = ref
    assert np.array_equal(out["idx"], ref_idx)
    assert np.array_equal(out["d2"], ref_d2)
    assert np.array_equal(out["rgba"], ref_rgba)
    assert np.allclose(out["normal"], ref_nrm, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("n_slabs,k,radius", [(2, 16, None), (3, 20, None), (4, 8, 0.6)])
def test_sharded_host_equals_oracle(n_slabs, k, radius, pkg, pto, torch_cuda):
    ndev = torch_cuda.cuda.device_count()
    P = pkg.synth.cloud_host(150_000, seed=17, side=60.0)
    V = pkg.synth.samples_host(60, side=60.0)
    rng = np.random.default_rng(2)
    V = V[rng.permutation(len(V))]                       # samples arrive in arbitrary order
    ref_idx, ref_d2 = pto.KdTree(P).knn(V, k, radius=-1.0 if radius is None else radius)
    ref = (ref_idx, ref_d2) + pto.blend(P, ref_idx, ref_d2)
    devices = [r % ndev for r in range(n_slabs)]
    with pkg.ShardedTree(P, devices, k_hint=k) as st:
        info = st.info()
        assert info["n_slabs"] == n_slabs and sum(info["slab_points"]) == len(P)
        assert all(g > 0 for g in info["slab_ghosts"])           # every slab carries a ghost zone
        _check(st.transfer(V, k, radius=radius, want_idx=True, want_d2=True), ref)
        idx, d2 = st.knn(V, k, radius=radius)
        assert np.array_equal(idx, ref_idx) and np.array_equal(d2, ref_d2)
        assert st.info()["rebuilds"] == 0
    # a ghost zone that is far too narrow: the call widens it until the result is provably exact
    with pkg.ShardedTree(P, devices, halo=1e-4, k_hint=k) as st:
        _check(st.transfer(V, k, radius=radius, want_idx=True, want_d2=True), ref)
        info = st.info()
        assert info["rebuilds"] > 0 and info["halo"] > 1e-4


def test_texture_from_lists_equals_oracle(pkg, pto, torch_cuda):
    side, g, k, res = 30.0, 20, 20, 400
    P = pkg.synth.cloud_host(90_000, seed=5, side=side)
    V = pkg.synth.samples_host(g, side=side)
    V["U"] = V["ver"][:, 0] / side * 0.9 + 0.05
    V["V"] = V["ver"][:, 1] / side * 0.9 + 0.05
    V["color"] = np.array([200, 90, 30])
    F = pkg.synth.grid_faces(g, g)
    with pkg.ShardedTree(P, [0, 0]) as st:
        idx, _ = st.knn(V, k)
    ref_idx, _ = pto.knn_bruteforce(P, V, k)
    assert np.array_equal(idx, ref_idx)
    img, stats = pkg.texture_from_lists(P, V, F, idx, resolution=res, pad=True)
    ref, (ntri, nin) = pto.texture(P, V, ref_idx, F, res, pad=True)
    assert stats["triangles"] == ntri and stats["inside_points"] == nin
    assert np.array_equal(img, ref)


def test_cli_with_two_slabs(pkg, pto, torch_cuda, tmp_path):
    """`pointsTransfer -g 2`: the sharded C++ host end to end, same texture.png as the oracle."""
    from test_cli import CLI, read_png_bgra, write_cloud, write_mesh
    if not os.path.exists(CLI):
        subprocess.run(["make", "-C", os.path.dirname(CLI)], check=True, stdout=subprocess.DEVNULL)
    P = pkg.synth.cloud_host(20_000, 3, side=20.0)
    V = pkg.synth.samples_host(12, side=20.0)
    F = pkg.synth.grid_faces(12, 12)
    V["U"] = V["ver"][:, 0] / 20.0 * 0.9 + 0.05
    V["V"] = V["ver"][:, 1] / 20.0 * 0.9 + 0.05
    write_cloud(tmp_path / "c.ply", P)
    write_mesh(tmp_path / "m.ply", V, F)
    r = subprocess.run([CLI, "-g", "2", "-R", "512", str(tmp_path / "c.ply"), str(tmp_path / "m.ply")],
                       capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and "Draw triangles total time:" in r.stdout, r.stderr
    png = read_png_bgra(tmp_path / "texture.png")
    Vm = V.copy()
    Vm["color"] = np.array([10, 20, 30])
    idx, _ = pto.knn_bruteforce(P, Vm, 20)
    ref_img, _ = pto.texture(P, Vm, idx, F, 512, pad=True)
    assert np.array_equal(png, ref_img)
