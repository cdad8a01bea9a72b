"""Rows N1 / N3 / N4 of SURVEY.md section 8: the per-face transfer and the texture output
(/root/reference src/pointsTransfer.cpp:462-611, draw_triangle :66-107).

CPU part: the oracle's restatement (oracle/pt_texture_oracle.c) -- its post-process is pinned on
OpenCV's own dilate / bitwise_not / bitwise_and / add (the calls of :593-611), stored as golden
data and, where the cv2 wheel is installed, recomputed; its Delaunay-by-definition is checked
against scipy's Qhull Delaunay; the PNG the CLI writes is decoded back (test_cli.read_png_bgra,
and cv2 where installed).  GPU part: pt_texture_render must equal the oracle bit for bit."""
import os

import numpy as np
import pytest


def _mesh(pkg, g, side, colour=(200, 90, 30)):
    V = pkg.synth.samples_host(g, side=side)
    V["U"] = V["ver"][:, 0] / side * 0.9 + 0.05
    V["V"] = V["ver"][:, 1] / side * 0.9 + 0.05
    V["color"] = np.array(colour)
    return V, pkg.synth.grid_faces(g, g)


def _opencv_pad(cv2, img):
    kern = cv2.getStructuringElement(cv2.MORPH_RECT, (25, 25))      # :595
    dilated = cv2.dilate(img, kern)                                 # :598
    bgra = cv2.split(img)                                           # :601
    alpha_mask = cv2.bitwise_not(cv2.merge([bgra[3]] * 4))          # :603-607
    return cv2.add(img, cv2.bitwise_and(dilated, alpha_mask))       # :609-612


def test_pad_is_opencv_dilate_and_gutter(pto, golden_dir):
    """Against OpenCV's results on the same images, stored in tests/golden/opencv/pad.npz
    (tools/make_golden_opencv.py), and against the cv2 wheel itself where it is installed."""
    try:
        import cv2
    except ImportError:
        cv2 = None
    z = np.load(os.path.join(golden_dir, "opencv", "pad.npz"))
    for res in (256, 200, 64):
        img, padded = z[f"in_{res}"], z[f"padded_{res}"]
        assert np.array_equal(pto.texture_pad(img), padded)
        if cv2 is not None:
            assert np.array_equal(_opencv_pad(cv2, img), padded)


def test_oracle_texture_covers_the_mesh_and_triangulates(pkg, pto):
    side, g, res = 20.0, 12, 512
    P = pkg.synth.cloud_host(40_000, seed=3, side=side)
    V, F = _mesh(pkg, g, side)
    idx, _ = pto.knn_bruteforce(P, V, 20)
    img, (ntri, nin) = pto.texture(P, V, idx, F, res, pad=False)
    assert nin > 0 and ntri > len(F)
    alpha = img[..., 3]
    assert set(np.unique(alpha).tolist()) <= {0, 255}
    # the UV image of the mesh is the square [0.05, 0.95]^2: fully covered inside, empty outside
    assert (alpha[40:470, 40:470] == 255).all()
    assert (alpha[:20] == 0).all() and (alpha[:, :20] == 0).all()
    # without inside points a face is drawn flat with its corners' colour
    far = pto.make_points(P["ver"] + 1000.0, normal=P["normal"], color=P["color"])
    img2, (ntri2, nin2) = pto.texture(far, V, idx, F, res, pad=False)
    assert nin2 == 0 and ntri2 == len(F)
    assert np.array_equal(np.unique(img2[alpha == 255].reshape(-1, 4), axis=0), [[30, 90, 200, 255]])


def test_delaunay_by_definition_matches_qhull(pkg, pto):
    """One big face over a planar cloud: the oracle's sub-triangle count equals Qhull's Delaunay of
    the same 2-D points (general position), and the drawn area is the face."""
    scipy_spatial = pytest.importorskip("scipy.spatial")
    rng = np.random.default_rng(7)
    n = 40
    xy = rng.random((n, 2)) * 0.6 + 0.1
    xy = xy[xy.sum(1) < 0.95]                       # strictly inside the triangle (0,0) (1,0) (0,1)
    P = pto.make_points(np.c_[xy, np.zeros(len(xy))], color=rng.integers(0, 256, (len(xy), 3)))
    V = pto.make_points(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0.0]]), color=[[9, 9, 9]] * 3,
                        uv=[[0.1, 0.1], [0.9, 0.1], [0.1, 0.9]])
    k = 32
    idx = np.full((3, k), -1, np.int32)
    ids = np.arange(len(xy))
    for c in range(3):                              # every point is some corner's neighbour
        part = ids[c::3][:k]
        idx[c, :len(part)] = part
    _, (ntri, nin) = pto.texture(P, V, idx, np.array([[0, 1, 2]]), 256, pad=False)
    assert nin == len(xy)
    tri = scipy_spatial.Delaunay(np.r_[[[0, 0], [1, 0], [0, 1.0]], xy])
    assert ntri == len(tri.simplices)


@pytest.mark.gpu
@pytest.mark.parametrize("k,res,pad", [(20, 512, True), (8, 256, False), (32, 300, True)])
def test_gpu_texture_equals_oracle(k, res, pad, pkg, pto):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    side, g = 30.0, 20
    P = pkg.synth.cloud_host(90_000, seed=11 + k, side=side)
    V, F = _mesh(pkg, g, side)
    with pkg.Tree(P) as tree:
        idx, _ = tree.knn(V, k)
        img, st = tree.texture(V, F, k=k, resolution=res, pad=pad)
    ref_idx, _ = pto.knn_bruteforce(P, V, k)
    assert np.array_equal(idx, ref_idx)
    ref, (ntri, nin) = pto.texture(P, V, ref_idx, F, res, pad=pad)
    assert st["triangles"] == ntri and st["inside_points"] == nin
    assert np.array_equal(img, ref)


@pytest.mark.gpu
def test_gpu_texture_degenerate_inputs(pkg, pto):
    """Lattice cloud (co-circular quadruples everywhere), points exactly on edges and corners,
    a degenerate face, fp64 coordinates: the GPU image still equals the oracle's."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    gx, gy = np.meshgrid(np.arange(41) * 0.25, np.arange(41) * 0.25)
    xyz = np.c_[gx.ravel(), gy.ravel(), np.zeros(gx.size)]
    rng = np.random.default_rng(5)
    P = pkg.make_points(xyz, normal=np.tile([0, 0, 1.0], (len(xyz), 1)), color=rng.integers(0, 256, (len(xyz), 3)))
    Vx = np.array([[0, 0, 0], [10, 0, 0], [10, 10, 0], [0, 10, 0], [5, 5, 0], [5, 5, 0.0]])
    V = pkg.make_points(Vx, color=[[1, 2, 3]] * 6, uv=Vx[:, :2] / 10 * 0.8 + 0.1)
    F = np.array([[0, 1, 4], [1, 2, 4], [2, 3, 4], [3, 0, 4], [4, 5, 4]], np.int32)    # the last one is degenerate
    for pts in (P, pkg.make_points(xyz + 1e-9 * rng.random(xyz.shape), normal=P["normal"], color=P["color"])):
        with pkg.Tree(pts) as tree:
            idx, _ = tree.knn(V, 20)
            img, st = tree.texture(V, F, k=20, resolution=400, pad=True)
        ref, (ntri, nin) = pto.texture(pts, V, idx, F, 400, pad=True)
        assert st["triangles"] == ntri and st["inside_points"] == nin
        assert np.array_equal(img, ref)


def test_png_writer_round_trip(tmp_path):
    """host/pt_png.h (replaces cv::imwrite, :613): the file decodes back to the same B G R A bytes,
    through a strict reader of its own and through OpenCV where it is installed."""
    import subprocess
    from test_cli import read_png_bgra
    try:
        import cv2
    except ImportError:
        cv2 = None
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    host = os.path.join(root, "3d-reconstruction-from-point-cloud_b200", "host")
    src = tmp_path / "t.cpp"
    src.write_text('#include "pt_png.h"\n#include <fstream>\n#include <iterator>\n'
                   "int main(int c, char **v) { std::ifstream f(v[1], std::ios::binary);\n"
                   "  std::vector<uint8_t> b((std::istreambuf_iterator<char>(f)), {});\n"
                   "  int w = atoi(v[3]), h = atoi(v[4]);\n"
                   "  return ptb::write_png_bgra(v[2], b.data(), w, h) ? 0 : 1; }\n")
    exe = tmp_path / "t"
    subprocess.run(["/usr/bin/g++", "-O1", "-std=c++17", "-I", host, str(src), "-o", str(exe), "-lz"], check=True)
    rng = np.random.default_rng(0)
    for w, h in ((37, 19), (640, 480)):
        img = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
        img[: h // 2] = 0                                     # long zero runs as in a real texture
        (tmp_path / "raw.bin").write_bytes(img.tobytes())
        assert subprocess.run([str(exe), str(tmp_path / "raw.bin"), str(tmp_path / "o.png"), str(w), str(h)]).returncode == 0
        assert np.array_equal(read_png_bgra(tmp_path / "o.png"), img)
        if cv2 is not None:
            back = cv2.imread(str(tmp_path / "o.png"), cv2.IMREAD_UNCHANGED)
            assert back is not None and np.array_equal(back, img)
