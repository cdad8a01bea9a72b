"""The C++ front end keeps the reference CLI's contract (src/pointsTransfer.cpp:109-141,
269-273, 587-625): usage text and exit codes, stdout labels, ASCII PLY formats."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "3d-reconstruction-from-point-cloud_b200", "host", "pointsTransfer")


@pytest.fixture(scope="module")
def cli():
    if not os.path.exists(CLI):
        subprocess.run(["make", "-C", os.path.dirname(CLI)], check=True, stdout=subprocess.DEVNULL)
    return CLI


def write_cloud(path, P):
    with open(path, "w") as f:
        f.write("ply\nformat ascii 1.0\nelement vertex %d\nproperty float x\nend_header\n" % len(P))
        for p in P:
            f.write("%.17g %.17g %.17g %.9g %.9g %.9g %d %d %d\n" % (
                *p["ver"], *p["normal"], *p["color"]))


def write_mesh(path, V, F):
    with open(path, "w") as f:
        f.write("ply\nformat ascii 1.0\nelement vertex %d\nelement face %d\nend_header\n" % (len(V), len(F)))
        for v in V:
            f.write("%.17g %.17g %.17g 0 0 1 %.17g %.17g 10 20 30\n" % (*v["ver"], v["U"], v["V"]))
        for a, b, c in F:
            f.write("3 %d %d %d\n" % (a, b, c))


def read_png_bgra(path):
    """Decode an 8-bit RGBA, non-interlaced PNG (every chunk CRC checked, all five scanline
    filters) into B G R A rows, the layout cv::imread(..., IMREAD_UNCHANGED) returns."""
    import struct
    import zlib
    data = open(path, "rb").read()
    assert data[:8] == b"\x89PNG\r\n\x1a\n", "not a PNG"
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
        elif kind == b"IEND":
            break
    w, h, depth, ctype, _, _, interlace = hdr
    assert (depth, ctype, interlace) == (8, 6, 0), hdr
    raw = zlib.decompress(idat)
    stride, bpp = 4 * w, 4
    assert len(raw) == h * (stride + 1)
    out = np.zeros((h, stride), np.uint8)
    prev = np.zeros(stride, np.int64)
    for y in range(h):
        f, line = raw[y * (stride + 1)], np.frombuffer(raw, np.uint8, stride, y * (stride + 1) + 1)
        cur = line.astype(np.int64)
        if f == 2:
            cur = (cur + prev) & 255
        elif f in (1, 3, 4):
            cur = cur.copy()
            for x in range(stride):
                a = cur[x - bpp] if x >= bpp else 0
                c = prev[x - bpp] if x >= bpp else 0
                if f == 1:
                    pred = a
                elif f == 3:
                    pred = (a + prev[x]) // 2
                else:
                    pa, pb, pc = abs(prev[x] - c), abs(a - c), abs(a + prev[x] - 2 * c)
                    pred = a if pa <= pb and pa <= pc else (prev[x] if pb <= pc else c)
                cur[x] = (cur[x] + pred) & 255
        else:
            assert f == 0, f"scanline filter {f}"
        out[y], prev = cur, cur
    return out.reshape(h, w, 4)[..., [2, 1, 0, 3]]


def test_usage_and_missing_files(cli, tmp_path):
    r = subprocess.run([cli], capture_output=True, text=True)
    assert r.returncode == 0       # the reference returns 0 on usage (:116-120)
    assert r.stdout.strip() == "Usage: ./pointTransfer <input-point-cloud> <input-mesh>"
    r = subprocess.run([cli, str(tmp_path / "nope.ply"), str(tmp_path / "nope2.ply")],
                       capture_output=True, text=True)
    assert r.returncode == 0       # :137-141
    assert "Cannot read or find point cloud file:" in r.stderr


def test_no_gpu_fails_loudly(cli, pkg, tmp_path):
    if pkg.device_count() > 0:
        pytest.skip("a GPU is present")
    P = pkg.synth.cloud_host(50, 1)
    write_cloud(tmp_path / "c.ply", P)
    write_mesh(tmp_path / "m.ply", pkg.synth.samples_host(3), pkg.synth.grid_faces(3, 3))
    r = subprocess.run([cli, str(tmp_path / "c.ply"), str(tmp_path / "m.ply")],
                       capture_output=True, text=True, cwd=tmp_path)
    assert "PC Point count: 50" in r.stdout
    assert "no CUDA device" in r.stderr and not (tmp_path / "texture.png").exists()


def test_header_announcing_more_than_memory_is_a_message_not_a_crash(cli, tmp_path):
    with open(tmp_path / "huge.ply", "w") as f:
        f.write("ply\nformat ascii 1.0\nelement vertex 99999999999999\nend_header\n1 2 3 0 0 1 1 2 3\n")
    r = subprocess.run([cli, str(tmp_path / "huge.ply"), str(tmp_path / "huge.ply")],
                       capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and "pointsTransfer:" in r.stderr


def test_bad_k_is_a_message_not_a_crash(cli, tmp_path):
    # every error path of the reference prints and returns 0 (:116-120, :137-141)
    for k in ("-3", "0", "99"):
        r = subprocess.run([cli, "-k", k, "a.ply", "b.ply"], capture_output=True, text=True, cwd=tmp_path)
        assert r.returncode == 0 and "-k must be" in r.stderr


@pytest.mark.gpu
def test_cli_end_to_end(cli, pkg, pto, tmp_path):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    P = pkg.synth.cloud_host(20_000, 3, side=20.0)
    V = pkg.synth.samples_host(12, side=20.0)
    F = pkg.synth.grid_faces(12, 12)
    write_cloud(tmp_path / "c.ply", P)
    V["U"] = V["ver"][:, 0] / 20.0 * 0.9 + 0.05
    V["V"] = V["ver"][:, 1] / 20.0 * 0.9 + 0.05
    write_mesh(tmp_path / "m.ply", V, F)
    r = subprocess.run([cli, "-R", "512", "-p", "transferred.ply", str(tmp_path / "c.ply"), str(tmp_path / "m.ply")],
                       capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    for label in ("PC Point count: 20000", "Read point set in:", "Built Kd tree in:",
                  "Mesh vertex count: 144", "Mesh face count: %d" % len(F), "Read mesh faces:",
                  "Neighbor search total time:", "Draw triangles total time:", "Output time:",
                  "Total real time:", "VIRT:", "RES:"):
        assert label in r.stdout, label
    # the reference's artefact: texture.png in the working directory (:613), equal to the oracle's
    # restatement of the face loop + post-process on the same inputs (K = 20, :128)
    png = read_png_bgra(tmp_path / "texture.png")                                # BGRA, as cv::Mat
    assert png.shape == (512, 512, 4)
    Vm = V.copy()
    Vm["color"] = np.array([10, 20, 30])                  # what write_mesh put in the file
    idx, d2 = pto.knn_bruteforce(P, Vm, 20)
    ref_img, (ntri, nin) = pto.texture(P, Vm, idx, F, 512, pad=True)
    assert ntri > len(F) and nin > 0
    assert np.array_equal(png, ref_img)
    rows = [l.split() for l in open(tmp_path / "transferred.ply").read().split("end_header\n")[1].splitlines()]
    verts = np.array(rows[:144], dtype=np.float64)
    faces = np.array(rows[144:], dtype=np.int64)
    assert np.array_equal(faces[:, 1:], F)
    # %.17g text round-trips the fp64 values exactly
    rgba, nrm = pto.blend(P, idx, d2)
    assert np.array_equal(verts[:, 8:11].astype(np.uint8), rgba[:, :3])
    assert np.allclose(verts[:, 3:6], nrm, rtol=1e-5, atol=1e-7)
    assert np.array_equal(verts[:, :3], V["ver"])
