"""Per-texel bake on one GPU (DESIGN.md section 8, "Per-texel bake").

The cfg2 cloud (50 M points, generated on the device) and the g = 448 grid mesh on the noise-free
surface with UV = (x / L, y / L); bakes at 2048^2 with k = 32 and at 4096^2 with k = 16, plus a
2-face quad covering a 16384^2 atlas (k = 1: the case that splits one face over many warps).  Per
shape: one warm-up bake, then `--reps` timed bakes; prints the per-stage device ms of
pt_bake_stats (median), the wall time, texels/s, and the kNN stage's samples/s next to
DeviceTree.query on the same number of pt_synth_samples_device(center=1) samples.  A seeded subset
of texels is checked against the CPU oracle in the same run (exit 1 on a mismatch).  The L2 is not
flushed between passes; the cloud alone (800 MB of records) is several times its size.

    python tools/prof_bake.py [--reps 3] [--verify 256] [--out report.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--verify", type=int, default=256, help="texels checked against the oracle")
    ap.add_argument("--out", default=None, help="also write the report as JSON to this file")
    args = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    from oracle import pto, pto_bake
    pkg = ge.package()
    if not torch.cuda.is_available():
        sys.exit("prof_bake needs a CUDA device")
    torch.cuda.set_device(0)
    L = pkg.synth.L_DOMAIN
    w = pkg.synth.CONFIGS["cfg2"]
    g = w.gu
    pos, attrs = pkg.synth.cloud_device(w.n_points, seed=w.seed)
    tree = pkg.DeviceTree(pos, attrs)
    V = pkg.synth.queries_to_host(pkg.synth.samples_device(g, g))
    V["U"], V["V"] = V["ver"][:, 0] / L, V["ver"][:, 1] / L
    F = pkg.synth.grid_faces(g, g)
    corners = np.array([[0, 0, 0], [L, 0, 0], [L, L, 0], [0, L, 0.0]])
    quad = pkg.make_points(corners, uv=corners[:, :2] / L)
    quad_faces = np.array([[0, 1, 2], [0, 2, 3]], np.int32)

    report = {"card": card(), "cloud": w.n_points, "mesh_faces": int(len(F)), "l2_flushed": False, "shapes": []}
    print("card (name, power limit):", report["card"])
    last = None
    for name, verts, faces, res, k, want in (("grid g=448, 2048^2, k=32", V, F, 2048, 32, ("bgra", "normal_bgra", "normal")),
                                             ("grid g=448, 4096^2, k=16", V, F, 4096, 16, ("bgra", "normal_bgra", "normal")),
                                             ("2-face quad, 16384^2, k=1", quad, quad_faces, 16384, 1, ("bgra",))):
        tree.bake(verts, faces, k=k, resolution=res, want=want)                  # warm-up
        runs = []
        for _ in range(args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = tree.bake(verts, faces, k=k, resolution=res, want=want)
            wall = time.perf_counter() - t0
            runs.append(dict(out["stats"], wall_s=wall))
        med = {key: float(np.median([r[key] for r in runs])) for key in ("raster_ms", "knn_ms", "pad_ms", "wall_s")}
        texels = runs[0]["texels"]
        # the same number of analytic texel-centre samples through DeviceTree.query
        q = pkg.synth.samples_device(res, max(1, texels // res), center=True)
        m = q.shape[0]
        rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
        nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
        tree.query(q, k, rgba=rgba, normal=nrm)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        qms = []
        for _ in range(args.reps):
            e0.record()
            tree.query(q, k, rgba=rgba, normal=nrm)
            e1.record()
            torch.cuda.synchronize()
            qms.append(e0.elapsed_time(e1))
        del q, rgba, nrm
        row = {"shape": name, "resolution": res, "k": k, "texels": texels, "empty": runs[0]["empty"], **med,
               "texels_per_s": texels / med["wall_s"], "knn_samples_per_s": texels / (med["knn_ms"] * 1e-3),
               "query_samples": m, "query_ms": float(np.median(qms)),
               "query_samples_per_s": m / (float(np.median(qms)) * 1e-3)}
        report["shapes"].append(row)
        print(json.dumps(row))
        if res == 2048:
            last = (verts, faces, res, k, out)
        del out

    # oracle check on a seeded subset of the 2048^2 bake: texel list and positions in full (device
    # piece vs oracle), blend of the subset by brute force over the whole cloud
    verts, faces, res, k, out = last
    xyzuv = torch.from_numpy(np.c_[verts["ver"], verts["U"], verts["V"]]).cuda()
    texels, xyz = pkg.bake_texels_device(xyzuv, torch.from_numpy(faces).cuda(), res)
    ref_t, ref_xyz = pto_bake.bake_texels(verts, faces, res)
    ok = np.array_equal(texels.cpu().numpy().astype(np.uint32), ref_t) and \
        np.array_equal(xyz.cpu().numpy().view(np.uint64), ref_xyz.view(np.uint64))
    rng = np.random.default_rng(20261020)
    pick = rng.choice(len(ref_t), size=min(args.verify, len(ref_t)), replace=False)
    P = pkg.synth.points_to_host(pos, attrs)
    idx, d2 = pto.knn_bruteforce(P, pto.make_points(ref_xyz[pick]), k)
    rgba, nrm = pto.blend(P, idx, d2)
    t = ref_t[pick]
    got_bgra = out["bgra"].reshape(-1, 4)[t]
    got_n = out["normal"].reshape(-1, 3)[t]
    ok &= np.array_equal(got_bgra[:, :3], rgba[:, 2::-1]) and np.array_equal(got_n.view(np.uint32), nrm.view(np.uint32))
    ok &= all(np.array_equal(out["normal_bgra"].reshape(-1, 4)[t][:, c], [pto_bake.bake_encode(x) for x in nrm[:, 2 - c]])
              for c in range(3))
    report["verified_texels"] = int(len(pick))
    report["verified"] = bool(ok)
    print(f"oracle check ({len(pick)} texels + full texel list): {'ok' if ok else 'MISMATCH'}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    tree.close()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
