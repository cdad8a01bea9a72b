"""Height bake on one GPU (DESIGN.md section 8, "Height bake").

The cfg2 cloud (50 M points, generated on the device) and the g = 448 grid mesh of tools/prof_bake.py
(noise-free surface, UV = (x / L, y / L), zero vertex normals, so the frames come from the summed
face normals); bakes at 2048^2 with k = 32 and at 4096^2 with k = 16.  Per shape:
* device time (CUDA events, median of --reps) of the k-NN + blend of the bake's samples through
  DeviceTree.query, without and with the neighbour lists (idx) written;
* device time of the height stage through pt_bake_compose_height_device: the float map alone
  (NaN fill + height kernel + range reduction), and with the padded 16-bit map (+ encode + pad);
* the bake's kernels by name from one torch.profiler pass over pt_texture_bake_height;
* wall time of pt_texture_bake_ex (six outputs) against pt_texture_bake_height (the same six plus
  both height maps), alternated in one process after a warm-up of each, maps copied to pageable
  host memory; the six common outputs compared byte for byte.
Then, at 2048^2, the heights of a seeded subset of texels are checked against the CPU oracle, fed
with the device's neighbour lists and the listed points (exit 1 on a mismatch).  The card's name
and power limit are read in the same run.  The L2 is not flushed; the cloud alone is several times
its size.

    python tools/prof_bake_height.py [--reps 5] [--verify 4096] [--out report.json]
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

ALL = ("bgra", "normal_bgra", "normal", "tangent_bgra", "tangent_normal", "tangents")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--verify", type=int, default=4096, help="texels of the height map checked against the oracle")
    ap.add_argument("--out", default=None, help="also write the report as JSON to this file")
    args = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    import bake_height_oracle as hgo
    import bake_tangent_oracle as tgo
    from prof_bake import card
    pkg = ge.package()
    if not torch.cuda.is_available():
        sys.exit("prof_bake_height needs a CUDA device")
    torch.cuda.set_device(0)
    api, L = pkg.api, pkg.lib()
    w = pkg.synth.CONFIGS["cfg2"]
    g, side = w.gu, pkg.synth.L_DOMAIN
    pos, attrs = pkg.synth.cloud_device(w.n_points, seed=w.seed)
    tree = pkg.DeviceTree(pos, attrs)
    V = pkg.synth.queries_to_host(pkg.synth.samples_device(g, g))
    V["U"], V["V"] = V["ver"][:, 0] / side, V["ver"][:, 1] / side
    F = pkg.synth.grid_faces(g, g)
    ptr = api._np_ptr
    xyzuv = torch.from_numpy(np.c_[V["ver"], V["U"], V["V"]]).cuda()
    xyzuvn = torch.from_numpy(np.c_[V["ver"], V["U"], V["V"], V["normal"]]).cuda()
    faces = torch.from_numpy(F).cuda()
    cloud = pos[:, :3].to(torch.float64).contiguous()          # original order: DeviceTree ids are row numbers

    report = {"card": card(), "cloud": w.n_points, "mesh_vertices": int(len(V)), "mesh_faces": int(len(F)),
              "l2_flushed": False, "shapes": []}
    print("card (name, power limit):", report["card"])
    med = lambda xs: float(np.median(xs))                                       # noqa: E731
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    verify = None
    for res, k in ((2048, 32), (4096, 16)):
        out6 = {"bgra": np.empty((res, res, 4), np.uint8), "normal_bgra": np.empty((res, res, 4), np.uint8),
                "normal": np.empty((res, res, 3), np.float32), "tangent_bgra": np.empty((res, res, 4), np.uint8),
                "tangent_normal": np.empty((res, res, 3), np.float32), "tangents": np.empty((len(V), 4), np.float32)}
        out8 = {n: np.empty_like(a) for n, a in out6.items()}
        hmap, h16 = np.empty((res, res), np.float32), np.empty((res, res), np.uint16)
        o6 = api.BakeOutputs(*[out6[n].ctypes.data for n in ALL])
        o8 = api.BakeOutputs(*[out8[n].ctypes.data for n in ALL])
        hb = api.BakeHeight(hmap.ctypes.data, h16.ctypes.data)

        def bake_ex():
            st = api.BakeStats()
            api._check(L.pt_texture_bake_ex(tree.handle, ptr(V), len(V), ptr(F), len(F), k, -1.0, res, 1,
                                            ctypes.byref(o6), ctypes.byref(st)), "bake_ex")
            return st

        def bake_height():
            st = api.BakeStats()
            api._check(L.pt_texture_bake_height(tree.handle, ptr(V), len(V), ptr(F), len(F), k, -1.0, res, 1,
                                                ctypes.byref(o8), ctypes.byref(hb), ctypes.byref(st)), "bake_height")
            return st

        bake_ex(), bake_height()                                                # warm-up
        walls = {"bake_ex": [], "bake_height": []}
        stats = {"bake_ex": [], "bake_height": []}
        for _ in range(args.reps):
            for name, fn in (("bake_ex", bake_ex), ("bake_height", bake_height)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                st = fn()
                walls[name].append(time.perf_counter() - t0)
                stats[name].append((st.raster_ms, st.knn_ms, st.pad_ms))
        same = all(out6[n].tobytes() == out8[n].tobytes() for n in ALL)

        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            bake_height()
        kernels = {}
        for ev in prof.key_averages():
            if ev.device_type == torch.autograd.DeviceType.CUDA and ev.device_time_total > 0:
                kernels[ev.key[:90]] = round(ev.device_time_total / 1e3, 4)

        # the stages on their own, on the bake's samples
        texels, xyz, owner = pkg.bake_samples_device(xyzuv, faces, res)
        xyz = xyz.contiguous()
        m = texels.numel()
        frames, _ = pkg.bake_frames_device(xyzuvn, faces, tangents=False)
        rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
        nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
        idx = torch.empty((m, k), dtype=torch.int32, device="cuda")
        dh = torch.empty((res, res), dtype=torch.float32, device="cuda")
        dh16 = torch.empty((res, res), dtype=torch.uint16, device="cuda")
        knn_ms, knn_idx_ms, height_ms, height_u16_ms = [], [], [], []
        for _ in range(args.reps + 1):
            knn_ms.append(timed(lambda: tree.query(xyz, k, rgba=rgba, normal=nrm)))
            knn_idx_ms.append(timed(lambda: tree.query(xyz, k, rgba=rgba, normal=nrm, idx=idx)))
            height_ms.append(timed(lambda: pkg.bake_compose_height_device(
                xyzuvn, frames, faces, texels, owner, xyz, idx, k, cloud, res, height=dh)))
            height_u16_ms.append(timed(lambda: pkg.bake_compose_height_device(
                xyzuvn, frames, faces, texels, owner, xyz, idx, k, cloud, res, height=dh, height_u16=dh16)))
        pieces_same = dh.cpu().numpy().tobytes() == hmap.tobytes() and np.array_equal(dh16.cpu().numpy(), h16)
        row = {"resolution": res, "k": k, "texels": int(m), "height_texels": int(hb.texels),
               "height_range": [hb.range_used[0], hb.range_used[1]],
               "knn_ms": med(knn_ms[1:]), "knn_with_idx_ms": med(knn_idx_ms[1:]),
               "height_float_ms": med(height_ms[1:]), "height_float_u16_pad_ms": med(height_u16_ms[1:]),
               "bake_ex_wall_ms": 1e3 * med(walls["bake_ex"]), "bake_height_wall_ms": 1e3 * med(walls["bake_height"]),
               "bake_ex_stage_ms": [med([s[j] for s in stats["bake_ex"]]) for j in range(3)],
               "bake_height_stage_ms": [med([s[j] for s in stats["bake_height"]]) for j in range(3)],
               "bake_ex_walls_ms": [1e3 * x for x in walls["bake_ex"]],
               "bake_height_walls_ms": [1e3 * x for x in walls["bake_height"]],
               "profiler_kernels_ms": kernels,
               "common_outputs_identical": bool(same), "device_piece_identical": bool(pieces_same)}
        report["shapes"].append(row)
        print(json.dumps(row))
        if res == 2048:
            rng = np.random.default_rng(20261020)
            pick = np.sort(rng.choice(m, size=min(args.verify, m), replace=False))
            d2 = torch.empty((m, k), dtype=torch.float64, device="cuda")
            tree.query(xyz, k, idx=idx, d2=d2)
            verify = (res, pick, texels.cpu().numpy()[pick].astype(np.uint32), owner.cpu().numpy()[pick],
                      xyz.cpu().numpy()[pick], idx.cpu().numpy()[pick], d2.cpu().numpy()[pick],
                      frames.cpu().numpy(), hmap.copy())
        del texels, xyz, owner, rgba, nrm, idx, dh, dh16, frames
        torch.cuda.empty_cache()

    # oracle check at 2048^2 on a seeded subset: the listed points only, ids renumbered
    res, pick, t, own, xyz, idx, d2, frames, hmap = verify
    ids, inv = np.unique(idx[idx >= 0], return_inverse=True)
    sub = np.full(idx.shape, -1, np.int32)
    sub[idx >= 0] = inv
    pts = pkg.make_points(cloud[torch.from_numpy(ids).cuda()].cpu().numpy())
    ref_frames, _ = tgo.bake_frames(V, F)
    ref = hgo.bake_height(V, ref_frames, F, t, own, xyz, pts, sub, d2, res)
    ok = frames.tobytes() == ref_frames.tobytes()
    ok &= ref.reshape(-1)[t].tobytes() == hmap.reshape(-1)[t].tobytes()
    report["verified_texels"] = int(len(pick))
    report["verified"] = bool(ok and all(r["common_outputs_identical"] and r["device_piece_identical"]
                                         for r in report["shapes"]))
    print(f"oracle check ({len(pick)} texels of the height map): {'ok' if report['verified'] else 'MISMATCH'}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    tree.close()
    sys.exit(0 if report["verified"] else 1)


if __name__ == "__main__":
    main()
