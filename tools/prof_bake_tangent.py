"""Tangent-space bake on one GPU (DESIGN.md section 8, "Tangent-space bake").

The cfg2 cloud (50 M points, generated on the device) and the g = 448 grid mesh of tools/prof_bake.py
(noise-free surface, UV = (x / L, y / L), zero vertex normals, so every frame starts from the summed
face normals); bakes at 2048^2 with k = 32 and at 4096^2 with k = 16.  Per shape:
* device time (CUDA events, median of --reps) of the frames stage (pt_bake_frames_device) and of
  the tangent composition + padding (pt_bake_compose_tangent_device) on the bake's own samples;
* wall time of pt_texture_bake (3 object-space maps) against pt_texture_bake_ex with all six
  outputs, alternated in one process after a warm-up of each, maps copied to pageable host memory;
* the outputs of pt_texture_bake and the object-space outputs of pt_texture_bake_ex compared byte
  for byte.
Then, at 2048^2, the vertex frames and tangents in full and the tangent maps of a seeded subset of
texels are checked against the CPU oracle (exit 1 on a mismatch).  The card's name and power limit
are read in the same run.  The L2 is not flushed; the cloud alone is several times its size.

    python tools/prof_bake_tangent.py [--reps 5] [--verify 4096] [--out report.json]
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
    ap.add_argument("--verify", type=int, default=4096, help="texels of the tangent maps checked against the oracle")
    ap.add_argument("--out", default=None, help="also write the report as JSON to this file")
    args = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    import bake_tangent_oracle as tgo
    from prof_bake import card
    pkg = ge.package()
    if not torch.cuda.is_available():
        sys.exit("prof_bake_tangent needs a CUDA device")
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

    report = {"card": card(), "cloud": w.n_points, "mesh_vertices": int(len(V)), "mesh_faces": int(len(F)),
              "l2_flushed": False, "shapes": []}
    print("card (name, power limit):", report["card"])
    verify = None
    for res, k in ((2048, 32), (4096, 16)):
        maps3 = [np.empty((res, res, 4), np.uint8), np.empty((res, res, 4), np.uint8), np.empty((res, res, 3), np.float32)]
        out6 = {"bgra": np.empty((res, res, 4), np.uint8), "normal_bgra": np.empty((res, res, 4), np.uint8),
                "normal": np.empty((res, res, 3), np.float32), "tangent_bgra": np.empty((res, res, 4), np.uint8),
                "tangent_normal": np.empty((res, res, 3), np.float32), "tangents": np.empty((len(V), 4), np.float32)}
        o6 = api.BakeOutputs(*[out6[n].ctypes.data for n in ALL])

        def bake3():
            st = api.BakeStats()
            api._check(L.pt_texture_bake(tree.handle, ptr(V), len(V), ptr(F), len(F), k, -1.0, res, 1,
                                         ptr(maps3[0]), ptr(maps3[1]), ptr(maps3[2]), ctypes.byref(st)), "bake")
            return st

        def bake6():
            st = api.BakeStats()
            api._check(L.pt_texture_bake_ex(tree.handle, ptr(V), len(V), ptr(F), len(F), k, -1.0, res, 1,
                                            ctypes.byref(o6), ctypes.byref(st)), "bake_ex")
            return st

        bake3(), bake6()                                                         # warm-up
        walls = {"bake": [], "bake_ex": []}
        stats = {"bake": [], "bake_ex": []}
        for _ in range(args.reps):
            for name, fn in (("bake", bake3), ("bake_ex", bake6)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                st = fn()
                walls[name].append(time.perf_counter() - t0)
                stats[name].append((st.raster_ms, st.knn_ms, st.pad_ms))
        same = all(a.tobytes() == out6[n].tobytes() for a, n in zip(maps3, ("bgra", "normal_bgra", "normal")))

        # the two tangent stages on their own, on the bake's samples
        texels, xyz, owner = pkg.bake_samples_device(xyzuv, faces, res)
        m = texels.numel()
        rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
        nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
        tree.query(xyz.contiguous(), k, rgba=rgba, normal=nrm)
        tb = torch.empty((res, res, 4), dtype=torch.uint8, device="cuda")
        tn = torch.empty((res, res, 3), dtype=torch.float32, device="cuda")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        frames_ms, compose_ms = [], []
        for _ in range(args.reps + 1):
            e0.record()
            frames, tangents = pkg.bake_frames_device(xyzuvn, faces)
            e1.record()
            torch.cuda.synchronize()
            frames_ms.append(e0.elapsed_time(e1))
            e0.record()
            pkg.bake_compose_tangent_device(xyzuvn, frames, faces, texels, owner, rgba, nrm, res, pad=True,
                                            tangent_bgra=tb, tangent_normal=tn)
            e1.record()
            torch.cuda.synchronize()
            compose_ms.append(e0.elapsed_time(e1))
        pieces_same = np.array_equal(tb.cpu().numpy(), out6["tangent_bgra"]) and \
            tn.cpu().numpy().tobytes() == out6["tangent_normal"].tobytes()
        med = lambda xs: float(np.median(xs))                                   # noqa: E731
        row = {"resolution": res, "k": k, "texels": int(m),
               "frames_ms": med(frames_ms[1:]), "tangent_compose_pad_ms": med(compose_ms[1:]),
               "bake_wall_ms": 1e3 * med(walls["bake"]), "bake_ex_wall_ms": 1e3 * med(walls["bake_ex"]),
               "bake_stage_ms": [med([s[j] for s in stats["bake"]]) for j in range(3)],
               "bake_ex_stage_ms": [med([s[j] for s in stats["bake_ex"]]) for j in range(3)],
               "bake_walls_ms": [1e3 * x for x in walls["bake"]], "bake_ex_walls_ms": [1e3 * x for x in walls["bake_ex"]],
               "object_maps_identical": bool(same), "device_pieces_identical": bool(pieces_same)}
        report["shapes"].append(row)
        print(json.dumps(row))
        if res == 2048:
            verify = (res, out6, frames.cpu().numpy(), tangents.cpu().numpy())
        del texels, xyz, owner, rgba, nrm, tb, tn, frames, tangents
        torch.cuda.empty_cache()

    # oracle check at 2048^2: frames and tangents in full; the tangent maps on a seeded subset, from
    # the bake's own float normal map (= the blended normal m of each covered texel)
    res, out6, frames, tangents = verify
    ref_frames, ref_tangents = tgo.bake_frames(V, F)
    ok = frames.tobytes() == ref_frames.tobytes() and tangents.tobytes() == ref_tangents.tobytes()
    ok &= out6["tangents"].tobytes() == ref_tangents.tobytes()
    ref_t, _, ref_owner = tgo.bake_samples(V, F, res)
    rng = np.random.default_rng(20261020)
    pick = np.sort(rng.choice(len(ref_t), size=min(args.verify, len(ref_t)), replace=False))
    t = ref_t[pick]
    m = out6["normal"].reshape(-1, 3)[t]
    rgba = np.zeros((len(t), 4), np.uint8)
    rgba[:, 3] = np.where(m.any(1), 255, 0)          # an empty neighbour list leaves the float map at 0
    tb, tn = tgo.bake_compose_tangent(V, ref_frames, F, t, ref_owner[pick], rgba, m, res, pad=False)
    ok &= tn.reshape(-1, 3)[t].tobytes() == out6["tangent_normal"].reshape(-1, 3)[t].tobytes()
    report["verified_texels"] = int(len(pick))
    report["verified"] = bool(ok and all(r["object_maps_identical"] and r["device_pieces_identical"]
                                         for r in report["shapes"]))
    print(f"oracle check (frames + tangents in full, {len(pick)} texels of the tangent maps): "
          f"{'ok' if report['verified'] else 'MISMATCH'}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    tree.close()
    sys.exit(0 if report["verified"] else 1)


if __name__ == "__main__":
    main()
