"""Per-texel bake on one GPU (DESIGN.md section 8: "Per-texel bake", "Tangent-space bake", "Height
bake").

The cfg2 cloud (50 M points, generated on the device) and the g = 448 grid mesh on the noise-free
surface with UV = (x / L, y / L) and zero vertex normals (so every frame starts from the summed face
normals); bakes at 2048^2 with k = 32 and at 4096^2 with k = 16.  Per shape:
* wall time of pt_texture_bake (3 object-space maps), pt_texture_bake_ex (those plus the tangent
  maps and tangents) and pt_texture_bake_height (those plus both height maps), alternated in one
  process after a warm-up of each, maps copied to pageable host memory; the per-stage device ms of
  pt_bake_stats (median of --reps); texels/s; the outputs they share compared byte for byte;
* the kNN stage's samples/s next to DeviceTree.query on as many pt_synth_samples_device(center=1)
  samples;
* the bake's kernels by name from one torch.profiler pass over pt_texture_bake_height;
* device time (CUDA events, median of --reps) of the stages on the bake's own samples: the k-NN +
  blend through DeviceTree.query without and with the neighbour lists (idx) written, the frames
  stage (pt_bake_frames_device), the tangent composition + padding
  (pt_bake_compose_tangent_device), and the height stage (pt_bake_compose_height_device) for the
  float map alone and with the padded 16-bit map; each piece's output equals the bake's.
Then a 2-face quad covering a 16384^2 atlas (k = 1: the case that splits one face over many warps)
through pt_texture_bake.  At 2048^2 three checks against the CPU oracle (exit 1 on a mismatch):
the texel list and positions in full and the object-space maps of --verify-blend texels blended by
brute force over the whole cloud; the vertex frames and tangents in full and the tangent maps of
--verify texels; the heights of --verify texels, fed with the device's neighbour lists.  The card's
name and power limit are read in the same run.  The L2 is not flushed between passes; the cloud
alone (800 MB of records) is several times its size.

    python tools/prof_bake.py [--reps 5] [--verify 4096] [--verify-blend 256] [--out report.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ALL = ("bgra", "normal_bgra", "normal", "tangent_bgra", "tangent_normal", "tangents")


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--verify", type=int, default=4096, help="texels of the tangent and height maps checked")
    ap.add_argument("--verify-blend", type=int, default=256, help="texels blended by brute force and checked")
    ap.add_argument("--out", default=None, help="also write the report as JSON to this file")
    args = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    from oracle import pto, pto_bake
    pkg = ge.package()
    if not torch.cuda.is_available():
        sys.exit("prof_bake needs a CUDA device")
    torch.cuda.set_device(0)
    api, L = pkg.api, pkg.lib()
    ptr = api._np_ptr
    w = pkg.synth.CONFIGS["cfg2"]
    g, side = w.gu, pkg.synth.L_DOMAIN
    pos, attrs = pkg.synth.cloud_device(w.n_points, seed=w.seed)
    tree = pkg.DeviceTree(pos, attrs)
    V = pkg.synth.queries_to_host(pkg.synth.samples_device(g, g))
    V["U"], V["V"] = V["ver"][:, 0] / side, V["ver"][:, 1] / side
    F = pkg.synth.grid_faces(g, g)
    xyzuv = torch.from_numpy(np.c_[V["ver"], V["U"], V["V"]]).cuda()
    xyzuvn = torch.from_numpy(np.c_[V["ver"], V["U"], V["V"], V["normal"]]).cuda()
    faces = torch.from_numpy(F).cuda()
    cloud = pos[:, :3].to(torch.float64).contiguous()          # original order: DeviceTree ids are row numbers

    report = {"card": card(), "cloud": w.n_points, "mesh_vertices": int(len(V)), "mesh_faces": int(len(F)),
              "l2_flushed": False, "shapes": []}
    print("card (name, power limit):", report["card"])
    med = lambda xs: float(np.median(xs))                                       # noqa: E731
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, ms):
        """fn()'s result; its device ms appended to ms."""
        e0.record()
        r = fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
        return r

    def maps(res, n_vertices):
        return {"bgra": np.empty((res, res, 4), np.uint8), "normal_bgra": np.empty((res, res, 4), np.uint8),
                "normal": np.empty((res, res, 3), np.float32), "tangent_bgra": np.empty((res, res, 4), np.uint8),
                "tangent_normal": np.empty((res, res, 3), np.float32),
                "tangents": np.empty((n_vertices, 4), np.float32)}

    def alternate(fns):
        """Wall time and pt_bake_stats of each bake, alternated after a warm-up of each."""
        for fn in fns.values():
            fn()
        walls, stats = {n: [] for n in fns}, {n: [] for n in fns}
        for _ in range(args.reps):
            for name, fn in fns.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                st = fn()
                walls[name].append(time.perf_counter() - t0)
                stats[name].append(st)
        row = {}
        for name in fns:
            row[f"{name}_wall_ms"] = 1e3 * med(walls[name])
            row[f"{name}_stage_ms"] = [med([getattr(s, f) for s in stats[name]]) for f in ("raster_ms", "knn_ms", "pad_ms")]
            row[f"{name}_walls_ms"] = [1e3 * x for x in walls[name]]
        first = stats[next(iter(fns))]
        knn_ms = med([s.knn_ms for s in first])
        row.update(texels=int(first[0].texels), empty=int(first[0].empty),
                   texels_per_s=first[0].texels / (row[f"{next(iter(fns))}_wall_ms"] * 1e-3),
                   knn_samples_per_s=first[0].texels / (knn_ms * 1e-3))
        return row

    def query_rate(res, k, texels):
        """The same number of analytic texel-centre samples through DeviceTree.query."""
        q = pkg.synth.samples_device(res, max(1, texels // res), center=True)
        m = q.shape[0]
        rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
        nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
        tree.query(q, k, rgba=rgba, normal=nrm)
        qms = []
        for _ in range(args.reps):
            timed(lambda: tree.query(q, k, rgba=rgba, normal=nrm), qms)
        qms = med(qms)
        return {"query_samples": m, "query_ms": qms, "query_samples_per_s": m / (qms * 1e-3)}

    verify = None
    for res, k in ((2048, 32), (4096, 16)):
        out6, out8 = maps(res, len(V)), maps(res, len(V))
        out3 = {n: np.empty_like(out6[n]) for n in ALL[:3]}
        hmap, h16 = np.empty((res, res), np.float32), np.empty((res, res), np.uint16)
        o6 = api.BakeOutputs(*[out6[n].ctypes.data for n in ALL])
        o8 = api.BakeOutputs(*[out8[n].ctypes.data for n in ALL])
        hb = api.BakeHeight(hmap.ctypes.data, h16.ctypes.data)

        def bake():
            st = api.BakeStats()
            api._check(L.pt_texture_bake(tree.handle, ptr(V), len(V), ptr(F), len(F), k, -1.0, res, 1,
                                         ptr(out3["bgra"]), ptr(out3["normal_bgra"]), ptr(out3["normal"]),
                                         ctypes.byref(st)), "bake")
            return st

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

        row = {"shape": f"grid g={g}, {res}^2, k={k}", "resolution": res, "k": k,
               **alternate({"bake": bake, "bake_ex": bake_ex, "bake_height": bake_height})}
        row["object_maps_identical"] = all(out3[n].tobytes() == out6[n].tobytes() for n in out3)
        row["common_outputs_identical"] = all(out6[n].tobytes() == out8[n].tobytes() for n in ALL)
        row["height_texels"] = int(hb.texels)
        row["height_range"] = [hb.range_used[0], hb.range_used[1]]
        row.update(query_rate(res, k, row["texels"]))

        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            bake_height()
        row["profiler_kernels_ms"] = {ev.key[:90]: round(ev.device_time_total / 1e3, 4) for ev in prof.key_averages()
                                      if ev.device_type == torch.autograd.DeviceType.CUDA and ev.device_time_total > 0}

        # the stages on their own, on the bake's samples
        texels, xyz, owner = pkg.bake_samples_device(xyzuv, faces, res)
        xyz = xyz.contiguous()
        m = texels.numel()
        rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
        nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
        idx = torch.empty((m, k), dtype=torch.int32, device="cuda")
        tb = torch.empty((res, res, 4), dtype=torch.uint8, device="cuda")
        tn = torch.empty((res, res, 3), dtype=torch.float32, device="cuda")
        dh = torch.empty((res, res), dtype=torch.float32, device="cuda")
        dh16 = torch.empty((res, res), dtype=torch.uint16, device="cuda")
        ms = {n: [] for n in ("knn", "knn_idx", "frames", "tangent", "height", "height_u16")}
        for _ in range(args.reps + 1):
            timed(lambda: tree.query(xyz, k, rgba=rgba, normal=nrm), ms["knn"])
            timed(lambda: tree.query(xyz, k, rgba=rgba, normal=nrm, idx=idx), ms["knn_idx"])
            frames, tangents = timed(lambda: pkg.bake_frames_device(xyzuvn, faces), ms["frames"])
            timed(lambda: pkg.bake_compose_tangent_device(xyzuvn, frames, faces, texels, owner, rgba, nrm, res, pad=True,
                                                          tangent_bgra=tb, tangent_normal=tn), ms["tangent"])
            timed(lambda: pkg.bake_compose_height_device(xyzuvn, frames, faces, texels, owner, xyz, idx, k, cloud, res,
                                                         height=dh), ms["height"])
            timed(lambda: pkg.bake_compose_height_device(xyzuvn, frames, faces, texels, owner, xyz, idx, k, cloud, res,
                                                         height=dh, height_u16=dh16), ms["height_u16"])
        row.update({"knn_ms": med(ms["knn"][1:]), "knn_with_idx_ms": med(ms["knn_idx"][1:]),
                    "frames_ms": med(ms["frames"][1:]), "tangent_compose_pad_ms": med(ms["tangent"][1:]),
                    "height_float_ms": med(ms["height"][1:]), "height_float_u16_pad_ms": med(ms["height_u16"][1:])})
        row["device_pieces_identical"] = bool(
            np.array_equal(tb.cpu().numpy(), out6["tangent_bgra"]) and
            tn.cpu().numpy().tobytes() == out6["tangent_normal"].tobytes() and
            dh.cpu().numpy().tobytes() == hmap.tobytes() and np.array_equal(dh16.cpu().numpy(), h16))
        report["shapes"].append(row)
        print(json.dumps({n: v for n, v in row.items() if n != "profiler_kernels_ms"}))
        if res == 2048:
            rng = np.random.default_rng(20261020)
            pick = np.sort(rng.choice(m, size=min(args.verify, m), replace=False))
            d2 = torch.empty((m, k), dtype=torch.float64, device="cuda")
            tree.query(xyz, k, idx=idx, d2=d2)
            verify = {"res": res, "k": k, "out3": out3, "out6": out6, "hmap": hmap, "pick": pick,
                      "frames": frames.cpu().numpy(), "tangents": tangents.cpu().numpy(),
                      "texels": texels.cpu().numpy()[pick].astype(np.uint32), "owner": owner.cpu().numpy()[pick],
                      "xyz": xyz.cpu().numpy()[pick],
                      "idx": idx.cpu().numpy()[pick], "d2": d2.cpu().numpy()[pick]}
            del d2
        del texels, xyz, owner, rgba, nrm, idx, tb, tn, dh, dh16, frames, tangents
        torch.cuda.empty_cache()

    # one face split over many warps
    corners = np.array([[0, 0, 0], [side, 0, 0], [side, side, 0], [0, side, 0.0]])
    quad = pkg.make_points(corners, uv=corners[:, :2] / side)
    quad_faces = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    res, k = 16384, 1
    qbgra = np.empty((res, res, 4), np.uint8)

    def bake_quad():
        st = api.BakeStats()
        api._check(L.pt_texture_bake(tree.handle, ptr(quad), len(quad), ptr(quad_faces), len(quad_faces), k, -1.0,
                                     res, 1, ptr(qbgra), None, None, ctypes.byref(st)), "bake")
        return st

    row = {"shape": f"2-face quad, {res}^2, k={k}", "resolution": res, "k": k, **alternate({"bake": bake_quad})}
    row.update(query_rate(res, k, row["texels"]))
    report["shapes"].append(row)
    print(json.dumps(row))
    del qbgra

    res, k, pick = verify["res"], verify["k"], verify["pick"]
    # object-space maps: the texel list and positions in full (device piece vs oracle), the blend of
    # a seeded subset by brute force over the whole cloud
    texels, xyz = pkg.bake_texels_device(xyzuv, faces, res)
    ref_t, ref_xyz, ref_owner = pto_bake.bake_samples(V, F, res)
    ok_obj = np.array_equal(texels.cpu().numpy().astype(np.uint32), ref_t) and \
        np.array_equal(xyz.cpu().numpy().view(np.uint64), ref_xyz.view(np.uint64))
    bpick = np.random.default_rng(20261020).choice(len(ref_t), size=min(args.verify_blend, len(ref_t)), replace=False)
    P = pkg.synth.points_to_host(pos, attrs)
    idx, d2 = pto.knn_bruteforce(P, pto.make_points(ref_xyz[bpick]), k)
    rgba, nrm = pto.blend(P, idx, d2)
    del P
    t = ref_t[bpick]
    out3 = verify["out3"]
    ok_obj &= np.array_equal(out3["bgra"].reshape(-1, 4)[t][:, :3], rgba[:, 2::-1]) and \
        np.array_equal(out3["normal"].reshape(-1, 3)[t].view(np.uint32), nrm.view(np.uint32))
    ok_obj &= all(np.array_equal(out3["normal_bgra"].reshape(-1, 4)[t][:, c], [pto_bake.bake_encode(x) for x in nrm[:, 2 - c]])
                  for c in range(3))

    # tangent space: frames and tangents in full; the tangent maps of the subset from the bake's own
    # float normal map (= the blended normal m of each covered texel)
    out6 = verify["out6"]
    ref_frames, ref_tangents = pto_bake.bake_frames(V, F)
    ok_tan = verify["frames"].tobytes() == ref_frames.tobytes() and verify["tangents"].tobytes() == ref_tangents.tobytes()
    ok_tan &= out6["tangents"].tobytes() == ref_tangents.tobytes()
    t = ref_t[pick]
    m = out6["normal"].reshape(-1, 3)[t]
    rgba = np.zeros((len(t), 4), np.uint8)
    rgba[:, 3] = np.where(m.any(1), 255, 0)          # an empty neighbour list leaves the float map at 0
    _, tn = pto_bake.bake_compose_tangent(V, ref_frames, F, t, ref_owner[pick], rgba, m, res, pad=False)
    ok_tan &= tn.reshape(-1, 3)[t].tobytes() == out6["tangent_normal"].reshape(-1, 3)[t].tobytes()

    # heights of the subset, on the device's samples and neighbour lists: the listed points only, ids
    # renumbered
    t, idx = verify["texels"], verify["idx"]
    ids, inv = np.unique(idx[idx >= 0], return_inverse=True)
    sub = np.full(idx.shape, -1, np.int32)
    sub[idx >= 0] = inv
    pts = pkg.make_points(cloud[torch.from_numpy(ids).cuda()].cpu().numpy())
    ref = pto_bake.bake_height(V, ref_frames, F, t, verify["owner"], verify["xyz"], pts, sub, verify["d2"], res)
    ok_h = ref.reshape(-1)[t].tobytes() == verify["hmap"].reshape(-1)[t].tobytes()

    report["oracle"] = {"object_maps": bool(ok_obj), "tangent": bool(ok_tan), "height": bool(ok_h),
                        "blend_texels": int(len(bpick)), "tangent_height_texels": int(len(pick))}
    report["verified"] = bool(ok_obj and ok_tan and ok_h and all(
        r.get(c, True) for r in report["shapes"]
        for c in ("object_maps_identical", "common_outputs_identical", "device_pieces_identical")))
    print(f"oracle check at {res}^2: object maps ({len(bpick)} texels + full texel list) "
          f"{'ok' if ok_obj else 'MISMATCH'}; frames + tangents in full and {len(pick)} texels of the tangent "
          f"maps {'ok' if ok_tan else 'MISMATCH'}; {len(pick)} texels of the height map {'ok' if ok_h else 'MISMATCH'}")
    print("verified:", report["verified"])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    tree.close()
    sys.exit(0 if report["verified"] else 1)


if __name__ == "__main__":
    main()
