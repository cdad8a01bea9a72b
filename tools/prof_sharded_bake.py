"""Per-texel bake of a sharded cloud (DESIGN.md section 8, "Sharded bake") against the single index.

The cfg2 cloud (50 M points) and the g = 448 grid mesh of tools/prof_bake.py, all eight outputs
(object-space, tangent-space and height maps, vertex tangents), at 2048^2 with k = 32 and at 4096^2
with k = 16.  Arms: Tree.bake on one index, ShardedTree.bake with 1, 2 and 4 slabs on device 0 (the
cost of the routing and the copies alone) and, where the box has them, on 2, 4 and 8 distinct GPUs.
Per shape every arm runs once as a warm-up and its outputs are compared byte for byte with the
single index's (exit 1 on a mismatch); then --reps rounds run the arms alternated.  Reported per arm:
the median wall time of the call (maps copied to pageable host memory) and the medians of its
stats (raster_ms and pad_ms: device time on the home device; knn_ms: for the sharded arms the host
wall time of routing, copies, the slabs' queries, checks and heights, and the scatter back), and the
rebuilds.  The card's name and power limit are read in the same run.

    python tools/prof_sharded_bake.py [--reps 5] [--out report.json]
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

WANT = ("bgra", "normal_bgra", "normal", "tangent_bgra", "tangent_normal", "tangents", "height", "height_u16")


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def same(a, b):
    for key in WANT:
        if a[key].tobytes() != b[key].tobytes():
            return key
    if np.array(a["height_range"]).tobytes() != np.array(b["height_range"]).tobytes():
        return "height_range"
    for s in ("texels", "empty", "height_texels"):
        if a["stats"][s] != b["stats"][s]:
            return s
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the report as JSON to this file")
    args = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    pkg = ge.package()
    if not torch.cuda.is_available():
        sys.exit("prof_sharded_bake needs a CUDA device")
    torch.cuda.set_device(0)
    ndev = torch.cuda.device_count()
    w = pkg.synth.CONFIGS["cfg2"]
    g, side = w.gu, pkg.synth.L_DOMAIN
    pos, attrs = pkg.synth.cloud_device(w.n_points, seed=w.seed)
    P = pkg.synth.points_to_host(pos, attrs)
    del pos, attrs
    V = pkg.synth.queries_to_host(pkg.synth.samples_device(g, g))
    V["U"], V["V"] = V["ver"][:, 0] / side, V["ver"][:, 1] / side
    F = pkg.synth.grid_faces(g, g)
    torch.cuda.empty_cache()

    t0 = time.perf_counter()
    arms = {"tree": pkg.Tree(P)}
    build_s = {"tree": time.perf_counter() - t0}
    layouts = [(f"slabs{r}_dev0", [0] * r) for r in (1, 2, 4)]
    layouts += [(f"gpus{r}", list(range(r))) for r in (2, 4, 8) if r <= ndev]
    for name, devices in layouts:
        t0 = time.perf_counter()
        arms[name] = pkg.ShardedTree(P, devices, k_hint=20)
        build_s[name] = time.perf_counter() - t0
    report = {"card": card(), "devices": ndev, "cloud": w.n_points, "mesh_vertices": int(len(V)),
              "mesh_faces": int(len(F)), "build_s": build_s, "shapes": []}
    ok = True
    for res, k in ((2048, 32), (4096, 16)):
        def run(name):
            t = time.perf_counter()
            out = arms[name].bake(V, F, k=k, resolution=res, want=WANT)
            return out, (time.perf_counter() - t) * 1e3
        ref, _ = run("tree")
        equal = {}
        for name in arms:
            if name != "tree":
                bad = same(run(name)[0], ref)
                equal[name] = bad is None
                if bad is not None:
                    ok = False
                    print(f"MISMATCH {name} at {res}^2: {bad}", flush=True)
        wall = {n: [] for n in arms}
        stats = {n: {"raster_ms": [], "knn_ms": [], "pad_ms": []} for n in arms}
        for _ in range(args.reps):
            for name in arms:
                out, ms = run(name)
                wall[name].append(ms)
                for s in stats[name]:
                    stats[name][s].append(out["stats"][s])
        shape = {"res": res, "k": k, "texels": ref["stats"]["texels"], "equal": equal, "arms": {}}
        for name in arms:
            row = {"wall_ms": float(np.median(wall[name]))}
            row.update({s: float(np.median(v)) for s, v in stats[name].items()})
            if name != "tree":
                row["rebuilds"] = arms[name].info()["rebuilds"]
                row["slabs"] = arms[name].info()["n_slabs"]
            shape["arms"][name] = row
            print(f"{res}^2 k={k} {name:12s} " + " ".join(f"{a}={b:.2f}" if isinstance(b, float) else f"{a}={b}"
                                                            for a, b in row.items()), flush=True)
        report["shapes"].append(shape)
    report["verified"] = ok
    for t in arms.values():
        t.close()
    print(json.dumps(report, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
