"""Normal orientation on a sharded cloud (DESIGN.md section 8, "Sharded normal orientation") against
the single index.

The cfg2 cloud (50 M points, generated on the device, its analytic normals with seeded random signs
as input normals) at k = 8, 18 and 32.  Arms: Tree.orient_normals on one index,
ShardedTree.orient_normals with 1, 2 and 4 slabs on device 0 and, where the box has them, on 2, 4
and 8 distinct GPUs.  Per k every arm runs once as a warm-up, and its normal, root and the four
counts are compared byte for byte with the single index's (exit 1 on a mismatch); the growth of the
library's memory pool over that first call is the arm's peak, per device (the pools are emptied
before it; device 0 is the home device).  Then --reps rounds run the arms alternated.  Reported per
arm: the medians of the call's wall time (outputs copied to pageable host memory) and of its stats
(the single index: knn_ms / mst_ms device times; the sharded cloud: host wall times of the slab
stage and of the rest), the rebuilds and the slabs' ghost points.  --big N also orients an N-point
cloud at k = 32 on 2 slabs of device 0 once, to show a cloud past the single index's n k <= 2^31 - 1
limit completes.  The card's name and power limit are read in the same run.

    python tools/prof_sharded_orient.py [--reps 3] [--big 0] [--out report.json]
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


def same(a, b):
    if a["normal"].view(np.uint32).tobytes() != b["normal"].view(np.uint32).tobytes():
        return "normal"
    if a["root"].tobytes() != b["root"].tobytes():
        return "root"
    for key in ("oriented", "flipped", "components", "edges"):
        if a["stats"][key] != b["stats"][key]:
            return key
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--big", type=int, default=0, help="points of the cloud past the single index's limit (0: none)")
    ap.add_argument("--out", default=None, help="also write the report as JSON to this file")
    args = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    pkg = ge.package()
    if not torch.cuda.is_available():
        sys.exit("prof_sharded_orient needs a CUDA device")
    torch.cuda.set_device(0)
    pkg.set_option("pool_keep_mb", 0)           # a build or a free hands the pool's spare memory back
    ndev = torch.cuda.device_count()
    w = pkg.synth.CONFIGS["cfg2"]
    pos, attrs = pkg.synth.cloud_device(w.n_points, seed=w.seed)
    P = pkg.synth.points_to_host(pos, attrs)
    del pos, attrs
    P["normal"] *= np.where(np.random.default_rng(w.seed).random(len(P)) < 0.5, -1.0, 1.0)[:, None]
    torch.cuda.empty_cache()
    tiny = pkg.make_points(np.random.default_rng(0).random((64, 3)))

    def empty_pool():
        free = []
        for d in range(ndev):
            pkg.Tree(tiny, device=d).close()    # the free trims the device's pool to nothing
            torch.cuda.synchronize(d)
            free.append(torch.cuda.mem_get_info(d)[0])
        return free

    t0 = time.perf_counter()
    arms = {"tree": pkg.Tree(P)}
    build_s = {"tree": time.perf_counter() - t0}
    layouts = [(f"slabs{r}_dev0", [0] * r) for r in (1, 2, 4)]
    layouts += [(f"gpus{r}", list(range(r))) for r in (2, 4, 8) if r <= ndev]
    for name, devices in layouts:
        t0 = time.perf_counter()
        arms[name] = pkg.ShardedTree(P, devices, k_hint=18)
        build_s[name] = time.perf_counter() - t0
    report = {"card": card(), "devices": ndev, "cloud": w.n_points, "build_s": build_s, "ks": []}
    print("card (name, power limit):", report["card"], flush=True)
    ok = True
    for k in (8, 18, 32):
        def run(name):
            t = time.perf_counter()
            out = arms[name].orient_normals(k)
            return out, (time.perf_counter() - t) * 1e3
        equal, growth = {}, {}
        ref = None
        for name in arms:
            free0 = empty_pool()
            out, _ = run(name)
            growth[name] = [int(f - torch.cuda.mem_get_info(d)[0]) for d, f in enumerate(free0)]
            if name == "tree":
                ref = out
                continue
            bad = same(out, ref)
            equal[name] = bad is None
            if bad is not None:
                ok = False
                print(f"MISMATCH {name} at k={k}: {bad}", flush=True)
        wall = {n: [] for n in arms}
        stats = {n: {"knn_ms": [], "mst_ms": []} for n in arms}
        for _ in range(args.reps):
            for name in arms:
                out, ms = run(name)
                wall[name].append(ms)
                for s in stats[name]:
                    stats[name][s].append(out["stats"][s])
        row_k = {"k": k, "counts": {c: ref["stats"][c] for c in ("oriented", "flipped", "components", "edges")},
                 "equal": equal, "arms": {}}
        for name in arms:
            row = {"wall_ms": float(np.median(wall[name]))}
            row.update({s: float(np.median(v)) for s, v in stats[name].items()})
            row["pool_growth_mb"] = [round(g / 2**20, 1) for g in growth[name]]
            if name != "tree":
                row["rebuilds"] = arms[name].info()["rebuilds"]
                row["slabs"] = arms[name].info()["n_slabs"]
                row["ghosts"] = sum(arms[name].info()["slab_ghosts"])
            row_k["arms"][name] = row
            print(f"k={k} {name:12s} " + " ".join(f"{a}={b:.2f}" if isinstance(b, float) else f"{a}={b}"
                                                  for a, b in row.items()), flush=True)
        report["ks"].append(row_k)
    report["verified"] = ok
    for t in arms.values():
        t.close()
    del arms
    if args.big:
        pos, attrs = pkg.synth.cloud_device(args.big, seed=w.seed + 1, u1=1400.0, v1=1400.0)
        B = pkg.synth.points_to_host(pos, attrs)
        del pos, attrs
        torch.cuda.empty_cache()
        free0 = empty_pool()
        with pkg.ShardedTree(B, [0, 0], k_hint=32) as st:
            t = time.perf_counter()
            out = st.orient_normals(32)
            big = {"points": args.big, "k": 32, "n_k": args.big * 32, "wall_ms": (time.perf_counter() - t) * 1e3,
                   "stats": out["stats"], "slab_records": [a + b for a, b in zip(st.info()["slab_points"],
                                                                                st.info()["slab_ghosts"])],
                   "rebuilds": st.info()["rebuilds"],
                   "pool_growth_mb": [round((f - torch.cuda.mem_get_info(d)[0]) / 2**20, 1) for d, f in enumerate(free0)]}
        print("big:", big, flush=True)
        report["big"] = big
    print(json.dumps(report, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
