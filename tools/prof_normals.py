"""Normal estimation on one GPU (DESIGN.md section 8, "Normal estimation").

The cfg2 cloud (50 M points, generated on the device) as a DeviceTree; pt_index_estimate_normals at
k = 8, 16 and 32: after one warm-up call per k, the median of --reps calls of the device time of the
k-NN self-queries (knn_ms, the row kernel included) and of the PCA kernel (pca_ms) from
pt_normals_stats (CUDA events), points/s over their sum, and the device piece
(pt_estimate_normals_device) timed with CUDA events around it.  The outputs of --verify seeded points
are compared bit for bit with the CPU oracle (exit 1 on a mismatch), and the oracle path (exact k-NN
on a kd-tree + the C statement, all host cores) is timed over --cpu-rows seeded points.  The card's
name and power limit are read in the same run.  The L2 is not flushed between calls; the cloud alone
(800 MB of records) is several times its size.

    python tools/prof_normals.py [--reps 5] [--verify 4096] [--cpu-rows 200000] [--out report.json]
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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--verify", type=int, default=4096, help="points checked bit for bit against the oracle")
    ap.add_argument("--cpu-rows", type=int, default=200_000, help="points of the timed oracle path")
    ap.add_argument("--out", default=None, help="also write the report as JSON to this file")
    args = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    from oracle import pto, pto_normals

    pkg = ge.package()
    assert torch.cuda.is_available(), "prof_normals.py needs a CUDA device"
    w = pkg.synth.CONFIGS["cfg2"]
    n = w.n_points
    report = {"card": card(), "workload": w.name, "n_points": n, "rows": []}
    print("card (name, power limit):", report["card"])
    pos, attrs = pkg.synth.cloud_device(n, seed=w.seed)
    tree = pkg.DeviceTree(pos, attrs)
    normal = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    variation = torch.empty(n, dtype=torch.float32, device="cuda")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    P = pkg.synth.points_to_host(pos, attrs)
    xyz, nrm = np.ascontiguousarray(P["ver"]), P["normal"].astype(np.float32)
    rng = np.random.default_rng(20261021)
    check_rows = np.sort(rng.choice(n, args.verify, replace=False))
    cpu_rows = np.sort(rng.choice(n, args.cpu_rows, replace=False))
    t0 = time.perf_counter()
    kd = pto.KdTree(P)
    kd_s = time.perf_counter() - t0
    report["cpu"] = {"threads": pto.max_threads(), "kdtree_build_s": kd_s, "rows": args.cpu_rows, "by_k": {}}
    failed = False
    for k in (8, 16, 32):
        pkg.Tree.estimate_normals(tree, k)                               # warm-up
        knn, pca, dev = [], [], []
        for _ in range(args.reps):
            r = pkg.Tree.estimate_normals(tree, k)
            knn.append(r["stats"]["knn_ms"])
            pca.append(r["stats"]["pca_ms"])
            ev[0].record()
            tree.estimate_normals(k, normal=normal, variation=variation)
            ev[1].record()
            torch.cuda.synchronize()
            dev.append(ev[0].elapsed_time(ev[1]))
        row = {"k": k, "knn_ms": float(np.median(knn)), "pca_ms": float(np.median(pca)),
               "device_piece_ms": float(np.median(dev)), "estimated": r["stats"]["estimated"],
               "knn_ms_all": knn, "pca_ms_all": pca}
        row["points_per_s"] = n / ((row["knn_ms"] + row["pca_ms"]) * 1e-3)
        # bit-exact check of a seeded subset (host call's result and the device piece's)
        idx, _ = kd.knn(pto.make_points(P["ver"][check_rows]), k, exact_ties=True, want_d2=False)
        ref_n, ref_v, _ = pto_normals.estimate(xyz, nrm, idx, rows=check_rows)
        dn, dv = normal.cpu().numpy(), variation.cpu().numpy()
        row["verified"] = bool(np.array_equal(r["normal"][check_rows].view(np.uint32), ref_n.view(np.uint32)) and
                               np.array_equal(r["variation"][check_rows].view(np.uint32), ref_v.view(np.uint32)) and
                               np.array_equal(dn.view(np.uint32), r["normal"].view(np.uint32)) and
                               np.array_equal(dv.view(np.uint32), r["variation"].view(np.uint32)))
        failed |= not row["verified"]
        ref = P["normal"] / np.linalg.norm(P["normal"], axis=1)[:, None]
        ang = np.degrees(np.arccos(np.clip(np.abs((r["normal"].astype(np.float64) * ref).sum(1)), 0, 1)))
        row["angle_deg_mean"], row["angle_deg_p99"] = float(ang.mean()), float(np.percentile(ang, 99))
        # the oracle path on all host cores
        t0 = time.perf_counter()
        idx, _ = kd.knn(pto.make_points(P["ver"][cpu_rows]), k, exact_ties=True, want_d2=False)
        t1 = time.perf_counter()
        pto_normals.estimate(xyz, nrm, idx, rows=cpu_rows)
        t2 = time.perf_counter()
        report["cpu"]["by_k"][k] = {"knn_s": t1 - t0, "pca_s": t2 - t1, "points_per_s": args.cpu_rows / (t2 - t0)}
        report["rows"].append(row)
        print(json.dumps({a: b for a, b in row.items() if not a.endswith("_all")}), json.dumps(report["cpu"]["by_k"][k]))
    print("cpu:", json.dumps({a: b for a, b in report["cpu"].items() if a != "by_k"}))
    tree.close()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    sys.exit(1 if failed else 0)


if __name__ == "__main__":
    main()
