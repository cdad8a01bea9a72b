"""Normal orientation on one GPU (DESIGN.md section 8, "Normal orientation").

The cfg2 cloud (50 M points, generated on the device) as a DeviceTree, its analytic normals given
seeded random signs; pt_index_orient_normals at k = 8, 18 and 32: after one warm-up call per k, the
median of --reps calls of the device time of the k-NN self-queries (knn_ms) and of the rest (mst_ms:
edges, spanning forest, signs) from pt_orient_stats (CUDA events), points/s over their sum, the edge,
component and flip counts, and the fraction of points whose oriented normal agrees in sign with the
analytic one.  A separate torch.profiler pass per k splits mst_ms into the edge build (unit normals,
edge masks, scan, edge writes) and Boruvka + signs by kernel, and counts the Boruvka rounds (launches
of orient_min_w_kernel).  Peak memory is the growth of the library's memory pool from before the first
call to after the first call at each k: the pool keeps what it maps and k ascends, so each figure is
that k's peak, an upper bound (fragmentation, the outputs' device buffers included).
Same-run checks (exit 1 on a failure): two calls give identical outputs, and a --check-points cloud
of cfg2's density equals the CPU oracle bit for bit; the oracle path (exact k-NN on a kd-tree + the C
statement of tests/orient_oracle.c) is timed on it.  The card's name and power limit are read in the
same run.

    python tools/prof_orient.py [--reps 5] [--check-points 4000000] [--out report.json]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

EDGE_KERNELS = ("orient_unit_kernel", "orient_mask_kernel", "orient_edges_kernel", "DeviceScan")


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def random_signs(attrs, seed):
    import torch
    g = torch.Generator(device=attrs.device).manual_seed(seed)
    f = attrs.view(torch.float32)                 # pt_attr: nx ny nz, then 4 colour bytes
    s = torch.randint(0, 2, (f.shape[0], 1), generator=g, device=attrs.device, dtype=torch.int32) * 2 - 1
    f[:, :3] *= s.to(torch.float32)


def kernel_split(tree, k):
    """(edge-build ms, Boruvka + signs ms, rounds) of one call, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        tree.orient_normals(k)
        torch.cuda.synchronize()
    edge = rest = 0.0
    rounds = 0
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA or "orient" not in e.name and "DeviceScan" not in e.name \
                and "DeviceSelect" not in e.name:
            continue
        us = e.time_range.elapsed_us()
        if any(s in e.name for s in EDGE_KERNELS):
            edge += us
        else:
            rest += us
        rounds += "orient_min_w_kernel" in e.name
    return edge * 1e-3, rest * 1e-3, rounds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--check-points", type=int, default=4_000_000)
    ap.add_argument("--out", default=None, help="also write the report as JSON to this file")
    args = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    import orient_oracle
    from oracle import pto, pto_normals

    pkg = ge.package()
    assert torch.cuda.is_available(), "prof_orient.py needs a CUDA device"
    pkg.set_option("pool_keep_mb", 0)               # the pool starts empty, so its growth is the peak
    w = pkg.synth.CONFIGS["cfg2"]
    n = w.n_points
    report = {"card": card(), "workload": w.name, "n_points": n, "rows": []}
    print("card (name, power limit):", report["card"])
    pos, attrs = pkg.synth.cloud_device(n, seed=w.seed)
    analytic = attrs.view(torch.float32)[:, :3].cpu().numpy().astype(np.float64)
    random_signs(attrs, 20261021)
    tree = pkg.DeviceTree(pos, attrs)
    failed = False
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for k in (8, 18, 32):
        first = tree.orient_normals(k)                                    # warm-up
        peak = free0 - torch.cuda.mem_get_info()[0]
        knn, mst = [], []
        for _ in range(args.reps):
            r = tree.orient_normals(k)
            knn.append(r["stats"]["knn_ms"])
            mst.append(r["stats"]["mst_ms"])
        same = bool(np.array_equal(r["normal"].view(np.uint32), first["normal"].view(np.uint32)) and
                    np.array_equal(r["root"], first["root"]) and r["stats"]["edges"] == first["stats"]["edges"])
        failed |= not same
        edge_ms, boruvka_ms, rounds = kernel_split(tree, k)
        agree = (r["normal"].astype(np.float64) * analytic).sum(1) > 0
        row = {"k": k, "knn_ms": float(np.median(knn)), "mst_ms": float(np.median(mst)),
               "edge_kernels_ms": edge_ms, "boruvka_signs_kernels_ms": boruvka_ms, "rounds": rounds,
               **{key: r["stats"][key] for key in ("edges", "components", "oriented", "flipped")},
               "sign_agreement": float(agree.mean()), "disagree": int((~agree).sum()),
               "pool_growth_bytes": int(peak), "bytes_per_point": peak / n, "two_calls_identical": same,
               "knn_ms_all": knn, "mst_ms_all": mst}
        row["points_per_s"] = n / ((row["knn_ms"] + row["mst_ms"]) * 1e-3)
        report["rows"].append(row)
        print(json.dumps({a: b for a, b in row.items() if not a.endswith("_all")}))
    tree.close()
    del pos, attrs

    # a cloud of cfg2's density, small enough for the oracle's whole graph
    m = args.check_points
    side = pkg.synth.L_DOMAIN * np.sqrt(m / n)
    pos, attrs = pkg.synth.cloud_device(m, seed=w.seed + 1, u1=side, v1=side)
    random_signs(attrs, 7)
    P = pkg.synth.points_to_host(pos, attrs)
    xyz, nrm = np.ascontiguousarray(P["ver"]), np.ascontiguousarray(P["normal"]).astype(np.float32)
    tree = pkg.DeviceTree(pos, attrs)
    check = {"points": m, "threads": pto.max_threads()}
    for k in (18,):
        got = tree.orient_normals(k)
        t0 = time.perf_counter()
        idx = pto_normals.neighbours(xyz, k)
        t1 = time.perf_counter()
        ref = orient_oracle.orient(xyz, nrm, idx)
        t2 = time.perf_counter()
        ok = bool(np.array_equal(got["normal"].view(np.uint32), ref["normal"].view(np.uint32)) and
                  np.array_equal(got["root"], ref["root"]) and
                  all(got["stats"][key] == ref[key] for key in ("oriented", "flipped", "components", "edges")))
        failed |= not ok
        check[f"k{k}"] = {"verified": ok, "gpu_ms": got["stats"]["knn_ms"] + got["stats"]["mst_ms"],
                          "cpu_knn_s": t1 - t0, "cpu_orient_s": t2 - t1, "cpu_points_per_s": m / (t2 - t0)}
    tree.close()
    report["check"] = check
    print("check:", json.dumps(check))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    sys.exit(1 if failed else 0)


if __name__ == "__main__":
    main()
