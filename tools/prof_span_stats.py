"""Work counters and warp finish times of knn_grid_span_kernel, from the -DPT_STATS build
(`make -C 3d-reconstruction-from-point-cloud_b200 stats` first; never the product library).
One DeviceTree.query per workload, as the bench's step.  Prints per sample: parent look-ups, bulk
copies, copies that continue another copy of the same half in the sorted cloud (what merging spans
across parents would save), halves redone by the whole warp; and the spread of the persistent
warps' finish times against the kernel's duration (%globaltimer: first warp start to last warp
finish).  The stats build's times are those of a slower kernel (its counters are atomics): read
them as shares, not as the product's times.
usage: prof_span_stats.py [--workloads cfg2,cfg5]"""
import argparse
import os
import sys

os.environ["PT_LIB_NAME"] = "libpoints_transfer_b200_stats.so"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import __graft_entry__ as ge

ap = argparse.ArgumentParser()
ap.add_argument("--workloads", default="cfg2,cfg5")
a = ap.parse_args()

pkg = ge.package()
torch.cuda.set_device(0)
print("card:", torch.cuda.get_device_name(0))
for name in a.workloads.split(","):
    w = pkg.synth.CONFIGS[name]
    pos, attrs = pkg.synth.cloud_device(w.n_points, w.seed, kind=w.kind, sigma=w.sigma)
    q = pkg.synth.samples_device(w.gu, w.gv, center=w.center)
    tree = pkg.DeviceTree(pos, attrs)
    del pos, attrs
    m, k = q.shape[0], w.k
    idx = torch.empty((m, k), dtype=torch.int32, device="cuda")
    rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
    nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
    for _ in range(2):
        tree.query(q, k, radius=w.radius, idx=idx, rgba=rgba, normal=nrm)
    pkg.api.debug_stats(reset=True)
    tree.query(q, k, radius=w.radius, idx=idx, rgba=rgba, normal=nrm)
    st = pkg.api.debug_stats(reset=True)
    assert pkg.get_option("grid_span_used") == 1, "the span kernel did not run"
    ns = max(st["grid_attempts"], 1)                 # first attempts of the span kernel: one per sample
    warps = max(st["span_warps"], 1)
    start = (~st["span_first_start_ns_inv"]) & (2**64 - 1)
    dur = st["span_last_finish_ns"] - start
    mean_busy = st["span_warp_busy_ns_sum"] / warps
    print(f"{name}: {m} samples, k={k}; per sample: look-ups {st['span_lookups'] / ns:.3f}, "
          f"copies {st['span_copies'] / ns:.3f}, mergeable copies {st['span_copies_mergeable'] / ns:.3f} "
          f"(-> {(st['span_copies'] - st['span_copies_mergeable']) / ns:.3f} copies merged), "
          f"candidates {st['grid_candidates'] / ns:.1f}, redone halves {st['span_redo_halves']}, "
          f"handed over {tree.fallback_counts()[1]}")
    print(f"{name}: {st['span_warps']} warps; kernel {dur / 1e3:.1f} us (first start -> last finish); "
          f"warp busy time mean {mean_busy / 1e3:.1f} us, max {st['span_warp_busy_ns_max'] / 1e3:.1f} us; "
          f"last finish - mean finish {(dur - mean_busy) / 1e3:.1f} us ({100.0 * (dur - mean_busy) / max(dur, 1):.1f} % of the kernel)")
    tree.close()
    del q, idx, rgba, nrm
    torch.cuda.empty_cache()
