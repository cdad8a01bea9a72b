"""knn_grid_span_kernel against knn_grid_pair_kernel on one index of a workload (default cfg2):
option "grid_span" 1 and 0 alternated round by round in one process, the bench's step (one
DeviceTree.query with idx, rgba and normal out), a 256 MiB L2 flush before every step, CUDA events
around the query only.  Prints per-round ms per step, medians and min / max per arm, the card's
name, power limit and SM clock read in the same run, and checks that both arms give identical
outputs.  --trace DIR: instead, one torch.profiler run per arm, kernel names and device times.
usage: prof_span.py [--workload cfg2] [--rounds 6] [--steps 20] [--trace DIR]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import __graft_entry__ as ge

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="cfg2")
ap.add_argument("--rounds", type=int, default=6)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--trace", default=None)
a = ap.parse_args()

pkg = ge.package()
w = pkg.synth.CONFIGS[a.workload]
torch.cuda.set_device(0)
smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                      "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("card:", torch.cuda.get_device_name(0), "|", smi)
pos, attrs = pkg.synth.cloud_device(w.n_points, w.seed, kind=w.kind, sigma=w.sigma)
q = pkg.synth.samples_device(w.gu, w.gv, center=w.center)
m, k = q.shape[0], w.k
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
tree = pkg.DeviceTree(pos, attrs)
e1.record()
torch.cuda.synchronize()
print(f"{a.workload}: {w.n_points} points, {m} samples, k={k}; build {e0.elapsed_time(e1):.1f} ms")
idx = torch.empty((m, k), dtype=torch.int32, device="cuda")
rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")


def step():
    tree.query(q, k, radius=w.radius, idx=idx, rgba=rgba, normal=nrm)


outs = {}
for span in (0, 1):
    pkg.set_option("grid_span", span)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    outs[span] = (idx.clone(), rgba.clone(), nrm.clone(), pkg.get_option("grid_span_used"),
                  pkg.get_option("grid_pair_used"))
same = all(torch.equal(x, y) for x, y in zip(outs[0][:3], outs[1][:3]))
print(f"outputs identical: {same}; grid_span_used / grid_pair_used: span 0 -> {outs[0][3]} / {outs[0][4]}, "
      f"span 1 -> {outs[1][3]} / {outs[1][4]}")

if a.trace:
    from torch.profiler import profile, ProfilerActivity
    os.makedirs(a.trace, exist_ok=True)
    for span in (0, 1):
        pkg.set_option("grid_span", span)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                flush.zero_()
                step()
            torch.cuda.synchronize()
        table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=12)
        print(f"--- grid_span {span} ---\n{table}")
        open(os.path.join(a.trace, f"span{span}.txt"), "w").write(table)
    sys.exit(0 if same else 1)

times = {0: [], 1: []}
for r in range(a.rounds):
    for span in ((0, 1) if r % 2 == 0 else (1, 0)):
        pkg.set_option("grid_span", span)
        step()
        tot = 0.0
        for _ in range(a.steps):
            flush.zero_()
            e0.record()
            step()
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        times[span].append(tot / a.steps)
    print(f"round {r}: span0 {times[0][-1]:.4f} ms  span1 {times[1][-1]:.4f} ms")
for span in (0, 1):
    t = times[span]
    print(f"grid_span {span}: median {statistics.median(t):.4f} ms/step, min {min(t):.4f}, max {max(t):.4f}")
print(f"span1 / span0 (medians): {statistics.median(times[1]) / statistics.median(times[0]):.3f}")
print("SM clock after:", subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=clocks.sm,power.limit",
                                         "--format=csv,noheader"], capture_output=True, text=True).stdout.strip())
tree.close()
sys.exit(0 if same else 1)
