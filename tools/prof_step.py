"""The bench's step with library options on and off: every combination of the named 0 / 1 options
(default: "chain_pdl") is one arm, the arms alternate round by round in one process, each step is
one DeviceTree.query with idx, rgba and normal out after a 256 MiB L2 flush, CUDA events around the
query only.  Prints per-round ms per step, medians and min / max per arm, the card's name, power
limit and SM clock read in the same run, and checks that every arm gives identical outputs.
--trace DIR: instead, one torch.profiler run per arm (kernel names and device times, so the kernel
and the gaps around it can be told apart), written to DIR.
usage: prof_step.py [--workload cfg2] [--options chain_pdl] [--rounds 6] [--steps 20] [--trace DIR]"""
import argparse
import itertools
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import __graft_entry__ as ge

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="cfg2")
ap.add_argument("--options", default="chain_pdl", help="comma-separated 0 / 1 library options")
ap.add_argument("--rounds", type=int, default=6)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--trace", default=None)
a = ap.parse_args()

pkg = ge.package()
w = pkg.synth.CONFIGS[a.workload]
names = [n for n in a.options.split(",") if n]
arms = list(itertools.product((1, 0), repeat=len(names)))
label = lambda arm: " ".join(f"{n}={v}" for n, v in zip(names, arm))
torch.cuda.set_device(0)
smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                      "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("card:", torch.cuda.get_device_name(0), "|", smi)
pos, attrs = pkg.synth.cloud_device(w.n_points, w.seed, kind=w.kind, sigma=w.sigma)
q = pkg.synth.samples_device(w.gu, w.gv, center=w.center)
m, k = q.shape[0], w.k
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
tree = pkg.DeviceTree(pos, attrs)
torch.cuda.synchronize()
idx = torch.empty((m, k), dtype=torch.int32, device="cuda")
rgba = torch.empty((m, 4), dtype=torch.uint8, device="cuda")
nrm = torch.empty((m, 3), dtype=torch.float32, device="cuda")
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
print(f"{a.workload}: {w.n_points} points, {m} samples, k={k}; arms: {[label(x) for x in arms]}")


def set_arm(arm):
    for n, v in zip(names, arm):
        pkg.set_option(n, v)


def step():
    tree.query(q, k, radius=w.radius, idx=idx, rgba=rgba, normal=nrm)


outs = {}
for arm in arms:
    set_arm(arm)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    outs[arm] = (idx.clone(), rgba.clone(), nrm.clone())
same = all(torch.equal(x, y) for arm in arms[1:] for x, y in zip(outs[arms[0]], outs[arm]))
rerun, handed = tree.fallback_counts()
print(f"outputs identical across arms: {same}; grid_span_used {pkg.get_option('grid_span_used')}; "
      f"samples handed over by the grid kernel {handed}, re-run by the warp kernel {rerun}")

if a.trace:
    from torch.profiler import profile, ProfilerActivity
    os.makedirs(a.trace, exist_ok=True)
    for arm in arms:
        set_arm(arm)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                flush.zero_()
                step()
            torch.cuda.synchronize()
        table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=14, max_name_column_width=60)
        print(f"--- {label(arm)} ---\n{table}")
        open(os.path.join(a.trace, "step_" + "_".join(f"{n}{v}" for n, v in zip(names, arm)) + ".txt"), "w").write(table)
        prof.export_chrome_trace(os.path.join(a.trace, "step_" + "_".join(f"{n}{v}" for n, v in zip(names, arm)) + ".json"))
    tree.close()
    sys.exit(0 if same else 1)

times = {arm: [] for arm in arms}
for r in range(a.rounds):
    for arm in (arms if r % 2 == 0 else arms[::-1]):
        set_arm(arm)
        step()
        tot = 0.0
        for _ in range(a.steps):
            flush.zero_()
            e0.record()
            step()
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        times[arm].append(tot / a.steps)
    print(f"round {r}: " + "  ".join(f"[{label(arm)}] {times[arm][-1]:.4f} ms" for arm in arms))
for arm in arms:
    t = times[arm]
    print(f"{label(arm)}: median {statistics.median(t):.4f} ms/step, min {min(t):.4f}, max {max(t):.4f}")
base = statistics.median(times[arms[-1]])
for arm in arms[:-1]:
    print(f"[{label(arm)}] / [{label(arms[-1])}] (medians): {statistics.median(times[arm]) / base:.3f}")
print("SM clock after:", subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=clocks.sm,power.limit",
                                         "--format=csv,noheader"], capture_output=True, text=True).stdout.strip())
set_arm(arms[0])
tree.close()
sys.exit(0 if same else 1)
