#!/usr/bin/env python
"""bench.py -- mesh-sample kNN transfers/sec on B200 (BASELINE.json metric).

One "step" = one pass of the hot path (exact k-NN + fused colour/normal blend of every mesh
sample against the resident spatial index) over one batch of synthetic samples.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload auto|cfgN] [--impl reference]

Workload (``--workload auto``): N = 1 -> cfg2 (50 M points, 200 704 samples, k = 16, the
configuration the metric is quoted on); N = 2, 4 -> cfg3 (300 M points in N x-slabs, 1 M samples,
k = 16, ghost zones); N = 8 -> cfg4 (1 B points in 8 slabs, 4.19 M texel samples, k = 32, no ghost
zone: halo exchange + K5 merge over NCCL every step).  For N > 1 the samples arrive in ONE
unsorted array, every rank holds an arbitrary share, and routing them to the owning slab is part
of the timed step (sharded.ShardedTransfer).

`value`   : samples/s with inputs resident in HBM (CUDA events around the step, L2 flushed
            between steps), whole job = all samples / max-over-ranks time.
`e2e`     : same metric through the host-buffer entry (N = 1: the C ABI pt_transfer; N > 1:
            ShardedTransfer.transfer_host) with pinned HOST buffers: H2D + step + D2H timed.
`roofline`: algorithmic bytes (32 + 36k per sample, SURVEY 8 M3) / step time vs the measured
            HBM copy peak (MEASURED_PEAKS.json), per GPU.
`cpu_baseline` / ``--impl reference``: the oracle's CGAL-style kd-tree (a port: the reference
            tool needs CGAL, absent here) on the host cores -- same workload, generated on the
            host by oracle/pt_synth_host.c, no CUDA library loaded.
"""
import argparse
import hashlib
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "mesh-sample kNN transfers/sec"
UNIT = "samples/s"
CPU_POINT_BUDGET = 64_000_000     # host arm: larger clouds are timed on a same-density patch
DUMP_BYTES = 64 << 20             # --dump-outputs: larger outputs are written as a seeded row sample


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="auto")
    ap.add_argument("--points", type=int, default=0, help="override total points")
    ap.add_argument("--grid", type=int, default=0, help="override sample grid side")
    ap.add_argument("--k", type=int, default=0)
    ap.add_argument("--variant", type=int, default=-1, help="knn kernel variant (tuning)")
    ap.add_argument("--order", type=int, default=-1, help="0 Morton, 1 Hilbert, 2 + kd refinement (tuning)")
    ap.add_argument("--sort", type=int, default=-1, help="1 hand-written radix sort, 0 CUB (tuning)")
    ap.add_argument("--halo", type=float, default=-1.0, help="N > 1: ghost-zone width (0 = none)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--profile-steps", type=int, default=0,
                    help="diagnosis: after the timed region run this many steps under torch.profiler and "
                         "print rank 0's kernel table to stderr (never part of a reported number)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (idx, rgba, normal) as DIR/<name>.npy "
                         "in float64 / float32, for comparing two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU arm's outputs")
    return args


def algorithmic_bytes_per_sample(k):
    # SURVEY.md 8 M3: 16 (query) + 16k (winner positions) + 16k (winner attrs) + 4k (idx out)
    # + 16 (blended rgba8 + normal out)
    return 32 + 36 * k


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload, k, kernel):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/r2_traffic.json); reported only while the kernel source it was captured on is
    unchanged (sha256 of the file), otherwise null -- never a stale constant."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        e = d.get(f"{workload}:k{k}:{kernel}")
        if not e:
            return None
        src = os.path.join(ROOT, e["source"])
        if hashlib.sha256(open(src, "rb").read()).hexdigest() != e["source_sha256"]:
            return None
        return e
    except Exception:
        return None


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md): NVML polled
    from a thread every ~0.5 ms (the region is tens of milliseconds, too short for nvidia-smi's
    loop mode, which is only the fallback)."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"),
               (0x4, "sw_power_cap"))

    def __init__(self, index, pci_bus_id=None):
        self.index, self.sm, self.mask, self.max_mhz = index, [], 0, None
        self.stop_flag, self.thread, self.proc, self.rows = False, None, None, []
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if pci_bus_id:
                try:
                    h = pynvml.nvmlDeviceGetHandleByPciBusId(pci_bus_id.encode())
                except Exception:
                    h = None
            self.handle = h or pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml = pynvml
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _poll(self):
        n, h = self.nvml, self.handle
        reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag:
            try:
                self.sm.append(int(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)))
                self.mask |= int(reasons(h))
            except Exception:
                pass
            time.sleep(0.0005)

    def start(self):
        if self.nvml:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml:
            self.stop_flag = True
            self.thread.join(timeout=1)
            sm = sorted(self.sm)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(name for bit, name in self.REASONS if self.mask & bit),
                    "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4)
                          if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": "nvidia-smi"}


def pick_workload(args, world):
    if args.workload != "auto":
        return args.workload
    return {1: "cfg2", 2: "cfg3", 4: "cfg3", 8: "cfg4"}.get(world, "cfg3")


def resolve_workload(args, pkg, world):
    name = pick_workload(args, world)
    w = pkg.synth.CONFIGS[name]
    n = args.points or w.n_points
    gu = args.grid or w.gu
    gv = args.grid or w.gv
    k = args.k or w.k
    return name, w, n, gu, gv, k


def make_config(w, n, gu, gv, k, world):
    """The workload both arms run -- identical keys and values on the GPU arm and on
    ``--impl reference``."""
    return {"workload": w.name, "points": n, "samples": gu * gv, "k": k, "radius": w.radius,
            "parallelism": f"slab x{world}",
            "l2": "flushed between steps (256 MiB write)"}


def pin_to_gpu_cores(local_rank, world):
    """Multi-GPU host side: keep each rank on its own cores next to its GPU (the ranks otherwise
    share the cores of one socket and the host copies of the end-to-end step fight)."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        cpus = open(f"/sys/bus/pci/devices/{bus}/local_cpulist").read().strip()
        ids = []
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids += list(range(int(a), int(b or a) + 1))
        ids = sorted(set(ids) & os.sched_getaffinity(0))
        if len(ids) >= 2 * world:
            per = len(ids) // world
            mine = ids[local_rank * per:(local_rank + 1) * per]
            os.sched_setaffinity(0, mine)
            return f"cores {mine[0]}-{mine[-1]} of local_cpulist {cpus}"
        return f"local_cpulist {cpus} (not split)"
    except Exception as e:          # no sysfs / no permission: stay where the launcher put us
        return f"unpinned ({type(e).__name__})"


# ---------------------------------------------------------------------------------------------
# CPU leg: the oracle's kd-tree port on the host cores (no CUDA library involved)
def cpu_leg(pto, w, n, gu, gv, k, steps, warmup):
    L = 1000.0
    frac = min(1.0, CPU_POINT_BUDGET / float(n))
    side = L * math.sqrt(frac)
    n_cpu = n if frac >= 1.0 else int(n * frac)
    gu_c = gu if frac >= 1.0 else max(2, int(round(gu * side / L)))
    gv_c = gv if frac >= 1.0 else max(2, int(round(gv * side / L)))
    t0 = time.perf_counter()
    P = pto.synth_cloud(n_cpu, w.seed, kind=w.kind, u1=side, v1=side, sigma=w.sigma)
    Q = pto.synth_samples(gu_c, gv_c, u1=side, v1=side, center=w.center)
    gen_s = time.perf_counter() - t0
    threads = pto.max_threads()
    t0 = time.perf_counter()
    tree = pto.KdTree(P)
    build_s = time.perf_counter() - t0
    r = -1.0 if w.radius is None else w.radius
    for _ in range(max(1, warmup)):
        tree.knn(Q[: max(1, len(Q) // 8)], k, radius=r, exact_ties=False, want_d2=False)
    times = []
    for _ in range(max(1, steps)):
        t0 = time.perf_counter()
        idx, d2 = tree.knn(Q, k, radius=r, exact_ties=False)
        pto.blend(P, idx, d2)
        times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    # SURVEY 8 M4: the single-thread rate (the reference is single-threaded unless built with
    # -DMULTI_THREADING=ON) and the reference's own query set -- a K-NN at each of the 3 corners
    # of every face (src/pointsTransfer.cpp:465-479)
    Q1 = Q[: max(1, len(Q) // 16)]
    t0 = time.perf_counter()
    tree.knn(Q1, k, radius=r, exact_ties=False, nthreads=1, want_d2=False)
    t1 = time.perf_counter() - t0
    import numpy as np
    jj, ii = np.meshgrid(np.arange(gv_c - 1), np.arange(gu_c - 1), indexing="ij")
    a = (jj * gu_c + ii).ravel()
    faces = np.stack([np.stack([a, a + 1, a + gu_c], 1), np.stack([a + 1, a + gu_c + 1, a + gu_c], 1)], 1)
    faces = faces.reshape(-1, 3).astype(np.int32)
    t0 = time.perf_counter()
    tree.reference_face_loop(Q, faces, k)
    tf = time.perf_counter() - t0
    tree.close()
    same = frac >= 1.0
    what = (f"the full workload: {n_cpu} points, {len(Q)} unique-vertex samples, k={k}" if same else
            f"a same-density {side:.0f} x {side:.0f} patch of the workload: {n_cpu} of {n} points, "
            f"{len(Q)} samples, k={k} (host memory / time bound)")
    return {"value": len(Q) / t, "unit": UNIT, "cores": threads, "kind": "port",
            "same_config": same, "points": n_cpu, "samples": len(Q),
            "single_thread_knn_value": len(Q1) / t1,
            "face_corner_queries_per_s": 3 * len(faces) / tf,
            "sample": what + "; CGAL-style kd-tree (sliding midpoint, bucket 10) + blend, OpenMP "
                             f"over samples; generated on the host in {gen_s:.1f} s, tree build "
                             f"{build_s:.1f} s, both excluded",
            "build_s": build_s, "ms_per_step": t * 1e3, "steps": max(1, steps)}


def run_reference_arm(args, pkg, world, rank):
    """The reference's own CPU implementation of the path (kd-tree k-NN per sample), all host
    threads: the CGAL-linked original cannot be built here, so this is the oracle port
    (cpu_baseline.kind = "port").  Rank 0 only; loads no CUDA library."""
    if rank != 0:
        return
    from oracle import pto
    name, w, n, gu, gv, k = resolve_workload(args, pkg, world)
    leg = cpu_leg(pto, w, n, gu, gv, k, steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": leg["value"], "unit": UNIT,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": leg["ms_per_step"], "higher_is_better": True,
        "scaling": "weak" if world == 1 else "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": make_config(w, n, gu, gv, k, world),
        "cpu_baseline": leg,
        "e2e": {"value": leg["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
def verify_by_ball(pkg, pto, torch, dist, world, rank, dev, own_pos, own_attrs, first_id, q, res, k,
                   radius, n_check, cuts=None):
    """Exact check of sampled results against the oracle by restriction: every true neighbour of
    a sample lies within its reported k-th distance (or the radius bound), so the oracle's brute
    force over the points of ALL slabs inside that ball must reproduce ids, colours and normals.
    own_pos / own_attrs: this rank's OWN slab points (ids first_id + i); q / res: this rank's
    samples and results."""
    import numpy as np
    m = q.shape[0]
    sel = torch.linspace(0, m - 1, min(n_check, m), device=dev).long()
    if cuts is not None and m:
        # half of the checked samples are the ones closest to a slab boundary: the samples whose
        # neighbours really come from two ranks (ghost zone / halo exchange + merge)
        inner = torch.tensor([c for c in cuts if math.isfinite(c)], dtype=torch.float64, device=dev)
        gap = (q[:, :1] - inner[None, :]).abs().min(dim=1).values
        near = torch.topk(gap, min(n_check // 2, m), largest=False).indices
        sel = torch.cat([sel[: sel.numel() - near.numel()], near])       # same count on every rank
    d_idx = res["idx"][sel]
    pos_k = None
    # k-th distance of each checked sample: recompute from the last valid neighbour -- its
    # coordinates may live on another rank, so use the ball radius carried by d2 if present
    if "d2" in res:
        kth = res["d2"][sel][:, k - 1]
    else:
        raise RuntimeError("verify_by_ball needs d2")
    if radius is not None:
        kth = torch.clamp(kth, max=float(radius) ** 2)
    balls = torch.cat([q[sel], kth[:, None]], dim=1)                  # [c, 4]
    if world > 1:
        allb = [torch.empty_like(balls) for _ in range(world)]
        dist.all_gather(allb, balls)
    else:
        allb = [balls]
    xyz = own_pos[:, :3].double()
    found = []                                                     # per source rank: list per ball
    for src in range(world):
        per = []
        for b in allb[src].tolist():
            if not math.isfinite(b[3]):
                per.append(None)
                continue
            dd = ((xyz - torch.tensor(b[:3], dtype=torch.float64, device=dev)) ** 2).sum(1)
            c = torch.nonzero(dd <= b[3] * (1 + 1e-9)).view(-1)
            per.append((c.cpu().numpy() + first_id, own_pos[c, :3].cpu().numpy(),
                        own_attrs[c].cpu().numpy()))
        found.append(per)
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, found)
        mine = [[gathered[r][rank][i] for r in range(world)] for i in range(len(sel))]
    else:
        mine = [[found[0][i]] for i in range(len(sel))]
    checked = 0
    for i, parts in enumerate(mine):
        if any(p is None for p in parts):
            continue                                               # short unbounded list: nothing to restrict
        ids = np.concatenate([p[0] for p in parts])
        xyzs = np.concatenate([p[1] for p in parts]).astype(np.float64)
        at = np.concatenate([p[2] for p in parts]).view(pkg.ATTR_DTYPE).reshape(-1)
        order = np.argsort(ids, kind="stable")
        ids, xyzs, at = ids[order], xyzs[order], at[order]
        sub = pkg.make_points(xyzs, normal=np.stack([at["nx"], at["ny"], at["nz"]], 1),
                              color=at["rgba"][:, :3].astype(np.int32))
        qp = pkg.make_points(q[sel[i]].cpu().numpy()[None])
        ridx, rd2 = pto.knn_bruteforce(sub, qp, k, radius=-1.0 if radius is None else radius)
        rrgba, rnrm = pto.blend(sub, ridx, rd2)
        want = np.where(ridx[0] >= 0, ids[np.maximum(ridx[0], 0)], -1)
        got = d_idx[i].cpu().numpy()
        if not np.array_equal(want, got):
            raise SystemExit(f"rank {rank}: verification failed (neighbour ids) at sample {int(sel[i])}")
        if not np.array_equal(rrgba[0], res["rgba"][sel[i]].cpu().numpy()):
            raise SystemExit(f"rank {rank}: verification failed (colour) at sample {int(sel[i])}")
        if not np.allclose(rnrm[0], res["normal"][sel[i]].cpu().numpy(), rtol=1e-5, atol=1e-7):
            raise SystemExit(f"rank {rank}: verification failed (normal) at sample {int(sel[i])}")
        checked += 1
    return checked


def dump_outputs(directory, dist, world, rank, out, rows, M, k):
    """Write the step's outputs as DIR/<name>.npy: idx (float64, -1 where a list is short),
    rgba and normal (float32), one row per sample, and sample_index (float64), the row of the
    one global sample array each output row belongs to.  Where M rows would exceed DUMP_BYTES, a
    fixed, seeded subset of rows is written.  rows: this rank's global sample rows (numpy)."""
    import numpy as np
    row_bytes = 8 * k + 4 * 4 + 4 * 3 + 8
    n_keep = min(M, DUMP_BYTES // row_bytes)
    keep = np.arange(M) if n_keep == M else \
        np.random.default_rng(20261020).choice(M, n_keep, replace=False)
    mask = np.isin(rows, keep)
    parts = [(rows[mask], {name: t.cpu().numpy()[mask] for name, t in out.items()})]
    if world > 1:
        mine, parts = parts[0], [None] * world
        dist.all_gather_object(parts, mine)
    if rank != 0:
        return
    ids = np.concatenate([p[0] for p in parts])
    order = np.argsort(ids)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "sample_index.npy"), ids[order].astype(np.float64))
    for name, dtype in (("idx", np.float64), ("rgba", np.float32), ("normal", np.float32)):
        a = np.concatenate([p[1][name] for p in parts])[order]
        np.save(os.path.join(directory, name + ".npy"), a.astype(dtype))


def timed_steps(pkg, torch, dist, world, dev, step, flush, steps, warmup):
    for _ in range(max(3, warmup)):
        flush.zero_()
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
           for _ in range(steps)]
    torch.cuda.synchronize()
    launches0 = pkg.kernel_launch_count()
    host_t0 = time.perf_counter()
    for a, b in evs:
        flush.zero_()
        a.record()
        step()
        b.record()
    host_issue_ms = (time.perf_counter() - host_t0) * 1e3 / steps
    launches = pkg.kernel_launch_count() - launches0       # this library's kernels, timed steps only
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    ms_per_rank = [dev_ms / steps]
    if world > 1:
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        ms_per_rank = [float(x.item()) / steps for x in allt]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / steps, ms_per_rank, host_issue_ms, launches


def main():
    args = parse_args()
    if args.impl == "reference":
        # torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm must use all the
        # host cores it can (rank 0 runs alone), so set it before any OpenMP runtime loads
        os.environ["OMP_NUM_THREADS"] = str(len(os.sched_getaffinity(0)))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    import __graft_entry__ as ge
    pkg = ge.package()
    if args.impl == "reference":
        return run_reference_arm(args, pkg, world, rank)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    pinned = None
    if world > 1:
        pinned = pin_to_gpu_cores(local_rank, world)
        dist.init_process_group("nccl", device_id=dev)
    if args.variant >= 0:
        pkg.set_option("knn_variant", args.variant)
    if args.order >= 0:
        pkg.set_option("order", args.order)
    if args.sort >= 0:
        pkg.set_option("sort", args.sort)

    name, w, n_total, gu, gv, k = resolve_workload(args, pkg, world)
    L = pkg.synth.L_DOMAIN
    M = gu * gv
    # ---- this rank's slab of the cloud (x-range [u0, u1), global ids first .. first + n) ------
    # Inner cuts sit 0.45 sample spacings off the regular L*r/N positions: with regular cuts no
    # k-NN ball of the mesh grids of cfg3 / cfg4 reaches a cut (the nearest sample column is half
    # a spacing away) and the ghost zones / the halo exchange would never carry a neighbour.
    cut_at = [0.0] + [r * L / world + 0.45 * L / gu for r in range(1, world)] + [L]
    counts_per_slab = [int(round(n_total * (cut_at[r + 1] - cut_at[r]) / L)) for r in range(world)]
    counts_per_slab[-1] = n_total - sum(counts_per_slab[:-1])
    first = sum(counts_per_slab[:rank])
    n = counts_per_slab[rank]
    u0, u1 = cut_at[rank], cut_at[rank + 1]
    pos, attrs = pkg.synth.cloud_device(n, w.seed, u0=u0, u1=u1, kind=w.kind, sigma=w.sigma,
                                        first_index=first, device=dev)
    own_pos, own_attrs = pos, attrs
    torch.cuda.synchronize()
    ids = own_box = halo = None
    if world > 1:
        ids = torch.arange(first, first + n, dtype=torch.int32, device=dev)
        own_box = pkg.dist.points_box(pos)
        if args.halo >= 0:
            halo = args.halo or None
        elif world >= 8:
            halo = None                  # pure slabs: halo exchange + K5 merge over NCCL every step
        else:
            rk = math.sqrt(k / (math.pi * (n_total / (L * L))))     # expected k-th neighbour distance
            halo = max(6.0 * rk, 2.0 * (w.radius or 0.0))
        if halo is not None:
            # slab + ghost zone: the other slabs' points within `halo` of this slab's box are
            # exchanged ONCE here, so the owner step needs no collective (DESIGN.md section 6)
            boxes = pkg.dist.gather_boxes(own_box)
            pos, attrs, ids = pkg.dist.exchange_ghosts(pos, attrs, ids, boxes, halo)
    # the timed build is a REBUILD (the first one also loads the module and maps the library's
    # private memory pool, which stays mapped in between: option pool_keep_mb)
    t0 = time.perf_counter()
    pkg.DeviceTree(pos, attrs, ids).close()     # first build (module load, pool mapping)
    first_build_wall_ms = (time.perf_counter() - t0) * 1e3
    # three rebuilds, the median reported (a rebuild that has to map fresh pool memory is 2-3x slower)
    rebuilds = []
    tree = None
    for _ in range(3 if world == 1 else 1):
        if tree is not None:
            tree.close()
        t0 = time.perf_counter()
        tree = pkg.DeviceTree(pos, attrs, ids)
        rebuilds.append((tree.info().build_ms, (time.perf_counter() - t0) * 1e3))
    build_ms, build_wall_ms = sorted(rebuilds)[len(rebuilds) // 2]
    info = tree.info()
    if pos is not own_pos:
        del pos, attrs                          # the index holds its own copy

    # ---- samples: one array in arbitrary order; every rank holds a share -----------------------
    q_all = pkg.synth.samples_device(gu, gv, center=w.center, device=dev)
    if world > 1:
        g = torch.Generator(device="cpu")
        g.manual_seed(20261018)
        perm = torch.randperm(M, generator=g).to(dev)
        q = q_all[perm[rank::world]].contiguous()
    else:
        q = q_all
    del q_all
    m = q.shape[0]
    out = {"idx": torch.empty((m, k), dtype=torch.int32, device=dev),
           "rgba": torch.empty((m, 4), dtype=torch.uint8, device=dev),
           "normal": torch.empty((m, 3), dtype=torch.float32, device=dev)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    st = None
    if world > 1:
        cuts = [-math.inf] + cut_at[1:-1] + [math.inf]
        st = pkg.sharded.ShardedTransfer(pkg.dist.CudaSlabEngine(tree), cuts, k, (M + world - 1) // world,
                                         own_box=own_box, halo=halo)

    def step():
        if st is None:
            tree.query(q, k, radius=w.radius, idx=out["idx"], rgba=out["rgba"], normal=out["normal"])
        else:
            st.transfer(q, out, radius=w.radius)

    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    except Exception:
        bus = None
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank, bus)
    sampler.start()
    ms_per_step, ms_per_rank, host_issue_ms, launches = timed_steps(pkg, torch, dist, world, dev, step, flush,
                                                                    args.steps, args.warmup)
    clocks = sampler.stop()
    if args.dump_outputs:
        import numpy as np
        rows = np.arange(M) if world == 1 else perm[rank::world].cpu().numpy()
        dump_outputs(args.dump_outputs, dist, world, rank, out, rows, M, k)
    if args.profile_steps > 0:
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            for _ in range(args.profile_steps):
                flush.zero_()
                step()
            torch.cuda.synchronize()
        if rank == 0:
            print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=40, max_name_column_width=70),
                  file=sys.stderr)
    if st is not None and not st.validate():
        raise SystemExit("a routing / halo block overflowed or a sample left the ghost zone during the "
                         "timed steps: results invalid")
    value = M / (ms_per_step * 1e-3)
    fallback = tree.fallback_counts()
    exchange = st.stats() if st is not None else None
    if exchange is not None:
        # whole-job totals (every rank only knows its own samples' crossings)
        rows = exchange.get("halo_rows_per_peer") or [0] * world
        tot = torch.tensor([exchange.get("crossing") or 0, exchange["routed_to_other_slabs"]] + list(rows),
                           dtype=torch.int64, device=dev)
        per_rank = [torch.empty_like(tot) for _ in range(world)]
        dist.all_gather(per_rank, tot)
        exchange["crossing_all_ranks"] = int(sum(int(t[0]) for t in per_rank))
        exchange["routed_to_other_slabs_all_ranks"] = int(sum(int(t[1]) for t in per_rank))
        if exchange.get("path") == "fast":
            exchange["halo_rows_rank_to_peer"] = [[int(v) for v in t[2:].tolist()] for t in per_rank]

    # ---- exact verification of sampled results (oracle by restriction; fails the run) ------------
    verified = None
    if not args.no_verify:
        from oracle import pto
        res = dict(out)
        d2 = torch.empty((m, k), dtype=torch.float64, device=dev)
        if st is None:
            tree.query(q, k, radius=w.radius, idx=res["idx"], d2=d2)
        else:
            # k-th distances of this rank's samples: recomputed from the returned ids is not
            # possible locally (neighbours may live on other ranks), so ask the owners once
            # more for d2 through the same routed path
            res["d2"] = d2
            st_d2 = _routed_d2(pkg, torch, dist, st, tree, q, k, w.radius, d2)
            assert st_d2
        res["d2"] = d2
        torch.cuda.synchronize()
        verified = verify_by_ball(pkg, pto, torch, dist, world, rank, dev, own_pos, own_attrs, first, q, res,
                                  k, w.radius, 200 if world == 1 else 96,
                                  cuts=None if st is None else cuts)

    # ---- e2e with pinned host buffers ------------------------------------------------------------
    out_idx = torch.empty((m, k), dtype=torch.int32, pin_memory=True)
    out_rgba = torch.empty((m, 4), dtype=torch.uint8, pin_memory=True)
    out_nrm = torch.empty((m, 3), dtype=torch.float32, pin_memory=True)
    if st is None:
        q_host = pkg.synth.queries_to_host(q, pinned=True)                  # [m,80] uint8 pinned
        qh_np = q_host.numpy().view(pkg.POINT_DTYPE).reshape(-1)
        o_np = {"idx": out_idx.numpy(), "rgba": out_rgba.numpy(), "normal": out_nrm.numpy()}

        def e2e_step():
            tree.transfer(qh_np, k, radius=w.radius, out=o_np)      # pt_transfer: host in, host out
        h2d = m * 80
    else:
        q_xyz_host = torch.empty((m, 3), dtype=torch.float64, pin_memory=True)
        q_xyz_host.copy_(q)
        o_t = {"idx": out_idx, "rgba": out_rgba, "normal": out_nrm}
        scratch = [None]

        def e2e_step():
            scratch[0] = st.transfer_host(q_xyz_host, o_t, radius=w.radius, scratch=scratch[0])
        h2d = m * 24
    for _ in range(3):
        e2e_step()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    e2e_s = (time.perf_counter() - t0) / args.steps
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if not st.validate():
            raise SystemExit("overflow during the end-to-end steps")
    e2e_s = float(t.item())
    info2 = tree.info()
    assert bool((out_idx.to(dev) == out["idx"]).all()), "host-buffer and device-buffer paths disagree"
    # the same call asking only for what the reference's transfer produces per sample (blended
    # colour + normal; the neighbour lists stay on the device): 80 % less to copy back
    blend_only = None
    if st is None:
        o_b = {"rgba": out_rgba.numpy(), "normal": out_nrm.numpy()}
        for _ in range(3):
            tree.transfer(qh_np, k, radius=w.radius, want_idx=False, out=o_b)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            tree.transfer(qh_np, k, radius=w.radius, want_idx=False, out=o_b)
        b_s = (time.perf_counter() - t0) / args.steps
        blend_only = {"value": M / b_s, "ms_per_step": b_s * 1e3, "d2h_bytes_per_step": m * 16}

    variant_used = pkg.get_option("knn_variant")
    kernel = {6: "knn_grid_kernel", 5: "knn_scan_kernel", 2: "knn_thread_kernel", 0: "knn_warp_kernel",
              -1: "knn_grid_kernel"}[variant_used]
    if kernel == "knn_grid_kernel" and pkg.get_option("grid_pair_used"):
        kernel = "knn_grid_pair_kernel"          # two samples per warp (pt_knn_grid.cuh)
    peak, peak_src = measured_peaks()
    alg_bytes = algorithmic_bytes_per_sample(k) * M / world          # per GPU and step
    achieved = alg_bytes / (ms_per_step * 1e-3) / 1e9
    tr = ncu_traffic(name, k, kernel) if world == 1 and not (args.points or args.grid) else None
    build_achieved = 36.0 * (int(info.n_points)) / (build_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": make_config(w, n_total, gu, gv, k, world),
        "details": {"points_this_gpu": n, "ghost_points_this_gpu": int(info.n_points) - n,
                    "samples_this_gpu": m, "halo": halo,
                    "coord_storage": "f32x4" if info.coord_mode == 1 else "f64",
                    "knn_variant": variant_used, "kernel": kernel, "order": pkg.get_option("order"),
                    "grid_handed_over_samples": fallback[1], "warp_fallback_samples": fallback[0],
                    "verified_samples_per_rank": verified, "cpu_pinning": pinned},
        "e2e": {"value": M / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": m * (4 * k + 4 + 12), "ms_per_step": e2e_s * 1e3,
                "kernel_ms": info2.last_query_ms if st is None else None,
                "without_neighbour_lists": blend_only},
        "gpu_launches": int(launches), "ms_per_rank": ms_per_rank,
        "host_issue_ms_per_step": host_issue_ms,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak,
                     "frac_of_nominal_8tbs": achieved / 8000.0,
                     "traffic": tr["dram_bytes"] if tr else None,
                     "traffic_gbs": tr["dram_bytes"] / (ms_per_step * 1e-3) / 1e9 if tr else None,
                     "traffic_source": tr["capture"] if tr else None,
                     "over_read_factor": tr.get("over_read_factor") if tr else None,
                     "l2_hit_pct": tr.get("l2_hit_pct") if tr else None,
                     "peak_source": peak_src, "per": "GPU",
                     "algorithmic_bytes_per_launch": alg_bytes, "kernel": kernel,
                     "kernel_ms": ms_per_step},
        "build": {"ms": build_ms, "wall_ms": build_wall_ms, "first_build_wall_ms": first_build_wall_ms,
                  "rebuilds_ms": [round(b[0], 3) for b in rebuilds],
                  "note": "median rebuild; the library's memory pool stays mapped in between (pool_keep_mb)",
                  "points_per_s": int(info.n_points) / (build_ms * 1e-3),
                  "roofline_frac": build_achieved / peak, "achieved_gbs": build_achieved,
                  "leaves": int(info.n_leaves), "index_bytes": int(info.device_bytes)},
    }
    if exchange is not None:
        line["exchange"] = dict(exchange, samples=M)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import pto
        line["cpu_baseline"] = cpu_leg(pto, w, n_total, gu, gv, k, steps=2, warmup=1)
    if rank == 0:
        print(json.dumps(line))
    tree.close()
    if world > 1:
        dist.destroy_process_group()


def _routed_d2(pkg, torch, dist, st, tree, q, k, radius, d2_out):
    """k-th-neighbour distances of this rank's (unsorted) samples for the verification: route the
    samples to their owners like a step, ask each owner for the squared distances of its FINAL
    lists (same slab path, want_d2), return them and scatter into sample order."""
    R, cap = st.R, st.cap
    send, sel, counts, overflow = pkg.dist.route_samples(q, st.cuts, cap)
    recv = torch.empty_like(send)
    dist.all_to_all_single(recv.view(R, -1), send.view(R, -1))
    rows = recv.view(R * cap, 4)
    res = st.slab.transfer(rows[:, :3].contiguous(), k, radius=radius, want_d2=True, validate=False,
                           r2pq=rows[:, 3].contiguous())
    back = torch.empty((R * cap, k), dtype=torch.float64, device=q.device)
    dist.all_to_all_single(back.view(R, -1), res["d2"].contiguous().view(R, -1))
    pkg.dist.scatter_rows(back, sel.view(-1), d2_out)
    return st.slab.validate()


if __name__ == "__main__":
    main()
