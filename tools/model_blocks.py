"""CPU model of the block runs (pt_knn_span.cuh, build_blocks) for a bench workload: the host
restatement of the cloud generator (oracle/pt_synth_host.c, the same Philox stream), the lattice
and level counts of build_grid, the level grid_plan picks for k = 16, and per occupied cell the
records of its 3^3 block.  Reports the runs' size in records and bytes, the largest run, the
blocks the span kernel would not stage (a parent over the 16-bit counts or more than PAIR_CAP
records), the share of samples whose cell is empty, the candidates staged per sample, and the
parents a run touches (a lower bound of its span heads: the curve order can split a parent's
children into up to four spans).
usage: model_blocks.py [--workload cfg2] [--patch F]   (F < 1: the same-density patch
[0, F L]^2 of the domain with F^2 of the points, for the slabbed workloads)"""
import argparse
import math
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as ge  # noqa: E402
from oracle import pto  # noqa: E402

PAIR_CAP = 192
ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="cfg2")
ap.add_argument("--patch", type=float, default=1.0)
a = ap.parse_args()

synth = ge.package().synth
w = synth.CONFIGS[a.workload]
L = synth.L_DOMAIN
span_u = L * a.patch
n = int(round(w.n_points * a.patch * a.patch))
print(f"{a.workload}: {n} points over [0, {span_u:g}]^2 (patch {a.patch:g}), "
      f"{w.gu} x {w.gv} samples, k = {w.k}")

# the cloud, in chunks of the generator's counter space: coordinates as the index stores them
xyz = np.empty((n, 3), dtype=np.float32)
CH = 4_000_000
for c0 in range(0, n, CH):
    cn = min(CH, n - c0)
    p = pto.synth_cloud(cn, w.seed, kind=w.kind, u0=0.0, u1=span_u, v0=0.0, v1=span_u, sigma=w.sigma,
                        first_index=c0)
    xyz[c0:c0 + cn] = p["ver"]
    del p
lo = xyz.min(0).astype(np.float64)
ext = float((xyz.max(0).astype(np.float64) - lo).max())
inv21 = 2097152.0 / ext


def lattice(v):
    t = (v.astype(np.float64) - lo) * inv21
    return np.minimum(np.maximum(t, 0.0), 2097151.0).astype(np.int64)


c21 = lattice(xyz)
del xyz
# levels whose cells are contiguous runs of the sorted cloud (40 sorted key bits up to 2^27 points)
sort_bits = 40 if n <= (1 << 27) else 48
first_bit = 63 - 8 * ((sort_bits + 7) // 8)
max_level = min(16, (63 - first_bit) // 3)


def keys_at(level):
    s = 21 - level
    return (c21[:, 0] >> s) | ((c21[:, 1] >> s) << 21) | ((c21[:, 2] >> s) << 42)


fine_keys, fine_counts = np.unique(keys_at(max_level), return_counts=True)
cells = {0: 1}
for lv in range(max_level, 0, -1):
    s = max_level - lv
    k3 = ((fine_keys & 0x1fffff) >> s) | ((((fine_keys >> 21) & 0x1fffff) >> s) << 21) | \
         ((((fine_keys >> 42) & 0x1fffff) >> s) << 42)
    cells[lv] = len(np.unique(k3))
lf = max([lv for lv in range(1, max_level + 1) if n / cells[lv] >= 4.0] or [1])
tables = [lf - t for t in range(4) if lf - t >= 1]

# grid_plan(k = 16, r2 = inf) with the default lookup cost 8 and admission 100 %
best = None
for t, lv in enumerate(tables):
    occ = n / cells[lv]
    d = min(max(math.log2(max(cells[lv] / max(cells[lv - 1], 1), 1.0)), 1.0), 3.0)
    vd = 2.0 + (d - 1.0) * (math.pi - 2.0) if d <= 2.0 else math.pi + (d - 2.0) * (4.18879 - math.pi)
    rk = (16 / (vd * occ)) ** (1.0 / d)
    for rc in (1, 2):
        if rc < rk:
            continue
        cost = (2 * rc + 1) ** d * occ + 8 * (8 if rc == 1 else 27)
        if best is None or cost < best[0]:
            best = (cost, lv, rc, (2 * rc + 1) ** d * occ)
_, lv, rc, expect = best
print(f"tables at levels {tables}; k = 16 plans level {lv}, rc {rc}, ~{expect:.1f} candidates expected")
if rc != 1 or expect > 0.74 * PAIR_CAP:
    print("no block runs: the first attempt is not one the span kernel runs")
    sys.exit(0)

keys = keys_at(lv)
del c21
ukeys, counts = np.unique(keys, return_counts=True)
del keys
ncell = 1 << lv
cx, cy, cz = ukeys & 0x1fffff, (ukeys >> 21) & 0x1fffff, (ukeys >> 42) & 0x1fffff
# parents over the 16-bit counts of the cell tables
pkeys = (cx >> 1) | ((cy >> 1) << 21) | ((cz >> 1) << 42)
pu, pinv = np.unique(pkeys, return_inverse=True)
pcount = np.bincount(pinv, weights=counts)
dense_parent = pcount >= 0xffff


def block_of(qx, qy, qz):
    """(records, any dense parent in the block, parents touched) of the 3^3 blocks around cells q"""
    tot = np.zeros(len(qx), dtype=np.int64)
    dense = np.zeros(len(qx), dtype=bool)
    parents = set()
    par_ids = []
    for dx in (-1, 0, 1):
        for dy in (-1, 0, 1):
            for dz in (-1, 0, 1):
                x, y, z = qx + dx, qy + dy, qz + dz
                inside = (x >= 0) & (x < ncell) & (y >= 0) & (y < ncell) & (z >= 0) & (z < ncell)
                kk = np.where(inside, x | (y << 21) | (z << 42), -1)
                j = np.searchsorted(ukeys, kk)
                j = np.minimum(j, len(ukeys) - 1)
                hit = inside & (ukeys[j] == kk)
                tot += np.where(hit, counts[j], 0)
                dense |= hit & dense_parent[pinv[j]]
                par_ids.append(np.where(hit, pinv[j], -1))
    P = np.stack(par_ids, 1)
    P.sort(1)
    touched = ((P[:, 1:] != P[:, :-1]) & (P[:, 1:] >= 0)).sum(1) + (P[:, 0] >= 0)
    del parents
    return tot, dense, touched


tot, dense, touched = block_of(cx, cy, cz)
ok = ~dense & (tot <= PAIR_CAP)
rec = int(tot[ok].sum())
units_lb = rec + int(((touched[ok] + 1) // 2).sum())
tab_cap = (3 * len(ukeys) + 8) & ~3
print(f"occupied cells at level {lv}: {len(ukeys)}; mean points per cell {n / len(ukeys):.2f}")
print(f"runs: {rec} records = {rec / n:.2f} per point, {rec * 16 / 1e9:.3f} GB of records; "
      f"with heads (lower bound) and table {(units_lb * 16 + tab_cap * 16) / 1e9:.3f} GB")
print(f"largest stageable run {int(tot[ok].max())} records; blocks not staged: {int((~ok).sum())} "
      f"({int(dense.sum())} with a dense parent, {int(((tot > PAIR_CAP) & ~dense).sum())} over {PAIR_CAP})")
print(f"parents touched per run (heads >= this): mean {touched[ok].mean():.2f}, max {int(touched[ok].max())}")

s = pto.synth_samples(w.gu, w.gv, 0.0, span_u if a.patch < 1 else L, 0.0, span_u if a.patch < 1 else L,
                      center=w.center)["ver"]
sc = lattice(s) >> (21 - lv)
skeys = sc[:, 0] | (sc[:, 1] << 21) | (sc[:, 2] << 42)
j = np.minimum(np.searchsorted(ukeys, skeys), len(ukeys) - 1)
occupied = ukeys[j] == skeys
st, sd, _ = block_of(sc[:, 0], sc[:, 1], sc[:, 2])
stage = ~sd & (st <= PAIR_CAP) & (st >= 16)
print(f"samples: {len(s)}; cell empty: {int((~occupied).sum())} ({100.0 * (~occupied).mean():.3f} %)")
print(f"candidates per sample (staged blocks; 0 for blocks not staged): {np.where(stage, st, 0).mean():.1f}; "
      f"over staged samples only {st[stage].mean():.1f}")
print(f"samples staging from a run: {100.0 * (stage & occupied).mean():.2f} %; staged by spans but "
      f"without a run (empty cell): {int((stage & ~occupied).sum())}")
