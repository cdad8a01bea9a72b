"""CPU test of bench.py's driver contract on the arm that runs without a GPU: the reference arm
(`--impl reference`) prints ONE JSON line with the keys the driver reads (task brief, section 4)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")          # what torchrun exports to every rank
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                        "--steps", "1", "--warmup", "1", "--workload", "cfg1"],
                       capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "mesh-sample kNN transfers/sec"
    assert d["unit"] == "samples/s" and d["higher_is_better"] is True and d["value"] > 0
    for key in ("n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config"):
        assert key in d, key
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["sample"]
    # the arm must use every core it can even though OMP_NUM_THREADS=1 was exported
    assert cb["cores"] == len(os.sched_getaffinity(0))
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0
    assert cb["same_config"] is True and cb["points"] == d["config"]["points"]


def test_reference_arm_loads_no_cuda_library():
    """The reference arm must be self-contained: it generates the workload on the host
    (oracle/pt_synth_host.c) and never dlopens the product's CUDA libraries."""
    code = ("import sys, os; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '1', "
            "'--workload', 'cfg1']; sys.path.insert(0, %r); import runpy; runpy.run_path(%r, run_name='__main__'); "
            "maps = open('/proc/self/maps').read(); "
            "assert 'libpoints_transfer_b200' not in maps and 'libpt_synth_b200' not in maps, 'CUDA library loaded'; "
            "assert 'libpt_oracle' in maps" % (ROOT, os.path.join(ROOT, "bench.py")))
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]


def test_both_arms_emit_the_same_config():
    sys.path.insert(0, ROOT)
    import importlib
    bench = importlib.import_module("bench")
    import __graft_entry__ as ge
    pkg = ge.package()
    w = pkg.synth.CONFIGS["cfg2"]
    a = bench.make_config(w, w.n_points, w.gu, w.gv, w.k, 1)
    assert a["points"] == 50_000_000 and a["samples"] == 200_704 and a["k"] == 16
    assert bench.pick_workload(type("A", (), {"workload": "auto"})(), 1) == "cfg2"
    assert bench.pick_workload(type("A", (), {"workload": "auto"})(), 2) == "cfg3"
    assert bench.pick_workload(type("A", (), {"workload": "auto"})(), 4) == "cfg3"
    assert bench.pick_workload(type("A", (), {"workload": "auto"})(), 8) == "cfg4"


def test_traffic_record_belongs_to_the_shipped_kernel_source():
    """roofline.traffic in the bench line comes from one committed `ncu --set full` capture and is
    reported only while the kernel source it was captured on is unchanged (sha256): editing
    pt_knn_grid.cuh without a fresh capture must be noticed here, not as a silent `null`."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rec = bench.ncu_traffic("cfg2", 16, "knn_grid_pair_kernel")
    assert rec is not None and rec["dram_bytes"] > 0



def test_dump_outputs_writes_the_step_outputs(tmp_path):
    """--dump-outputs: every output of the step as float64 / float32 .npy in sample order; above
    the byte budget the same seeded rows on every call."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import importlib
    bench = importlib.import_module("bench")
    rng = np.random.default_rng(5)
    M, k = 1000, 4
    out = {"idx": torch.from_numpy(rng.integers(-1, 10**6, (M, k), dtype=np.int32)),
           "rgba": torch.from_numpy(rng.integers(0, 256, (M, 4), dtype=np.uint8)),
           "normal": torch.from_numpy(rng.standard_normal((M, 3)).astype(np.float32))}
    bench.dump_outputs(str(tmp_path / "all"), None, 1, 0, out, np.arange(M), M, k)
    got = {n: np.load(tmp_path / "all" / (n + ".npy")) for n in ("idx", "rgba", "normal", "sample_index")}
    assert got["idx"].dtype == np.float64 and got["rgba"].dtype == np.float32
    assert got["normal"].dtype == np.float32 and got["sample_index"].dtype == np.float64
    assert np.array_equal(got["sample_index"], np.arange(M))
    for n in ("idx", "rgba", "normal"):
        assert np.array_equal(got[n], out[n].numpy())
    # a share of the rows in another order (one rank of several), over a small budget
    bench.DUMP_BYTES, budget = 100 * (8 * k + 36), bench.DUMP_BYTES
    try:
        perm = rng.permutation(M)          # local row i holds global sample perm[i]
        bench.dump_outputs(str(tmp_path / "a"), None, 1, 0, out, np.arange(M), M, k)
        bench.dump_outputs(str(tmp_path / "b"), None, 1, 0,
                           {n: t[torch.from_numpy(perm)] for n, t in out.items()}, perm, M, k)
    finally:
        bench.DUMP_BYTES = budget
    a = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in got}
    b = {n: np.load(tmp_path / "b" / (n + ".npy")) for n in got}
    assert len(a["sample_index"]) == 100
    sel = a["sample_index"].astype(np.int64)
    for n in got:
        assert np.array_equal(a[n], b[n])
    assert np.array_equal(a["idx"], got["idx"][sel])
