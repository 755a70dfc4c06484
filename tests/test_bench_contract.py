"""The bench contract, as far as it can be checked without a GPU: `bench.py --impl reference` (the reference's own CPU
path on the host cores, here on the 64x smaller --small matrices) prints exactly ONE JSON line on stdout with the keys
a reader of the result expects and times exactly --steps calls, and the GPU arm's helpers (keyed traffic table, the
row sample of --dump-outputs) behave.  On a GPU: what --dump-outputs writes is y of the timed SpMV."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--small", "--steps", "5", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    line = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "impl"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == "spmv_gflops_fp64_csr" and line["higher_is_better"] is True
    assert line["vs_baseline"] is None and line["dtype"] == "f64" and line["value"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"]
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["config"]["same_config"] is True and "workload" in line["config"]
    assert line["steps"] == 5 and "; 5 timed calls," in line["cpu_baseline"]["sample"]


def test_y_sample_is_a_fixed_seeded_sample_when_y_is_large(monkeypatch):
    import torch
    sys.path.insert(0, ROOT)
    import bench
    y = torch.arange(5000, dtype=torch.float64) * 0.5
    vals, rows = bench.y_sample(torch, y)                   # at most DUMP_ROWS rows: all of them
    assert np.array_equal(rows, np.arange(5000)) and np.array_equal(vals, y.numpy())
    monkeypatch.setattr(bench, "DUMP_ROWS", 700)
    vals, rows = bench.y_sample(torch, y)
    vals2, rows2 = bench.y_sample(torch, y)
    assert vals.dtype == rows.dtype == np.float64 and len(rows) == 700
    assert (np.diff(rows) > 0).all() and rows[0] >= 0 and rows[-1] < 5000 and rows[-1] - rows[0] > 2500
    assert np.array_equal(vals, rows * 0.5) and np.array_equal(rows, rows2) and np.array_equal(vals, vals2)


@pytest.mark.gpu
def test_dump_outputs_writes_y_of_the_timed_steps(tmp_path, libpath, port):
    """--dump-outputs: y of the last timed step, as float arrays under 64 MiB, equal to a host SpMV of the same seeded
    matrix and x, and identical for two runs with different step counts; the launches counted in the timed region
    grow with --steps."""
    sys.path.insert(0, ROOT)
    import bench
    from spmv_b200 import matrices as M
    A = bench.host_c2(small=True)
    x = M.make_x(A.n, M.SEED_C2, np.float64)
    y_ex = port.spmv_exact(A.rowptr, A.col, A.val, x)
    eps = np.finfo(np.float64).eps
    tol = 8 * eps * port.row_abs_sum(A.rowptr, A.col, A.val, x) + 0.5 * eps * np.abs(y_ex)
    ys, launches = [], []
    for steps in (1, 4):
        out = tmp_path / f"s{steps}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--small", "--steps", str(steps), "--warmup", "3",
                            "--extras", "", "--c5", "0", "--no-cpu", "--also", "", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout)
        assert line["steps"] == steps
        launches.append(line["gpu_launches"])
        y, rows = np.load(out / "y.npy"), np.load(out / "y_rows.npy")
        assert y.dtype == np.float64 and rows.dtype == np.float64 and len(y) == len(rows) == A.m == line["config"]["m_per_gpu"]
        assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
        idx = rows.astype(np.int64)
        assert (np.abs(y - y_ex[idx]) <= tol[idx]).all()
        ys.append(y)
    assert np.array_equal(ys[0].view(np.uint64), ys[1].view(np.uint64))
    assert launches[0] > 0 and launches[1] == 4 * launches[0]


def test_traffic_table_is_keyed_by_workload_and_kernel():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.traffic_for("c2", "csr_vector") == 7292376984
    assert bench.traffic_for("c1", "csr_vector") not in (None, bench.traffic_for("c2", "csr_vector"))
    assert bench.traffic_for("c4", "sell") > 5e9 and bench.traffic_for("c3", "csr5") > 2e9
    assert bench.traffic_for("c1", "no_such_kernel") is None
    table = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    assert all("/" in k for k in table if not k.startswith("_"))
