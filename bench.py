#!/usr/bin/env python
"""bench.py -- SpMV GFLOP/s + effective HBM GB/s on the BASELINE.json configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2] [--method parallel]
    python bench.py --impl reference ...      # the reference's own CPU path on the host cores

N = 1: a "step" is one spmv() over BASELINE.json configs[1] (uniform-random 2^24 x 2^24, 32 nnz/row, fp64: "C2"),
everything resident in HBM.  The same line carries sub-records for the other configurations (`extras`: C1 flushed and
L2-warm, C3, C4, the C5 shard) and, with --c5, the full C5 power-method iteration on one GPU (the strong-scaling
baseline of the multi-GPU record).

N > 1 (strong scaling, `"scaling": "strong"`): a step is one iteration x <- A x of the power method on the SAME square
C2 matrix, row-sharded over the N ranks by equal nnz (the reference's splitter), INCLUDING the y -> x exchange.  Three
loops run on the same handles (spmv_b200/multigpu.py) and must agree bit for bit: the plain loop (SpMV, then
ncclAllGather, timed separately -- the reported baseline), the pipelined loop over NCCL send/recv, and the pipelined
loop whose exchange runs on the copy engines (peer DMA + stream flags) under the band-staged SpMV of the next
iteration; `value` comes from the fastest of them, `power_method` holds all their numbers (SpMV alone, exchange alone,
exposed exchange).  `c5` holds the same record for BASELINE.json configs[4] (uniform-random 2^28 x 2^28, 16 nnz/row,
50 iterations) at this N.  Every multi-GPU leg runs under a watchdog (see Watchdog).

Other workloads (`--workload c1|c3|c4|c5shard`) time the remaining configurations as the primary one (single GPU).
`--also` names further methods timed after the primary one; their numbers land in "methods".
`--dump-outputs DIR` (N = 1) writes y of the primary method's last timed step to DIR (see --help); the matrix and x
come from fixed seeds, so two builds run with the same arguments can be compared output for output.

One JSON line on stdout (rank 0).  `value` = whole-job GFLOP/s with everything resident in HBM; `e2e` = the same
metric with HOST x / y (pinned), H2D + kernels + D2H inside the timed region (N = 1: one spmv() call of the C-ABI with
host pointers; N > 1: every rank uploads only ITS slice of x, the slices are all-gathered over NVLink, every rank
returns its slice of y); `roofline` = algorithmic bytes (B_min, BASELINE.md) / kernel time vs the measured HBM copy
peak; `cpu_baseline` = the compiled reference's best method on the host cores, on the FULL C2 matrix.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # no __pycache__ in the tree: it may be read-only

METHODS = {"serial": 0, "parallel": 1, "balanced": 2, "balanced2": 3, "balanced_yid": 4, "sell": 5, "csr5": 6}
REF_METHOD_NAMES = ["Method_Serial", "Method_Parallel", "Method_Balanced", "Method_Balanced2", "Method_BalancedYid",
                    "Method_SellCSigma", "Method_Csr5Spmv"]
LOG2_ROWS_C2 = 24
SAMPLE_LOG2_ROWS = 21  # method selection on the CPU: the first 2^21 rows of C2, full-length x (the timing is on ALL rows)
LOG2_ROWS_C5 = 28


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout.  Native libraries write to file descriptor 1 behind Python's back
# (NCCL prints its version banner there), so descriptor 1 is pointed at stderr for the whole run and the result
# line goes to a private duplicate of the original stdout.
RESULT = None


def claim_stdout():
    global RESULT
    if RESULT is None:
        sys.stdout.flush()
        RESULT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = RESULT if RESULT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


# A hung collective or a lost flag on one rank would otherwise block every rank until the driver's own limit: each
# multi-GPU leg runs under a deadline.  When it passes, rank 0 prints the line built from what HAS been measured (the
# plain loop comes first) with a "watchdog" note, and every rank leaves the process.
PROGRESS = {}


class Watchdog:
    def __init__(self, rank):
        self.rank, self.deadline, self.what, self.fallback = rank, None, "", None
        t = threading.Thread(target=self._run, daemon=True)
        t.start()

    def arm(self, seconds, what, fallback=None):
        self.what, self.fallback, self.deadline = what, fallback, time.monotonic() + seconds

    def disarm(self):
        self.deadline = None

    def _run(self):
        while True:
            time.sleep(1.0)
            d = self.deadline
            if d is not None and time.monotonic() > d:
                log(f"[watchdog] '{self.what}' did not finish in time: giving up on it")
                try:
                    if self.rank == 0 and self.fallback is not None:
                        line = self.fallback()
                        if line is not None:
                            line["watchdog"] = f"leg '{self.what}' exceeded its deadline; numbers measured before it are reported"
                            emit(line)
                finally:
                    os._exit(0)


WATCHDOG = None


# ------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------
def make_workload(name: str, small: bool):
    """Device-resident matrix + (n, dtype size, description, seed, default method)."""
    from spmv_b200 import api, matrices as M
    sh = 6 if small else 0  # --small: 64x fewer rows, for debugging the script itself
    if name == "c2":
        rows = 1 << (LOG2_ROWS_C2 - sh)
        A = api.gen_uniform(rows, rows, 32, M.SEED_C2, 0, False, 8)
        return A, rows, 8, f"C2 uniform-random {rows}x{rows}, 32 nnz/row, fp64 CSR", M.SEED_C2, "parallel"
    if name == "c5shard":
        # exactly one GPU's share of C5 at 8 GPUs, on ONE GPU: 2^25 rows of the 2^28-column matrix (x = 2 GiB)
        rows = 1 << (25 - sh)
        n = rows * 8
        A = api.gen_uniform(rows, n, 16, M.SEED_C5, 0, False, 8)
        return A, n, 8, f"C5 shard: rows [0, {rows}) of uniform-random {n}x{n}, 16 nnz/row, fp64 CSR", M.SEED_C5, "parallel"
    if name == "c1":
        g = 1024 >> (sh // 2)
        A = api.gen_laplacian2d(g, g, 8)
        return A, A.n, 8, f"C1 5-point 2-D Laplacian {g}x{g} grid, fp64 CSR", 1, "parallel"
    if name == "c3":
        A = api.gen_rmat(24 - sh, 16, M.SEED_C3, 4)
        return A, A.n, 4, f"C3 R-MAT scale {24 - sh} edge-factor 16 (duplicates kept), fp32 CSR", M.SEED_C3, "csr5"
    if name == "c4":
        g = 256 >> (sh // 3)
        A = api.gen_stencil27(g, g, g, 8)
        return A, A.n, 8, f"C4 27-point stencil {g}^3, fp64 CSR", 4, "sell"
    raise SystemExit(f"unknown workload {name}")


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons of one GPU, polled through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.stop_flag, self.max_mhz = [], set(), False, None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.nv = None
            log("clock sampler unavailable:", e)

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksEventReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.002)

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (device copy, of measured)"
        except Exception:
            pass
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


def traffic_for(workload: str, kernel: str):
    """dram bytes per SpMV of the kernel family on THIS workload, from the committed ncu capture (profiles/traffic.json,
    keyed "workload/kernel"); None when no capture of that pair exists."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(f"{workload}/{kernel}")
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------------
# CPU side: the reference (oracle/_ref) or the port, on the FULL C2 matrix
# ------------------------------------------------------------------------------------------------
def host_c2(small: bool, device_matrix=None):
    """The full C2 matrix in host memory: copied back from the device generator when the GPU arm already holds it,
    otherwise generated with numpy in row chunks (bit-identical: tests/test_gpu_structures.py)."""
    from spmv_b200 import matrices as M
    sh = 6 if small else 0
    rows = 1 << (LOG2_ROWS_C2 - sh)
    if device_matrix is not None:
        return device_matrix.to_host()
    chunk = min(rows, 1 << 20)
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=min(8, len(os.sched_getaffinity(0)))) as ex:
        parts = list(ex.map(lambda r0: M.uniform_random(chunk, rows, 32, seed=M.SEED_C2, row0=r0), range(0, rows, chunk)))
    rowptr = (np.arange(rows + 1, dtype=np.int64) * 32).astype(np.int32)
    return M.CSR(rows, rows, rowptr, np.concatenate([p.col for p in parts]), np.concatenate([p.val for p in parts]), "c2")


def cpu_time_reference(steps: int, warmup: int, small: bool, device_matrix=None):
    """Best OpenMP+AVX2 method of the reference on all host threads (protocol of src/samples/test_spmv.c:87-124: create
    with nthreads = team size, warm-up, timed spmv() calls).  The method is chosen from 10 calls each on a 2^21-row
    sample (creating CSR5 / SELL handles for half a billion non-zeros six times over would take minutes); the two
    fastest are then created and timed on the FULL matrix, `steps` calls each, and the better one is reported."""
    from oracle import oracle as O
    from spmv_b200 import matrices as M
    A = host_c2(small, device_matrix)
    x = M.make_x(A.n, M.SEED_C2, np.float64)
    flops = 2.0 * A.nnz
    desc = f"full C2 ({A.m} rows, {A.nnz} nnz)"
    if O.have_reference():
        R = O.Reference()
        # all host cores this process may use (torchrun exports OMP_NUM_THREADS=1: override it explicitly,
        # the reference sizes its team from omp_set_num_threads, src/samples/test_spmv.c:88)
        T = max(R.max_threads(), len(os.sched_getaffinity(0)))
        srows = min(A.m, 1 << (SAMPLE_LOG2_ROWS - (6 if small else 0)))
        S = M.CSR(srows, A.n, A.rowptr[:srows + 1], A.col[:srows * 32], A.val[:srows * 32], "sample")
        # spin the OpenMP team up first: the first ~second of parallel regions in a fresh process runs
        # 100x slow on these hosts (thread creation + cgroup ramp-up) and would bias the method choice
        h = R.create(S.m, S.n, S.rowptr, S.col, S.val, T, 1)
        y = np.zeros(S.m)
        t_end = time.perf_counter() + 1.5
        while time.perf_counter() < t_end:
            R.spmv(h, x, y)
        h.destroy()
        sample_ms = {}
        for method in (1, 2, 3, 4, 5, 6):
            h = R.create(S.m, S.n, S.rowptr, S.col, S.val, T, method)
            R.spmv(h, x, y)
            best = 1e9
            for _ in range(10):
                t0 = time.perf_counter()
                R.spmv(h, x, y)
                best = min(best, time.perf_counter() - t0)
            h.destroy()
            sample_ms[method] = best * 1e3
            log(f"  cpu reference, sample, {REF_METHOD_NAMES[method]}: best of 10 {best * 1e3:.2f} ms")
        ranked = sorted(sample_ms, key=sample_ms.get)[:2]
        best = None
        y = np.zeros(A.m)
        for method in ranked:
            h = R.create(A.m, A.n, A.rowptr, A.col, A.val, T, method)
            for _ in range(max(warmup, 2)):
                R.spmv(h, x, y)
            times = []
            for _ in range(steps):
                t0 = time.perf_counter()
                R.spmv(h, x, y)
                times.append(time.perf_counter() - t0)
            h.destroy()
            log(f"  cpu reference, full C2, {REF_METHOD_NAMES[method]}: {steps} calls, avg {np.mean(times) * 1e3:.1f} ms, best {min(times) * 1e3:.1f} ms")
            if best is None or np.mean(times) < np.mean(best[1]):
                best = (method, times)
        method, times = best
        kind, cores, name = "reference", T, REF_METHOD_NAMES[method]
    else:
        P = O.Port()
        T = len(os.sched_getaffinity(0))
        __import__("ctypes").CDLL("libgomp.so.1").omp_set_num_threads(T)
        P.spmv_serial(A.rowptr, A.col, A.val, x, parallel=True)
        times = []
        for _ in range(steps):
            t0 = time.perf_counter()
            P.spmv_serial(A.rowptr, A.col, A.val, x, parallel=True)
            times.append(time.perf_counter() - t0)
        kind, cores, name = "port", T, "oracle_spmv_parallel_d"
    avg = float(np.mean(times))
    return {"value": flops / avg / 1e9, "unit": "GFLOP/s", "cores": cores, "kind": kind,
            "sample": desc + f"; best method {name}; {len(times)} timed calls, avg {avg * 1e3:.2f} ms, best {min(times) * 1e3:.2f} ms",
            "best_value": flops / min(times) / 1e9, "same_config": True}, len(times), avg, A


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs and prints; the others exit 0 without work
    cb, steps, avg, A = cpu_time_reference(args.steps, args.warmup, args.small)
    line = {"metric": "spmv_gflops_fp64_csr", "value": cb["value"], "unit": "GFLOP/s", "impl": "reference",
            "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": avg * 1e3,
            "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": f"C2 uniform-random {A.m}x{A.n}, 32 nnz/row, fp64 CSR", "sample": cb["sample"],
                       "same_config": True},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------------
# GPU arm: timing helpers
# ------------------------------------------------------------------------------------------------
def time_steps(fn, steps, warmup, torch, dist, flush=None):
    """W untimed + K timed steps, CUDA events on the launching stream, barrier + sync on both sides,
    max over ranks.  With `flush`, L2 is overwritten before every timed step and steps are timed one by one."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    if flush is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
    else:
        ms = 0.0
        for _ in range(steps):
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms += e0.elapsed_time(e1)
    if dist is not None:
        ms = max_over_ranks(torch, dist, [ms])[0]
        dist.barrier()
    torch.cuda.synchronize()
    return ms


def max_over_ranks(torch, dist, values):
    if dist is None:
        return [float(v) for v in values]
    t = torch.tensor([float(v) for v in values], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t.tolist()]


DUMP_ROWS = 1 << 21  # rows of y written by --dump-outputs: 2^21 x (8 B value + 8 B row index) = 32 MiB at most


def y_sample(torch, y):
    """Host copy of y at a fixed, seeded set of rows (all rows when y has at most DUMP_ROWS): (values, rows)."""
    m = y.numel()
    if m <= DUMP_ROWS:
        rows = np.arange(m, dtype=np.int64)
    else:
        rows = np.sort(np.random.default_rng(0).choice(m, size=DUMP_ROWS, replace=False))
    vals = y.index_select(0, torch.from_numpy(rows).to(y.device)).cpu().numpy()
    return vals, rows.astype(np.float64)


def bench_matrix(name, args, torch, steps, warmup, methods, want_e2e, outputs=None):
    """One single-GPU workload: every method in `methods` timed device-resident (L2 flushed between steps when the
    matrix would fit L2), the first one also L2-warm and through host pointers.  Returns a record.  With `outputs`
    (a dict), y of the first method's last timed step is sampled into outputs["y"] / outputs["y_rows"]."""
    from spmv_b200 import api
    A, n, vsize, desc, seed, _ = make_workload(name, args.small)
    tdt = torch.float64 if vsize == 8 else torch.float32
    m, nnz, bmin = A.m, A.nnz, A.min_bytes()
    flops = 2.0 * nnz
    dev = torch.device("cuda", torch.cuda.current_device())
    x = torch.empty(n, dtype=tdt, device=dev)
    api.gen_x(x, n, seed, False, vsize)
    y = torch.zeros(m, dtype=tdt, device=dev)
    l2_bytes = torch.cuda.get_device_properties(dev).L2_cache_size
    fits_l2 = bmin < 2 * l2_bytes
    flush_buf = torch.zeros(max(2 * l2_bytes, 1 << 28), dtype=torch.uint8, device=dev) if fits_l2 else None
    # read-only flush: evicts the working set without leaving dirty lines to be written back under the timer
    flush = (lambda: flush_buf.max()) if fits_l2 else None
    peak, peak_src = measured_peak()
    rec = {"workload": desc, "m": m, "n": n, "nnz": nnz, "min_bytes": bmin, "dtype": "f64" if vsize == 8 else "f32",
           "l2": ("L2 flushed (%d MiB read of a scratch buffer) before every timed step" % (flush_buf.numel() >> 20)) if fits_l2
           else "inputs larger than L2 (%.1f GB per step vs %d MiB L2); no flush" % (bmin / 1e9, l2_bytes >> 20),
           "methods": {}}
    handles = {}
    launches = clocks = None
    for i, mname in enumerate(methods):
        t0 = time.perf_counter()
        h = A.handle(METHODS[mname])
        torch.cuda.synchronize()
        create_ms = (time.perf_counter() - t0) * 1e3
        handles[mname] = h
        fn = lambda h=h: h.spmv(x, y)  # noqa: E731
        if i == 0:
            sampler = ClockSampler(dev.index or 0)
            for _ in range(warmup):
                fn()
            torch.cuda.synchronize()
            sampler.start()
            l0 = api.launch_count()
            ms = time_steps(fn, steps, 0, torch, None, flush)
            launches = api.launch_count() - l0
            clocks = sampler.result()
            if outputs is not None:
                outputs["y"], outputs["y_rows"] = y_sample(torch, y)
        else:
            ms = time_steps(fn, steps, warmup, torch, None, flush)
        per = ms / steps
        rec["methods"][mname] = {"kernel": h.kernel, "ms_per_step": per, "gflops": flops / per / 1e6,
                                 "gbs_effective": bmin / per / 1e6, "frac_of_measured_peak": bmin / per / 1e6 / peak,
                                 "create_ms": create_ms, "traffic": traffic_for(name, h.kernel)}
        log(f"[{name}] {mname:13s} [{h.kernel}] {per:.4f} ms/step  {flops / per / 1e6:9.1f} GFLOP/s  "
            f"{bmin / per / 1e6:8.1f} GB/s eff  frac {bmin / per / 1e6 / peak:.3f}  (create {create_ms:.1f} ms)")
    primary = methods[0]
    rec["primary"] = primary
    rec["launches"], rec["clocks"] = int(launches), clocks
    if fits_l2:  # L2-warm figure next to the flushed one
        ms = time_steps(lambda: handles[primary].spmv(x, y), steps, warmup, torch, None, None)
        rec["l2_warm"] = {"ms_per_step": ms / steps, "gflops": flops / (ms / steps) / 1e6,
                          "frac_of_measured_peak": bmin / (ms / steps) / 1e6 / peak}
    if want_e2e:
        # host (pinned) x and y through the same C-ABI call; the fastest method's handle is used when it differs
        best = min(rec["methods"], key=lambda k: rec["methods"][k]["ms_per_step"])
        hx = torch.empty(n, dtype=tdt, pin_memory=True)
        hx.copy_(x)
        hy = torch.empty(m, dtype=tdt, pin_memory=True)
        out = {}
        for mname in dict.fromkeys([primary, best]):
            h = handles[mname]
            k = max(3, min(steps, 20))
            for _ in range(3):
                h.spmv(hx, hy)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(k):
                h.spmv(hx, hy)  # H2D x, kernel, D2H y, stream sync -- all inside
            torch.cuda.synchronize()
            per = (time.perf_counter() - t0) * 1e3 / k
            y_chk = torch.empty_like(y)
            h.spmv(x, y_chk)
            torch.cuda.synchronize()
            assert torch.equal(y_chk.cpu(), hy), "host-pointer path and device-pointer path disagree"
            out[mname] = {"ms_per_step": per, "gflops": flops / per / 1e6, "steps": k, "pipelined": bool(h.info("pipeline"))}
        rec["e2e"] = {"by_method": out, "h2d_bytes_per_step": n * vsize, "d2h_bytes_per_step": m * vsize}
    for h in handles.values():
        h.destroy()
    A.destroy()
    del x, y, flush_buf
    torch.cuda.empty_cache()
    return rec


# ------------------------------------------------------------------------------------------------
# power method on a square uniform-random matrix, row-sharded over the ranks
# ------------------------------------------------------------------------------------------------
def power_method_record(tag, log2_n, k, seed, iters, args, torch, dist, rank, world):
    """x <- A x, `iters` times, on the 2^log2_n square uniform-random matrix with k entries per row; this rank owns
    rows [rank n/N, (rank+1) n/N) as one handle per 2^26 rows (the int32 ABI: < 2^31 non-zeros per handle).
    Three loops on the same handles: the SpMV alone (band-staged, no exchange), the plain loop (SpMV, then
    ncclAllGather, timed separately) and the pipelined loop (exchange k under SpMV k+1)."""
    from spmv_b200 import api, multigpu as G
    n = 1 << log2_n
    mp = n // world
    split = [g * mp for g in range(world + 1)]
    rows_per_part = min(mp, (1 << 30) // k)
    parts = []
    t0 = time.perf_counter()
    # Column bands aligned with the owners' slices (band g = the rows rank g produces) when that is no coarser than
    # what L2 needs: then the band of a rank's own slice can start at once and every other band exactly one exchange
    # step after the previous one.  (C2 at 8 GPUs with the default 3 bands: no band is complete before step 3 of 7.)
    aligned = args.align_bands and world >= 3 and tag == "C2"
    if aligned:
        api.set_option("x_bands", world)
    try:
        for p0 in range(0, mp, rows_per_part):
            A = api.gen_uniform(rows_per_part, n, k, seed, rank * mp + p0, False, 8)
            h = A.handle(METHODS["parallel"])
            parts.append((h, p0, p0 + rows_per_part, A))
    finally:
        if aligned:
            api.set_option("x_bands", 0)
    for h, _, _, A in parts:
        if h.kernel == "band_seg":
            A.destroy()  # band segments keep their own copy of everything: give the generated CSR back
    torch.cuda.synchronize()
    create_s = time.perf_counter() - t0
    dev = torch.device("cuda", torch.cuda.current_device())
    x0 = torch.empty(n, dtype=torch.float64, device=dev)
    api.gen_x(x0, n, seed, False, 8)
    x0 *= 1.0 / k if k >= 32 else 1.0 / 8.0  # un-normalised loop: keep `iters` iterations far inside the fp64 range
    nnz_total = float(n) * k
    hparts = [(h, r0, r1) for h, r0, r1, _ in parts]
    kernel = parts[0][0].kernel
    bands = parts[0][0].bands()
    warm = 2

    # (1) the plain loop: SpMV, then in-place ncclAllGather, timed separately
    def spmv_local(xf, ys):
        for h, r0, r1 in hparts:
            h.spmv(xf, ys[r0:r1])
    pm = G.PowerMethod(spmv_local, split, x0)
    pm.run(warm)
    pm = G.PowerMethod(spmv_local, split, x0)
    x_plain, t_spmv, t_comm = pm.run(iters)
    x_plain = x_plain.clone()
    del pm
    t_spmv, t_comm = max_over_ranks(torch, dist, [t_spmv, t_comm])
    PROGRESS[tag] = {"spmv_ms": t_spmv, "allgather_ms": t_comm, "kernel": kernel, "n": n, "k": k, "mp": mp, "iters": iters}
    if WATCHDOG is not None:
        WATCHDOG.arm(240, f"{tag}: pipelined loops", FALLBACK.get("fn"))

    # (2) the pipelined loop and (3) its SpMV alone / its exchange alone
    pp = G.PipelinedPowerMethod(hparts, split, x0)
    pp.run(warm)
    pp = G.PipelinedPowerMethod(hparts, split, x0)
    if dist is not None:
        dist.barrier()
    x_pipe, t_iter = pp.run(iters)
    same = bool(torch.equal(x_pipe, x_plain))
    finite = bool(torch.isfinite(x_pipe).all())
    _, t_staged = pp.run(iters, exchange=False)
    t_xchg = pp.exchange_only(max(3, iters // 5))
    t_iter, t_staged, t_xchg, bad = max_over_ranks(torch, dist, [t_iter, t_staged, t_xchg, 0.0 if same else 1.0])
    sched = [[(pi, b0, c) for pi, b0, c in step] for step in pp.schedule]
    del pp, x_pipe
    # (4) the same pipelined loop with the exchange on the COPY ENGINES (peer DMA + stream flags, no kernels)
    ce = None
    if world > 1 and not args.no_ce:
        try:
            cp = G.CopyEnginePowerMethod(hparts, split, x0, lanes=args.ce_lanes)
            cp.run(warm)
            cp.close()
            cp = G.CopyEnginePowerMethod(hparts, split, x0, lanes=args.ce_lanes)
            t_ce = cp.run(iters)
            x_ce = cp.result()
            same_ce = bool(torch.equal(x_ce, x_plain))
            t_ce_alone = cp.run(iters, exchange=False)
            t_ce_xchg = cp.run(max(3, iters // 3), compute=False)
            t_ce, t_ce_alone, t_ce_xchg, bad_ce = max_over_ranks(torch, dist, [t_ce, t_ce_alone, t_ce_xchg, 0.0 if same_ce else 1.0])
            ce = {"iter_ms": t_ce, "spmv_alone_ms": t_ce_alone, "exchange_alone_ms": t_ce_xchg,
                  "exposed_exchange_ms": max(t_ce - t_ce_alone, 0.0),
                  "bands_launched_after_step": [sum(c for _, _, c in step) for step in cp.schedule],
                  "bitwise_equal_to_plain_loop": bad_ce == 0.0, "direct_peer_flags": cp.direct_flags, "lanes": cp.lanes,
                  "transport": "per step one cudaMemcpyAsync of the y slice into the peer's next-x buffer (CUDA-IPC mapping, "
                               "copy engine over NVLink) + cuStreamWriteValue32 arrival flag; the band-staged SpMV waits per "
                               "band with cuStreamWaitValue32; no kernel and no collective in the exchange"}
            cp.close()
            del x_ce
            log(f"[{tag} x{world}] copy-engine loop {t_ce:.3f} ms (spmv alone {t_ce_alone:.3f}, exchange alone {t_ce_xchg:.3f}) | bitwise equal {bad_ce == 0.0}")
        except Exception as e:
            log("copy-engine loop unavailable:", repr(e))
            ce = {"error": repr(e)}
    del x_plain
    if WATCHDOG is not None:
        WATCHDOG.disarm()
    rec = {"matrix": f"{tag}: uniform-random {n}x{n}, {k} nnz/row, fp64 CSR, rows sharded over {world} GPU(s) by equal nnz",
           "iters": iters, "rows_per_gpu": mp, "handles_per_gpu": len(parts), "kernel": kernel, "column_bands": bands,
           "create_s": create_s,
           "plain_loop": {"spmv_ms_per_iter": t_spmv, "allgather_ms_per_iter": t_comm, "iter_ms": t_spmv + t_comm,
                          "collective": "ncclAllGather in place (torch.distributed)" if world > 1 else "none (1 GPU)"},
           "pipelined_loop": {"iter_ms": t_iter, "spmv_alone_ms": t_staged, "exchange_alone_ms": t_xchg,
                              "exposed_exchange_ms": max(t_iter - t_staged, 0.0),
                              "transport": "N-1 NCCL send/recv permutation steps on a side stream, nearest neighbours first; "
                                           "band-staged SpMV waits per band on the steps it needs",
                              "bands_launched_after_step": [sum(c for _, _, c in step) for step in sched],
                              "bitwise_equal_to_plain_loop": bad == 0.0, "finite": finite},
           "copy_engine_loop": ce,
           "allgather_bytes_recv_per_gpu": (world - 1) * mp * 8,
           "gflops_plain": 2.0 * nnz_total / (t_spmv + t_comm) / 1e6, "gflops_pipelined": 2.0 * nnz_total / t_iter / 1e6,
           "gflops_spmv_alone": 2.0 * nnz_total / t_staged / 1e6}
    log(f"[{tag} x{world}] plain {t_spmv:.3f} + {t_comm:.3f} ms | pipelined {t_iter:.3f} ms (spmv alone {t_staged:.3f}, "
        f"exchange alone {t_xchg:.3f}) | bitwise equal {bad == 0.0}")
    return rec, parts, split, x0


FALLBACK = {}


def free_parts(parts):
    for h, _, _, A in parts:
        h.destroy()
        A.destroy()


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_gpu_arm(args):
    import torch
    from spmv_b200 import api, build
    build.build()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        log(f"note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes y of the single-GPU SpMV; it is not available with N > 1")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # belt and braces: see RESULT below
        import torch.distributed as dist_mod
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    if world == 1:
        line = single_gpu(args, torch, api)
    else:
        line = multi_gpu(args, torch, api, dist, rank, world, local)
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


def single_gpu(args, torch, api):
    name = args.workload
    default_method = {"c1": "parallel", "c2": "parallel", "c3": "csr5", "c4": "sell", "c5shard": "parallel"}[name]
    primary = args.method or default_method
    methods = [primary] + [mname for mname in args.also.split(",") if mname and mname != primary]
    outputs = {} if args.dump_outputs else None
    rec = bench_matrix(name, args, torch, args.steps, args.warmup, methods, want_e2e=True, outputs=outputs)
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for key, arr in outputs.items():
            np.save(os.path.join(args.dump_outputs, key + ".npy"), arr)
        log(f"wrote {', '.join(k + '.npy' for k in outputs)} ({len(outputs['y'])} of {rec['m']} rows of y) to {args.dump_outputs}")
    r = rec["methods"][primary]
    per = r["ms_per_step"]
    peak, peak_src = measured_peak()
    bmin = rec["min_bytes"]
    achieved = bmin / per / 1e6  # GB/s, algorithmic bytes of ONE launch / its average duration
    e2e = rec["e2e"]["by_method"][primary]
    e2e_best_name = min(rec["e2e"]["by_method"], key=lambda k: rec["e2e"]["by_method"][k]["ms_per_step"])
    line = {
        "metric": "spmv_gflops_fp64_csr" if rec["dtype"] == "f64" else "spmv_gflops_fp32_csr",
        "value": r["gflops"], "unit": "GFLOP/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": per, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": rec["dtype"], "data": "synthetic",
        "config": {"workload": rec["workload"], "method": api.METHOD_NAMES[METHODS[primary]], "kernel": r["kernel"],
                   "m_per_gpu": rec["m"], "n": rec["n"], "nnz_per_gpu": rec["nnz"], "min_bytes_per_gpu": bmin, "l2": rec["l2"],
                   "timing": "CUDA events on the launch stream around K back-to-back spmv() calls",
                   "scaling_note": "N > 1 runs the power-method iteration (SpMV + exchange) on this same matrix, row-sharded"},
        "gbs_effective": achieved, "frac_of_8TBps_nominal": achieved / 8000.0,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": r["traffic"], "kernel": r["kernel"], "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": bmin},
        "methods": rec["methods"],
        "e2e": {"value": e2e["gflops"], "unit": "GFLOP/s", "ms_per_step": e2e["ms_per_step"],
                "h2d_bytes_per_step": rec["e2e"]["h2d_bytes_per_step"], "d2h_bytes_per_step": rec["e2e"]["d2h_bytes_per_step"],
                "steps": e2e["steps"], "api": "spmv() of include/spmv.h with pinned HOST x and y",
                "fastest_method": {"method": e2e_best_name, **rec["e2e"]["by_method"][e2e_best_name]}},
        "gpu_launches": rec["launches"], "clocks": rec["clocks"],
    }
    if "l2_warm" in rec:
        line["l2_warm"] = rec["l2_warm"]
    # ---- the other BASELINE.json configurations, same protocol, as sub-records ----
    extras = {}
    for ex in [e for e in args.extras.split(",") if e and e != name]:
        try:
            m_ex = {"c1": ["parallel", "sell"], "c2": ["parallel", "sell"], "c3": ["csr5", "balanced2", "parallel"],
                    "c4": ["sell", "parallel"], "c5shard": ["parallel"]}[ex]
            er = bench_matrix(ex, args, torch, max(5, min(args.steps, 20)), max(3, min(args.warmup, 5)), m_ex, want_e2e=False)
            extras[ex] = {k: er[k] for k in ("workload", "nnz", "min_bytes", "dtype", "l2", "methods", "primary")}
            if "l2_warm" in er:
                extras[ex]["l2_warm"] = er["l2_warm"]
        except Exception as e:  # a sub-record must never take the headline down
            log(f"extra workload {ex} failed:", repr(e))
            extras[ex] = {"error": repr(e)}
    if extras:
        line["configs"] = extras
    # ---- C5 on ONE GPU (4 handles of 2^26 rows): the strong-scaling baseline of the multi-GPU record ----
    if args.c5 and name == "c2":
        try:
            c5, parts, _, _ = power_method_record("C5", LOG2_ROWS_C5 - (6 if args.small else 0), 16, __import__("spmv_b200.matrices", fromlist=["x"]).SEED_C5,
                                                  min(args.power_iters, 10), args, torch, None, 0, 1)
            free_parts(parts)
            line["c5"] = c5
        except Exception as e:
            log("C5 record failed:", repr(e))
            line["c5"] = {"error": repr(e)}
    # ---- CPU baseline on the box's host cores: the FULL C2 matrix ----
    if not args.no_cpu and name == "c2":
        try:
            A, *_ = make_workload("c2", args.small)
            cpu, _, _, _ = cpu_time_reference(20, 3, args.small, device_matrix=A)
            A.destroy()
            line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "same_config")}
        except Exception as e:  # the GPU numbers stand on their own
            log("cpu baseline failed:", repr(e))
    return line


def multi_gpu(args, torch, api, dist, rank, world, local):
    from spmv_b200 import matrices as M, multigpu as G
    if args.workload != "c2":
        raise SystemExit("--gpus N > 1 runs the C2 power-method iteration (plus the C5 record)")
    sh = 6 if args.small else 0
    dev = torch.device("cuda", local)
    iters = max(args.steps, 1)
    global WATCHDOG
    WATCHDOG = Watchdog(rank)

    def fallback_line():
        p = PROGRESS.get("C2")
        if not p:
            return None
        t = p["spmv_ms"] + p["allgather_ms"]
        nn, mpp = p["n"], p["mp"]
        bmin = mpp * 32 * 12 + (mpp + 1) * 4 + mpp * 8 + nn * 8
        pk, src = measured_peak()
        ach = bmin / p["spmv_ms"] / 1e6
        line = {"metric": "spmv_gflops_fp64_csr", "value": 2.0 * nn * 32 / t / 1e6, "unit": "GFLOP/s", "n_gpus": world,
                "steps": p["iters"], "warmup": 2, "ms_per_step": t, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"C2 uniform-random {nn}x{nn}, 32 nnz/row, fp64 CSR: one power-method iteration x <- A x "
                                       f"(SpMV + y->x exchange), rows sharded over {world} GPUs by equal nnz",
                           "method": "Method_Parallel", "kernel": p["kernel"], "loop": "plain"},
                "roofline": {"bound": "hbm", "achieved": ach, "peak": pk, "unit": "GB/s", "frac": ach / pk, "traffic": None,
                             "kernel": p["kernel"], "peak_source": src, "algorithmic_bytes_per_launch": bmin},
                "power_method": {"plain_loop": {"spmv_ms_per_iter": p["spmv_ms"], "allgather_ms_per_iter": p["allgather_ms"], "iter_ms": t}},
                "e2e": None, "gpu_launches": int(api.launch_count()), "c5_progress": PROGRESS.get("C5")}
        return line
    FALLBACK["fn"] = fallback_line
    sampler = ClockSampler(local)
    sampler.start()
    l0 = api.launch_count()
    WATCHDOG.arm(300, "C2: create + plain loop", fallback_line)
    rec, parts, split, x0 = power_method_record("C2", LOG2_ROWS_C2 - sh, 32, M.SEED_C2, iters, args, torch, dist, rank, world)
    launches = api.launch_count() - l0
    clocks = sampler.result()
    n = 1 << (LOG2_ROWS_C2 - sh)
    mp = n // world
    nnz_total = float(n) * 32
    h0 = parts[0][0]
    bmin_gpu = mp * 32 * 12 + (mp + 1) * 4 + mp * 8 + n * 8
    loops = {"plain": rec["plain_loop"]["iter_ms"]}
    if rec["pipelined_loop"]["bitwise_equal_to_plain_loop"] and rec["pipelined_loop"]["finite"]:
        loops["pipelined_nccl"] = rec["pipelined_loop"]["iter_ms"]
    ce = rec.get("copy_engine_loop")
    if ce and ce.get("bitwise_equal_to_plain_loop"):
        loops["pipelined_copy_engine"] = ce["iter_ms"]
    best_loop = min(loops, key=loops.get)
    t_iter = loops[best_loop]
    t_spmv = rec["pipelined_loop"]["spmv_alone_ms"]
    peak, peak_src = measured_peak()
    achieved = bmin_gpu / t_spmv / 1e6

    # ---- fused variant of round 1 (peer stores from the kernel that writes y): kept as a measured alternative ----
    fused = None
    if len(parts) == 1 and not args.no_fused:
        WATCHDOG.arm(180, "C2: fused peer-store loop", fallback_line)
        try:
            xs = x0
            fp = G.FusedPowerMethod(h0, split, xs)
            fp.run(2)
            fp2 = G.FusedPowerMethod(h0, split, xs)
            t_f, t_sync = fp2.run(iters)
            t_f, t_sync = max_over_ranks(torch, dist, [t_f, t_sync])
            fused = {"iter_ms": t_f + t_sync, "spmv_plus_peer_stores_ms_per_iter": t_f, "rank_sync_ms_per_iter": t_sync,
                     "transport": "st.global to CUDA-IPC peer mappings over NVLink from the kernel that writes y"}
            fp.close()
            fp2.close()
        except Exception as e:  # IPC may be unavailable in some containers: the other loops stand
            log("fused power method unavailable:", repr(e))

    # ---- e2e: host x / y; every rank uploads ITS slice of x, NVLink all-gather, SpMV, its slice of y back ----
    WATCHDOG.arm(180, "C2: end-to-end leg", fallback_line)
    lo, hi = split[rank], split[rank + 1]
    hx = torch.empty(mp, dtype=torch.float64, pin_memory=True)
    hx.copy_(x0[lo:hi])
    hy = torch.empty(mp, dtype=torch.float64, pin_memory=True)
    xd = torch.empty(n, dtype=torch.float64, device=dev)
    yd = torch.empty(mp, dtype=torch.float64, device=dev)

    def e2e_step():
        xd[lo:hi].copy_(hx, non_blocking=True)
        dist.all_gather_into_tensor(xd, xd[lo:hi])
        h0.spmv(xd, yd) if len(parts) == 1 else [h.spmv(xd, yd[r0:r1]) for h, r0, r1, _ in parts]
        hy.copy_(yd, non_blocking=True)
        torch.cuda.synchronize()
    for _ in range(3):
        e2e_step()
    dist.barrier()
    k = max(3, min(iters, 20))
    t0 = time.perf_counter()
    for _ in range(k):
        e2e_step()
    e2e_ms = max_over_ranks(torch, dist, [(time.perf_counter() - t0) * 1e3 / k])[0]
    free_parts(parts)
    del x0, xd, yd
    torch.cuda.empty_cache()

    # ---- the line so far: what the watchdog prints if the C5 record hangs ----
    def build_line(c5):
        return {
            "metric": "spmv_gflops_fp64_csr", "value": 2.0 * nnz_total / t_iter / 1e6, "unit": "GFLOP/s", "n_gpus": world,
            "steps": iters, "warmup": 2, "ms_per_step": t_iter, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"C2 uniform-random {n}x{n}, 32 nnz/row, fp64 CSR: one power-method iteration x <- A x "
                                   f"(SpMV + y->x exchange), rows sharded over {world} GPUs by equal nnz",
                       "method": "Method_Parallel", "kernel": rec["kernel"], "m_per_gpu": mp, "n": n, "nnz_per_gpu": mp * 32,
                       "min_bytes_per_gpu": bmin_gpu,
                       "l2": "inputs larger than L2 (%.2f GB per GPU and step); no flush" % (bmin_gpu / 1e9),
                       "timing": "CUDA events around `steps` back-to-back iterations incl. the exchange, max over ranks",
                       "loop": best_loop, "loops_ms": loops},
            "gbs_effective": world * achieved, "frac_of_8TBps_nominal": achieved / 8000.0,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "kernel": rec["kernel"], "peak_source": peak_src, "algorithmic_bytes_per_launch": bmin_gpu,
                         "note": "per GPU, from the SpMV-alone time of the row shard"},
            "power_method": rec, "power_method_fused": fused, "c5": c5,
            "e2e": {"value": 2.0 * nnz_total / e2e_ms / 1e6, "unit": "GFLOP/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": n * 8, "d2h_bytes_per_step": n * 8, "steps": k,
                    "api": "per rank: its slice of x from pinned host memory, ncclAllGather of x over NVLink, spmv() on device "
                           "pointers, its slice of y back to pinned host memory (bytes are totals over all ranks)"},
            "gpu_launches": int(launches), "clocks": clocks,
        }
    FALLBACK["fn"] = lambda: build_line({"progress": PROGRESS.get("C5"), "note": "the C5 record did not complete"})

    # ---- BASELINE.json configs[4]: C5 at this N ----
    c5 = None
    if args.c5:
        WATCHDOG.arm(420, "C5: create + plain loop", FALLBACK["fn"])
        try:
            c5, parts5, _, _ = power_method_record("C5", LOG2_ROWS_C5 - sh, 16, M.SEED_C5, min(args.power_iters, 50), args, torch, dist,
                                                   rank, world)
            free_parts(parts5)
        except Exception as e:
            log("C5 record failed:", repr(e))
            c5 = {"error": repr(e)}

    WATCHDOG.disarm()
    return build_line(c5)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c3", "c4", "c5shard"])
    ap.add_argument("--method", default="", choices=[""] + list(METHODS))
    ap.add_argument("--also", default="balanced2,sell", help="comma list of further methods timed after the primary")
    ap.add_argument("--extras", default="c1,c3,c4,c5shard", help="other configurations timed as sub-records (N = 1, workload c2)")
    ap.add_argument("--c5", type=int, default=1, help="1 = add the C5 power-method record (N = 1: ten iterations on one GPU)")
    ap.add_argument("--power-iters", type=int, default=50)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-fused", action="store_true")
    ap.add_argument("--no-ce", action="store_true", help="skip the copy-engine exchange loop")
    ap.add_argument("--ce-lanes", type=int, default=1, help="streams (copy engines) a slice is spread over in the copy-engine exchange")
    ap.add_argument("--align-bands", type=int, default=1, help="N >= 3: as many column bands as ranks for the C2 shards")
    ap.add_argument("--small", action="store_true", help="64x smaller matrices (script debugging only; not a bench)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write y of the last timed step as DIR/y.npy (values) and DIR/y_rows.npy "
                         "(their row indices): all rows up to 2^21, else a fixed seeded sample of 2^21 rows")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; it is not available with --impl reference")
    claim_stdout()
    args.warmup = max(args.warmup, 3)
    if args.workload != "c2":
        args.extras = ""
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
