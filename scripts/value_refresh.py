"""What refreshing a handle's values costs: spmv_b200_set_values (option "refresh") against spmv_b200_update_values
(a full rebuild) and against one SpMV, at the BASELINE sizes, fp64.

    python scripts/value_refresh.py [--out profiles/r03_value_refresh.json] [--small]

Per configuration (matrix generated on the device, handle adopting it):
  * set_values from a device source: the adopted values scaled in place with torch, then set_values(NULL) -- the
    timed calls re-read the same array (>= 20 calls after warm-up, CUDA events);
  * set_values from a pinned host array, on a handle that owns its upload (built from host copies of the matrix);
  * update_values(NULL): 3 calls, each ending in a device synchronise (option "refresh" off, as a client without it);
  * one spmv (mean of 20);
  * modelled bytes of a refresh: per stored slot 4 B of map + 2 x 8 B (read the source, write the slot), plus nnz x 8 B
    for a copied identity target (the host copy or the upload); GB/s and its share of the measured 6 534.8 GB/s
    device-copy peak;
  * create time and memory of the maps: create with the option on against off (host clock around create, which ends
    in a stream synchronise; live_allocations and cudaMemGetInfo deltas);
and after the timed calls, y of the refreshed handle against a handle newly created on the same values, bitwise.
The card's name and power limit are read in the same run.  --small: 64x fewer rows, for checking the script."""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK_GBS = 6534.8  # measured device-copy peak of a B200 (BASELINE.md)
VSIZE = 8


@contextlib.contextmanager
def options(api, **kw):
    old = {k: api.get_option(k) for k in kw}
    for k, v in kw.items():
        api.set_option(k, v)
    try:
        yield
    finally:
        for k, v in old.items():
            api.set_option(k, v)


class _DeviceArray:
    """A raw device pointer as something torch.as_tensor can view in place."""

    def __init__(self, ptr, count):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f8", "data": (int(ptr), False), "version": 3,
                                         "strides": None}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # pragma: no cover
        return {"error": repr(e)}


def configs(api, M, small):
    sh = 6 if small else 0
    return [
        ("C2", f"uniform-random 2^{24 - sh} x 2^{24 - sh}, 32 nnz/row, fp64",
         lambda: api.gen_uniform(1 << (24 - sh), 1 << (24 - sh), 32, M.SEED_C2, 0, False, 8), M.SEED_C2,
         [api.Method_Parallel, api.Method_SellCSigma]),
        ("C3", f"R-MAT scale {24 - sh} edge-factor 16, fp64", lambda: api.gen_rmat(24 - sh, 16, M.SEED_C3, 8), M.SEED_C3,
         [api.Method_CSR5SPMV]),
        ("C4", f"27-point stencil {256 >> (sh // 3)}^3, fp64", lambda: api.gen_stencil27(256 >> (sh // 3), 256 >> (sh // 3), 256 >> (sh // 3), 8),
         4, [api.Method_SellCSigma]),
        ("C5 shard", f"rows [0, 2^{25 - sh}) of uniform-random 2^{28 - sh} x 2^{28 - sh}, 16 nnz/row, fp64",
         lambda: api.gen_uniform(1 << (25 - sh), 1 << (28 - sh), 16, M.SEED_C5, 0, False, 8), M.SEED_C5, [api.Method_Parallel]),
    ]


def stored_slots(h, nnz):
    """(slots of every value array the handle stores, whether it keeps its own upload in the caller's order)."""
    slots = {}
    kernel = h.info("kernel")
    if h.info("x_bands") > 1 and kernel != 8:
        slots["band_copy"] = nnz
    if kernel == 6:
        slots["sell"] = h.info("padded_nnz")
    if kernel == 7:
        slots["csr5"] = nnz
    if kernel == 8:
        slots["band_segments"] = int(h.structure("seg_ptr", np.int32)[-1])
    return slots, h.info("owns_csr") == 1


def refresh_bytes(slots, nnz, copied):
    return (4 + 2 * VSIZE) * sum(slots.values()) + (nnz * VSIZE if copied else 0)


def time_events(torch, fn, calls, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def rate(nbytes, ms):
    gbs = nbytes / (ms * 1e-3) / 1e9
    return {"ms": round(ms, 4), "modelled_bytes": int(nbytes), "gb_s": round(gbs, 1), "of_copy_peak": round(gbs / PEAK_GBS, 3)}


def run_method(api, torch, A, seed, method, log):
    nnz, m, n = A.nnz, A.m, A.n
    vals = torch.as_tensor(_DeviceArray(A.Val, nnz), device="cuda")
    x = torch.empty(n, dtype=torch.float64, device="cuda")
    api.gen_x(x, n, seed, False, 8)
    y = torch.empty(m, dtype=torch.float64, device="cuda")
    rec = {"method": api.METHOD_NAMES[method]}

    # create with the option off, then on: time and memory of the maps
    create = {}
    for refresh in (0, 1):
        torch.cuda.synchronize()
        free0, live0 = torch.cuda.mem_get_info()[0], api.live_allocations()
        t0 = time.perf_counter()
        with options(api, refresh=refresh):
            h = A.handle(method)
        torch.cuda.synchronize()
        create[refresh] = {"ms": (time.perf_counter() - t0) * 1e3, "bytes": free0 - torch.cuda.mem_get_info()[0],
                           "allocations": api.live_allocations() - live0}
        if refresh == 0:
            h.destroy()
    assert h.info("refreshable") == 1
    slots, owns = stored_slots(h, nnz)
    rec["kernel"] = api.KERNEL_NAMES[h.info("kernel")]
    rec["x_bands"] = h.info("x_bands")
    rec["stored_slots"] = slots
    rec["maps"] = {"create_ms_without": round(create[0]["ms"], 1), "create_ms_with": round(create[1]["ms"], 1),
                   "create_ms_overhead": round(create[1]["ms"] - create[0]["ms"], 1),
                   "extra_allocations": create[1]["allocations"] - create[0]["allocations"],
                   "extra_bytes_cudaMemGetInfo": create[1]["bytes"] - create[0]["bytes"],
                   "modelled_map_bytes": 4 * sum(slots.values())}
    log(rec["method"], rec["kernel"], slots, rec["maps"])

    rec["spmv_ms"] = round(time_events(torch, lambda: h.spmv(x, y), 20, 5), 4)
    ms = time_events(torch, lambda: h.set_values(), 20, 3)
    rec["set_values_device"] = rate(refresh_bytes(slots, nnz, False), ms)
    rec["set_values_device"]["calls"] = 20
    rec["set_values_device"]["spmvs"] = round(ms / rec["spmv_ms"], 2)
    log("device source", rec["set_values_device"], "spmv", rec["spmv_ms"])

    # new values in place, refresh, and y against a handle created on them
    vals.mul_(-0.75)
    h.set_values()
    h.spmv(x, y)
    fresh = A.handle(method)
    y_fresh = torch.empty_like(y)
    fresh.spmv(x, y_fresh)
    torch.cuda.synchronize()
    rec["bitwise_equal_to_fresh_create"] = bool(torch.equal(y.view(torch.int64), y_fresh.view(torch.int64)))
    fresh.destroy()
    log("bitwise", rec["bitwise_equal_to_fresh_create"])

    times = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        h.update_values()
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
    rec["update_values_ms"] = [round(t, 1) for t in times]
    rec["speedup_over_update_values"] = round(float(np.median(times)) / ms, 1)
    log("update_values", rec["update_values_ms"], "speed-up", rec["speedup_over_update_values"])
    h.destroy()
    return rec


def run_host_source(api, torch, host, method, log):
    """set_values from a pinned host array on a handle that owns its upload."""
    rp, ci, va = host.rowptr, host.col, host.val
    with options(api, refresh=1):
        h = api.Handle(host.m, host.n, rp, ci, va, method)
    slots, owns = stored_slots(h, host.nnz)
    src = torch.from_numpy(va).pin_memory()
    ms = time_events(torch, lambda: h.set_values(src), 20, 2)
    out = rate(refresh_bytes(slots, host.nnz, True), ms)
    out["calls"] = 20
    out["copied_to"] = "upload" if owns else "staging"
    h.destroy()
    log("host pinned source", out)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_value_refresh.json"))
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    import torch
    from spmv_b200 import api, matrices as M

    def log(*a):
        print(*a, file=sys.stderr, flush=True)

    assert torch.cuda.is_available(), "needs a GPU"
    result = {"card": card(), "copy_peak_gb_s": PEAK_GBS, "dtype": "fp64", "configs": []}
    log(result["card"])
    for name, desc, gen, seed, methods in configs(api, M, args.small):
        A = gen()
        log("==", name, desc, "nnz", A.nnz)
        entry = {"config": name, "matrix": desc, "m": A.m, "n": A.n, "nnz": A.nnz, "methods": []}
        for method in methods:
            entry["methods"].append(run_method(api, torch, A, seed, method, log))
        host = A.to_host()
        A.destroy()
        for rec, method in zip(entry["methods"], methods):
            rec["set_values_host_pinned"] = run_host_source(api, torch, host, method, log)
        del host
        result["configs"].append(entry)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"out": args.out, "all_bitwise": all(r["bitwise_equal_to_fresh_create"] for c in result["configs"]
                                                         for r in c["methods"])}))


if __name__ == "__main__":
    main()
