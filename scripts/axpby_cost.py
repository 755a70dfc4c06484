"""What y <- alpha A x + beta y costs: spmv_b200_spmv_axpby against spmv() and against the caller's alternative (spmv()
into a temporary, then eager torch mul, mul, add), on the workloads bench.py records, one B200.

    python scripts/axpby_cost.py [--out profiles/r04_axpby.json] [--steps 20] [--rounds 5] [--small]

Per workload and method (the matrices and x of bench.py's make_workload):
  * the modes below, timed with CUDA events over `steps` calls each, in `rounds` rounds that alternate the modes:
      spmv           h.spmv(x, y)
      axpby_beta0    h.spmv_axpby(alpha, x, 0, y)
      axpby          h.spmv_axpby(alpha, x, beta, y)            (alpha = 0.5, beta = -0.75)
      torch_3pass    h.spmv(x, t); y = torch.add(t * alpha, y * beta)
      axpby_scratch  (fold / main-kernel handles) spmv_axpby(alpha, x, beta, y) on a second handle of the same matrix
                     created with option "axpby_fused" = 0: the scratch pass the fused kernel replaces
    C1 fits L2 and is flushed before every call and timed call by call, as bench.py does; the others are larger
    than L2 and are not flushed (C1 also: spmv and axpby_beta0 L2-warm, calls back to back without a flush).
    ms = median over the rounds, spread = (max - min) / median;
  * modelled bytes (B_min of BASELINE.md: nnz (v + 4) + (m + 1) 4 + m v + n v): spmv B_min; the fused scaled store
    adds m v (the old y) when beta != 0; the scratch pass adds 2 m v (s written and read back) and the old y; the
    caller's three passes add 7 m v (mul: m v in, m v out, twice; add: 2 m v in, m v out);
  * the path the handle takes (spmv_b200_info "axpby_path": 0 scratch pass, 1 main kernel, 2 fold);
  * bitwise check at full size: spmv_axpby's y (and the scratch-pass handle's) against the torch formula on spmv()'s
    y (beta != 0 and beta == 0).
The card's name and power limit are read in the same run.  --small: 64x fewer rows, for checking the script."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ALPHA, BETA = 0.5, -0.75
PATHS = {0: "scratch pass", 1: "main kernel", 2: "fold"}
# (workload of bench.py, method, whether bench.py flushes L2 before every timed call)
RUNS = [("c1", "parallel", True), ("c2", "parallel", False), ("c2", "sell", False), ("c3", "csr5", False),
        ("c4", "sell", False), ("c4", "parallel", False), ("c4", "balanced", False), ("c5shard", "parallel", False)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # pragma: no cover
        return {"error": repr(e)}


def timed(torch, fn, steps, flush):
    """ms per call: events around `steps` calls, or (flush) around each call after an L2 flush."""
    if flush is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps
    total = 0.0
    for _ in range(steps):
        flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
    return total / steps


def run_one(api, torch, bench, name, method, flushed, steps, rounds, small, log):
    A, n, vsize, desc, seed, _ = bench.make_workload(name, small)
    tdt = torch.float64 if vsize == 8 else torch.float32
    m, nnz, bmin = A.m, A.nnz, A.min_bytes()
    x = torch.empty(n, dtype=tdt, device="cuda")
    api.gen_x(x, n, seed, False, vsize)
    y0 = torch.empty(m, dtype=tdt, device="cuda")
    api.gen_x(y0, m, seed + 1, False, vsize)
    y, t = y0.clone(), torch.empty_like(y0)
    h = A.handle(bench.METHODS[method])
    path = h.info("axpby_path")
    hs = None
    if path != 0:  # the same layout with the scratch pass, for the fused path to be timed against
        api.set_option("axpby_fused", 0)
        try:
            hs = A.handle(bench.METHODS[method])
        finally:
            api.set_option("axpby_fused", 1)
        assert hs.info("axpby_path") == 0
    flush_buf = torch.zeros(max(2 * torch.cuda.get_device_properties(0).L2_cache_size, 1 << 28), dtype=torch.uint8,
                            device="cuda") if flushed else None
    flush = (lambda: flush_buf.max()) if flushed else None

    def caller_alternative():
        h.spmv(x, t)
        torch.add(t * ALPHA, y * BETA, out=y)

    modes = {"spmv": lambda: h.spmv(x, y), "axpby_beta0": lambda: h.spmv_axpby(ALPHA, x, 0.0, y),
             "axpby": lambda: h.spmv_axpby(ALPHA, x, BETA, y), "torch_3pass": caller_alternative}
    if hs is not None:
        modes["axpby_scratch"] = lambda: hs.spmv_axpby(ALPHA, x, BETA, y)
    for fn in modes.values():  # warm-up: module loads, the scratch array, torch's allocator
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    samples = {k: [] for k in modes}
    for r in range(rounds):
        order = list(modes) if r % 2 == 0 else list(reversed(modes))
        for k in order:
            y.copy_(y0)  # |beta| < 1: y stays bounded however many calls run
            samples[k].append(timed(torch, modes[k], steps, flush))
    mv = m * vsize
    scratch = path == 0
    model = {"spmv": bmin, "axpby_beta0": bmin + (2 * mv if scratch else 0),
             "axpby": bmin + mv + (2 * mv if scratch else 0), "torch_3pass": bmin + 7 * mv, "axpby_scratch": bmin + 3 * mv}
    rec = {"workload": desc, "method": method, "kernel": h.kernel, "x_bands": h.info("x_bands"),
           "axpby_path": f"{path} ({PATHS[path]})", "m": m, "n": n, "nnz": nnz,
           "l2": "flushed before every timed call, timed call by call" if flushed else "larger than L2, not flushed",
           "steps_per_round": steps, "rounds": rounds, "modes": {}}
    base = float(np.median(samples["spmv"]))
    for k, v in samples.items():
        med = float(np.median(v))
        rec["modes"][k] = {"ms": round(med, 5), "spread": round((max(v) - min(v)) / med, 4),
                           "ms_rounds": [round(s, 5) for s in v], "modelled_bytes": int(model[k]),
                           "time_over_spmv": round(med / base, 4), "bytes_over_spmv": round(model[k] / bmin, 4)}
    if flushed:  # the same calls back to back, L2-warm: host entry cost overlaps the previous call's kernel
        warm = {k: [] for k in ("spmv", "axpby_beta0")}
        for r in range(rounds):
            for k in (warm if r % 2 == 0 else list(reversed(warm))):
                warm[k].append(timed(torch, modes[k], steps, None))
        rec["l2_warm"] = {k: {"ms": round(float(np.median(v)), 5), "spread": round((max(v) - min(v)) / float(np.median(v)), 4)}
                          for k, v in warm.items()}
    # bits at full size: spmv_axpby against the torch formula on spmv()'s y
    s = torch.empty_like(y0)
    h.spmv(x, s)
    bits = {}
    itype = torch.int64 if vsize == 8 else torch.int32
    for beta in (BETA, 0.0):
        want = s * ALPHA if beta == 0.0 else torch.add(s * ALPHA, y0 * beta)
        for tag, hh in (("", h), ("scratch handle, ", hs)):
            if hh is None:
                continue
            y.copy_(y0)
            hh.spmv_axpby(ALPHA, x, beta, y)
            torch.cuda.synchronize()
            bits[f"{tag}beta={beta}"] = bool(torch.equal(y.view(itype), want.view(itype)))
    rec["bitwise_equal_to_torch_formula"] = bits
    ax, alt = rec["modes"]["axpby"], rec["modes"]["torch_3pass"]
    rec["axpby_vs_caller_alternative"] = round(ax["ms"] / alt["ms"], 4)
    if hs is not None:
        rec["axpby_vs_scratch_pass"] = round(ax["ms"] / rec["modes"]["axpby_scratch"]["ms"], 4)
        hs.destroy()
    log(f"[{name} {method}] path {rec['axpby_path']} | " +
        " | ".join(f"{k} {v['ms']:.4f} ms (x{v['time_over_spmv']:.3f}, bytes x{v['bytes_over_spmv']:.3f}, spread {v['spread']:.3f})"
                   for k, v in rec["modes"].items()) + f" | {rec.get('l2_warm', '')} | bits {bits}")
    h.destroy()
    A.destroy()
    del x, y, y0, t, s, flush_buf
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_axpby.json"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    import torch
    import bench
    from spmv_b200 import api

    def log(*a):
        print(*a, file=sys.stderr, flush=True)

    assert torch.cuda.is_available(), "needs a GPU"
    result = {"card": card(), "alpha": ALPHA, "beta": BETA, "runs": []}
    log(result["card"])
    for name, method, flushed in RUNS:
        result["runs"].append(run_one(api, torch, bench, name, method, flushed, args.steps, args.rounds, args.small, log))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"out": args.out,
                      "all_bitwise": all(all(r["bitwise_equal_to_torch_formula"].values()) for r in result["runs"]),
                      "axpby_vs_caller_alternative": {f"{r['workload'][:2]} {r['method']}": r["axpby_vs_caller_alternative"]
                                                      for r in result["runs"]},
                      "axpby_vs_scratch_pass": {f"{r['workload'][:2]} {r['method']}": r.get("axpby_vs_scratch_pass")
                                                for r in result["runs"]}}))


if __name__ == "__main__":
    main()
