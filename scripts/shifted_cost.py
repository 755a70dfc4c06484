"""What spmv_b200_spmv_shifted saves a Chebyshev / KPM step: y <- alpha (A - sigma I) x + beta y with x . y and y . y
in one call, against what a client does without it, on one B200, fp64.

    python scripts/shifted_cost.py [--out profiles/r06_shifted.json] [--steps 20] [--rounds 5] [--small]

Workloads (square matrices only: the shift needs m == n): bench.py's C1, C2 and C4 with their methods, C3 (bench.py's
R-MAT) in fp64 with CSR5, and a square matrix of the C5 shard's shape (2^25 rows, 16 non-zeros per row, uniform
random columns; the shard itself, 2^25 rows of a 2^28-column matrix, is not square).  Per workload, the arms, timed
with CUDA events as scripts/axpby_cost.py times them (C1 flushed before every call, the others larger than L2), in
`rounds` rounds that alternate the arms; alpha = 0.5, sigma = 0.25, beta = -0.75, dots into device doubles (no host
synchronisation in the loop):
  axpby           h.spmv_axpby(alpha, x, beta, y)                                   (no shift, no dots: the floor)
  shifted         spmv_b200_spmv_shifted(h, alpha, sigma, x, beta, y, NULL)
  shifted_dots    h.spmv_shifted(alpha, sigma, x, beta, y, dots)
  separate        h.spmv_axpby(alpha, x, beta, y); y.add_(x, alpha=-alpha sigma); torch.dot(x, y); torch.dot(y, y)
  dots_scratch    shifted_dots on a second handle created with option "axpby_fused" = 0 (fold / main-kernel handles)
ms = median over the rounds, spread = (max - min) / median.  Modelled bytes: axpby's (scripts/axpby_cost.py's model)
plus m v for the read of x[i] (the shift or dots[0]); the separate arm adds the axpy (3 m v) and the two dots (3 m v:
x and y, then y again).  "dot_path" (0 scratch pass, 1 main kernel, 2 fold).
A full-size check: y of the shifted call against fl(fl(alpha fl(s - fl(sigma x))) + fl(beta y_old)) in numpy, s =
spmv()'s y on the same handle, bit for bit; both dots within the header's bound L 2^-53 sum |p_i| of math.fsum of the
products (plus the one rounding of fsum).
The card's name and power limit are read in the same run.  --small: 64x fewer rows, for checking the script."""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from axpby_cost import ALPHA, BETA, PATHS, card, timed  # noqa: E402
from axpby_dot_cost import within_bound  # noqa: E402

SIGMA = 0.25
# (workload, method, whether bench.py flushes L2 before every timed call)
RUNS = [("c1", "parallel", True), ("c2", "parallel", False), ("c3", "csr5", False), ("c4", "sell", False),
        ("c5sq", "parallel", False)]


def make_workload(bench, name, small):
    """(device matrix, description, seed): bench.py's workload, or the fp64 / square variants named above."""
    from spmv_b200 import api, matrices as M
    sh = 6 if small else 0
    if name == "c3":
        A = api.gen_rmat(24 - sh, 16, M.SEED_C3, 8)
        return A, f"C3 R-MAT scale {24 - sh} edge-factor 16 (duplicates kept), fp64 CSR", M.SEED_C3
    if name == "c5sq":
        rows = 1 << (25 - sh)
        A = api.gen_uniform(rows, rows, 16, M.SEED_C5, 0, False, 8)
        return A, f"C5-shaped square: uniform-random {rows}x{rows}, 16 nnz/row, fp64 CSR", M.SEED_C5
    A, n, vsize, desc, seed, _ = bench.make_workload(name, small)
    assert vsize == 8 and n == A.m, name
    return A, desc, seed


def run_one(api, torch, bench, name, method, flushed, steps, rounds, small, log):
    A, desc, seed = make_workload(bench, name, small)
    handles = []
    try:
        return measure(api, torch, bench, A, desc, seed, name, method, flushed, steps, rounds, log, handles)
    finally:  # also when a step fails, so that the next workload finds the memory free
        for hh in handles:
            hh.destroy()
        A.destroy()
        torch.cuda.empty_cache()


def measure(api, torch, bench, A, desc, seed, name, method, flushed, steps, rounds, log, handles):
    m, nnz, bmin = A.m, A.nnz, A.min_bytes()
    x = torch.empty(m, dtype=torch.float64, device="cuda")
    api.gen_x(x, m, seed, False, 8)
    y0 = torch.empty(m, dtype=torch.float64, device="cuda")
    api.gen_x(y0, m, seed + 1, False, 8)
    y = y0.clone()
    dots = torch.zeros(2, dtype=torch.float64, device="cuda")
    h = A.handle(bench.METHODS[method])
    handles.append(h)
    path = h.info("dot_path")
    hs = None
    if path != 0:
        api.set_option("axpby_fused", 0)
        try:
            hs = A.handle(bench.METHODS[method])
            handles.append(hs)
        finally:
            api.set_option("axpby_fused", 1)
        assert hs.info("dot_path") == 0
    flush_buf = torch.zeros(max(2 * torch.cuda.get_device_properties(0).L2_cache_size, 1 << 28), dtype=torch.uint8,
                            device="cuda") if flushed else None
    flush = (lambda: flush_buf.max()) if flushed else None
    L = api.lib()

    def shifted():
        if L.spmv_b200_spmv_shifted(h.h, ALPHA, SIGMA, x.data_ptr(), BETA, y.data_ptr(), None) != 0:
            raise RuntimeError(api.last_error())

    def separate():
        h.spmv_axpby(ALPHA, x, BETA, y)
        y.add_(x, alpha=-ALPHA * SIGMA)
        torch.dot(x, y, out=dots[0])
        torch.dot(y, y, out=dots[1])

    arms = {"axpby": lambda: h.spmv_axpby(ALPHA, x, BETA, y), "shifted": shifted,
            "shifted_dots": lambda: h.spmv_shifted(ALPHA, SIGMA, x, BETA, y, dots), "separate": separate}
    if hs is not None:
        arms["dots_scratch"] = lambda: hs.spmv_shifted(ALPHA, SIGMA, x, BETA, y, dots)
    for fn in arms.values():  # warm-up: module loads, the partials, the scratch array, torch's allocator
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    samples = {k: [] for k in arms}
    for r in range(rounds):
        for k in (list(arms) if r % 2 == 0 else list(reversed(arms))):
            y.copy_(y0)
            samples[k].append(timed(torch, arms[k], steps, flush))
    mv = m * 8
    ax_bytes = bmin + mv + (2 * mv if path == 0 else 0)
    model = {"axpby": ax_bytes, "shifted": ax_bytes + mv, "shifted_dots": ax_bytes + mv,
             "separate": ax_bytes + 6 * mv, "dots_scratch": bmin + 4 * mv}
    rec = {"workload": desc, "method": method, "kernel": h.kernel, "x_bands": h.info("x_bands"),
           "dot_path": f"{path} ({PATHS[path]})", "m": m, "n": m, "nnz": nnz,
           "l2": "flushed before every timed call, timed call by call" if flushed else "larger than L2, not flushed",
           "steps_per_round": steps, "rounds": rounds, "arms": {}}
    base = float(np.median(samples["axpby"]))
    for k, v in samples.items():
        med = float(np.median(v))
        rec["arms"][k] = {"ms": round(med, 5), "spread": round((max(v) - min(v)) / med, 4),
                          "ms_rounds": [round(s, 5) for s in v], "modelled_bytes": int(model[k]),
                          "time_over_axpby": round(med / base, 4)}
    # full-size check
    s = torch.empty(m, dtype=torch.float64, device="cuda")
    h.spmv(x, s)
    y.copy_(y0)
    xy, yy = h.spmv_shifted(ALPHA, SIGMA, x, BETA, y)
    torch.cuda.synchronize()
    sn, xn, y0n, yn = s.cpu().numpy(), x.cpu().numpy(), y0.cpu().numpy(), y.cpu().numpy()
    want = ALPHA * (sn - SIGMA * xn) + BETA * y0n
    rec["full_size_check"] = {"y_bits_equal_formula": bool(np.array_equal(yn.view(np.int64), want.view(np.int64))),
                              "x.y": within_bound(xy, xn, yn), "y.y": within_bound(yy, yn, yn)}
    rec["shifted_dots_vs_separate"] = round(rec["arms"]["shifted_dots"]["ms"] / rec["arms"]["separate"]["ms"], 4)
    rec["shifted_vs_axpby"] = round(rec["arms"]["shifted"]["ms"] / base, 4)
    if hs is not None:
        rec["shifted_dots_vs_scratch_pass"] = round(rec["arms"]["shifted_dots"]["ms"] / rec["arms"]["dots_scratch"]["ms"], 4)
    c = rec["full_size_check"]
    log(f"[{name} {method}] path {rec['dot_path']} | " +
        " | ".join(f"{k} {v['ms']:.4f} ms (x{v['time_over_axpby']:.3f}, spread {v['spread']:.3f})" for k, v in rec["arms"].items()) +
        f" | y bits {c['y_bits_equal_formula']}, x.y {c['x.y']['ok']}, y.y {c['y.y']['ok']}")
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_shifted.json"))
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
    result = {"card": card(), "alpha": ALPHA, "sigma": SIGMA, "beta": BETA, "runs": []}
    log(result["card"])
    for name, method, flushed in RUNS:
        free, total = torch.cuda.mem_get_info()
        try:
            result["runs"].append(run_one(api, torch, bench, name, method, flushed, args.steps, args.rounds, args.small, log))
        except RuntimeError as e:  # the card is shared: a workload that does not fit next to other work is not measured
            log(f"[{name} {method}] not measured: {e} ({free / 2**30:.1f} of {total / 2**30:.1f} GiB free before it)")
            result["runs"].append({"workload": name, "method": method, "not_measured": str(e),
                                   "free_gib_before": round(free / 2**30, 1)})
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    key = lambda r: f"{r['workload'][:2]} {r['method']}"
    runs = [r for r in result["runs"] if "not_measured" not in r]
    print(json.dumps({"out": args.out, "not_measured": [key(r) for r in result["runs"] if "not_measured" in r],
                      "all_checks": all(r["full_size_check"]["y_bits_equal_formula"] and r["full_size_check"]["x.y"]["ok"]
                                        and r["full_size_check"]["y.y"]["ok"] for r in runs),
                      "shifted_dots_vs_separate": {key(r): r["shifted_dots_vs_separate"] for r in runs},
                      "shifted_vs_axpby": {key(r): r["shifted_vs_axpby"] for r in runs},
                      "shifted_dots_vs_scratch_pass": {key(r): r.get("shifted_dots_vs_scratch_pass") for r in runs}}))


if __name__ == "__main__":
    main()
