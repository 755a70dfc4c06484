"""What the fused dot of spmv_b200_spmv_axpby_dot costs: against spmv_b200_spmv_axpby alone, against the caller's
alternative (spmv_b200_spmv_axpby, then torch.dot over the new y), and against its own scratch pass, on the workloads
of scripts/axpby_cost.py (bench.py's matrices, all three paths), one B200.

    python scripts/axpby_dot_cost.py [--out profiles/r05_axpby_dot.json] [--steps 20] [--rounds 5] [--small]

Per workload and method:
  * the arms below, timed with CUDA events as axpby_cost.py times them (C1 flushed before every call, the others
    larger than L2), in `rounds` rounds that alternate the arms; alpha = 0.5, beta = -0.75, the dot into a device
    double (no host synchronisation in the loop):
      axpby          h.spmv_axpby(alpha, x, beta, y)
      dot_wy         h.spmv_axpby_dot(alpha, x, beta, y, y, d)      (|y|^2)
      dot_wx         h.spmv_axpby_dot(alpha, x, beta, y, x, d)      (square matrices: CG's p . Ap)
      axpby_torchdot h.spmv_axpby(alpha, x, beta, y); torch.dot(y, y, out=d)   (what a client does without the dot)
      dot_scratch    dot_wy on a second handle created with option "axpby_fused" = 0 (fold / main-kernel handles)
    ms = median over the rounds, spread = (max - min) / median;
  * modelled bytes: axpby's (axpby_cost.py's model) plus m v when w is x (w = y costs nothing more); the caller's
    alternative reads y again (m v); the scratch pass adds 2 m v;
  * "dot_path" (0 scratch pass, 1 main kernel, 2 fold);
  * a full-size check: y of spmv_axpby_dot equals spmv_axpby's bits, and the dot lies within the header's bound
    L 2^-53 sum |p_i| of math.fsum of the products (plus the one rounding of fsum).
The card's name and power limit are read in the same run.  --small: 64x fewer rows, for checking the script."""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from axpby_cost import ALPHA, BETA, PATHS, RUNS, card, timed  # noqa: E402


def within_bound(dot, w, y):
    p = w.astype(np.float64) * y.astype(np.float64)
    L = 18 + -(-(len(y) + 2) // 1024)
    exact = math.fsum(p)
    err, bound = abs(dot - exact), L * 2.0 ** -53 * float(np.sum(np.abs(p))) + 2.0 ** -53 * abs(exact)
    return {"dot": dot, "fsum": exact, "error": err, "bound": bound, "ok": bool(err <= bound)}


def run_one(api, torch, bench, name, method, flushed, steps, rounds, small, log):
    wl = bench.make_workload(name, small)
    A, handles = wl[0], []
    try:
        return measure(api, torch, bench, wl, name, method, flushed, steps, rounds, log, handles)
    finally:  # also when a step fails, so that the next workload finds the memory free
        for hh in handles:
            hh.destroy()
        A.destroy()
        torch.cuda.empty_cache()


def measure(api, torch, bench, wl, name, method, flushed, steps, rounds, log, handles):
    A, n, vsize, desc, seed, _ = wl
    tdt = torch.float64 if vsize == 8 else torch.float32
    m, nnz, bmin = A.m, A.nnz, A.min_bytes()
    x = torch.empty(n, dtype=tdt, device="cuda")
    api.gen_x(x, n, seed, False, vsize)
    y0 = torch.empty(m, dtype=tdt, device="cuda")
    api.gen_x(y0, m, seed + 1, False, vsize)
    y = y0.clone()
    d = torch.zeros(1, dtype=torch.float64, device="cuda")
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
    y64 = torch.empty(m, dtype=torch.float64, device="cuda")

    def caller_alternative():
        h.spmv_axpby(ALPHA, x, BETA, y)
        if vsize == 8:
            torch.dot(y, y, out=d[0])
        else:  # the contract's dot of an fp32 handle is taken in double
            y64.copy_(y)
            torch.dot(y64, y64, out=d[0])

    arms = {"axpby": lambda: h.spmv_axpby(ALPHA, x, BETA, y),
            "dot_wy": lambda: h.spmv_axpby_dot(ALPHA, x, BETA, y, y, d),
            "axpby_torchdot": caller_alternative}
    if m == n:
        arms["dot_wx"] = lambda: h.spmv_axpby_dot(ALPHA, x, BETA, y, x, d)
    if hs is not None:
        arms["dot_scratch"] = lambda: hs.spmv_axpby_dot(ALPHA, x, BETA, y, y, d)
    for fn in arms.values():  # warm-up: module loads, the partials, the scratch array, torch's allocator
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    samples = {k: [] for k in arms}
    for r in range(rounds):
        for k in (list(arms) if r % 2 == 0 else list(reversed(arms))):
            y.copy_(y0)
            samples[k].append(timed(torch, arms[k], steps, flush))
    mv = m * vsize
    ax_bytes = bmin + mv + (2 * mv if path == 0 else 0)
    model = {"axpby": ax_bytes, "dot_wy": ax_bytes, "dot_wx": ax_bytes + mv, "axpby_torchdot": ax_bytes + mv,
             "dot_scratch": bmin + 3 * mv}
    rec = {"workload": desc, "method": method, "kernel": h.kernel, "x_bands": h.info("x_bands"),
           "dot_path": f"{path} ({PATHS[path]})", "m": m, "n": n, "nnz": nnz,
           "l2": "flushed before every timed call, timed call by call" if flushed else "larger than L2, not flushed",
           "steps_per_round": steps, "rounds": rounds, "arms": {}}
    base = float(np.median(samples["axpby"]))
    for k, v in samples.items():
        med = float(np.median(v))
        rec["arms"][k] = {"ms": round(med, 5), "spread": round((max(v) - min(v)) / med, 4),
                          "ms_rounds": [round(s, 5) for s in v], "modelled_bytes": int(model[k]),
                          "time_over_axpby": round(med / base, 4)}
    # full-size check
    itype = torch.int64 if vsize == 8 else torch.int32
    y.copy_(y0)
    h.spmv_axpby(ALPHA, x, BETA, y)
    want = y.clone()
    checks = {}
    for tag, hh, w in (("w=y", h, None), ("w=x", h, x if m == n else False), ("scratch handle, w=y", hs, None)):
        if hh is None or w is False:
            continue
        y.copy_(y0)
        dot = hh.spmv_axpby_dot(ALPHA, x, BETA, y, w)
        torch.cuda.synchronize()
        yy = y.cpu().numpy()
        checks[tag] = {"y_bits_equal_axpby": bool(torch.equal(y.view(itype), want.view(itype))),
                       **within_bound(dot, yy if w is None else x.cpu().numpy(), yy)}
    rec["full_size_check"] = checks
    rec["dot_vs_axpby_torchdot"] = round(rec["arms"]["dot_wy"]["ms"] / rec["arms"]["axpby_torchdot"]["ms"], 4)
    if hs is not None:
        rec["dot_vs_scratch_pass"] = round(rec["arms"]["dot_wy"]["ms"] / rec["arms"]["dot_scratch"]["ms"], 4)
    log(f"[{name} {method}] path {rec['dot_path']} | " +
        " | ".join(f"{k} {v['ms']:.4f} ms (x{v['time_over_axpby']:.3f}, spread {v['spread']:.3f})" for k, v in rec["arms"].items()) +
        f" | checks {{{', '.join(f'{k}: {v['y_bits_equal_axpby']} {v['ok']}' for k, v in checks.items())}}}")
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_axpby_dot.json"))
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
                      "all_checks": all(c["y_bits_equal_axpby"] and c["ok"] for r in runs
                                        for c in r["full_size_check"].values()),
                      "dot_vs_axpby_torchdot": {key(r): r["dot_vs_axpby_torchdot"] for r in runs},
                      "dot_vs_scratch_pass": {key(r): r.get("dot_vs_scratch_pass") for r in runs}}))


if __name__ == "__main__":
    main()
