"""Cost of residual checks and what a tolerance saves (admm_solve_tol, DESIGN.md section 10), on bench.py's workloads.

    python tools/tol_bench.py [--workloads cfg2,cfg3] [--reps 7] [--warmup 2] [--out FILE.json]

For cfg2 (64x3x512x512, 31x31 motion PSF, 100 iterations) and cfg3 (1x3x2160x3840, 63x63 Gaussian PSF, 200 iterations), on
bench.py's seeded inputs and lambda / rho, inference, it times one call with CUDA events (after --warmup untimed calls;
median, min and max of --reps):
  fixed        admm_solve at maxit (as shipped: the cluster / split-stream choices of the library included)
  hist_M10     admm_solve_tol, rtol = atol = 0, check_every = 10: maxit iterations with a residual history
  hist_M1      the same with a check after every iteration
  rtol_1e-3    admm_solve_tol, rtol = 1e-3, check_every = 10: iterations reached, time, and the largest difference of the
  rtol_1e-4    early-stopped output to the `fixed` output, relative to its largest magnitude
  rtol_needed_M10  per check (M = 10) the smallest rtol (atol = 0) at which every plane would have converged there
The card name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench                                               # noqa: E402  (definitions only; its main() is not run)
from torch_admm_deconv_b200.eops.deconv import admm_solve, admm_solve_tol   # noqa: E402
sys.path.insert(0, os.path.join(ROOT, "tools"))
from f64_bench import card_info                            # noqa: E402


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms, res = [], None
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        res = fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return {"ms_median": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms)}, res


def run(name, reps, warmup, dev):
    B, C, H, W, kind, k, sigma, maxit = bench.WORKLOADS[name]
    x, kern = bench.make_inputs_torch((B, C, H, W), kind, k, sigma)
    x, kern = x.to(dev), kern.to(dev)
    lam, rho = bench.LAMBDA, bench.RHO
    rows = {}
    with torch.no_grad():
        t, ref = timed(lambda: admm_solve(x, lam, rho, kern, False, maxit), reps, warmup)
        rows["fixed"] = dict(t, iters=maxit)
        scale = float(ref.abs().max())
        for label, rtol, every in (("hist_M10", 0.0, 10), ("hist_M1", 0.0, 1), ("rtol_1e-3", 1e-3, 10), ("rtol_1e-4", 1e-4, 10)):
            t, (out, info) = timed(lambda: admm_solve_tol(x, lam, rho, kern, False, maxit, rtol=rtol, check_every=every),
                                   reps, warmup)
            row = dict(t, iters=info.iters, checks=int(info.residuals.shape[0]),
                       overhead_vs_fixed=t["ms_median"] / rows["fixed"]["ms_median"] - 1.0,
                       max_rel_diff_to_fixed=float((out - ref).abs().max()) / scale)
            if rtol == 0.0 and info.residuals.shape[0]:
                last = info.residuals[-1]
                row["last_check_max_r"] = float(last[..., 0].max())
                row["last_check_max_s"] = float(last[..., 1].max())
            rows[label] = row
        # the smallest rtol (atol = 0) that every plane meets at each check of M = 10: from a run whose tolerance is
        # never met, eps / rtol = the norms
        small = float(np.float32(1e-9))
        _, info = admm_solve_tol(x, lam, rho, kern, False, maxit, rtol=small, check_every=10)
        h = info.residuals.double()
        need = torch.maximum(h[..., 0] / (h[..., 2] / small), h[..., 1] / (h[..., 3] / small)).amax(dim=(1, 2))
        rows["rtol_needed_M10"] = {"checks_after": [10 * (i + 1) for i in range(len(need))],
                                   "rtol": [float(v) for v in need]}
    return {"workload": name, "shape": [B, C, H, W], "psf": [kind, k], "maxit": maxit, "runs": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg2,cfg3")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tol_bench.py measures on a CUDA device; none found")
    dev = torch.device("cuda:0")
    name, power = card_info(dev)
    res = {"card": name, "power_limit_w": power, "reps": a.reps, "warmup": a.warmup,
           "timing": "CUDA events around one call, no L2 flush", "results": []}
    for w in a.workloads.split(","):
        r = run(w, a.reps, a.warmup, dev)
        res["results"].append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"card": name, "power_limit_w": power}))


if __name__ == "__main__":
    main()
