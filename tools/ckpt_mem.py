"""Memory and time of checkpointed training (admm_solve(..., ckpt_interval=K)) on large frames.

    python tools/ckpt_mem.py [--reps 5] [--warmup 2] [--out FILE.json]

One training step = forward + backward of admm_solve with a learnable PSF, lambda and rho (the input is data: no
gradient for it).  For each workload and K in {0 (every iteration kept), 10, -1 (ceil(sqrt(maxit - 1)))} it reports
  peak_gb        torch.cuda.max_memory_allocated over one step, minus what was allocated before it (inputs, parameters):
                 the saved state, the forward and backward workspaces and the gradients
  saved_gb       the saved-state buffer alone (admm_query_saved_ex)
  ms             median step time over --reps steps after --warmup untimed ones, CUDA events around each step
The card name and power limit are read in the same run.  Both K = 0 workloads fit in 180 GB.
"""
import argparse
import json
import math
import os
import statistics
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from f64_bench import card_info                          # noqa: E402
from oracle import admm_oracle as O                       # noqa: E402
from torch_admm_deconv_b200 import _lib                   # noqa: E402
from torch_admm_deconv_b200.eops.deconv import admm_solve  # noqa: E402

# name: (shape, gaussian PSF size, sigma, maxit)
WORKLOADS = {
    "cfg3_1x3x2160x3840_k63_n200": ((1, 3, 2160, 3840), 63, 10.0, 200),
    "hd_8x3x1080x1920_k15_n100": ((8, 3, 1080, 1920), 15, 2.5, 100),
}
KS = (0, 10, -1)


def run(name, reps, warmup, dev):
    shape, k, sigma, maxit = WORKLOADS[name]
    psf = O.make_psf("gauss", k, sigma)
    g = torch.Generator(dev).manual_seed(11)
    x = torch.rand(shape, device=dev, generator=g)
    gout = torch.randn(shape, device=dev, generator=g)
    kern = torch.tensor(psf[None, None], device=dev, requires_grad=True)
    lam = torch.tensor([0.02], device=dev, requires_grad=True)
    rho = torch.tensor([0.04], device=dev, requires_grad=True)
    lib = _lib.load()
    B, C, H, W = shape
    rows = []
    for K in KS:
        Keff = int(math.ceil(math.sqrt(maxit - 1))) if K < 0 else K

        def step():
            admm_solve(x, lam, rho, kern, False, maxit, ckpt_interval=K).backward(gout)

        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        kern.grad = lam.grad = rho.grad = None
        base = torch.cuda.memory_allocated(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        step()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated(dev) - base
        times = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step()
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b))
        saved = lib.admm_query_saved_ex(B * C, H, W, k, 0, maxit, Keff if Keff >= 2 else 0)
        r = {"workload": name, "shape": list(shape), "k": k, "maxit": maxit, "K": K, "K_eff": Keff,
             "peak_gb": round(peak / 1e9, 3), "saved_gb": round(saved / 1e9, 3),
             "ms": round(statistics.median(times), 3), "ms_min_max": [round(min(times), 3), round(max(times), 3)]}
        rows.append(r)
        print(json.dumps(r), flush=True)
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="write the result lines (JSON) to this file too")
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ckpt_mem.py measures on a CUDA device; none found")
    dev = torch.device("cuda:0")
    name, power = card_info(dev)
    head = {"card": name, "power_limit_w": power, "reps": a.reps, "warmup": a.warmup, "statistic": "median",
            "peak": "max_memory_allocated over one step minus the allocation before it"}
    print(json.dumps(head), flush=True)
    lines = [head]
    for n in (a.only.split(",") if a.only else list(WORKLOADS)):
        lines += run(n, a.reps, a.warmup, dev)
    print("\n%-30s %4s %10s %10s %10s" % ("workload", "K", "peak GB", "saved GB", "ms/step"))
    for r in lines[1:]:
        print("%-30s %4d %10.2f %10.2f %10.1f" % (r["workload"], r["K"], r["peak_gb"], r["saved_gb"], r["ms"]))
    if a.out:
        with open(a.out, "w") as f:
            for l in lines:
                f.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()
