"""Cost of a λ map (spatially varying regularisation, DESIGN.md section 11) against the scalar solve, on bench.py's inputs.

    python tools/lmap_bench.py [--reps 7] [--warmup 2] [--out FILE.json]

Times, with CUDA events around one call (after --warmup untimed calls; median, min and max of --reps; the variants of one
workload alternate call by call, no L2 flush):
  cfg2 inference (64x3x512x512, 31x31 motion PSF, 100 iterations): scalar λ, a shared (1, 1, H, W) map, a full (B, C, H, W)
       map.  The map solves run their iterations on the generic row kernel, the scalar one on the power-of-two kernel.
  cfg4 training step (32x3x256x256, no PSF, 10 iterations; ADMMDeconv, loss = mean(out^2), forward + backward): the
       scalar learnable λ and a learnable shared map Parameter.
  1x3x2160x3840 inference (63x63 Gaussian PSF, 200 iterations): scalar λ (large-frame row and column kernels) and a
       shared map (generic rows, large-frame columns on the row-major layout).
The card name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench                                               # noqa: E402  (definitions only; its main() is not run)
from torch_admm_deconv_b200 import ADMMDeconv             # noqa: E402
from torch_admm_deconv_b200.eops.deconv import admm_solve  # noqa: E402
sys.path.insert(0, os.path.join(ROOT, "tools"))
from f64_bench import card_info                            # noqa: E402


def timed_alternating(fns, reps, warmup):
    """{label: timing} for callables run in turn, one call each per round."""
    for _ in range(warmup):
        for fn in fns.values():
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ms[k].append(a.elapsed_time(b))
    return {k: {"ms_median": statistics.median(v), "ms_min": min(v), "ms_max": max(v)} for k, v in ms.items()}


def smooth_map(shape, dev, seed=5):
    """A positive λ map around bench.LAMBDA (0.5x .. 1.5x), smooth in space, as a predicted or hand-made map would be."""
    g = torch.Generator().manual_seed(seed)
    m = torch.rand(shape, generator=g)
    m = torch.nn.functional.avg_pool2d(m.reshape(-1, 1, *shape[-2:]), 9, 1, 4, count_include_pad=False).reshape(shape)
    return (bench.LAMBDA * (0.5 + m)).to(dev)


def inference(name, shape, kind, k, sigma, maxit, variants, reps, warmup, dev):
    B, C, H, W = shape
    x, kern = bench.make_inputs_torch(shape, kind, k, sigma)
    x, kern = x.to(dev), kern.to(dev)
    maps = {"scalar": bench.LAMBDA, "shared_map": smooth_map((1, 1, H, W), dev), "full_map": smooth_map((B, C, H, W), dev, 6)}
    fns = {v: (lambda m=maps[v]: admm_solve(x, m, bench.RHO, kern, False, maxit)) for v in variants}
    with torch.no_grad():
        t = timed_alternating(fns, reps, warmup)
        ref = fns["scalar"]()
        # a map filled with the scalar λ: the same iterate up to the row kernel's rounding (different kernel route)
        const = admm_solve(x, torch.full((1, 1, H, W), bench.LAMBDA, device=dev), bench.RHO, kern, False, maxit)
        diff = float((const - ref).abs().max() / ref.abs().max())
    elems = B * C * H * W
    for v in t:
        t[v]["ns_per_element_iteration"] = t[v]["ms_median"] * 1e6 / (elems * maxit)
        t[v]["vs_scalar"] = t[v]["ms_median"] / t["scalar"]["ms_median"]
    return {"workload": name, "shape": list(shape), "psf": [kind, k], "maxit": maxit, "runs": t,
            "constant_map_max_rel_diff_to_scalar": diff}


def training(reps, warmup, dev):
    B, C, H, W, kind, k, sigma, maxit = bench.WORKLOADS["cfg4"]
    g = torch.Generator().manual_seed(1234)
    x = torch.rand(B, C, H, W, generator=g).to(dev)
    models = {}
    for v in ("scalar", "shared_map"):
        m = ADMMDeconv((), max_iters=maxit, lmbda=None, rho=None, iso=False).to(dev)
        with torch.no_grad():
            m.rho.fill_(bench.RHO)
            m.lmbda.fill_(bench.LAMBDA)
        if v == "shared_map":
            m.lmbda = torch.nn.Parameter(smooth_map((1, 1, H, W), dev))
        models[v] = m

    def step(m):
        m.zero_grad(set_to_none=True)
        (m(x) ** 2).mean().backward()

    t = timed_alternating({v: (lambda m=m: step(m)) for v, m in models.items()}, reps, max(warmup, 3))
    t["shared_map"]["vs_scalar"] = t["shared_map"]["ms_median"] / t["scalar"]["ms_median"]
    return {"workload": "cfg4_train_step", "shape": [B, C, H, W], "maxit": maxit, "runs": t}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("lmap_bench.py measures on a CUDA device; none found")
    dev = torch.device("cuda:0")
    name, power = card_info(dev)
    res = {"card": name, "power_limit_w": power, "reps": a.reps, "warmup": a.warmup,
           "timing": "CUDA events around one call, variants alternating, no L2 flush", "results": []}
    def infer(name, variants):
        B, C, H, W, kind, k, sigma, maxit = bench.WORKLOADS[name]
        return inference(name, (B, C, H, W), kind, k, sigma, maxit, variants, a.reps, a.warmup, dev)
    jobs = [lambda: infer("cfg2", ("scalar", "shared_map", "full_map")), lambda: training(a.reps, a.warmup, dev),
            lambda: infer("cfg3", ("scalar", "shared_map"))]
    for job in jobs:
        r = job()
        res["results"].append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"card": name, "power_limit_w": power}))


if __name__ == "__main__":
    main()
