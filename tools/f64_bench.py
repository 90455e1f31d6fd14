"""Float64 solve (fft_admm_tv_f64) against the float32 solver on the same workloads.

    python tools/f64_bench.py [--reps 15] [--warmup 3] [--out FILE.json]

For each workload it times, with CUDA events around one call (median of --reps after --warmup untimed calls):
  f64          fft_admm_tv_f64: the generic kernels in double
  f32_generic  fft_admm_tv with option force_generic = 1 and one stream: the same kernels and schedule in float, so the
               ratio f64 / f32_generic is the cost of the precision alone
  f32_default  fft_admm_tv as shipped (specialised power-of-two / cluster / large-frame kernels, split streams)
and reports G pixel-it/s (B*C*H*W*maxit / time) and the share of the HBM roofline the float64 run reaches for its
algorithmic traffic: 72 B per element-iteration for a forward (row pass 48, column pass 24), 192 B for a training step,
at 6551 GB/s (the bandwidth measured on this card type, DESIGN.md section 4).  L2 (126 MB) is flushed before every timed
call by a 256 MB fill outside the timed interval.  The card name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import admm_oracle as O                       # noqa: E402
from torch_admm_deconv_b200 import _lib, fft_admm_tv, fft_admm_tv_f64   # noqa: E402
from torch_admm_deconv_b200.eops import deconv as D      # noqa: E402

HBM_GBS = 6551.0
# name: (shape, psf kind, k, sigma, iso, maxit, training)
WORKLOADS = {
    "cfg1x8_256_k15_n50": ((8, 3, 256, 256), "gauss", 15, 2.5, False, 50, False),
    "cfg2_512_k31_n100": ((2, 3, 512, 512), "motion", 31, None, False, 100, False),
    "hd_1080x1920_k15_n50": ((1, 3, 1080, 1920), "gauss", 15, 2.5, False, 50, False),
    "ref_eval_256_iso_n100": ((8, 3, 256, 256), None, 0, None, True, 100, False),
    "train_32x3x256_k15_n10": ((32, 3, 256, 256), "gauss", 15, 2.5, False, 10, True),
}


def card_info(dev):
    name = torch.cuda.get_device_name(dev)
    power = None
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev.index or 0)
        power = pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
    except Exception:
        try:
            r = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=30)
            power = float(r.stdout.strip().splitlines()[0])
        except Exception:
            pass
    return name, power


def make_inputs(shape, kind, k, sigma, dtype, dev):
    psf = O.make_psf(kind, k, sigma) if kind else None
    x = torch.from_numpy(O.make_blurred(shape, psf, seed=1234)).to(dev, dtype)
    kern = torch.from_numpy(psf[None, None]).to(dev, dtype) if kind else torch.empty(0, dtype=dtype, device=dev)
    return x, kern


def time_call(fn, reps, warmup, flush):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times), min(times), max(times)


def run(name, reps, warmup, dev, flush):
    shape, kind, k, sigma, iso, maxit, training = WORKLOADS[name]
    res = {"workload": name, "shape": list(shape), "k": k, "iso": iso, "maxit": maxit, "training": training}
    for arm in ("f64", "f32_generic", "f32_default"):
        dtype = torch.float64 if arm == "f64" else torch.float32
        x, kern = make_inputs(shape, kind, k, sigma, dtype, dev)
        lam = torch.tensor([0.02], dtype=dtype, device=dev, requires_grad=training)
        rho = torch.tensor([0.04], dtype=dtype, device=dev, requires_grad=training)
        solve = fft_admm_tv_f64 if arm == "f64" else fft_admm_tv
        if training:
            x.requires_grad_(True)
            gout = torch.randn(shape, dtype=dtype, device=dev, generator=torch.Generator(dev).manual_seed(7))

            def fn():
                solve(x, lam, rho, kern, iso, maxit).backward(gout)
        else:
            def fn():
                with torch.no_grad():
                    solve(x, lam, rho, kern, iso, maxit)
        split = D.SPLIT_STREAMS
        try:
            _lib.set_option("force_generic", 1 if arm == "f32_generic" else 0)
            D.SPLIT_STREAMS = 1 if arm == "f32_generic" else split
            med, lo, hi = time_call(fn, reps, warmup, flush)
        finally:
            _lib.set_option("force_generic", 0)
            D.SPLIT_STREAMS = split
        res[arm + "_ms"] = round(med, 4)
        res[arm + "_ms_min_max"] = [round(lo, 4), round(hi, 4)]
        del x, kern
    elems = int(np.prod(shape)) * maxit
    res["f64_gpix_it_s"] = round(elems / (res["f64_ms"] * 1e-3) / 1e9, 3)
    res["f32_generic_gpix_it_s"] = round(elems / (res["f32_generic_ms"] * 1e-3) / 1e9, 3)
    res["f32_default_gpix_it_s"] = round(elems / (res["f32_default_ms"] * 1e-3) / 1e9, 3)
    bpe = 192 if training else 72
    res["f64_bytes_per_elem_it"] = bpe
    res["f64_hbm_roofline_share"] = round(bpe * elems / (res["f64_ms"] * 1e-3) / (HBM_GBS * 1e9), 4)
    res["f64_over_f32_generic"] = round(res["f64_ms"] / res["f32_generic_ms"], 3)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="write the result lines (JSON) to this file too")
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("f64_bench.py measures on a CUDA device; none found")
    if a.reps < 10:
        raise SystemExit("--reps must be >= 10")
    dev = torch.device("cuda:0")
    name, power = card_info(dev)
    head = {"card": name, "power_limit_w": power, "reps": a.reps, "warmup": a.warmup, "statistic": "median",
            "l2": "flushed before every timed call (256 MB fill, outside the timed interval)", "hbm_gbs": HBM_GBS}
    lines = [head]
    print(json.dumps(head), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    names = a.only.split(",") if a.only else list(WORKLOADS)
    for n in names:
        r = run(n, a.reps, a.warmup, dev, flush)
        lines.append(r)
        print(json.dumps(r), flush=True)
    print("\n%-26s %10s %14s %14s %10s %8s" % ("workload", "f64 ms", "f32 generic ms", "f32 default ms", "f64 Gpix-it/s", "f64 HBM"))
    for r in lines[1:]:
        print("%-26s %10.3f %14.3f %14.3f %10.2f %7.1f%%" % (r["workload"], r["f64_ms"], r["f32_generic_ms"], r["f32_default_ms"],
                                                          r["f64_gpix_it_s"], 100 * r["f64_hbm_roofline_share"]))
    if a.out:
        with open(a.out, "w") as f:
            for l in lines:
                f.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()
