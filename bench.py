#!/usr/bin/env python
"""bench.py -- headline benchmark of the ADMM-TV deconvolution hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg5|cfg3|cfg1|cfg4]

A "step" is ONE full solve (`fft_admm_tv`) over one batch of synthetic blurred images.  The default
workload is BASELINE.json configs[1]: batch 64 RGB 512x512, 31x31 motion-blur PSF, 100 ADMM iterations,
fp32, iso=False.  With N > 1 (launched by torchrun, one rank per GPU) every rank solves its own batch of
the same size (weak scaling, no collective on the solve path: planes are independent for iso=False).

Output: ONE JSON line on rank 0 (see the keys below).  `value` is whole-job Mpixel*ADMM-iterations/s with
inputs resident in HBM, timed with the per-kernel profiling events OFF; `e2e` is the same metric through the
public Python API with pinned-host inputs and outputs (H2D + D2H inside the timed region); `roofline` holds the
achieved algorithmic HBM bandwidth of the iteration's two kernels (CUDA events around every launch, taken in a
SECOND identical pass so they do not perturb `value`) against the measured copy peak in MEASURED_PEAKS.json:
`frac` is the WHOLE iteration (row pass + column pass, 36 B/element), `frac_rows` / `frac_cols` the two kernels;
`cpu_baseline` is the UNMODIFIED reference (`admmtor.eops.deconv.fft_admm_tv`, pip-installed into baseline/_ref
by baseline/install_ref.py) timed on this box's host cores on a bounded sample (`kind: "reference"`), with the
numpy/scipy oracle port beside it (`port`); `scaling_cfg5` is BASELINE configs[4]: 4096 images split over the N
GPUs (strong scaling), device-timed and end to end.

`--impl reference` times the reference alone on the host cores (rank 0 only): exactly --warmup + --steps steps, each
step a bounded sample of the workload sized from a calibration run so the whole command takes a few minutes; the
line reports the sample, the steps actually run and the measured ms per (sample) step, with "impl": "reference".

`--dump-outputs DIR` (our arm, rank 0) writes what the last timed step returned to its caller as DIR/<name>.npy, so
that two builds can be compared output for output on the same seeded inputs: `out.npy` (float32) for a solve;
`loss.npy`, `grad_lmbda.npy`, `grad_rho.npy` for the cfg4 training step.  An output larger than 64 MB is stored as a
fixed sample of 8 Mi elements (flat indices drawn with torch.Generator seed 0, sorted; the same for every run with
the same arguments).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Mpixel*ADMM-iters/s"
UNIT = "Mpixel*it/s"
LAMBDA, RHO = 0.02, 0.04

WORKLOADS = {
    # name: (B, C, H, W, psf kind, k, psf sigma, maxit)   -- BASELINE.json configs
    "cfg1": (1, 1, 256, 256, "gauss", 15, 2.5, 50),
    "cfg2": (64, 3, 512, 512, "motion", 31, None, 100),
    "cfg3": (1, 3, 2160, 3840, "gauss", 63, 8.0, 200),
    "cfg5": (512, 3, 256, 256, "gauss", 15, 2.5, 50),      # per-GPU shard of the 4096-image sweep at 8 GPUs
    "cfg5full": (4096, 3, 256, 256, "gauss", 15, 2.5, 50), # the whole 4096-image batch on ONE GPU (22 GB of state)
    # unrolled-layer TRAINING step (fwd + bwd, learnable lambda / rho, no kernel): a "step" is one fwd+bwd of the layer
    "cfg4": (32, 3, 256, 256, "gauss", 0, None, 10),
}
TRAIN_BYTES_PER_ELEM = 96.0  # fwd 36 + saved state 8 + bwd 52 per element-iteration (SURVEY.md section 8d)
ROW_BYTES_PER_ELEM = 24.0    # row-pass kernel: read col-spectrum 4 + read q_x,q_y 8 + write q_x,q_y 8 + write row-spectrum 4
COL_BYTES_PER_ELEM = 12.0    # column-pass kernel: read 4 + read A 4 + write 4   (SURVEY.md section 8d)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def make_inputs_torch(shape, kind, k, sigma, seed=1234):
    """Pinned synthetic inputs of SURVEY.md section 8d (torch generator, CPU)."""
    import torch
    from oracle.admm_oracle import make_psf
    B, C, H, W = shape
    g = torch.Generator().manual_seed(seed)
    sharp = torch.rand(B, C, H, W, generator=g)
    psf = torch.from_numpy(make_psf(kind, k, sigma))
    s = int(math.ceil((k - 1) / 2))
    pad = torch.zeros(H, W); pad[:k, :k] = psf
    blurred = torch.fft.irfft2(torch.fft.rfft2(sharp) * torch.fft.rfft2(pad), s=(H, W))
    blurred = torch.roll(blurred, (-s, -s), dims=(-2, -1)) + 0.01 * torch.randn(B, C, H, W, generator=g)
    return blurred.float().contiguous(), psf.float()[None, None].contiguous()


DUMP_MAX_BYTES = 64 << 20
DUMP_SAMPLE = 8 << 20


def dump_array(t):
    """`t` on the host as numpy (float32 / float64); beyond DUMP_MAX_BYTES a fixed seeded sample of its flat elements."""
    import torch
    t = t.detach()
    if t.numel() * t.element_size() > DUMP_MAX_BYTES:
        idx = torch.randint(0, t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
        t = t.reshape(-1)[idx.to(t.device)]
    return t.cpu().numpy()


def write_dump(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index, period=0.1):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------ CPU port
def cpu_port_run(workload, sample_images, sample_iters, repeats=1):
    """Time the oracle port (oracle/admm_oracle.py, spectral form, float32) on the host cores.
    Returns (Mpixel*it/s, seconds, cores, description)."""
    from oracle import admm_oracle as O
    B, C, H, W, kind, k, sigma, maxit = WORKLOADS[workload]
    cores = os.cpu_count() or 1
    nb = max(1, min(sample_images, B))
    psf = O.make_psf(kind, k, sigma)
    x = O.make_blurred((nb, C, H, W), psf, seed=1234)
    # all host threads: images are independent for iso=False, so the batch is split over a thread pool (numpy and
    # pocketfft release the GIL); a single image falls back to multi-threaded FFTs
    from concurrent.futures import ThreadPoolExecutor
    nthreads = min(cores, nb)

    def solve_all(iters):
        if nthreads <= 1:
            return O.admm_tv_spectral_form(x, LAMBDA, RHO, psf[None, None], False, iters, workers=cores)
        chunks = np.array_split(np.arange(nb), nthreads)
        with ThreadPoolExecutor(max_workers=nthreads) as ex:
            return list(ex.map(lambda idx: O.admm_tv_spectral_form(x[idx[0]:idx[-1] + 1], LAMBDA, RHO, psf[None, None],
                                                                    False, iters, workers=1), chunks))
    solve_all(1)                                                                                # warm-up
    best = 1e30
    for _ in range(repeats):
        t0 = time.perf_counter()
        solve_all(sample_iters)
        best = min(best, time.perf_counter() - t0)
    val = nb * H * W * sample_iters / best / 1e6
    desc = ("%d of %d images x %d of %d iterations of %s (per-iteration cost is constant: no data-dependent "
            "control flow, deconv.py:103-115); %d host threads (batch split over a thread pool)"
            % (nb, B, sample_iters, maxit, workload, max(nthreads, 1) if nthreads > 1 else cores))
    return val, best, cores, desc


# ------------------------------------------------------------------------------------------ the real reference on the CPU
def reference_available():
    from baseline import install_ref
    return install_ref.installed()


def make_inputs_numpy(workload, nb, seed=1234):
    from oracle import admm_oracle as O
    B, C, H, W, kind, k, sigma, maxit = WORKLOADS[workload]
    psf = O.make_psf(kind, k, sigma) if k else None
    return O.make_blurred((nb, C, H, W), psf, seed=seed), psf


def reference_run(workload, n_img, n_it, x=None, psf=None):
    """One bounded sample of `workload` through the UNMODIFIED reference (baseline/_ref, admmtor.eops.deconv.fft_admm_tv /
    admmtor.elayers.admmdeconv.ADMMDeconv) on the host cores, fp32, default intra-op threads.  cfg4: forward + backward of the
    reference layer through stock autograd.  Returns (Mpixel*it/s, seconds)."""
    import torch
    from baseline import install_ref
    ref_fft_admm_tv, RefADMMDeconv = install_ref.import_reference()
    B, C, H, W, kind, k, sigma, maxit = WORKLOADS[workload]
    if x is None:
        x, psf = make_inputs_numpy(workload, n_img)
    xt = torch.from_numpy(x[:n_img])
    if workload == "cfg4":
        m = RefADMMDeconv((), max_iters=n_it, lmbda=None, rho=None, iso=False)
        with torch.no_grad():
            m.lmbda.fill_(LAMBDA); m.rho.fill_(RHO)
        t0 = time.perf_counter()
        loss = (m(xt) ** 2).mean()
        loss.backward()
        secs = time.perf_counter() - t0
    else:
        kt = torch.from_numpy(psf[None, None]) if psf is not None else torch.tensor([])
        lam, rho = torch.tensor([LAMBDA]), torch.tensor([RHO])
        with torch.no_grad():
            t0 = time.perf_counter()
            ref_fft_admm_tv(xt, lam, rho, kt, False, n_it)
            secs = time.perf_counter() - t0
    return n_img * H * W * n_it / secs / 1e6, secs


def reference_sample_size(workload, budget_s):
    """Calibrate on a tiny run, then pick (images, iterations) so one step takes about `budget_s` seconds.  The reference's
    per-iteration cost is constant (no data-dependent control flow, deconv.py:103-115) and images are independent."""
    B, C, H, W, kind, k, sigma, maxit = WORKLOADS[workload]
    n_it = maxit if workload == "cfg4" else min(maxit, 3)         # cfg4 keeps its 10 unrolled iterations (autograd graph)
    cal_img = 1 if H * W >= 1 << 20 else min(B, 4)
    cal_it = n_it if workload == "cfg4" else 1
    x, psf = make_inputs_numpy(workload, cal_img)
    reference_run(workload, cal_img, cal_it, x, psf)             # first call: thread pool, mkldnn primitive caches
    _, secs = reference_run(workload, cal_img, cal_it, x, psf)
    per_img_it = secs / (cal_img * cal_it)
    n_img = int(max(1, min(B, budget_s / (per_img_it * n_it))))
    if n_img == 1 and per_img_it * n_it > 2 * budget_s and workload != "cfg4":
        n_it = max(1, int(budget_s / per_img_it))
    return n_img, n_it, per_img_it


def cpu_info():
    model = ""
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    model = ln.split(":", 1)[1].strip()
                    break
    except Exception:
        pass
    import torch
    return {"cpu_count": os.cpu_count(), "torch_threads": torch.get_num_threads(), "cpu_model": model}


CPU_SAMPLES = {"cfg1": (1, 200), "cfg2": (64, 100), "cfg3": (1, 8), "cfg5": (256, 100), "cfg5full": (256, 100),
               "cfg4": (32, 10)}


def cpu_port_train(sample_images):
    """cfg4 on the host cores: oracle forward + hand-derived adjoint (oracle/admm_oracle.py), images split over threads."""
    from oracle import admm_oracle as O
    from concurrent.futures import ThreadPoolExecutor
    B, C, H, W, kind, k, sigma, maxit = WORKLOADS["cfg4"]
    cores = os.cpu_count() or 1
    nb = max(1, min(sample_images, B))
    rng = np.random.default_rng(1234)
    x = rng.random((nb, C, H, W), dtype=np.float32)
    kern = np.zeros((0,), np.float32)
    nthreads = min(cores, nb)
    chunks = np.array_split(np.arange(nb), nthreads)

    def one(idx):
        xs = x[idx[0]:idx[-1] + 1].astype(np.float64)
        out = O.admm_tv_spectral_form(xs, LAMBDA, RHO, kern, False, maxit)
        return O.admm_tv_backward(xs, LAMBDA, RHO, kern, 2.0 * out / out.size, False, maxit)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=nthreads) as ex:
        list(ex.map(one, chunks))
    secs = time.perf_counter() - t0
    val = nb * H * W * maxit / secs / 1e6
    return val, secs, cores, ("%d of %d images, fwd + bwd of the %d-iteration layer (fp64 oracle and its adjoint), %d host threads"
                              % (nb, B, maxit, nthreads))


def bench_train(args, rank, world, local_rank, config):
    """cfg4: one training step = zero_grad, forward, loss, backward (+ the NCCL all-reduce of the layer gradients when
    world > 1).  e2e additionally copies the batch from pinned host memory and reads loss and gradients back."""
    import torch
    import torch.distributed as dist
    from torch_admm_deconv_b200 import ADMMDeconv, _lib
    from torch_admm_deconv_b200.sharding import GradAllReducer
    B, C, H, W, kind, k, sigma, maxit = WORKLOADS["cfg4"]
    dev = torch.device("cuda", local_rank)
    g = torch.Generator().manual_seed(1234 + rank)
    x_pin = torch.rand(B, C, H, W, generator=g).pin_memory()
    x_dev = x_pin.to(dev)
    model = ADMMDeconv((), max_iters=maxit, lmbda=None, rho=None, iso=False).to(dev)
    with torch.no_grad():
        model.lmbda.fill_(LAMBDA); model.rho.fill_(RHO)
    res_pin = torch.empty(3).pin_memory()

    reducer = GradAllReducer(model.parameters(), average=True)     # one NCCL all-reduce per step on a side stream

    def step(x):
        reducer.wait()                                             # the previous step's exchange has landed in .grad
        model.zero_grad(set_to_none=True)
        loss = (model(x) ** 2).mean()
        loss.backward()
        reducer.reduce()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(max(args.warmup, 10)):        # also settles NCCL's lazily created channels (first all-reduces are slow)
        step(x_dev)
    barrier()
    n0 = _lib.launch_count()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step(x_dev)
    reducer.wait()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    launches = _lib.launch_count() - n0
    dump = None
    if args.dump_outputs and rank == 0:
        dump = {"loss": dump_array(loss.reshape(1)), "grad_lmbda": dump_array(model.lmbda.grad),
                "grad_rho": dump_array(model.rho.grad)}
    # e2e: every step's batch comes from pinned host memory; like a prefetching data loader, the copy of step i+1 runs on
    # a side stream while step i computes (two device buffers), and loss + gradients go back to the host every step
    cur = torch.cuda.current_stream()
    copy_stream = torch.cuda.Stream(dev)
    bufs = [torch.empty_like(x_dev), torch.empty_like(x_dev)]
    done = [None, None]                                             # event: the step that last used the buffer finished
    f0 = torch.cuda.Event(enable_timing=True); f1 = torch.cuda.Event(enable_timing=True)
    f0.record()
    with torch.cuda.stream(copy_stream):
        copy_stream.wait_stream(cur)
        bufs[0].copy_(x_pin, non_blocking=True)
    for i in range(args.steps):
        cur.wait_stream(copy_stream)                                # batch i has landed
        if i + 1 < args.steps:
            with torch.cuda.stream(copy_stream):
                if done[(i + 1) % 2] is not None:
                    copy_stream.wait_event(done[(i + 1) % 2])
                bufs[(i + 1) % 2].copy_(x_pin, non_blocking=True)   # H2D of the next step's batch
        loss = step(bufs[i % 2])
        done[i % 2] = torch.cuda.Event(); done[i % 2].record(cur)
        reducer.wait()
        res_pin.copy_(torch.cat([loss.reshape(1), model.lmbda.grad, model.rho.grad]), non_blocking=True)   # D2H
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    if world > 1:
        t = torch.tensor([ms_total, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        return
    if dump is not None:
        write_dump(args.dump_outputs, dump)
    units = world * B * H * W * maxit * args.steps
    peak, peak_src = measured_peak()
    elems = B * C * H * W
    ach = TRAIN_BYTES_PER_ELEM * elems * maxit * args.steps / (ms_total * 1e-3) / 1e9
    line = {"metric": METRIC, "value": units / (ms_total * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 10), "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "e2e": {"value": units / (ms_e2e * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": x_pin.numel() * 4,
                    "d2h_bytes_per_step": 12, "ms_per_step": ms_e2e / args.steps,
                    "how": "every step: pinned H2D of its batch (on a side stream, overlapping the previous step, as a prefetching loader does), fwd + bwd, D2H of loss and the lambda / rho gradients"},
            "gpu_launches": launches, "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "training step (all forward and backward kernels)", "achieved": ach,
                         "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": TRAIN_BYTES_PER_ELEM * elems * maxit,
                         "avg_launch_ms": ms_total / args.steps, "launches_timed": args.steps,
                         "note": "96 B per element-iteration over the whole fwd+bwd step; L2 is flushed by the step's own "
                                 "0.6 GB of traffic"}}
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_block("cfg4")
    print(json.dumps(line), flush=True)


def cpu_baseline_block(workload):
    """`cpu_baseline` of our arm (rank 0, N = 1): the unmodified reference on a bounded sample (SURVEY.md section 8d:
    cfg2 = the full batch x 3 iterations after a 1-iteration warm-up), and the oracle port beside it."""
    B, C, H, W, kind, k, sigma, maxit = WORKLOADS[workload]
    info = cpu_info()
    block = None
    if reference_available():
        if workload == "cfg2":
            n_img, n_it = B, 3
            x, psf = make_inputs_numpy(workload, n_img)
            reference_run(workload, n_img, 1, x, psf)                                  # warm-up
        else:
            n_img, n_it, _ = reference_sample_size(workload, 15.0)
            x, psf = make_inputs_numpy(workload, n_img)
        v, secs = reference_run(workload, n_img, n_it, x, psf)
        block = {"value": v, "unit": UNIT, "cores": info["torch_threads"], "kind": "reference", "seconds": secs, "host": info,
                 "sample": "%d of %d images x %d of %d iterations of %s through the unmodified reference (baseline/_ref, "
                           "admmtor fft_admm_tv%s, fp32, torch CPU, %d intra-op threads); per-iteration cost is constant "
                           "(deconv.py:103-115), so the rate extrapolates by x%.1f to the full step"
                           % (n_img, B, n_it, maxit, workload, " + autograd backward" if workload == "cfg4" else "",
                              info["torch_threads"], (B / n_img) * (maxit / n_it))}
    ni, nit = CPU_SAMPLES[workload]
    if workload == "cfg4":
        pv, ps, pc, pd = cpu_port_train(ni)
    else:
        pv, ps, pc, pd = cpu_port_run(workload, ni, min(nit, 30))
    port = {"value": pv, "unit": UNIT, "cores": pc, "kind": "port", "seconds": ps, "sample": pd}
    if block is None:
        return port
    block["port"] = port
    return block


def bench_cfg5_strong(rank, world, dev, barrier, steps):
    """BASELINE configs[4]: 4096 synthetic 256 x 256 RGB patches, 15 x 15 Gaussian PSF, 50 iterations, split over the N GPUs
    of the job (STRONG scaling: 4096 / N images per rank, contiguous batch split, no collective), `steps` timed steps.  Device-timed with the
    whole shard resident (one fft_admm_tv call per step), and end to end through HostPipeline in chunks of 512 images from
    pinned host memory.  Returns the block on rank 0 (max over ranks)."""
    import torch
    import torch.distributed as dist
    from torch_admm_deconv_b200 import fft_admm_tv
    from torch_admm_deconv_b200.pipeline import HostPipeline
    from torch_admm_deconv_b200.sharding import shard_range
    B, C, H, W, kind, k, sigma, maxit = WORKLOADS["cfg5full"]
    lo, hi = shard_range(B, world, rank)
    nb = hi - lo
    chunk = min(512, nb)
    x_host, psf = make_inputs_torch((64, C, H, W), kind, k, sigma, seed=4321 + rank)
    base = x_host.to(dev)
    # nb images from the 64 seeded ones: every repeat is circularly shifted by a different offset, so all images differ
    x_dev = torch.empty(nb, C, H, W, device=dev)
    for j in range(0, nb, 64):
        n = min(64, nb - j)
        x_dev[j:j + n] = torch.roll(base[:n], shifts=(j // 64 * 3, j // 64 * 5), dims=(-2, -1))
    x_pin = torch.empty(chunk, C, H, W).pin_memory(); x_pin.copy_(x_dev[:chunk])
    outs = [torch.empty(chunk, C, H, W).pin_memory() for _ in range(2)]
    kern = psf.to(dev)
    lam = torch.tensor([LAMBDA], device=dev); rho = torch.tensor([RHO], device=dev)
    warm = 1
    for _ in range(warm):
        fft_admm_tv(x_dev, lam, rho, kern, False, maxit)
    barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fft_admm_tv(x_dev, lam, rho, kern, False, maxit)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    del x_dev
    torch.cuda.empty_cache()
    pipe = HostPipeline(dev, lam, rho, kern, False, maxit, depth=2)
    nchunks = (nb + chunk - 1) // chunk
    pipe.submit(x_pin, outs[0]); pipe.synchronize()
    barrier()
    f0 = torch.cuda.Event(enable_timing=True); f1 = torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(steps * nchunks):
        pipe.submit(x_pin, outs[i % 2])
    for st_ in pipe.streams:
        torch.cuda.current_stream().wait_stream(st_)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        return None
    peak, _ = measured_peak()
    units = B * H * W * maxit * steps
    e2e_units = world * nchunks * chunk * H * W * maxit * steps
    return {"workload": "cfg5: batch %d x %d ch %dx%d split over %d GPU(s) (%d images per rank), %dx%d %s PSF, %d ADMM "
                        "iterations, fp32, iso=False" % (B, C, H, W, world, nb, k, k, kind, maxit),
            "scaling": "strong", "global_batch": B, "per_gpu_batch": nb, "n_gpus": world, "steps": steps, "warmup": warm,
            "value": units / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms / steps,
            "frac_whole_step": 36.0 * B * C * H * W * maxit * steps / world / (ms * 1e-3) / 1e9 / peak,
            "e2e": {"value": e2e_units / (ms_e2e * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms_e2e / steps,
                    "h2d_bytes_per_step": nchunks * chunk * C * H * W * 4, "d2h_bytes_per_step": nchunks * chunk * C * H * W * 4,
                    "how": "HostPipeline over chunks of %d images from pinned host memory (H2D, solve, D2H on three streams)" % chunk},
            "note": "max over ranks of the device time; frac_whole_step = 36 B x elements per rank x iterations / time / measured HBM peak"}


# ------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cfg5", action="store_true", help="skip the scaling_cfg5 block (4096 images over the N GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    B, C, H, W, kind, k, sigma, maxit = WORKLOADS[args.workload]
    config = {"workload": ("%s: batch %d x %d ch %dx%d, %dx%d %s PSF, %d ADMM iterations, fp32, iso=False, lambda=%g rho=%g"
                           % (args.workload, B, C, H, W, k, k, kind, maxit, LAMBDA, RHO)) if args.workload != "cfg4" else
                          ("cfg4: training step (fwd+bwd) of the unrolled layer, batch %d x %d ch %dx%d, no kernel, learnable "
                           "lambda / rho, %d unrolled iterations, fp32, iso=False" % (B, C, H, W, maxit)),
              "per_gpu_batch": B, "global_batch": B * max(1, args.gpus), "sharding": "batch split, no collective",
              "l2": "working set per step >> 126 MB L2 (inputs larger than L2, no flush needed)"
                    if B * C * H * W * 4 * 6 > 2 * 126e6 else "working set fits L2: a 256 MB buffer is rewritten between steps"}

    # ---------------------------------------------------------------- reference arm: the reference on the host cores, rank 0 only
    if args.impl == "reference":
        if rank != 0:
            return 0
        steps, warm = max(1, args.steps), max(0, args.warmup)
        budget = float(os.environ.get("ADMM_REF_BUDGET_S", "150"))          # whole command: a few minutes
        # all host threads, also under torchrun (which exports OMP_NUM_THREADS=1 to every rank)
        import torch
        torch.set_num_threads(os.cpu_count() or 1)
        if reference_available():
            kind_ = "reference"
            n_img, n_it, per = reference_sample_size(args.workload, budget / (steps + warm))
            x, psf = make_inputs_numpy(args.workload, n_img)
            run_ref = lambda: reference_run(args.workload, n_img, n_it, x, psf)
            what = "the unmodified reference admmtor.eops.deconv.fft_admm_tv (baseline/_ref), fp32, torch CPU"
            if args.workload == "cfg4":
                what = "the unmodified reference ADMMDeconv layer (baseline/_ref), forward + stock autograd backward, fp32, torch CPU"
        else:                                                             # baseline/_ref missing: oracle port, labelled as such
            kind_ = "port"
            n_img, n_it = CPU_SAMPLES[args.workload]
            run_ref = ((lambda: cpu_port_train(n_img)[:2]) if args.workload == "cfg4"
                       else (lambda: cpu_port_run(args.workload, n_img, n_it)[:2]))
            what = "numpy/scipy oracle port (baseline/_ref not installed)"
        for _ in range(warm):
            run_ref()
        vals, secs = [], []
        for _ in range(steps):
            v, s_ = run_ref()
            vals.append(v); secs.append(s_)
        tot = float(np.sum(secs))
        v = n_img * H * W * n_it * steps / tot / 1e6
        info = cpu_info()
        desc = ("each step = %d of %d images x %d of %d iterations of %s through %s; per-iteration cost is constant "
                "(no data-dependent control flow, deconv.py:103-115) and images are independent, so the rate extrapolates "
                "to the full step" % (n_img, B, n_it, maxit, args.workload, what))
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
                "warmup": warm, "ms_per_step": tot / steps * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": info["torch_threads"] if kind_ == "reference" else info["cpu_count"],
                                 "kind": kind_, "sample": desc, "host": info},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0,
                "ms_per_full_step_extrapolated": B * H * W * maxit / (v * 1e6) * 1e3,
                "note": "a step is a bounded sample of the workload (see cpu_baseline.sample); steps / warmup / ms_per_step are "
                        "what actually ran; one CPU process with all host threads regardless of --gpus"}
        print(json.dumps(line), flush=True)
        return 0

    # ---------------------------------------------------------------- our arm
    import torch
    import torch.distributed as dist
    from torch_admm_deconv_b200 import fft_admm_tv, _lib, build as _build
    from torch_admm_deconv_b200.pipeline import HostPipeline
    _build.build()
    _lib.load()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback exists for this path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its banner / debug output (NCCL_DEBUG=VERSION|INFO) to the
        # process's stdout while the communicator is created, so fd 1 points at stderr for that moment
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier(device_ids=[local_rank])
            torch.cuda.synchronize()
        finally:
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    if args.workload == "cfg4":
        config["l2"] = "the saved state of the unrolled iterations (0.45 GB) and the step's 0.6 GB of traffic exceed the 126 MB L2: no flush"
        config["sharding"] = "batch split; one NCCL all-reduce of the lambda / rho gradients per step when n_gpus > 1"
        bench_train(args, rank, world, local_rank, config)
        if world > 1:
            dist.destroy_process_group()
        return 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    x_host, psf = make_inputs_torch((B, C, H, W), kind, k, sigma, seed=1234 + rank)
    x_pin = x_host.pin_memory()
    out_pin = torch.empty_like(x_host).pin_memory()
    out_pin2 = torch.empty_like(x_host).pin_memory()
    x_dev = x_pin.to(dev, non_blocking=True)
    kern = psf.to(dev)
    lam = torch.tensor([LAMBDA], device=dev); rho = torch.tensor([RHO], device=dev)
    flush = None
    if "rewritten" in config["l2"]:
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def step_resident():
        if flush is not None:
            flush.fill_(1)
        return fft_admm_tv(x_dev, lam, rho, kern, False, maxit)

    pipe = HostPipeline(dev, lam, rho, kern, False, maxit, depth=2)
    outs = [out_pin, out_pin2]

    def step_e2e(i=0):
        # public streaming API: H2D of this step's inputs, solve, D2H of this step's result; the copies of one step
        # overlap with the solve of the neighbouring step (two streams, double-buffered device input)
        pipe.submit(x_pin, outs[i % 2])

    # warm-up
    for _ in range(max(args.warmup, 3)):
        step_resident()
    step_e2e(0); step_e2e(1)
    pipe.synchronize()
    barrier()

    # ---- timed region 1: inputs resident in HBM, per-kernel profiling events OFF -> `value`, `gpu_launches`
    _lib.set_option("profile", 0)
    _lib.profile_reset()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    barrier()

    def timed_pass():
        """Returns (ms, output of the last step); every other step's output is released before the next step runs."""
        out = None
        if flush is None:
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                out = None
                out = step_resident()
            e1.record()
            barrier()
            return e0.elapsed_time(e1), out
        # small working set: L2 is flushed between steps and the flush is kept OUT of the timed intervals
        evs = []
        for _ in range(args.steps):
            out = None
            flush.fill_(1)
            a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
            a0.record()
            out = fft_admm_tv(x_dev, lam, rho, kern, False, maxit)
            a1.record()
            evs.append((a0, a1))
        barrier()
        return sum(a.elapsed_time(b) for a, b in evs), out

    ms_total, out = timed_pass()
    clocks = sampler.stop() if sampler else None
    launches = _lib.launch_count()
    dump = {"out": dump_array(out)} if args.dump_outputs and rank == 0 else None
    del out
    # ---- second pass with CUDA events around every kernel launch -> per-kernel times for `roofline`.  The kernels are
    # timed one at a time on ONE stream (the public call overlaps the two halves of the batch on two streams, which would
    # make the events of one half include the other half's kernels)
    from torch_admm_deconv_b200.eops import deconv as _deconv
    split = _deconv.SPLIT_STREAMS
    _deconv.SPLIT_STREAMS = 1
    _lib.set_option("profile", 1)
    _lib.profile_reset()
    ms_profiled = timed_pass()[0]
    prof = {kname: _lib.profile_read(kid) for kid, kname in enumerate(("rows", "cols", "other"))}
    _lib.set_option("profile", 0)
    _deconv.SPLIT_STREAMS = split

    # ---- timed region 2: end to end through the public API with host buffers -> `e2e`
    barrier()
    f0 = torch.cuda.Event(enable_timing=True); f1 = torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    f0.record()
    for i in range(args.steps):
        step_e2e(i)
    for st_ in pipe.streams:                                        # f1 fires after both pipeline streams drained
        torch.cuda.current_stream().wait_stream(st_)
    f1.record()
    barrier()
    ms_e2e_host = (time.perf_counter() - t0) * 1e3                  # host clock between two device syncs (cross-check)
    ms_e2e = f0.elapsed_time(f1)

    if world > 1:
        t = torch.tensor([ms_total, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e = float(t[0]), float(t[1])

    cfg5 = None
    if args.workload == "cfg2" and not args.no_cfg5:
        cfg5 = bench_cfg5_strong(rank, world, dev, barrier, args.steps)

    if rank == 0:
        if dump is not None:
            write_dump(args.dump_outputs, dump)
        units = world * B * H * W * maxit * args.steps            # pixel-iterations of the whole job
        value = units / (ms_total * 1e-3) / 1e6
        e2e_val = units / (ms_e2e * 1e-3) / 1e6
        peak, peak_src = measured_peak()
        elems = B * C * H * W
        kinds = {"rows": ROW_BYTES_PER_ELEM, "cols": COL_BYTES_PER_ELEM}
        avg = {n: (prof[n][0] / prof[n][1] if prof[n][1] else None) for n in kinds}      # ms per launch
        ach = {n: (kinds[n] * elems / (avg[n] * 1e-3) / 1e9 if avg[n] else None) for n in kinds}
        dom = max(kinds, key=lambda n: prof[n][0])
        bott = min((n for n in kinds if ach[n]), key=lambda n: ach[n] / peak, default=None)
        traffic = {}
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get(args.workload, {})
            except Exception:
                traffic = {}
        names = {"rows": "row pass (C2R + prox/dual/divergence + R2C)", "cols": "column pass (FFT + A+Bm*V + iFFT)"}
        roofline = None
        if avg["rows"] and avg["cols"]:
            # headline: ONE ADMM iteration = one row-pass launch + one column-pass launch, 24 + 12 = 36 B per element
            it_ms = avg["rows"] + avg["cols"]
            it_ach = 36.0 * elems / (it_ms * 1e-3) / 1e9
            step_ach = 36.0 * elems * maxit * args.steps / (ms_total * 1e-3) / 1e9
            tr = (traffic.get("rows") or 0) + (traffic.get("cols") or 0)
            roofline = {"bound": "hbm", "kernel": "one ADMM iteration = " + names["rows"] + " + " + names["cols"],
                        "achieved": it_ach, "peak": peak, "unit": "GB/s", "frac": it_ach / peak,
                        "traffic": tr or None, "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": 36.0 * elems, "avg_launch_ms": it_ms, "launches_timed": prof["rows"][1],
                        "frac_rows": ach["rows"] / peak, "frac_cols": ach["cols"] / peak, "frac_whole_iteration": it_ach / peak,
                        "frac_whole_step": step_ach / peak,
                        "bottleneck": names[bott], "dominant_by_time": names[dom],
                        "rows": {"bytes_per_element": ROW_BYTES_PER_ELEM, "avg_launch_ms": avg["rows"], "achieved": ach["rows"],
                                 "launches": prof["rows"][1], "traffic": traffic.get("rows")},
                        "cols": {"bytes_per_element": COL_BYTES_PER_ELEM, "avg_launch_ms": avg["cols"], "achieved": ach["cols"],
                                 "launches": prof["cols"][1], "traffic": traffic.get("cols")},
                        "kernel_ms": {n: prof[n][0] for n in prof}, "timed_region_ms": ms_total,
                        "profiled_pass_ms": ms_profiled,
                        "note": "kernel times from a second pass with CUDA events around every launch, one stream; `value` is "
                                "timed without them through the public call (batch halves on two streams).  frac_whole_step "
                                "also carries the one-off precompute and the last C2R"}
        elif prof["other"][1]:
            # cluster-resident solver: the whole solve is one launch and touches HBM only for y and x
            one_ms = ms_total / args.steps                   # the whole solve: tables + ONE cluster launch
            roofline = {"bound": "hbm", "kernel": "cluster-resident solver (whole solve in one launch)",
                        "achieved": 8.0 * elems / (one_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": 8.0 * elems / (one_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": 8.0 * elems, "avg_launch_ms": one_ms, "launches_timed": args.steps,
                        "note": "latency-bound: one plane lives in the shared memory of a thread-block cluster for all iterations; "
                                "report ms per solve, not a roofline fraction"}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config,
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": x_pin.numel() * 4,
                        "d2h_bytes_per_step": out_pin.numel() * 4, "ms_per_step": ms_e2e / args.steps,
                        "host_clock_ms_per_step": ms_e2e_host / args.steps,
                        "how": "HostPipeline: pinned H2D, solve and D2H of every step on three streams (copies overlap the neighbouring solve)"},
                "gpu_launches": launches, "clocks": clocks, "roofline": roofline}
        if cfg5 is not None:
            line["scaling_cfg5"] = cfg5
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_block(args.workload)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
