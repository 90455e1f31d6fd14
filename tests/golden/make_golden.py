"""Generate the golden fixtures in this directory by running the UNMODIFIED reference.

Run in the build container only (it needs /root/reference, which does not exist on the GPU box):

    python tests/golden/make_golden.py

The reference (`admmtor.eops.deconv.fft_admm_tv`, `admmtor.elayers.admmdeconv.ADMMDeconv`) is
imported from /root/reference/src and executed on the CPU in float32 and float64.  Each fixture
stores the inputs, the reference outputs in both precisions, and (for the *_grad cases) the
gradients produced by the reference's stock autograd in float64.  The reference has no tests or
golden vectors of its own (SURVEY.md section 4), so these files are the parity pins.
"""
import math
import os
import sys

import numpy as np
import torch

REF_SRC = "/root/reference/src"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REF_SRC)
sys.path.insert(0, os.path.join(HERE, "..", ".."))

from admmtor.eops.deconv import fft_admm_tv  # noqa: E402  (the reference)
from admmtor.elayers.admmdeconv import ADMMDeconv  # noqa: E402  (the reference)
from oracle.admm_oracle import make_psf, make_blurred  # noqa: E402  (input generators only)

torch.set_num_threads(8)


def run_ref(x, lam, rho, kern, iso, maxit, dtype):
    xt = torch.from_numpy(x).to(dtype)
    kt = torch.from_numpy(kern).to(dtype) if kern.size else torch.tensor([], dtype=dtype)
    out = fft_admm_tv(xt, torch.tensor([lam], dtype=dtype), torch.tensor([rho], dtype=dtype), kt, iso, maxit)
    return out.numpy()


def save_case(name, x, kern, lam, rho, iso, maxit, extra=None):
    k4 = kern[None, None].astype(np.float32) if kern is not None else np.zeros((0,), np.float32)
    out32 = run_ref(x, lam, rho, k4, iso, maxit, torch.float32)
    out64 = run_ref(x, lam, rho, k4, iso, maxit, torch.float64)
    d = dict(x=x.astype(np.float32), kern=k4, lam=np.float64(lam), rho=np.float64(rho),
             iso=np.bool_(iso), maxit=np.int32(maxit), out32=out32.astype(np.float32), out64=out64)
    if extra:
        d.update(extra)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **d)
    e = np.abs(out32 - out64).max() / max(np.abs(out64).max(), 1e-300)
    print(f"{name:28s} shape={x.shape} k={k4.shape} iso={iso} N={maxit}  ref32-vs-ref64={e:.2e}")


def grad_case(name, shape, k, iso, maxit, seed, lam=0.02, rho=0.04):
    rng = np.random.default_rng(seed)
    x = rng.random(shape)
    kern = None
    if k:
        kern = rng.random((k, k)); kern /= kern.sum()
    gout = rng.standard_normal(shape)
    xt = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    lt = torch.tensor([lam], dtype=torch.float64, requires_grad=True)
    rt = torch.tensor([rho], dtype=torch.float64, requires_grad=True)
    if k:
        kt = torch.tensor(kern[None, None], dtype=torch.float64, requires_grad=True)
    else:
        kt = torch.tensor([], dtype=torch.float64)
    out = fft_admm_tv(xt, lt, rt, kt, iso, maxit)
    (out * torch.tensor(gout)).sum().backward()
    d = dict(x=x, kern=(kern[None, None] if k else np.zeros((0,))), lam=lam, rho=rho, iso=np.bool_(iso),
             maxit=np.int32(maxit), gout=gout, out64=out.detach().numpy(), gx=xt.grad.numpy(),
             glam=(lt.grad.numpy() if lt.grad is not None else np.zeros(1)),   # N=1: tau is never consumed
             grho=(rt.grad.numpy() if rt.grad is not None else np.zeros(1)),
             gkern=(kt.grad.numpy() if k else np.zeros((0,))))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **d)
    print(f"{name:28s} shape={shape} k={k} iso={iso} N={maxit}  |gx|={np.abs(d['gx']).max():.3e} "
          f"glam={d['glam'][0]:.6e} grho={d['grho'][0]:.6e}")


def main():
    rng = np.random.default_rng(7)
    # cfg1 of BASELINE.json, in full: single 256x256 grayscale, 15x15 Gaussian, 50 iterations
    psf = make_psf("gauss", 15, 2.5)
    save_case("cfg1_256_gauss15_n50", make_blurred((1, 1, 256, 256), psf), psf, 0.02, 0.04, False, 50)
    # cfg2 reduced (same PSF family, 31-tap motion blur), small enough for a fixture: the first image of a seeded pair
    # (planes are independent for iso=False; one image keeps the file under 1 MB)
    psf = make_psf("motion", 31)
    save_case("cfg2r_128_motion31_n30", make_blurred((2, 3, 128, 128), psf, seed=11)[:1], psf, 0.02, 0.04, False, 30)
    # D5 pins: asymmetric odd and even kernels
    k7 = rng.random((7, 7)); k7 /= k7.sum()
    save_case("asym7_32x48_n20", make_blurred((2, 3, 32, 48), k7.astype(np.float32), seed=12), k7, 0.02, 0.04, False, 20)
    k8 = rng.random((8, 8)); k8 /= k8.sum()
    save_case("even8_64x32_n20", make_blurred((1, 2, 64, 32), k8.astype(np.float32), seed=13), k8, 0.03, 0.05, False, 20)
    # D6: empty kernel = TV denoise
    save_case("denoise_32x32_n25", make_blurred((2, 3, 32, 32), None, seed=14, noise=0.05), None, 0.05, 0.1, False, 25)
    # D2: iso=True (module default), with and without kernel; batch is coupled
    k5 = rng.random((5, 5)); k5 /= k5.sum()
    save_case("iso_k5_32x32_n15", make_blurred((4, 3, 32, 32), k5.astype(np.float32), seed=15), k5, 0.02, 0.04, True, 15)
    save_case("iso_denoise_32x32_n15", make_blurred((4, 3, 32, 32), None, seed=16, noise=0.05), None, 0.05, 0.1, True, 15)
    # odd and mixed-radix sizes (D7): 33x45, 60x90 (2^2*3*5 x 2*3^2*5), prime 31x37
    k3 = rng.random((3, 3)); k3 /= k3.sum()
    save_case("odd_33x45_n12", make_blurred((1, 2, 33, 45), k3.astype(np.float32), seed=17), k3, 0.02, 0.04, False, 12)
    save_case("mixed_60x90_n12", make_blurred((1, 1, 60, 90), k5.astype(np.float32), seed=18), k5, 0.02, 0.04, False, 12)
    save_case("prime_31x37_n8", make_blurred((1, 1, 31, 37), k3.astype(np.float32), seed=19), k3, 0.02, 0.04, False, 8)
    # maxit = 0 and 1 (known answers 1 and 4 of SURVEY.md section 4)
    save_case("n0_16x16", make_blurred((1, 1, 16, 16), k3.astype(np.float32), seed=20), k3, 0.02, 0.04, False, 0)
    save_case("n1_16x16", make_blurred((1, 1, 16, 16), k3.astype(np.float32), seed=20), k3, 0.02, 0.04, False, 1)

    # module level: ADMMDeconv with bias, fixed seed; records the RNG draw order (admmdeconv.py:15-23)
    torch.manual_seed(1234)
    m = ADMMDeconv((5, 5), max_iters=8, lmbda=None, rho=None, iso=False, bias=True)
    sd = {k_: v.detach().numpy().copy() for k_, v in m.state_dict().items()}
    xm = make_blurred((2, 3, 24, 24), None, seed=21)
    with torch.no_grad():
        m.w.copy_(torch.from_numpy(k5[None, None].astype(np.float32)))   # xavier w is zero-mean: den(0,0)~0
        ym = m(torch.from_numpy(xm)).numpy()
    sd_after = {k_: v.detach().numpy().copy() for k_, v in m.state_dict().items()}
    np.savez_compressed(os.path.join(HERE, "module_k5_bias.npz"), x=xm, out32=ym,
                        **{"init_" + k_: v for k_, v in sd.items()}, **{"sd_" + k_: v for k_, v in sd_after.items()},
                        is_param=np.array([isinstance(getattr(m, n), torch.nn.Parameter) for n in ("w", "lmbda", "rho", "b")]))
    m2 = ADMMDeconv((), max_iters=5, lmbda=0.02, rho=0.04)
    np.savez_compressed(os.path.join(HERE, "module_empty.npz"),
                        keys=np.array(list(m2.state_dict().keys())),
                        w_shape=np.array(m2.w.shape), iso=np.bool_(m2.iso),
                        is_param=np.array([isinstance(getattr(m2, n), torch.nn.Parameter) for n in ("w", "lmbda", "rho", "b")]))
    print("module fixtures written; state-dict keys", list(m.state_dict().keys()))

    # gradients from the reference's stock autograd, float64
    grad_case("grad_aniso_k5_16x20_n6", (2, 3, 16, 20), 5, False, 6, 31)
    grad_case("grad_aniso_k4_16x16_n5", (1, 2, 16, 16), 4, False, 5, 32)
    grad_case("grad_aniso_empty_16x20_n6", (2, 3, 16, 20), 0, False, 6, 33, lam=0.05, rho=0.1)
    grad_case("grad_iso_k4_16x16_n5", (2, 3, 16, 16), 4, True, 5, 34)
    grad_case("grad_iso_empty_16x16_n5", (2, 3, 16, 16), 0, True, 5, 35, lam=0.05, rho=0.1)
    grad_case("grad_aniso_k3_n1", (1, 1, 8, 8), 3, False, 1, 36)


if __name__ == "__main__":
    main()
