"""GPU tests of the float64 solve (fft_admm_tv_f64, admm_*_f64): the generic sm_100a kernels instantiated for double,
against the reference's float64 outputs and autograd gradients (tests/golden), the fp64 oracle, finite differences
(torch.autograd.gradcheck) and the float32 solver.  Tolerance metric: max|a-b| / max|b|."""
import numpy as np
import pytest
import torch

from conftest import golden, golden_names
from oracle import admm_oracle as O

pytestmark = pytest.mark.gpu

TOL_FWD = 1e-10          # forward vs the reference's / oracle's float64 result
TOL_GX = 1e-9            # x-gradient
TOL_P = 1e-8             # lambda / rho / kernel gradients (relative)
FWD_FIXTURES = golden_names(exclude=("module", "grad"))


def _dev():
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    return torch.device("cuda:0")


def _t(a, grad=False):
    return torch.tensor(np.asarray(a, np.float64), device=_dev(), requires_grad=grad)


def _kern(kern, grad=False):
    return _t(kern, grad) if np.size(kern) else torch.empty(0, dtype=torch.float64, device=_dev())


def _solve64(x, lam, rho, kern, iso, maxit):
    from torch_admm_deconv_b200 import fft_admm_tv_f64
    out = fft_admm_tv_f64(_t(x), _t([lam]), _t([rho]), _kern(kern), iso, maxit)
    torch.cuda.synchronize()
    assert out.dtype == torch.float64
    return out.cpu().numpy()


def _state(out, shape, maxit, iso):
    """The saved forward state: maxit-1 slots of [q_x, q_y] (B, C, H, W), then for iso the maxit-1 pairs of H x W norms."""
    saved = out.grad_fn.saved_tensors[4]
    n, hw = int(np.prod(shape)), shape[2] * shape[3]
    s = saved.view(torch.float64).cpu().numpy()
    q = s[: (maxit - 1) * 2 * n].reshape(maxit - 1, 2, *shape)
    nm = s[(maxit - 1) * 2 * n: (maxit - 1) * 2 * (n + hw)].reshape(maxit - 1, 2, *shape[2:]) if iso else None
    return [(q[k, 0], q[k, 1]) for k in range(maxit - 1)], nm


def _grads64(x, lam, rho, kern, gout, iso, maxit):
    from torch_admm_deconv_b200 import fft_admm_tv_f64
    xt, lt, rt, kt = _t(x, True), _t([lam], True), _t([rho], True), _kern(kern, bool(np.size(kern)))
    out = fft_admm_tv_f64(xt, lt, rt, kt, iso, maxit)
    state = _state(out, x.shape, maxit, iso) if maxit > 1 else ([], None)
    (out * _t(gout)).sum().backward()
    torch.cuda.synchronize()
    g = lambda t: None if t.grad is None else t.grad.cpu().numpy()
    return out.detach().cpu().numpy(), g(xt), g(lt), g(rt), (g(kt) if np.size(kern) else None), state


def _rel(a, b):
    return abs(float(a) - float(b)) / max(abs(float(b)), 1e-12)


# ------------------------------------------------------------------------------- forward
@pytest.mark.parametrize("name", FWD_FIXTURES)
def test_forward_matches_reference_float64_fixture(name):
    d = golden(name)
    out = _solve64(d["x"], float(d["lam"]), float(d["rho"]), d["kern"], bool(d["iso"]), int(d["maxit"]))
    e = O.rel_err(out, d["out64"])
    print("%s: float64 forward err vs reference float64 %.2e" % (name, e))
    assert out.shape == d["out64"].shape and e <= TOL_FWD


@pytest.mark.parametrize("shape,k,kind", [((2, 3, 512, 512), 31, "motion"), ((1, 3, 1080, 1920), 15, "gauss")])
def test_forward_matches_oracle_large(shape, k, kind):
    psf = O.make_psf(kind, k, 2.5)
    x = O.make_blurred(shape, psf, seed=21).astype(np.float64)
    out = _solve64(x, 0.02, 0.04, psf[None, None], False, 20)
    ref = O.admm_tv_spectral_form(x, 0.02, 0.04, psf[None, None], False, 20)
    e = O.rel_err(out, ref)
    print("%s k=%d: float64 forward err vs fp64 oracle %.2e" % (shape, k, e))
    assert e <= TOL_FWD


def test_agrees_with_float32_solver_on_specialised_kernels():
    from torch_admm_deconv_b200 import fft_admm_tv
    psf = O.make_psf("motion", 31)
    x = O.make_blurred((2, 3, 512, 512), psf, seed=5)
    lam, rho = torch.tensor([0.02], device=_dev()), torch.tensor([0.04], device=_dev())
    o32 = fft_admm_tv(torch.from_numpy(x).to(_dev()), lam, rho, torch.from_numpy(psf[None, None]).to(_dev()), False, 100)
    o64 = _solve64(x, 0.02, 0.04, psf[None, None], False, 100)
    e = O.rel_err(o32.cpu().numpy(), o64)
    print("cfg2-like (2,3,512,512) k=31 N=100: float32 vs float64 %.2e" % e)
    assert e <= 1e-4


# ------------------------------------------------------------------------------- gradients
def _kink_margin(state, nm, tau, iso):
    """Distance of the saved pre-threshold values to the kinks of the threshold (|q| = tau; q = 0 as well for tau < 0;
    iso: pixel norm = tau)."""
    if iso:
        return float(np.abs(nm - tau).min())
    qs = np.abs(np.stack([np.stack(s) for s in state]))
    m = float(np.abs(qs - abs(tau)).min())
    return min(m, float(qs.min())) if tau < 0 else m


@pytest.mark.parametrize("name", golden_names(prefix="grad"))
def test_gradients_match_reference_autograd(name):
    d = golden(name)
    iso, maxit, lam, rho = bool(d["iso"]), int(d["maxit"]), float(d["lam"]), float(d["rho"])
    out, gx, gl, gr, gk, (state, nm) = _grads64(d["x"], lam, rho, d["kern"], d["gout"], iso, maxit)
    e_out, e_x = O.rel_err(out, d["out64"]), O.rel_err(gx, d["gx"])
    e_l, e_r = _rel(gl[0], d["glam"][0]), _rel(gr[0], d["grho"][0])
    e_k = O.rel_err(gk, d["gkern"]) if d["kern"].size else 0.0
    margin = _kink_margin(state, nm, lam / rho, iso) if maxit > 1 else float("inf")
    print("%s: out %.1e gx %.1e glam %.1e grho %.1e gkern %.1e (state %.1e from a kink)"
          % (name, e_out, e_x, e_l, e_r, e_k, margin))
    assert e_out <= TOL_FWD
    assert e_x <= TOL_GX and e_l <= TOL_P and e_r <= TOL_P and e_k <= TOL_P


def _gradcheck_case(iso, lam, rho, seeds=range(64)):
    """First seed whose forward state keeps 1e-3 away from the threshold's kinks (so a finite-difference step cannot
    cross one), and the inputs for it.  The image is scaled by 10: at unit scale the gradient fields are so dense near
    tau (and, after a saturated first iteration, q_2 = D x_2 +- tau piles up at +-tau) that no small input keeps 1e-3
    clear of the kinks; scaled, about half the values lie past the threshold and the rest inside it."""
    from torch_admm_deconv_b200 import fft_admm_tv_f64
    psf = O.make_psf("gauss", 3, 0.8)
    for seed in seeds:
        x = 10.0 * O.make_blurred((1, 2, 12, 10), psf, seed=seed, noise=0.05).astype(np.float64)
        args = (_t(x, True), _t([lam], True), _t([rho], True), _t(psf[None, None], True))
        out = fft_admm_tv_f64(*args, iso, 3)
        state, nm = _state(out, x.shape, 3, iso)
        if _kink_margin(state, nm, lam / rho, iso) > 1e-3:
            return seed, args
    raise AssertionError("no input among the seeds keeps the saved state 1e-3 away from the threshold")


@pytest.mark.parametrize("iso,lam,rho", [(False, 0.2, 0.4), (True, 0.4, 0.4), (False, -0.04, 0.4)],
                         ids=["aniso", "iso", "aniso-negtau"])
def test_gradcheck_finite_differences(iso, lam, rho):
    from torch_admm_deconv_b200 import fft_admm_tv_f64
    seed, args = _gradcheck_case(iso, lam, rho)
    print("gradcheck iso=%s tau=%g: seed %d" % (iso, lam / rho, seed))
    assert torch.autograd.gradcheck(lambda x, l, r, k: fft_admm_tv_f64(x, l, r, k, iso, 3), args, eps=1e-6, atol=1e-7,
                                    rtol=1e-5)


@pytest.mark.parametrize("iso", [False, True])
def test_backward_is_bit_reproducible(iso):
    psf = O.make_psf("gauss", 5, 1.2)
    x = O.make_blurred((2, 3, 40, 36), psf, seed=3).astype(np.float64)
    gout = np.random.default_rng(4).standard_normal(x.shape)
    runs = [_grads64(x, 0.02, 0.04, psf[None, None], gout, iso, 6)[1:5] for _ in range(3)]
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert np.array_equal(a, b)


def test_parameter_gradients_in_their_own_dtype():
    from torch_admm_deconv_b200 import fft_admm_tv_f64
    x = _t(O.make_blurred((1, 2, 16, 20), None, seed=1))
    lam = torch.tensor([0.02], device=_dev(), requires_grad=True)            # float32 parameters
    rho = torch.tensor(0.04, device=_dev(), requires_grad=True)              # 0-d
    k = torch.tensor(O.make_psf("gauss", 3, 1.0)[None, None], dtype=torch.float32, device=_dev(), requires_grad=True)
    fft_admm_tv_f64(x, lam, rho, k, False, 4).square().sum().backward()
    assert lam.grad.dtype == torch.float32 and lam.grad.shape == (1,)
    assert rho.grad.dtype == torch.float32 and rho.grad.shape == ()
    assert k.grad.dtype == torch.float32 and k.grad.shape == (1, 1, 3, 3)


# ------------------------------------------------------------------------------- errors and edge cases
def test_errors():
    from torch_admm_deconv_b200 import fft_admm_tv_f64
    dev = _dev()
    lam, rho = torch.tensor([0.02], device=dev), torch.tensor([0.04], device=dev)
    e = torch.empty(0, device=dev)
    with pytest.raises(RuntimeError, match="shared memory"):
        fft_admm_tv_f64(torch.zeros(1, 1, 16, 3840, dtype=torch.float64, device=dev), lam, rho, e, False, 5)
    with pytest.raises(TypeError):
        fft_admm_tv_f64(torch.zeros(1, 1, 16, 16, device=dev), lam, rho, e, False, 5)
    x = torch.zeros(1, 1, 16, 16, dtype=torch.float64, device=dev)
    with pytest.raises(ValueError):
        fft_admm_tv_f64(x[0], lam, rho, e)                                              # 3-D
    with pytest.raises(ValueError):
        fft_admm_tv_f64(x, torch.ones(2, device=dev), rho, e)                           # two-element lambda
    with pytest.raises(RuntimeError):
        fft_admm_tv_f64(x, lam, rho, torch.ones(1, 1, 3, 5, device=dev))               # non-square PSF
    with pytest.raises(ValueError):
        fft_admm_tv_f64(x, lam, rho, torch.ones(1, 1, 17, 17, device=dev))             # PSF larger than the image


def test_maxit_zero_returns_zeros_with_zero_gradients():
    from torch_admm_deconv_b200 import fft_admm_tv_f64
    xt, lt, rt = _t(np.random.default_rng(0).random((1, 2, 16, 16)), True), _t([0.02], True), _t([0.04], True)
    kt = _t(O.make_psf("gauss", 3, 1.0)[None, None], True)
    out = fft_admm_tv_f64(xt, lt, rt, kt, False, 0)
    assert out.dtype == torch.float64 and torch.count_nonzero(out) == 0
    out.sum().backward()
    for t in (xt, lt, rt, kt):
        assert torch.count_nonzero(t.grad) == 0


def test_module_in_float64():
    from torch_admm_deconv_b200 import ADMMDeconv, fft_admm_tv_f64
    torch.manual_seed(0)
    m = ADMMDeconv((5, 5), 6, iso=True, bias=True, activation=torch.sigmoid).double().to(_dev())
    x = _t(O.make_blurred((2, 3, 32, 32), O.make_psf("gauss", 5, 1.2), seed=2))
    with pytest.raises(TypeError):
        m(x)                                                                            # default precision is float32
    m.precision = "float64"
    y = m(x)
    ref = torch.sigmoid(fft_admm_tv_f64(x, m.lmbda, m.rho, m.w, True, 6) + m.b)
    assert y.dtype == torch.float64 and torch.equal(y, ref)
    y.square().mean().backward()
    for name in ("w", "lmbda", "rho", "b"):
        g = getattr(m, name).grad
        assert g is not None and g.dtype == torch.float64 and torch.isfinite(g).all(), name
