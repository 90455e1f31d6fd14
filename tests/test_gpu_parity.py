"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the oracle and the golden
fixtures of the reference.  Tolerance: err(a,b) = max|a-b| / max|b| <= 1e-4 (BASELINE.json north_star),
checked against the reference's fp32 AND fp64 outputs."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import golden, golden_names
from oracle import admm_oracle as O
from oracle import packed_layout_model as M

pytestmark = pytest.mark.gpu

TOL = 1e-4
FWD_ANISO = [n for n in golden_names(exclude=("module", "grad")) if not n.startswith("iso")]


def _dev():
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    return torch.device("cuda:0")


def _solve(x, lam, rho, kern, iso, maxit):
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    xt = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(dev)
    kt = torch.from_numpy(np.asarray(kern, dtype=np.float32)).to(dev) if np.size(kern) else torch.empty(0, device=dev)
    out = fft_admm_tv(xt, torch.tensor([lam], dtype=torch.float32, device=dev),
                      torch.tensor([rho], dtype=torch.float32, device=dev), kt, iso, maxit)
    torch.cuda.synchronize()
    return out.cpu().numpy()


# ------------------------------------------------------------------------------- stage level
def _ws(lib, planes, H, W):
    n = lib.admm_query_workspace(planes, H, W, 0, 0, 1)
    assert n > 0
    return torch.empty(n, dtype=torch.uint8, device=_dev())


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def _cerr(a, b):
    """max|a-b| / max|b| for complex arrays."""
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


@pytest.mark.parametrize("shape", [(3, 16, 16), (2, 33, 45), (1, 60, 90), (2, 31, 37), (2, 256, 256), (1, 128, 512),
                                   (1, 30, 3840), (1, 2160, 16)])
def test_stage_kernels_match_layout_model(lib, shape):
    from torch_admm_deconv_b200 import _lib
    P, H, W = shape
    rng = np.random.default_rng(P * 1000 + H + W)
    x = rng.standard_normal(shape).astype(np.float32)
    Wc = (W + 1) // 2
    dev = _dev()
    ws = _ws(lib, P, H, W)
    xt = torch.from_numpy(x).to(dev)
    spec = torch.empty(P, H, Wc, 2, dtype=torch.float32, device=dev)
    _lib.check(lib.admm_dbg_rows_r2c(_p(xt), _p(spec), P, H, W, _p(ws), ws.numel(), None), "rows_r2c")
    ref = M.rows_r2c(x.astype(np.float64))
    got = torch.view_as_complex(spec).cpu().numpy()
    assert _cerr(got, ref) < 2e-6, "row R2C"
    # column FFT forward then inverse
    spec2 = torch.empty_like(spec)
    _lib.check(lib.admm_dbg_cols_fft(_p(spec), _p(spec2), P, H, W, 0, _p(ws), ws.numel(), None), "cols fwd")
    ref2 = np.fft.fft(ref, axis=-2)
    got2 = torch.view_as_complex(spec2).cpu().numpy()
    assert _cerr(got2, ref2) < 3e-6, "column FFT"
    spec3 = torch.empty_like(spec)
    _lib.check(lib.admm_dbg_cols_fft(_p(spec2), _p(spec3), P, H, W, 1, _p(ws), ws.numel(), None), "cols inv")
    got3 = torch.view_as_complex(spec3).cpu().numpy() / H
    assert _cerr(got3, ref) < 4e-6, "column iFFT"
    # row C2R (unnormalised)
    back = torch.empty_like(xt)
    _lib.check(lib.admm_dbg_rows_c2r(_p(spec3), _p(back), P, H, W, _p(ws), ws.numel(), None), "rows_c2r")
    torch.cuda.synchronize()
    assert O.rel_err(back.cpu().numpy() / (H * W), x) < 5e-6, "round trip"


# ------------------------------------------------------------------------------- golden fixtures
@pytest.mark.parametrize("name", FWD_ANISO)
def test_forward_matches_reference_fixture(name):
    d = golden(name)
    out = _solve(d["x"], float(d["lam"]), float(d["rho"]), d["kern"], bool(d["iso"]), int(d["maxit"]))
    assert out.shape == d["out32"].shape and out.dtype == np.float32
    e64, e32 = O.rel_err(out, d["out64"]), O.rel_err(out, d["out32"])
    print("%s: vs ref64 %.2e  vs ref32 %.2e" % (name, e64, e32))
    assert e64 < TOL and e32 < TOL


@pytest.mark.parametrize("rows,cols", [(2, 1), (4, 3), (6, 8), (32, 16), (64, 32)])
def test_tiling_independence(rows, cols):
    """Band / tile sizes must not change the answer beyond fp32 noise."""
    from torch_admm_deconv_b200 import _lib
    d = golden("asym7_32x48_n20")
    _lib.set_option("rows_per_band", rows); _lib.set_option("cols_per_tile", cols)
    try:
        out = _solve(d["x"], float(d["lam"]), float(d["rho"]), d["kern"], False, int(d["maxit"]))
    finally:
        _lib.set_option("rows_per_band", 0); _lib.set_option("cols_per_tile", 0)
    assert O.rel_err(out, d["out64"]) < TOL


# ------------------------------------------------------------------------------- oracle on seeded inputs
@pytest.mark.parametrize("shape,k,kind,maxit", [
    ((2, 3, 64, 64), 15, "gauss", 30),
    ((1, 1, 256, 256), 15, "gauss", 50),          # cfg1
    ((2, 3, 128, 256), 31, "motion", 40),
    ((1, 2, 96, 80), 9, "gauss", 25),             # 2^5*3 x 2^4*5
    ((1, 1, 45, 63), 5, "gauss", 10),             # odd x odd
    ((3, 1, 50, 34), 0, None, 20),                # empty kernel, even non-pow2
])
def test_forward_matches_oracle(shape, k, kind, maxit):
    psf = O.make_psf(kind, k, 2.5) if k else None
    x = O.make_blurred(shape, psf, seed=99)
    kern = psf[None, None] if k else np.zeros((0,), np.float32)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.02, 0.04, kern, False, maxit)
    out = _solve(x, 0.02, 0.04, kern, False, maxit)
    e = O.rel_err(out, ref)
    print("shape %s k=%d N=%d err %.2e" % (shape, k, maxit, e))
    assert e < TOL


# ------------------------------------------------------------------------------- properties (any size)
def test_known_answers_on_gpu():
    rng = np.random.default_rng(5)
    x = rng.random((2, 3, 64, 48)).astype(np.float32)
    k = rng.random((5, 5)); k /= k.sum(); k4 = k[None, None].astype(np.float32)
    assert np.all(_solve(x, 0.02, 0.04, k4, False, 0) == 0)                      # maxit = 0 -> zeros
    c = np.full((1, 2, 32, 32), 0.37, np.float32)
    assert O.rel_err(_solve(c, 0.02, 0.04, k4, False, 5), c) < 1e-5              # constant image fixed point
    delta = np.zeros((1, 1, 3, 3), np.float32); delta[0, 0, 1, 1] = 1
    a = _solve(x, 0.05, 0.1, delta, False, 7); b = _solve(x, 0.05, 0.1, np.zeros((0,)), False, 7)
    assert O.rel_err(a, b) < 1e-5                                                # centred delta == denoise
    r = _solve(np.roll(x, (3, 5), (-2, -1)), 0.02, 0.04, k4, False, 6)
    assert O.rel_err(r, np.roll(_solve(x, 0.02, 0.04, k4, False, 6), (3, 5), (-2, -1))) < 2e-5   # shift equivariance


def test_batch_items_independent_bit_exact():
    """iso=False: planes are independent, so a batched call equals per-item calls bit for bit
    (SURVEY.md section 4 item 6); this is what makes batch sharding across GPUs collective-free."""
    psf = O.make_psf("gauss", 7, 1.5)
    x = O.make_blurred((4, 3, 64, 64), psf, seed=5)
    full = _solve(x, 0.02, 0.04, psf[None, None], False, 12)
    for b in range(4):
        one = _solve(x[b:b + 1], 0.02, 0.04, psf[None, None], False, 12)
        assert np.array_equal(one, full[b:b + 1])


def test_full_size_cfg2_slice_properties():
    """BASELINE cfg2 shape (512x512, 31-tap motion PSF) on a batch slice: oracle parity at a few
    iterations plus shift equivariance at the full 100 iterations."""
    psf = O.make_psf("motion", 31)
    x = O.make_blurred((2, 3, 512, 512), psf, seed=1234)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.02, 0.04, psf[None, None], False, 100)
    out = _solve(x, 0.02, 0.04, psf[None, None], False, 100)
    e = O.rel_err(out, ref)
    print("cfg2 slice err %.2e" % e)
    assert e < TOL
    r = _solve(np.roll(x, (17, 250), (-2, -1)), 0.02, 0.04, psf[None, None], False, 100)
    assert O.rel_err(r, np.roll(out, (17, 250), (-2, -1))) < TOL


def test_module_forward_matches_reference_fixture():
    from torch_admm_deconv_b200 import ADMMDeconv
    d = golden("module_k5_bias")
    m = ADMMDeconv((5, 5), max_iters=8, lmbda=None, rho=None, iso=False, bias=True)
    m.load_state_dict({k: torch.from_numpy(d["sd_" + k]) for k in ("w", "lmbda", "rho", "b")}, strict=True)
    m = m.to(_dev())
    with torch.inference_mode():
        out = m(torch.from_numpy(d["x"]).to(_dev()))
    assert O.rel_err(out.cpu().numpy(), d["out32"]) < TOL


def test_errors_on_gpu():
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    lam, rho = torch.tensor([0.02], device=dev), torch.tensor([0.04], device=dev)
    x = torch.zeros(1, 1, 16, 16, device=dev)
    with pytest.raises(RuntimeError):                                            # non-square PSF, like the reference
        fft_admm_tv(x, lam, rho, torch.zeros(1, 1, 3, 5, device=dev))
    with pytest.raises(ValueError):                                              # PSF larger than the image
        fft_admm_tv(x, lam, rho, torch.zeros(1, 1, 17, 17, device=dev))
    with pytest.raises(TypeError):
        fft_admm_tv(x.double(), lam, rho, torch.empty(0, device=dev))


@pytest.mark.parametrize("shape", [(2, 1, 256, 256), (1, 3, 512, 512), (3, 1, 128, 128), (1, 2, 512, 128), (2, 1, 128, 512),
                                   (1, 1, 6, 256), (2, 1, 30, 512), (1, 2, 256, 24), (5, 1, 62, 128), (1, 1, 34, 256)])
def test_specialised_pow2_kernels_match_generic(shape):
    """The power-of-two kernels (rows_pow2.cu / cols_pow2.cu) against the generic kernels and the oracle,
    including bands that do not fill a CTA and mixed generic/specialised passes."""
    from torch_admm_deconv_b200 import _lib
    psf = O.make_psf("gauss", 5, 1.2)
    x = O.make_blurred(shape, psf, seed=77)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.02, 0.04, psf[None, None], False, 12)
    fast = _solve(x, 0.02, 0.04, psf[None, None], False, 12)
    _lib.set_option("force_generic", 1)
    try:
        slow = _solve(x, 0.02, 0.04, psf[None, None], False, 12)
    finally:
        _lib.set_option("force_generic", 0)
    e_fast, e_slow, e_fs = O.rel_err(fast, ref), O.rel_err(slow, ref), O.rel_err(fast, slow)
    print("shape %s: pow2 vs oracle %.2e, generic vs oracle %.2e, pow2 vs generic %.2e" % (shape, e_fast, e_slow, e_fs))
    assert e_fast < 1e-5 and e_slow < 1e-5 and e_fs < 1e-5


# ------------------------------------------------------------------------------- backward (a13)
GRAD_ANISO = [n for n in golden_names(prefix="grad") if "iso_" not in n or "aniso" in n]
# Gradient tolerances of the fp32 unrolled adjoint against fp64 (reference autograd fixtures / oracle adjoint):
#   x-gradient: max|a-b| / max|b| <= 1e-5 (observed 1e-7 .. 4e-7);  lambda / rho / kernel gradients: relative 1e-4.
# These hold whenever both sides decide the soft threshold's masks 1[|q| < tau] alike.  The ADMM iteration drives q to
# +-tau in flat regions (saturated duals), so on large inputs an fp32 forward decides a few borderline masks differently
# from an fp64 one (measured: ~1 element per 12 planes of 256 x 256 over 10 iterations; the fp32 numpy oracle flips as
# often), and each such element moves the gradient by O(1) locally -- for any fp32 implementation.  The oracle-based
# tests therefore (i) gate the saved forward state itself, (ii) gate the adjoint SHARPLY with the masks taken from that
# state (`qs_override`), and (iii) gate the end-to-end gradient in the relative L2 norm with a bound on the flip count.
GRAD_TOL_X = 1e-5
GRAD_TOL_P = 1e-4
GRAD_TOL_L2 = 1e-3
GRAD_TOL = GRAD_TOL_X


def _grads(x, lam, rho, kern, gout, iso, maxit, return_state=False):
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    xt = torch.tensor(np.asarray(x, np.float32), device=dev, requires_grad=True)
    lt = torch.tensor([lam], dtype=torch.float32, device=dev, requires_grad=True)
    rt = torch.tensor([rho], dtype=torch.float32, device=dev, requires_grad=True)
    if np.size(kern):
        kt = torch.tensor(np.asarray(kern, np.float32), device=dev, requires_grad=True)
    else:
        kt = torch.empty(0, device=dev)
    out = fft_admm_tv(xt, lt, rt, kt, iso, maxit)
    state = None
    if return_state:
        # the per-iteration pre-threshold fields the forward saved for its backward (ctx.save_for_backward, last entry):
        # slots 1 .. maxit-1, each [q_x (B,C,H,W), q_y (B,C,H,W)] in float32
        saved = out.grad_fn.saved_tensors[4]
        n = int(np.prod(x.shape))
        q = saved[: (maxit - 1) * 2 * n * 4].view(torch.float32).reshape(maxit - 1, 2, *x.shape).cpu().numpy()
        state = [(q[k, 0], q[k, 1]) for k in range(maxit - 1)]
    (out * torch.tensor(np.asarray(gout, np.float32), device=dev)).sum().backward()
    torch.cuda.synchronize()
    g = lambda t: None if t.grad is None else t.grad.cpu().numpy().astype(np.float64)
    res = (out.detach().cpu().numpy(), g(xt), g(lt), g(rt), (g(kt) if np.size(kern) else None))
    return res + (state,) if return_state else res


def _rel(a, b):
    return abs(float(a) - float(b)) / max(abs(float(b)), 1e-12)


def _check_grads_vs_oracle(x, kern, gout, iso, maxit, lam=0.02, rho=0.04, tag=""):
    """GPU forward + backward against the fp64 oracle: forward output, saved state, adjoint given that state (sharp),
    and the end-to-end gradient (L2 norm; borderline masks may differ, see the note at GRAD_TOL_X)."""
    x64 = np.asarray(x, np.float64)
    out, gx, gl, gr, gk, state = _grads(x, lam, rho, kern, gout, iso, maxit, return_state=True)
    ref, hist = O.admm_tv_spectral_form(x64, lam, rho, kern, iso, maxit, return_state=True)
    e_out = O.rel_err(out, ref)
    qmax = max(float(np.abs(h[0]).max()) for h in hist)
    e_q = max(float(np.abs(s_[0] - h[0]).max()) for s_, h in zip(state, hist)) / qmax if state else 0.0
    tau32 = float(np.float32(lam) / np.float32(rho))
    sx, sl, sr, sk = O.admm_tv_backward(x64, lam, rho, kern, gout, iso, maxit, qs_override=state, tau_override=tau32)
    fx, fl, fr, fk = O.admm_tv_backward(x64, lam, rho, kern, gout, iso, maxit)
    e_x = O.rel_err(gx, sx)
    # rho gradient = (spectral part) - taubar * lam / rho^2: the two parts can cancel almost completely (iso=True without a
    # kernel: 114.70 - 114.66 = 0.04 at the cfg4 shape), so its error is measured against the larger of the result and the
    # tau part  glam * lam / rho  (each part is accurate to fp32 level)
    r_scale = max(abs(float(sr)), abs(float(sl)) * abs(lam / rho), 1e-12)
    e_l, e_r = (_rel(gl[0], sl) if maxit > 1 else 0.0), abs(float(gr[0]) - float(sr)) / r_scale
    e_k = O.rel_err(gk, sk) if np.size(kern) else 0.0
    d = np.abs(gx - fx)
    l2 = float(np.linalg.norm(d) / np.linalg.norm(fx))
    flips = int((d > 1e-4 * np.abs(fx).max()).sum())
    print("%s %s k=%d iso=%s N=%d: out %.1e state %.1e | same-state: gx %.1e glam %.1e grho %.1e gkern %.1e | end-to-end: gx L2 %.1e "
          "max %.1e (%d of %d elements off by > 1e-4) glam %.1e grho %.1e"
          % (tag, tuple(x.shape), int(np.shape(kern)[-1]) if np.size(kern) else 0, iso, maxit, e_out, e_q, e_x, e_l, e_r, e_k,
             l2, d.max() / np.abs(fx).max(), flips, d.size, _rel(gl[0], fl) if maxit > 1 else 0.0, _rel(gr[0], fr)))
    assert e_out < TOL and e_q < 1e-5
    assert e_x < GRAD_TOL_X and e_l < GRAD_TOL_P and e_r < GRAD_TOL_P and e_k < GRAD_TOL_P
    assert l2 < GRAD_TOL_L2 and flips <= max(8, d.size // 50000)
    return gx, gl, gr, gk


def _close(a, b, tol, what):
    e = abs(float(a) - float(b)) / max(abs(float(b)), 1e-3)
    assert e < tol, "%s: got %r want %r (rel %.2e)" % (what, float(a), float(b), e)


@pytest.mark.parametrize("name", [n for n in golden_names(prefix="grad_aniso")])
def test_backward_matches_reference_autograd(name):
    d = golden(name)
    out, gx, gl, gr, gk = _grads(d["x"], float(d["lam"]), float(d["rho"]), d["kern"], d["gout"], False, int(d["maxit"]))
    assert O.rel_err(out, d["out64"]) < TOL
    e = O.rel_err(gx, d["gx"])
    print("%s: gx err %.2e  glam %g/%g  grho %g/%g" % (name, e, gl[0], d["glam"][0], gr[0], d["grho"][0]))
    assert e < GRAD_TOL_X
    _close(gl[0], d["glam"][0], GRAD_TOL_P, "grad lambda")
    _close(gr[0], d["grho"][0], GRAD_TOL_P, "grad rho")
    if d["kern"].size:
        assert O.rel_err(gk, d["gkern"]) < GRAD_TOL_P


@pytest.mark.parametrize("shape,k,maxit", [((2, 3, 64, 64), 7, 8), ((1, 2, 48, 40), 5, 6), ((2, 1, 33, 45), 3, 5),
                                           ((1, 1, 256, 256), 15, 10), ((2, 2, 32, 32), 0, 7),
                                           ((1, 1, 1080, 1920), 5, 4)])       # forward on the large-frame kernels
def test_backward_matches_oracle_adjoint(shape, k, maxit):
    rng = np.random.default_rng(sum(shape) + k)
    psf = O.make_psf("gauss", k, 1.5) if k else None
    x = O.make_blurred(shape, psf, seed=3, noise=0.02)
    kern = psf[None, None] if k else np.zeros((0,), np.float32)
    gout = rng.standard_normal(shape)
    _check_grads_vs_oracle(x, kern, gout, False, maxit)


def test_module_training_step():
    """Unrolled ADMM layer with learnable w / lmbda / rho / b: one fwd+bwd+SGD step runs and every parameter
    receives a finite gradient (cfg4 shape family, reduced)."""
    from torch_admm_deconv_b200 import ADMMDeconv
    dev = _dev()
    torch.manual_seed(0)
    m = ADMMDeconv((5, 5), max_iters=6, lmbda=None, rho=None, iso=False, bias=True).to(dev)
    with torch.no_grad():
        m.w.copy_(torch.from_numpy(O.make_psf("gauss", 5, 1.0)[None, None]).to(dev))
        m.lmbda.fill_(0.02); m.rho.fill_(0.04)
    x = torch.from_numpy(O.make_blurred((4, 3, 64, 64), O.make_psf("gauss", 5, 1.0), seed=9)).to(dev)
    opt = torch.optim.SGD(m.parameters(), lr=1e-4)
    loss = (m(x) ** 2).mean()
    loss.backward()
    for n, p in m.named_parameters():
        assert p.grad is not None and bool(torch.isfinite(p.grad).all()), n
    # bias gradient of mean(out^2) is 2*mean(out)
    with torch.no_grad():
        assert abs(float(m.b.grad) - 2 * float(m(x).mean())) < 1e-3
    opt.step()


# ------------------------------------------------------------------------------- iso=True (a10, module default)
@pytest.mark.parametrize("name", golden_names(prefix="iso"))
def test_iso_forward_matches_reference_fixture(name):
    d = golden(name)
    out = _solve(d["x"], float(d["lam"]), float(d["rho"]), d["kern"], True, int(d["maxit"]))
    e64, e32 = O.rel_err(out, d["out64"]), O.rel_err(out, d["out32"])
    print("%s: vs ref64 %.2e  vs ref32 %.2e" % (name, e64, e32))
    assert e64 < TOL and e32 < TOL


@pytest.mark.parametrize("shape,k,maxit", [((4, 3, 256, 256), 15, 20), ((2, 3, 45, 60), 5, 12), ((3, 1, 128, 512), 0, 15)])
def test_iso_forward_matches_oracle(shape, k, maxit):
    psf = O.make_psf("gauss", k, 2.0) if k else None
    x = O.make_blurred(shape, psf, seed=41)
    kern = psf[None, None] if k else np.zeros((0,), np.float32)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.02, 0.04, kern, True, maxit)
    out = _solve(x, 0.02, 0.04, kern, True, maxit)
    e = O.rel_err(out, ref)
    print("iso shape %s k=%d N=%d err %.2e" % (shape, k, maxit, e))
    assert e < TOL
    # the block threshold couples the batch: solving items separately must give a different answer
    if shape[0] > 1:
        one = _solve(x[:1], 0.02, 0.04, kern, True, maxit)
        assert O.rel_err(one, out[:1]) > 1e-4


@pytest.mark.parametrize("name", golden_names(prefix="grad_iso"))
def test_iso_backward_matches_reference_autograd(name):
    d = golden(name)
    out, gx, gl, gr, gk = _grads(d["x"], float(d["lam"]), float(d["rho"]), d["kern"], d["gout"], True, int(d["maxit"]))
    assert O.rel_err(out, d["out64"]) < TOL
    e = O.rel_err(gx, d["gx"])
    print("%s: gx err %.2e  glam %g/%g  grho %g/%g" % (name, e, gl[0], d["glam"][0], gr[0], d["grho"][0]))
    assert e < GRAD_TOL_X
    _close(gl[0], d["glam"][0], GRAD_TOL_P, "grad lambda")
    _close(gr[0], d["grho"][0], GRAD_TOL_P, "grad rho")
    if d["kern"].size:
        assert O.rel_err(gk, d["gkern"]) < GRAD_TOL_P


def test_module_default_is_iso_and_trains():
    """ADMMDeconv's defaults (iso=True, empty kernel, learnable lmbda/rho) are what the reference's training
    script uses (scripts/train.py:19-24); forward parity with the oracle and a backward through it."""
    from torch_admm_deconv_b200 import ADMMDeconv
    dev = _dev()
    m = ADMMDeconv((), max_iters=10, lmbda=None, rho=None).to(dev)
    assert m.iso is True
    with torch.no_grad():
        m.lmbda.fill_(0.05); m.rho.fill_(0.1)
    x = O.make_blurred((3, 3, 64, 64), None, seed=8, noise=0.05)
    xt = torch.from_numpy(x).to(dev).requires_grad_(True)
    y = m(xt)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.05, 0.1, np.zeros((0,)), True, 10)
    assert O.rel_err(y.detach().cpu().numpy(), ref) < TOL
    gout = np.random.default_rng(1).standard_normal(x.shape)
    (y * torch.from_numpy(gout.astype(np.float32)).to(dev)).sum().backward()
    gx64, gl64, gr64, _ = O.admm_tv_backward(x.astype(np.float64), 0.05, 0.1, np.zeros((0,)), gout, True, 10)
    assert O.rel_err(xt.grad.cpu().numpy(), gx64) < GRAD_TOL_X
    _close(float(m.lmbda.grad), gl64, GRAD_TOL_P, "grad lambda")
    _close(float(m.rho.grad), gr64, GRAD_TOL_P, "grad rho")


def test_host_pipeline_matches_direct_call():
    from torch_admm_deconv_b200 import fft_admm_tv
    from torch_admm_deconv_b200.pipeline import HostPipeline
    dev = _dev()
    psf = O.make_psf("gauss", 7, 1.5)
    lam, rho = torch.tensor([0.02], device=dev), torch.tensor([0.04], device=dev)
    kern = torch.from_numpy(psf[None, None]).to(dev)
    xs = [torch.from_numpy(O.make_blurred((2, 3, 64, 64), psf, seed=s)).pin_memory() for s in range(5)]
    outs = [torch.empty_like(x).pin_memory() for x in xs]
    pipe = HostPipeline(dev, lam, rho, kern, False, 9)
    for x, o in zip(xs, outs):
        pipe.submit(x, o)
    pipe.synchronize()
    for x, o in zip(xs, outs):
        ref = fft_admm_tv(x.to(dev), lam, rho, kern, False, 9).cpu()
        assert torch.equal(o, ref)


def test_cfg3_full_size_first_iterations():
    """BASELINE cfg3 shape (2160 x 3840 = 2^4 3^3 5 x 2^8 3 5, 63x63 PSF): mixed-radix generic engine at full
    size against the oracle for a few iterations (200 iterations would take the fp64 oracle minutes)."""
    psf = O.make_psf("gauss", 63, 8.0)
    x = O.make_blurred((1, 1, 2160, 3840), psf, seed=1234)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.02, 0.04, psf[None, None], False, 4)
    out = _solve(x, 0.02, 0.04, psf[None, None], False, 4)
    e = O.rel_err(out, ref)
    print("cfg3 full size, 4 iterations: err %.2e" % e)
    assert e < TOL


@pytest.mark.parametrize("H,W", [(1080, 1920), (1024, 1024), (720, 1280), (1440, 2560)])
def test_hd_frame_matches_oracle(H, W):
    """1080 x 1920 (rows 15*8*16, columns 15*9*8) and 1024 x 1024 (rows 8*8*16, columns 16*8*8, padded shared-memory
    maps) on the large-frame kernels against the fp64 oracle."""
    psf = O.make_psf("gauss", 21, 3.0)
    x = O.make_blurred((1, 2, H, W), psf, seed=77)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.02, 0.04, psf[None, None], False, 6)
    out = _solve(x, 0.02, 0.04, psf[None, None], False, 6)
    e = O.rel_err(out, ref)
    print("%dx%d, 6 iterations: err %.2e" % (H, W, e))
    assert e < TOL


@pytest.mark.parametrize("H,W", [(2160, 3840), (1080, 1920), (1080, 3840), (2160, 1920), (1024, 1024), (128, 2048),
                                 (64, 4096), (1024, 1920), (720, 1280), (1440, 2560), (720, 2560), (2048, 2048), (768, 768), (1536, 1536), (768, 3072)])
def test_large_frame_kernels_match_generic_engine(H, W):
    """2160 x 3840 (and the HD sizes 1080 / 1920) take the compile-time mixed-radix kernels (rows 15*16*16 / 15*8*16,
    columns 15*12*12 / 15*9*8; csrc/rows_big.cu, csrc/cols_big.cu).  They must agree with the generic engine (independent code: runtime plan, batch-fastest
    layout) on two planes -- plane indexing, band seams and the packed DC/Nyquist column included -- both with the
    clamped-dual state of inference and with the pre-clamp state that training saves for the backward."""
    from torch_admm_deconv_b200 import fft_admm_tv, _lib
    dev = _dev()
    psf = O.make_psf("motion", 31, 0.0)
    x = torch.from_numpy(O.make_blurred((1, 2, H, W), psf, seed=5)).to(dev)
    kern = torch.from_numpy(psf[None, None]).to(dev)
    lam, rho = torch.tensor([0.05], device=dev), torch.tensor([0.08], device=dev)
    _lib.set_option("use_big", 0)
    try:
        ref = fft_admm_tv(x, lam, rho, kern, False, 6).clone()
    finally:
        _lib.set_option("use_big", 3)
    for ub in (1, 2, 3):
        _lib.set_option("use_big", ub)
        try:
            out = fft_admm_tv(x, lam, rho, kern, False, 6)
            xg = x.clone().requires_grad_(True)
            out_train = fft_admm_tv(xg, lam, rho, kern, False, 6)       # saves q: ROWS_FULL instead of ROWS_FULL_U
        finally:
            _lib.set_option("use_big", 3)
        e = ((out - ref).abs().max() / ref.abs().max()).item()
        et = ((out_train.detach() - ref).abs().max() / ref.abs().max()).item()
        print("use_big %d: large kernels vs generic %.2e (inference), %.2e (state saved)" % (ub, e, et))
        assert e < 1e-5 and et < 1e-5


@pytest.mark.parametrize("shape", [(1, 2, 6, 3840), (2, 1, 4, 1920), (1, 2, 2160, 16), (1, 1, 1080, 48), (1, 1, 10, 3840)])
def test_large_axis_with_small_other_axis(shape):
    """Only ONE axis on the large-frame kernels (the other on the generic engine, row-major spectra in between): thin
    frames against the oracle -- a single band of 2..5 row pairs with wrap-around, column tiles with Wc = 8 and 24."""
    psf = O.make_psf("gauss", 3, 0.8)
    x = O.make_blurred(shape, psf, seed=sum(shape))
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.03, 0.05, psf[None, None], False, 7)
    out = _solve(x, 0.03, 0.05, psf[None, None], False, 7)
    e = O.rel_err(out, ref)
    print("%s: err %.2e" % (shape, e))
    assert e < TOL


@pytest.mark.parametrize("H,W", [(1080, 1920), (1024, 1024)])
def test_large_frame_iso_matches_oracle(H, W):
    """iso=True (the module default) on the large-frame sizes: C2R and R2C (divergence formed while loading) on the
    plain large-frame row kernel, tile-major spectra to and from the large column kernel; against the fp64 oracle."""
    psf = O.make_psf("gauss", 9, 2.0)
    x = O.make_blurred((1, 3, H, W), psf, seed=21)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.02, 0.04, psf[None, None], True, 5)
    out = _solve(x, 0.02, 0.04, psf[None, None], True, 5)
    e = O.rel_err(out, ref)
    print("iso %dx%d, 5 iterations: err %.2e" % (H, W, e))
    assert e < TOL


@pytest.mark.parametrize("H,W", [(1024, 512), (256, 1920), (512, 3840), (720, 512), (1440, 256), (2160, 1024),
                                 (720, 4096), (100, 1920), (1080, 100)])
@pytest.mark.parametrize("iso", [False, True])
def test_mixed_kernel_families_match_generic_engine(H, W, iso):
    """Every axis picks its own kernel family (power-of-two, large-frame or generic) and the spectra in between are
    row-major unless both axes are on the large-frame kernels: all combinations must agree with the generic engine."""
    from torch_admm_deconv_b200 import fft_admm_tv, _lib
    dev = _dev()
    g = torch.Generator().manual_seed(H * 7 + W)
    x = torch.rand(1, 2, H, W, generator=g).to(dev)
    kern = torch.rand(1, 1, 7, 7, generator=g).to(dev); kern /= kern.sum()
    lam, rho = torch.tensor([0.02], device=dev), torch.tensor([0.04], device=dev)
    _lib.set_option("force_generic", 1)
    try:
        ref = fft_admm_tv(x, lam, rho, kern, iso, 4).clone()
    finally:
        _lib.set_option("force_generic", 0)
    out = fft_admm_tv(x, lam, rho, kern, iso, 4)
    assert ((out - ref).abs().max() / ref.abs().max()).item() < 1e-5


def test_large_frame_kernels_are_deterministic():
    """The large-frame kernels reuse shared-memory buffers across passes and march steps under hand-placed barriers; a
    missing barrier shows up as run-to-run differences.  Three planes (more CTAs than resident slots), repeated."""
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    psf = O.make_psf("gauss", 15, 2.5)
    x = torch.from_numpy(O.make_blurred((1, 3, 2160, 3840), psf, seed=8)).to(dev)
    kern = torch.from_numpy(psf[None, None]).to(dev)
    lam, rho = torch.tensor([0.02], device=dev), torch.tensor([0.04], device=dev)
    first = fft_admm_tv(x, lam, rho, kern, False, 12).clone()
    for _ in range(4):
        assert torch.equal(fft_admm_tv(x, lam, rho, kern, False, 12), first)


def test_large_frame_band_height_independence():
    """The row kernel's result may not depend on how the frame is cut into bands (halo rows, wrap-around at the top
    and bottom edge)."""
    from torch_admm_deconv_b200 import fft_admm_tv, _lib
    dev = _dev()
    psf = O.make_psf("gauss", 9, 2.0)
    x = torch.from_numpy(O.make_blurred((1, 1, 2160, 3840), psf, seed=6)).to(dev)
    kern = torch.from_numpy(psf[None, None]).to(dev)
    lam, rho = torch.tensor([0.02], device=dev), torch.tensor([0.04], device=dev)
    outs = []
    for R in (0, 2, 10, 2160):
        _lib.set_option("rows_per_band", R)
        try:
            outs.append(fft_admm_tv(x, lam, rho, kern, False, 4).clone())
        finally:
            _lib.set_option("rows_per_band", 0)
    for o in outs[1:]:
        assert torch.equal(o, outs[0])


def test_cuda_graph_capture_and_replay():
    """The library only enqueues work on the current stream (no sync, no allocation inside the C ABI), so a whole
    solve can be captured in a CUDA graph and replayed -- the way to run small, launch-bound problems (cfg1)."""
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    psf = O.make_psf("gauss", 15, 2.5)
    x = torch.from_numpy(O.make_blurred((1, 1, 256, 256), psf, seed=1234)).to(dev)
    lam, rho = torch.tensor([0.02], device=dev), torch.tensor([0.04], device=dev)
    kern = torch.from_numpy(psf[None, None]).to(dev)
    ref = fft_admm_tv(x, lam, rho, kern, False, 20).clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fft_admm_tv(x, lam, rho, kern, False, 20)          # warm-up on the side stream
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fft_admm_tv(x, lam, rho, kern, False, 20)
    out.zero_()
    g.replay(); torch.cuda.synchronize()
    assert torch.equal(out, ref)
    x.mul_(0.5)                                            # new input in the same buffer, replay again
    g.replay(); torch.cuda.synchronize()
    assert torch.equal(out, fft_admm_tv(x, lam, rho, kern, False, 20))


@pytest.mark.parametrize("shape,k,maxit", [((2, 2, 128, 128), 5, 6), ((1, 2, 256, 128), 0, 5), ((2, 1, 128, 512), 7, 4),
                                           ((3, 1, 512, 256), 3, 5)])
def test_fused_backward_row_pass_matches_unfused(shape, k, maxit):
    """Power-of-two sizes take the fused backward row pass (ROWS_ADJ); force_generic takes the elementwise path.
    Both must agree with each other and with the fp64 oracle adjoint."""
    from torch_admm_deconv_b200 import _lib
    rng = np.random.default_rng(sum(shape))
    psf = O.make_psf("gauss", k, 1.2) if k else None
    x = O.make_blurred(shape, psf, seed=5, noise=0.02)
    kern = psf[None, None] if k else np.zeros((0,), np.float32)
    gout = rng.standard_normal(shape)
    _check_grads_vs_oracle(x, kern, gout, False, maxit, tag="fused")
    _lib.set_option("force_generic", 1)
    try:
        _check_grads_vs_oracle(x, kern, gout, False, maxit, tag="unfused")
    finally:
        _lib.set_option("force_generic", 0)


def test_multi_solver_fanout_matches_sequential():
    """MultiADMM / Deconvs (reference modelbuild/blocks.py:252-261, deconver.py:8-23): solvers on separate streams
    give exactly the sequential concatenation, forward and backward."""
    from torch_admm_deconv_b200 import MultiADMM, Deconvs
    import time
    dev = _dev()
    cfgs = [dict(kern_size=(), max_iters=12, lmbda=0.02, rho=0.04, iso=True),
            dict(kern_size=(5, 5), max_iters=8, lmbda=None, rho=None, iso=False),
            dict(kern_size=(), max_iters=10, lmbda=None, rho=None, iso=False, bias=True)]
    torch.manual_seed(3)
    m = MultiADMM(cfgs).to(dev)
    assert list(m.state_dict().keys())[:4] == ["admms.0.w", "admms.0.lmbda", "admms.0.rho", "admms.0.b"]
    with torch.no_grad():
        m.admms[1].w.copy_(torch.from_numpy(O.make_psf("gauss", 5, 1.0)[None, None]).to(dev))
        for a in m.admms[1:]:
            a.lmbda.fill_(0.03); a.rho.fill_(0.05)
    x = torch.from_numpy(O.make_blurred((3, 3, 256, 256), None, seed=2, noise=0.05)).to(dev).requires_grad_(True)
    y = m(x)
    assert y.shape == (3, 9, 256, 256)
    (y ** 2).mean().backward()
    gx = x.grad.clone(); gl = m.admms[1].lmbda.grad.clone()
    x.grad = None; m.zero_grad()
    m.concurrent = False
    y2 = m(x)
    (y2 ** 2).mean().backward()
    assert torch.equal(y, y2)
    assert torch.allclose(gx, x.grad, rtol=1e-5, atol=1e-7) and torch.allclose(gl, m.admms[1].lmbda.grad, rtol=1e-4)
    d = Deconvs(cfgs[:2]).to(dev)
    assert d(x.detach()).shape == (3, 6, 256, 256) and list(d.state_dict().keys())[0] == "blocks.0.w"
    # timing (informative): inference, concurrent vs sequential
    with torch.no_grad():
        for flag in (True, False):
            m.concurrent = flag
            m(x); torch.cuda.synchronize(); t0 = time.perf_counter()
            for _ in range(5):
                m(x)
            torch.cuda.synchronize()
            print("fan-out concurrent=%s: %.3f ms" % (flag, (time.perf_counter() - t0) / 5 * 1e3))


@pytest.mark.parametrize("lam,rho,iso,maxit,k", [(0.02, 0.02, True, 300, 7), (0.02, 0.04, False, 300, 7), (0.02, 0.005, False, 150, 7),
                                                 (0.5, 0.1, False, 200, 0)])
def test_many_iterations_and_stiff_parameters(lam, rho, iso, maxit, k):
    """Hundreds of iterations (the reference notebook runs 300, notebooks/test_torch_admm.ipynb:232-249), small rho and
    strong regularisation: fp32 error growth must stay far below the 1e-4 bar."""
    psf = O.make_psf("gauss", k, 1.5) if k else None
    x = O.make_blurred((2, 3, 128, 128), psf, seed=1, noise=0.08)
    kern = psf[None, None] if k else np.zeros((0,), np.float32)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), lam, rho, kern, iso, maxit)
    e = O.rel_err(_solve(x, lam, rho, kern, iso, maxit), ref)
    print("lam=%g rho=%g iso=%s N=%d: err %.2e" % (lam, rho, iso, maxit, e))
    assert e < TOL / 4


@pytest.mark.parametrize("shape,k", [((1, 1, 2, 2), 0), ((2, 1, 2, 3), 2), ((1, 2, 3, 2), 1), ((1, 1, 4, 4), 4), ((2, 2, 5, 7), 5),
                                     ((1, 1, 16, 16), 16)])
def test_tiny_images_and_image_sized_kernels(shape, k):
    """Degenerate geometry: 2x2 images, 1x1 PSF, PSF as large as the image."""
    rng = np.random.default_rng(sum(shape) + k)
    x = rng.random(shape).astype(np.float32)
    kern = np.zeros((0,), np.float32)
    if k:
        kern = rng.random((1, 1, k, k)).astype(np.float32); kern /= kern.sum()
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.02, 0.04, kern, False, 9)
    assert O.rel_err(_solve(x, 0.02, 0.04, kern, False, 9), ref) < TOL


def test_cfg2_full_batch_properties():
    """BASELINE cfg2 at FULL size (64 x 3 x 512 x 512, 31-tap motion PSF, 100 iterations): per-item independence
    (bit exact), circular-shift equivariance and oracle parity on one item."""
    psf = O.make_psf("motion", 31)
    x = O.make_blurred((64, 3, 512, 512), psf, seed=1234)
    full = _solve(x, 0.02, 0.04, psf[None, None], False, 100)
    assert np.isfinite(full).all()
    for b in (0, 37, 63):
        assert np.array_equal(_solve(x[b:b + 1], 0.02, 0.04, psf[None, None], False, 100), full[b:b + 1])
    r = _solve(np.roll(x[5:7], (100, 33), (-2, -1)), 0.02, 0.04, psf[None, None], False, 100)
    assert O.rel_err(r, np.roll(full[5:7], (100, 33), (-2, -1))) < TOL
    ref = O.admm_tv_spectral_form(x[11:12].astype(np.float64), 0.02, 0.04, psf[None, None], False, 100)
    assert O.rel_err(full[11:12], ref) < TOL


def test_cfg5_shard_properties():
    """BASELINE cfg5 per-GPU shard at 8 GPUs (512 x 3 x 256 x 256, 15x15 Gaussian, 50 iterations): sharding the
    batch in two halves (what two ranks would do) reproduces the unsharded result bit for bit."""
    psf = O.make_psf("gauss", 15, 2.5)
    x = O.make_blurred((512, 3, 256, 256), psf, seed=1234)
    full = _solve(x, 0.02, 0.04, psf[None, None], False, 50)
    lo = _solve(x[:256], 0.02, 0.04, psf[None, None], False, 50)
    hi = _solve(x[256:], 0.02, 0.04, psf[None, None], False, 50)
    assert np.array_equal(np.concatenate([lo, hi]), full)
    ref = O.admm_tv_spectral_form(x[300:301].astype(np.float64), 0.02, 0.04, psf[None, None], False, 50)
    assert O.rel_err(full[300:301], ref) < TOL


# ------------------------------------------------------------------------------- BASELINE configs at their REAL shape and length
def _cfg3_summary(out):
    d = golden("cfg3_2160x3840_gauss63_n200")
    crops = np.stack([out[0, :, r:r + 64, c:c + 64] for r, c in d["crops"]]).astype(np.float64)
    return crops, out[0].mean(axis=2, dtype=np.float64), out[0].mean(axis=1, dtype=np.float64)


def test_cfg3_full_length_matches_reference_fixture():
    """BASELINE configs[2] in full: 1 x 3 x 2160 x 3840, 63 x 63 Gaussian PSF, 200 iterations, against the fixture written by
    tests/golden/make_golden_cfg3.py: the fp64 oracle (spectral form) and the UNMODIFIED reference in fp32 on the same input
    (the reference cannot run this size in fp64: its 63 x 63 double conv wants 263 GB).  The fixture keeps six 64 x 64 crops of
    every channel (the four wrap-around corners included) plus all row and column means; tolerance max|a-b| / max|ref| <= 1e-4."""
    d = golden("cfg3_2160x3840_gauss63_n200")
    psf = O.make_psf("gauss", int(d["k"]), float(d["sigma"]))
    x = O.make_blurred(tuple(int(v) for v in d["shape"]), psf, seed=int(d["seed"]))
    # the input must be the one the fixture was made from (numpy generator + FFT are deterministic on the same image)
    assert np.array_equal(x[0, :, :8, :8], d["x_crop0"]) and abs(float(x.sum(dtype=np.float64)) - float(d["x_sum"])) < 1e-3
    out = _solve(x, float(d["lam"]), float(d["rho"]), psf[None, None], False, int(d["maxit"]))
    assert np.isfinite(out).all()
    crops, rowm, colm = _cfg3_summary(out)
    for tag in ("oracle64", "ref32"):
        if tag + "_crops" not in d.files:
            continue
        amax = float(d[tag + "_absmax"])
        e_c = float(np.abs(crops - d[tag + "_crops"]).max() / amax)
        e_r = float(np.abs(rowm - d[tag + "_rowmean"]).max() / amax)
        e_m = float(np.abs(colm - d[tag + "_colmean"]).max() / amax)
        print("cfg3, 200 iterations vs %s: crops %.2e  row means %.2e  column means %.2e" % (tag, e_c, e_r, e_m))
        assert e_c < TOL and e_r < TOL and e_m < TOL


@pytest.mark.parametrize("k", [0, 15])
@pytest.mark.parametrize("iso", [False, True])
def test_cfg4_real_shape_backward_matches_oracle_adjoint(k, iso):
    """BASELINE configs[3] at its own shape: 32 x 3 x 256 x 256, 10 unrolled iterations, learnable lambda / rho, with
    `kern_size=()` (what scripts/train.py:19-24 trains) and with a learnable 15 x 15 kernel, iso False and True (the module
    default): forward, saved state and all gradients against the fp64 oracle adjoint (itself pinned to the reference's
    autograd to 3e-15).  See the note at GRAD_TOL_X for the three gates."""
    shape, maxit = (32, 3, 256, 256), 10
    rng = np.random.default_rng(40 + k + int(iso))
    psf = O.make_psf("gauss", k, 2.5) if k else None
    x = O.make_blurred(shape, psf, seed=4, noise=0.02)
    kern = psf[None, None] if k else np.zeros((0,), np.float32)
    gout = rng.standard_normal(shape)
    _check_grads_vs_oracle(x, kern, gout, iso, maxit, tag="cfg4")


@pytest.mark.parametrize("shape,k,iso", [((32, 3, 256, 256), 15, False), ((32, 3, 256, 256), 0, True), ((2, 3, 60, 90), 5, False),
                                         ((1, 2, 1080, 1920), 5, False)])
def test_backward_is_bit_reproducible(shape, k, iso):
    """Every reduction of the backward is two-stage in a fixed order (per-CTA slots for the tau gradient, per-plane-group
    slices for the spectral sums; no floating-point atomics): repeated backward passes give bit-identical gradients."""
    rng = np.random.default_rng(7)
    psf = O.make_psf("gauss", k, 1.5) if k else None
    x = O.make_blurred(shape, psf, seed=6, noise=0.02)
    kern = psf[None, None] if k else np.zeros((0,), np.float32)
    gout = rng.standard_normal(shape)
    first = _grads(x, 0.02, 0.04, kern, gout, iso, 6)
    for _ in range(3):
        again = _grads(x, 0.02, 0.04, kern, gout, iso, 6)
        for a, b in zip(first, again):
            assert (a is None and b is None) or np.array_equal(a, b)


def test_maxit_zero_with_bias_returns_bias():
    """ADMMDeconv(max_iters=0, bias=True): the solve returns zeros (deconv.py:61,103,117) and the layer still adds b
    (admmdeconv.py:64)."""
    from torch_admm_deconv_b200 import ADMMDeconv
    dev = _dev()
    m = ADMMDeconv((3, 3), max_iters=0, lmbda=0.02, rho=0.04, iso=False, bias=True).to(dev)
    x = torch.rand(2, 3, 16, 16, device=dev, requires_grad=True)
    y = m(x)
    assert torch.equal(y, m.b.detach().expand_as(y))
    y.sum().backward()
    assert float(m.b.grad) == y.numel() and float(x.grad.abs().max()) == 0.0


@pytest.mark.parametrize("shape,k,maxit,K", [((2, 3, 64, 64), 5, 11, 3), ((1, 2, 128, 256), 0, 10, 4), ((2, 1, 60, 90), 3, 9, 2),
                                             ((2, 2, 256, 256), 7, 26, -1), ((1, 1, 48, 40), 3, 7, 10),
                                             # odd heights (generic rows, the last band's halo wraps to row 0); K = 6 of 7
                                             # slots re-runs a one-slot block, K = 8 of 8 slots keeps only the last one
                                             ((1, 2, 33, 45), 5, 10, 3), ((2, 3, 31, 37), 3, 9, -1), ((1, 1, 45, 63), 5, 8, 6),
                                             ((1, 2, 33, 45), 3, 9, 8), ((1, 1, 45, 256), 5, 6, 2)])
def test_checkpointed_training_matches_full_state(shape, k, maxit, K):
    """Memory-saving training (admm_ext.ckpt_interval): the forward keeps every K-th iteration's state, the backward re-runs
    each block from its checkpoint.  Gradients must equal those of the run that keeps every iteration and the saved buffer
    must be the promised size."""
    from torch_admm_deconv_b200.eops.deconv import admm_solve
    from torch_admm_deconv_b200 import _lib
    dev = _dev()
    rng = np.random.default_rng(sum(shape) + K)
    psf = O.make_psf("gauss", k, 1.5) if k else None
    x = O.make_blurred(shape, psf, seed=13, noise=0.02)
    gout = torch.tensor(rng.standard_normal(shape).astype(np.float32), device=dev)
    res = []
    for ck in (0, K):
        xt = torch.tensor(x, device=dev, requires_grad=True)
        lt = torch.tensor([0.02], device=dev, requires_grad=True); rt = torch.tensor([0.04], device=dev, requires_grad=True)
        kt = torch.tensor(psf[None, None], device=dev, requires_grad=True) if k else torch.empty(0, device=dev)
        out = admm_solve(xt, lt, rt, kt, False, maxit, ckpt_interval=ck)
        nbytes = out.grad_fn.saved_tensors[4].numel()
        (out * gout).sum().backward()
        res.append((out.detach(), xt.grad, lt.grad, rt.grad, kt.grad if k else None, nbytes))
    full, ck = res
    Keff = K if K > 0 else int(np.ceil(np.sqrt(maxit - 1)))
    field = int(np.prod(shape)) * 4
    assert ck[5] <= ((maxit - 1) // Keff) * 2 * field + 256 and full[5] >= (maxit - 1) * 2 * field
    assert torch.equal(full[0], ck[0])
    # the restart recomputes v_k with the forward's operation order, so the regenerated fields -- and with them every
    # threshold mask and gradient -- are bit-identical to the run that kept all iterations
    for a, b in zip(full[1:5], ck[1:5]):
        if a is not None:
            assert torch.equal(a, b), float((a - b).abs().max() / a.abs().max().clamp_min(1e-30))
    lib = _lib.load()
    assert lib.admm_query_saved_ex(6, 64, 64, 0, 1, 10, 3) == 0          # iso=True: not available, callers fall back


# ------------------------------------------------------------------------------- cluster-resident solver (cluster_pow2.cu)
def _with_cluster(mode, fn):
    from torch_admm_deconv_b200 import _lib
    _lib.set_option("use_cluster", mode)
    try:
        return fn()
    finally:
        _lib.set_option("use_cluster", 1)


@pytest.mark.parametrize("shape,k,maxit,lam", [((1, 1, 256, 256), 15, 50, 0.02),      # BASELINE configs[0]
                                               ((3, 1, 128, 128), 5, 12, 0.02), ((2, 2, 128, 256), 7, 9, 0.02),
                                               ((1, 3, 256, 128), 0, 10, 0.05), ((1, 1, 256, 256), 3, 1, 0.02),
                                               ((2, 1, 256, 256), 3, 2, 0.02), ((1, 2, 256, 256), 5, 7, -0.01),
                                               ((7, 3, 256, 256), 9, 6, 0.02)])       # 21 planes: more planes than clusters
def test_cluster_solver_matches_two_kernel_path(shape, k, maxit, lam):
    """One launch, a 16-CTA thread-block cluster per plane, spectra exchanged through distributed shared memory: the
    arithmetic is that of rows_pow2.cu / cols_pow2.cu in the same order (the compiler contracts a few multiply-adds
    differently inside the larger kernel, so the agreement is to the last fp32 digits, not bit for bit), and the result
    is gated against the fp64 oracle like every other path."""
    psf = O.make_psf("gauss", k, 1.5) if k else None
    x = O.make_blurred(shape, psf, seed=sum(shape) + k)
    kern = psf[None, None] if k else np.zeros((0,), np.float32)
    a = _with_cluster(2, lambda: _solve(x, lam, 0.04, kern, False, maxit))
    b = _with_cluster(0, lambda: _solve(x, lam, 0.04, kern, False, maxit))
    ref = O.admm_tv_spectral_form(x.astype(np.float64), lam, 0.04, kern, False, maxit)
    e_ab, e_a, e_b = O.rel_err(a, b), O.rel_err(a, ref), O.rel_err(b, ref)
    print("%s k=%d N=%d: cluster vs two-kernel %.1e; vs oracle: cluster %.1e, two-kernel %.1e" % (shape, k, maxit, e_ab, e_a, e_b))
    # tau < 0 makes u(q) jump by 2|tau| at q = 0: on this input the reference's own fp32 run is 0.49 away from its fp64 run
    # after 7 iterations, so only the agreement of the two GPU paths is checked there
    assert np.isfinite(a).all() and e_ab < 5e-6 and (e_a < TOL or lam < 0)


def test_cluster_solver_cfg1_reference_fixture_and_epilogues():
    """cfg1 in full against the reference's own fp32 / fp64 outputs, through the cluster solver (the default for a single
    plane); plus the fused layer epilogue / prologue (bias, sigmoid, uint8 input, channel-slice output) on that path."""
    from torch_admm_deconv_b200 import ADMMDeconv, _lib
    d = golden("cfg1_256_gauss15_n50")
    assert _lib.get_option("use_cluster") == 1
    n0 = _lib.launch_count()
    out = _solve(d["x"], float(d["lam"]), float(d["rho"]), d["kern"], False, int(d["maxit"]))
    assert _lib.launch_count() - n0 <= 6                # twiddles, tables, ONE solver launch (the two-kernel path: ~104)
    assert O.rel_err(out, d["out64"]) < TOL and O.rel_err(out, d["out32"]) < TOL
    dev = _dev()
    img = torch.randint(0, 256, (2, 3, 128, 128), dtype=torch.uint8, device=dev)
    m = ADMMDeconv((5, 5), max_iters=8, lmbda=0.02, rho=0.04, iso=False, bias=True, activation=torch.sigmoid).to(dev)
    with torch.no_grad():
        m.w.copy_(torch.from_numpy(O.make_psf("gauss", 5, 1.0)[None, None]).to(dev)); m.b.fill_(-0.3)
    big = torch.zeros(2, 7, 128, 128, device=dev)
    with torch.inference_mode():
        y1 = _with_cluster(2, lambda: m(img, out=big[:, 2:5]).clone())
        y0 = _with_cluster(0, lambda: m(img))
    assert float((y1 - y0).abs().max()) < 2e-6 and torch.equal(big[:, 2:5], y1) and float(big[:, :2].abs().max()) == 0.0


def test_two_stream_batch_split_is_bit_identical():
    """Large inference batches are solved as two halves on two streams (eops/deconv.py, SPLIT_STREAMS): same bits as the
    single-stream call, also for an odd batch, a channel-slice output and a fused activation."""
    from torch_admm_deconv_b200.eops import deconv as D
    dev = _dev()
    psf = O.make_psf("gauss", 7, 1.5)
    x = torch.from_numpy(O.make_blurred((11, 3, 256, 256), psf, seed=3)).to(dev)
    kern = torch.from_numpy(psf[None, None]).to(dev)
    lam, rho = torch.tensor([0.02], device=dev), torch.tensor([0.04], device=dev)
    b = torch.tensor([0.1], device=dev)
    old = (D.SPLIT_STREAMS, D.SPLIT_MIN_ELEMENTS)
    try:
        D.SPLIT_MIN_ELEMENTS = 1
        D.SPLIT_STREAMS = 1
        ref = D.admm_solve(x, lam, rho, kern, False, 9, bias=b, activation=torch.tanh)
        D.SPLIT_STREAMS = 2
        out = D.admm_solve(x, lam, rho, kern, False, 9, bias=b, activation=torch.tanh)
        big = torch.zeros(11, 8, 256, 256, device=dev)
        D.admm_solve(x, lam, rho, kern, False, 9, bias=b, activation=torch.tanh, out=big[:, 4:7])
    finally:
        D.SPLIT_STREAMS, D.SPLIT_MIN_ELEMENTS = old
    torch.cuda.synchronize()
    assert torch.equal(out, ref) and torch.equal(big[:, 4:7], ref) and float(big[:, :4].abs().max()) == 0.0


# ------------------------------------------------------------------------------- cooperative small-batch kernel (coop_small.cu)
@pytest.mark.parametrize("shape,k,iso,maxit", [((8, 3, 256, 256), 0, True, 30), ((3, 3, 256, 256), 5, True, 12), ((5, 3, 256, 256), 7, False, 15),
                                               ((1, 3, 512, 512), 9, True, 8), ((2, 2, 512, 256), 3, False, 9), ((3, 1, 128, 512), 0, True, 6),
                                               ((2, 1, 128, 128), 5, True, 1), ((2, 1, 128, 128), 5, False, 2), ((16, 3, 256, 256), 5, False, 5)])
def test_cooperative_small_batch_kernel_matches_two_kernel_path(shape, k, iso, maxit):
    """Option use_coop: iterations 1 .. maxit-1 in ONE cooperative launch (a grid barrier between the phases, the phase bodies
    are those of the stand-alone kernels).  Measured slower than the separate launches and off by default (coop_small.cu);
    the test keeps the shared kernel bodies honest: same bits as the separate launches, and oracle parity."""
    from torch_admm_deconv_b200 import _lib
    psf = O.make_psf("gauss", k, 1.5) if k else None
    x = O.make_blurred(shape, psf, seed=sum(shape) + k, noise=0.03)
    kern = psf[None, None] if k else np.zeros((0,), np.float32)
    outs = []
    _lib.set_option("use_cluster", 0)
    try:
        for mode in (2, 0):
            _lib.set_option("use_coop", mode)
            n0 = _lib.launch_count()
            outs.append(_solve(x, 0.02, 0.04, kern, iso, maxit))
            n = _lib.launch_count() - n0
            if mode == 2 and maxit > 1:
                assert n <= 8, n                      # twiddles, tables, R2C, INIT, ONE cooperative launch, C2R
    finally:
        _lib.set_option("use_coop", 0); _lib.set_option("use_cluster", 1)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.02, 0.04, kern, iso, maxit)
    e_ab, e_a = O.rel_err(outs[0], outs[1]), O.rel_err(outs[0], ref)
    print("%s k=%d iso=%s N=%d: cooperative vs separate launches %.1e; vs oracle %.1e" % (shape, k, iso, maxit, e_ab, e_a))
    assert np.isfinite(outs[0]).all() and e_ab < 5e-6 and e_a < TOL
