"""λ maps (spatially varying regularisation, DESIGN.md section 11) on the GPU: forward and backward.

A `lmbd` tensor that broadcasts to (B, C, H, W) gives the threshold tau = lmbd / rho element by element, as in the
reference (deconv.py:15-24, 44).  The gates:
  a. a map filled with the scalar λ gives, on the same kernel route, the scalar solve's output and x-gradient bit for bit,
     and its summed map gradient, ρ and kernel gradients within 1e-6 (the λ and ρ sums relative to the L1 norm of the
     summed terms: they cancel, and the two solves add them in different orders);
  b. one iteration at a time against an fp64 replay with a tau array (the pattern of test_gpu_routes.py): the GPU's saved
     states, its output and its adjoint (grad_tau, fixed-tau grad_rho, x and kernel gradients) from the same state;
  c. end to end against a float64 torch restatement of deconv.py:103-115 with a tensor tau, and gradcheck of that
     restatement's λ-map path against the library's on a small case;
  d. training: checkpointed = full-state gradients, bit-reproducible backward, an ADMMDeconv whose λ is a map Parameter;
  e. errors raised before anything runs."""
import numpy as np
import pytest
import torch

from oracle import admm_oracle as O

pytestmark = pytest.mark.gpu

STEP_TOL = 5e-6
GRAD_TOL_X = 1e-5
GRAD_TOL_P = 1e-4
RHO = 0.04


def _dev():
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    return torch.device("cuda:0")


def _with_options(opts, fn):
    from torch_admm_deconv_b200 import _lib
    old = {k: _lib.get_option(k) for k in opts}
    try:
        for k, v in opts.items():
            _lib.set_option(k, v)
        return fn()
    finally:
        for k, v in old.items():
            _lib.set_option(k, v)


def _inputs(shape, k, seed):
    psf = O.make_psf("gauss", k, 1.5) if k else None
    kern = psf[None, None] if k else np.zeros((0,), np.float32)
    x = O.make_blurred(shape, psf, seed=seed, noise=0.02)
    gout = np.random.default_rng(seed + 1).standard_normal(shape)
    return x, kern, gout


def make_map(shape, kind, seed, lam=0.02):
    """λ map of `kind`: "shared" (1, 1, H, W) positive, "full" (B, C, H, W) positive, "mixed" (1, 1, H, W) of both signs,
    "zeros" (B, C, H, W) with a fifth of the entries 0, "plane" (B, C, 1, 1)."""
    B, C, H, W = shape
    r = np.random.default_rng(seed)
    if kind == "plane":
        return (lam * r.uniform(0.5, 1.5, (B, C, 1, 1))).astype(np.float32)
    s = (1, 1, H, W) if kind in ("shared", "mixed") else (B, C, H, W)
    m = lam * r.uniform(0.3, 1.7, s)
    if kind == "mixed":
        m *= np.where(r.random(s) < 0.4, -1.0, 1.0)
    if kind == "zeros":
        m[r.random(s) < 0.2] = 0.0
    return m.astype(np.float32)


# ------------------------------------------------------------------------------------------------ fp64 oracle with maps
def _soft(q, tau):
    return np.sign(q) * np.maximum(np.abs(q) - tau, 0)


def replay_map(x, kern, states, tau, iso=False, nmaps=None):
    """`admm_tv_replay` (oracle/admm_oracle.py) with an array tau broadcasting to the image (iso: an (H, W) array)."""
    x = np.asarray(x, np.float64)
    B, C, H, W = x.shape
    k2d = O._kernel_2d(kern)
    sg, ph, L, den = O._spectral_tables(H, W, None if k2d is None else np.asarray(k2d, np.float64), RHO, np.float64)
    A = sg * ph * O._rfft2(x, -1) / den
    Bm = RHO / den

    def dual(qx, qy, nm):
        if iso:
            nx, ny = (np.asarray(n, np.float64) for n in nm)
            sx = np.maximum(1 - tau / (nx + 1e-15), 0); sy = np.maximum(1 - tau / (ny + 1e-15), 0)
            return (1 - sx) * qx, (1 - sy) * qy
        return qx - _soft(qx, tau), qy - _soft(qy, tau)

    def step(k):
        if k == 0:
            xn = O._irfft2(A, (H, W), -1)
            return xn, (O._dx(xn), O._dy(xn))
        qx, qy = (np.asarray(t, np.float64) for t in states[k - 1])
        ux, uy = dual(qx, qy, None if nmaps is None else nmaps[k - 1])
        v = O._dxt(qx - 2 * ux) + O._dyt(qy - 2 * uy)
        xn = O._irfft2(A + Bm * O._rfft2(v, -1), (H, W), -1)
        return xn, (O._dx(xn) + ux, O._dy(xn) + uy)

    preds = [step(k)[1] for k in range(len(states))]
    return preds, step(len(states))[0]


def adjoint_map(x, kern, gout, states, tau, maxit, iso=False, nmaps=None):
    """`admm_tv_backward` (oracle) from the saved states with an array tau.  Returns (grad_x, grad_tau per element of
    the image (aniso) or per pixel (iso), fixed-tau grad_rho, grad_kern)."""
    x = np.asarray(x, np.float64)
    g = np.asarray(gout, np.float64)
    B, C, H, W = x.shape
    k2d = O._kernel_2d(kern)
    k2d64 = None if k2d is None else np.asarray(k2d, np.float64)
    sg, ph, L, den = O._spectral_tables(H, W, k2d64, RHO, np.float64)
    Bm = RHO / den
    Fy = O._rfft2(x, -1)
    A = sg * ph * Fy / den
    N = int(maxit)
    eps = 1e-15
    qs = [tuple(np.asarray(t, np.float64) for t in s) for s in states]
    nm = [None if nmaps is None else tuple(np.asarray(t, np.float64) for t in nmaps[k]) for k in range(len(qs))]
    vs = [None] * N
    for k in range(1, N):
        qx, qy = qs[k - 1]
        if iso:
            sx = np.maximum(1 - tau / (nm[k - 1][0] + eps), 0); sy = np.maximum(1 - tau / (nm[k - 1][1] + eps), 0)
            wx, wy = (2 * sx - 1) * qx, (2 * sy - 1) * qy
        else:
            wx, wy = 2 * _soft(qx, tau) - qx, 2 * _soft(qy, tau) - qy
        vs[k] = O._dxt(wx) + O._dyt(wy)
    cw = np.full((W // 2 + 1,), 2.0); cw[0] = 1.0
    if W % 2 == 0:
        cw[-1] = 1.0
    xb = g.copy()
    ub = [np.zeros_like(x), np.zeros_like(x)]
    wb = [np.zeros_like(x), np.zeros_like(x)]
    tbar = np.zeros((H, W) if iso else x.shape)
    Gsum = np.zeros_like(A); GVsum = np.zeros_like(A)
    for k in range(N - 1, -1, -1):
        if k < N - 1:
            qb = []
            for f in range(2):
                q = qs[k][f]
                ut = ub[f] - 2 * wb[f]
                if iso:
                    n = nm[k][f]
                    s = np.maximum(1 - tau / (n + eps), 0)
                    act = (s > 0).astype(np.float64)
                    sb = np.sum((2 * wb[f] - ub[f]) * q, (0, 1))
                    qb.append((2 * s - 1) * wb[f] + (1 - s) * ub[f] + act * sb * tau / (n + eps) ** 2 * q / n)
                    tbar += act * sb * (-1.0 / (n + eps))
                else:
                    m = (np.abs(q) < tau).astype(np.float64)
                    qb.append(wb[f] + m * ut)
                    tbar += ut * (1 - m) * np.sign(q)
            xb = xb + O._dxt(qb[0]) + O._dyt(qb[1])
            ub = qb
        Fxb = O._rfft2(xb, -1)
        G = Fxb / (H * W)
        Gsum += G
        if k > 0:
            GVsum += np.conj(G) * O._rfft2(vs[k], -1)
        vb = O._irfft2(Bm * Fxb, (H, W), -1)
        wb = [O._dx(vb), O._dy(vb)]
        xb = np.zeros_like(x)
    wgt = cw[None, None, None, :]
    gy = O._irfft2(np.conj(sg * ph / den) * Gsum * (H * W), (H, W), -1)
    rho_bar = float(np.sum(wgt * np.real(np.conj(Gsum) * (-A * L / den) + GVsum * (np.abs(sg) ** 2 / den ** 2))))
    return gy, tbar, rho_bar


# ------------------------------------------------------------------------------------------------ GPU runs
def train_tau(x, kern, gout, tau, planes, iso, maxit, ckpt=0, need_k=True):
    """The autograd Function with tau itself as the leaf: returns the output, (grad_x, grad_tau, fixed-tau grad_rho,
    grad_kern), the saved states and (iso) their norm maps."""
    from torch_admm_deconv_b200.eops.deconv import _AdmmTV
    dev = _dev()
    xt = torch.tensor(x, device=dev, requires_grad=True)
    tt = torch.tensor(tau, device=dev).contiguous().requires_grad_(True)
    rt = torch.tensor([RHO], dtype=torch.float32, device=dev, requires_grad=True)
    kt = torch.tensor(np.asarray(kern, np.float32), device=dev, requires_grad=need_k) if np.size(kern) \
        else torch.empty(0, device=dev)
    out = _AdmmTV.apply(xt, tt, rt, kt, None, bool(iso), maxit, True, 0, None, None, ckpt, None, planes)
    saved = out.grad_fn.saved_tensors[4]
    n, hw, S = x.size, x.shape[-2] * x.shape[-1], maxit - 1
    states, nmaps = [], None
    if ckpt < 2:
        flt = saved[: (S * 2 * n + (S * 2 * hw if iso else 0)) * 4].view(torch.float32).cpu().numpy()
        q = flt[: S * 2 * n].reshape(S, 2, *x.shape)
        states = [(q[i, 0], q[i, 1]) for i in range(S)]
        if iso:
            m = flt[S * 2 * n:].reshape(S, 2, *x.shape[-2:])
            nmaps = [(m[i, 0], m[i, 1]) for i in range(S)]
    (out * torch.tensor(gout, dtype=torch.float32, device=dev)).sum().backward()
    torch.cuda.synchronize()
    gk = kt.grad if np.size(kern) and need_k else None
    return out.detach(), (xt.grad, tt.grad, rt.grad, gk), states, nmaps


# a. constant map = scalar, on the same route --------------------------------------------------------------------------
def _scalar_vs_map(shape, k, maxit, iso, lam, kind, opts):
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    x, kern, gout = _inputs(shape, k, 5)
    B, C, H, W = shape
    g = torch.tensor(gout, dtype=torch.float32, device=dev)

    def run(lmbd):
        xt = torch.tensor(x, device=dev, requires_grad=True)
        rt = torch.tensor([RHO], device=dev, requires_grad=True)
        kt = torch.tensor(np.asarray(kern, np.float32), device=dev, requires_grad=bool(k))
        lt = lmbd.clone().requires_grad_(True)
        out = fft_admm_tv(xt, lt, rt, kt, iso, maxit)
        (out * g).sum().backward()
        torch.cuda.synchronize()
        return out.detach(), xt.grad, lt.grad, rt.grad, kt.grad

    s = _with_options(opts, lambda: run(torch.tensor([lam], device=dev)))
    mshape = (1, 1, H, W) if kind == "shared" else (B, C, H, W)
    m = _with_options(opts, lambda: run(torch.full(mshape, lam, device=dev)))
    assert torch.equal(s[0], m[0]), "output"
    assert torch.equal(s[1], m[1]), "x-gradient"
    # the λ gradient is a sum of signed terms that partly cancel, added in another order by the two solves (per element
    # over the sweep for the map, per CTA for the scalar): measured against the larger of the sum and the terms' L1 norm
    l1 = float(m[2].double().abs().sum())
    e_l = abs(float(m[2].double().sum()) - float(s[2])) / max(abs(float(s[2])), l1, 1e-12)
    # grad_rho = (spectral part) - taubar lam / rho^2: the parts can cancel, so it is measured against the larger of the
    # result and the tau part (as test_gpu_routes.py does)
    e_r = abs(float(m[3]) - float(s[3])) / max(abs(float(s[3])), l1 * abs(lam / RHO), 1e-12)
    e_k = float((m[4] - s[4]).abs().max() / s[4].abs().max()) if k else 0.0
    print("%s %s iso=%s lam=%g: lambda %.1e rho %.1e kern %.1e" % (shape, kind, iso, lam, e_l, e_r, e_k))
    assert e_l <= 1e-6 and e_r <= 1e-6 and e_k <= 1e-6


# the scalar solve runs on the map's route: generic rows (force_generic on power-of-two widths also moves the columns to
# the generic kernel, for both solves; use_big = 2 keeps the large-frame column kernel and drops the large-frame rows)
SAME_ROUTE = [((2, 3, 256, 256), 5, 6, {"force_generic": 1}), ((1, 2, 33, 45), 3, 5, {}),
              ((1, 2, 1080, 1920), 5, 3, {"use_big": 2}), ((2, 1, 128, 128), 0, 4, {"force_generic": 1})]


@pytest.mark.parametrize("lam", [0.02, -0.02])
@pytest.mark.parametrize("kind", ["shared", "full"])
@pytest.mark.parametrize("shape,k,maxit,opts", SAME_ROUTE, ids=lambda v: "x".join(map(str, v)) if isinstance(v, tuple) else None)
def test_constant_map_equals_scalar(shape, k, maxit, opts, kind, lam):
    _scalar_vs_map(shape, k, maxit, False, lam, kind, dict(opts, use_cluster=0))


@pytest.mark.parametrize("lam", [0.02, -0.02])
@pytest.mark.parametrize("shape,k,maxit", [((2, 2, 256, 256), 5, 5), ((1, 3, 45, 33), 3, 4), ((1, 2, 720, 1280), 3, 3)])
def test_constant_map_equals_scalar_iso(shape, k, maxit, lam):
    _scalar_vs_map(shape, k, maxit, True, lam, "shared", {})


# b. one iteration at a time against fp64 -------------------------------------------------------------------------------
def _rel(a, b):
    return abs(float(a) - float(b)) / max(abs(float(b)), 1e-12)


def gate_map(shape, k, maxit, iso, kind, seed=3):
    x, kern, gout = _inputs(shape, k, seed)
    lmap = make_map(shape, kind, seed + 7)
    lt = torch.tensor(lmap)
    from torch_admm_deconv_b200.eops.deconv import _tau_map
    tau_t, planes = _tau_map(lt, torch.tensor([RHO]), shape, iso, torch.device("cpu"))
    tau = tau_t.numpy().astype(np.float64)                               # float32 division, as the library sees it
    out, (gx, gt, gr, gk), states, nmaps = train_tau(x, kern, gout, tau_t.numpy(), planes, iso, maxit)
    tau_o = tau[0, 0] if iso else tau
    preds, x_out = replay_map(x, kern, states, tau_o, iso, nmaps)
    e = {"step": O.pair_err(states, preds, np.abs(x_out).max()), "out": O.rel_err(out.cpu().numpy(), x_out)}
    sx, stau, sr = adjoint_map(x, kern, gout, states, tau_o, maxit, iso, nmaps)
    e["gx"] = O.rel_err(gx.cpu().numpy().astype(np.float64), sx)
    if maxit > 1:
        ref_t = stau if (iso or planes > 1) else stau.sum(axis=(0, 1))
        e["gtau"] = O.rel_err(gt.cpu().numpy().reshape(ref_t.shape).astype(np.float64), ref_t)
    e["grho"] = _rel(gr.item(), sr)
    print("%s %s iso=%s N=%d: %s" % ("x".join(map(str, shape)), kind, iso, maxit, "  ".join("%s %.1e" % kv for kv in e.items())))
    assert e["step"] <= STEP_TOL and e["out"] <= STEP_TOL
    assert e["gx"] <= GRAD_TOL_X
    assert max(e.get("gtau", 0.0), e["grho"]) <= GRAD_TOL_P
    return e


ROUTES = [((1, 2, 128, 128), 5, 5), ((1, 2, 256, 256), 7, 5), ((1, 2, 512, 512), 5, 3), ((1, 2, 33, 45), 3, 5),
          ((2, 1, 31, 37), 5, 4), ((1, 2, 1080, 1920), 3, 3), ((1, 1, 2160, 3840), 5, 3), ((1, 1, 256, 256), 5, 6)]


@pytest.mark.parametrize("kind", ["shared", "full", "mixed", "zeros"])
@pytest.mark.parametrize("shape,k,maxit", ROUTES, ids=lambda v: "x".join(map(str, v)) if isinstance(v, tuple) else None)
def test_map_step_and_adjoint(shape, k, maxit, kind):
    if shape[-1] * shape[-2] > 2_000_000 and kind in ("mixed", "zeros"):
        pytest.skip("the large frames take the shared and full maps; the sign cases are covered on the smaller shapes")
    gate_map(shape, k, maxit, False, kind)


@pytest.mark.parametrize("kind", ["shared", "mixed"])
@pytest.mark.parametrize("shape,k,maxit", [((2, 2, 128, 128), 5, 4), ((1, 3, 33, 45), 3, 4), ((1, 2, 720, 1280), 3, 3)],
                         ids=lambda v: "x".join(map(str, v)) if isinstance(v, tuple) else None)
def test_map_step_and_adjoint_iso(shape, k, maxit, kind):
    gate_map(shape, k, maxit, True, kind)


# c. end to end against a float64 torch restatement ---------------------------------------------------------------------
def restatement(x, lmbd, rho, kern, iso, maxit, history=None):
    """deconv.py:103-115 in float64 torch with a tensor lmbd, differentiable by autograd w.r.t. x, lmbd and rho: the
    spectral form of the x-update (the PSF tables of oracle/admm_oracle.py, den = |sigma|^2 + rho L recomputed in torch)
    and the soft / block threshold with tau = lmbd / rho broadcast to the image."""
    B, C, H, W = x.shape
    tau = lmbd / rho
    k2d = O._kernel_2d(np.asarray(kern))
    sg, ph, L, _ = O._spectral_tables(H, W, None if k2d is None else np.asarray(k2d, np.float64), 1.0, np.float64)
    sg, ph, L = torch.as_tensor(sg), torch.as_tensor(ph), torch.as_tensor(L)
    den = sg.abs() ** 2 + rho * L
    A = sg * ph * torch.fft.rfft2(x) / den
    dx = lambda a: a - torch.roll(a, 1, 3)
    dy = lambda a: a - torch.roll(a, 1, 2)
    dxt = lambda a: a - torch.roll(a, -1, 3)
    dyt = lambda a: a - torch.roll(a, -1, 2)
    wx = torch.zeros_like(x); wy = torch.zeros_like(x); ux = torch.zeros_like(x); uy = torch.zeros_like(x)
    xk = torch.zeros_like(x)
    for _ in range(maxit):
        xk = torch.fft.irfft2(A + rho * torch.fft.rfft2(dxt(wx) + dyt(wy)) / den, s=(H, W))
        qx, qy = dx(xk) + ux, dy(xk) + uy
        if iso:
            nx = (qx.pow(2).sum((0, 1)) + 1e-15).sqrt(); ny = (qy.pow(2).sum((0, 1)) + 1e-15).sqrt()
            zx = (1 - tau / (nx + 1e-15)).clamp_min(0) * qx; zy = (1 - tau / (ny + 1e-15)).clamp_min(0) * qy
        else:
            zx = qx.sign() * (qx.abs() - tau).clamp_min(0); zy = qy.sign() * (qy.abs() - tau).clamp_min(0)
        ux, uy = qx - zx, qy - zy
        wx, wy = zx - ux, zy - uy
        if history is not None:                          # the pre-threshold state (iso: its pixel norms) of every iteration
            history.append((nx, ny) if iso else (qx, qy))
    return xk


def test_restatement_matches_the_oracle():
    x, kern, _ = _inputs((1, 2, 32, 40), 5, 9)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), 0.02, RHO, kern, False, 6)
    got = restatement(torch.tensor(x, dtype=torch.float64), torch.tensor([0.02], dtype=torch.float64),
                      torch.tensor(RHO, dtype=torch.float64), kern, False, 6)
    assert O.rel_err(got.numpy(), ref) < 1e-12


def _kink_margin(hist, tau):
    """Distance of the fp64 trajectory's pre-threshold values (iso: pixel norms) to the kinks of the threshold: |q| = tau
    element by element, and q = 0 where tau < 0."""
    m = float("inf")
    for fx, fy in hist:
        for f in (fx, fy):
            a_ = f.detach().abs()
            m = min(m, float((a_ - tau.abs()).abs().min()))
            if bool((tau < 0).any()):
                m = min(m, float(a_[(tau < 0).expand_as(a_)].min()))
    return m


def _kink_safe_case(shape, kind, iso, maxit, rho, seeds=range(64)):
    """First seed whose float64 trajectory keeps 1e-3 away from every kink (the seed selection of test_gpu_f64.py), so
    that an fp32 and an fp64 run take the same branch of every threshold and their gradients compare tightly.  The image
    is scaled by 10 and tau is O(1): about half of the values lie past the threshold."""
    psf = O.make_psf("gauss", 3, 0.8)
    kern = psf[None, None]
    for seed in seeds:
        x = 10.0 * O.make_blurred(shape, psf, seed=seed, noise=0.05).astype(np.float64)
        lmap = make_map(shape, kind, seed + 100, lam=0.2)
        hist = []
        restatement(torch.tensor(x), torch.tensor(lmap, dtype=torch.float64), torch.tensor(rho, dtype=torch.float64),
                    kern, iso, maxit, hist)
        tau = torch.tensor(lmap, dtype=torch.float64) / rho
        if iso:
            tau = tau.reshape(tau.shape[-2:])
        if _kink_margin(hist, tau) > 1e-3:
            return seed, x, lmap, kern
    raise AssertionError("no input among the seeds keeps the trajectory 1e-3 away from the threshold's kinks")


@pytest.mark.parametrize("iso,kind", [(False, "full"), (False, "mixed"), (False, "plane"), (True, "shared")])
def test_end_to_end_against_restatement(iso, kind):
    """Output and every gradient against the float64 restatement, on a kink-safe input: tight relative gates."""
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    shape, maxit, rho = (1, 2, 12, 10), 3, 0.4
    seed, x, lmap, kern = _kink_safe_case(shape, kind, iso, maxit, rho)
    gout = np.random.default_rng(seed + 1).standard_normal(shape)
    lt = torch.tensor(lmap, device=dev, requires_grad=True)
    xt = torch.tensor(x, dtype=torch.float32, device=dev, requires_grad=True)
    rt = torch.tensor([rho], device=dev, requires_grad=True)
    kt = torch.tensor(kern, device=dev)
    out = fft_admm_tv(xt, lt, rt, kt, iso, maxit)
    (out * torch.tensor(gout, dtype=torch.float32, device=dev)).sum().backward()
    l64 = torch.tensor(lmap, dtype=torch.float64, requires_grad=True)
    x64 = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    r64 = torch.tensor(rho, dtype=torch.float64, requires_grad=True)
    ref = restatement(x64, l64, r64, kern, iso, maxit)
    (ref * torch.tensor(gout)).sum().backward()
    e_out = O.rel_err(out.detach().cpu().numpy(), ref.detach().numpy())
    e_gx = O.rel_err(xt.grad.cpu().double().numpy(), x64.grad.numpy())
    e_gl = O.rel_err(lt.grad.cpu().double().numpy(), l64.grad.numpy())
    e_gr = _rel(rt.grad.item(), r64.grad.item())
    print("%s iso=%s seed %d: out %.1e  gx %.1e  glam %.1e  grho %.1e" % (kind, iso, seed, e_out, e_gx, e_gl, e_gr))
    assert lt.grad.shape == lt.shape and lt.grad.dtype == lt.dtype
    assert e_out < 1e-5 and e_gx < 1e-4 and e_gl < 1e-4 and e_gr < 1e-4


def test_gradcheck_small():
    """torch.autograd.gradcheck of the float64 restatement's λ-map path on a small case, then the library's float32 λ-map
    gradient against that checked gradient."""
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    shape = (1, 1, 16, 16)
    x, kern, gout = _inputs(shape, 3, 21)
    lmap = make_map(shape, "shared", 23, lam=0.002)          # tau ~ 0.05: both sides of the threshold occur
    l64 = torch.tensor(lmap, dtype=torch.float64, requires_grad=True)
    f = lambda l: restatement(torch.tensor(x, dtype=torch.float64), l, torch.tensor(RHO, dtype=torch.float64),
                              kern, False, 4)
    assert torch.autograd.gradcheck(f, (l64,), eps=1e-7, atol=1e-5)
    lt = torch.tensor(lmap, device=dev, requires_grad=True)
    g = torch.tensor(gout, dtype=torch.float32, device=dev)
    loss = lambda l: (fft_admm_tv(torch.tensor(x, device=dev), l, torch.tensor([RHO], device=dev),
                                  torch.tensor(kern, device=dev), False, 4) * g).sum()
    loss(lt).backward()
    ref = torch.autograd.grad((f(l64) * torch.tensor(gout)).sum(), l64)[0]
    assert float((lt.grad.cpu().double() - ref).norm() / ref.norm()) < 1e-3


def test_reference_accepts_a_map():
    """The reference's own fft_admm_tv broadcasts a λ map (deconv.py:15-24, 44): same output as this library."""
    import os
    import sys
    refdir = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "baseline", "_ref")
    if not os.path.exists(os.path.join(refdir, "admmtor", "eops", "deconv.py")):
        pytest.skip("baseline/_ref is not installed (python baseline/install_ref.py in the build container)")
    if refdir not in sys.path:
        sys.path.insert(0, refdir)
    import admmtor.eops.deconv as ref
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    shape = (1, 2, 32, 32)
    x, kern, _ = _inputs(shape, 5, 31)
    lmap = make_map(shape, "shared", 33)
    r = ref.fft_admm_tv(torch.tensor(x), torch.tensor(lmap), torch.tensor([RHO]), torch.tensor(kern), False, 10)
    o = fft_admm_tv(torch.tensor(x, device=dev), torch.tensor(lmap, device=dev), torch.tensor([RHO], device=dev),
                    torch.tensor(kern, device=dev), False, 10)
    assert O.rel_err(o.cpu().numpy(), r.numpy()) < 1e-4


# c2. inference routes: without saved state a solve may take the cluster solver, the cooperative kernel, plane chunks or
# the two-stream split.  A map solve takes none of them: its no-grad output equals its training output bit for bit, and
# matches the float64 restatement
@pytest.mark.parametrize("shape,opts", [((1, 1, 256, 256), {}),                       # cluster-preferred (cfg1's shape)
                                        ((2, 3, 128, 128), {"use_coop": 2}),        # the cooperative kernel if it applied
                                        ((2, 3, 128, 128), {"chunk_mb": 1}),        # plane chunks if they applied
                                        ((4, 3, 1024, 1024), {})],                  # two-stream split size (>= 8 M elements)
                         ids=["cluster", "coop", "chunks", "split"])
@pytest.mark.parametrize("kind", ["shared", "full"])
def test_inference_map_solve(shape, opts, kind):
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    maxit = 4
    x, kern, _ = _inputs(shape, 5, 61)
    lmap = make_map(shape, kind, 63)
    args = lambda rg: (torch.tensor(x, device=dev), torch.tensor(lmap, device=dev, requires_grad=rg),
                       torch.tensor([RHO], device=dev), torch.tensor(kern, device=dev), False, maxit)

    def run():
        with torch.no_grad():
            a = fft_admm_tv(*args(False))
        b = fft_admm_tv(*args(True))
        torch.cuda.synchronize()
        return a, b.detach()
    a, b = _with_options(opts, run)
    assert torch.equal(a, b)
    n = 1                                                # the fp64 restatement on the first image
    ref = restatement(torch.tensor(x[:n], dtype=torch.float64), torch.tensor(lmap[:n] if kind == "full" else lmap,
                      dtype=torch.float64), torch.tensor(RHO, dtype=torch.float64), kern, False, maxit)
    e = O.rel_err(a[:n].cpu().numpy(), ref.numpy())
    print("%s %s %s: no-grad = training, vs fp64 %.1e" % (shape, opts, kind, e))
    assert e < 1e-4


# d. training ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,k,maxit", [((2, 2, 256, 256), 5, 10), ((1, 1, 1080, 1920), 3, 7), ((1, 2, 33, 45), 3, 10)],
                         ids=lambda v: "x".join(map(str, v)) if isinstance(v, tuple) else None)
@pytest.mark.parametrize("kind", ["shared", "full"])
def test_checkpointed_training_is_bit_identical(shape, k, maxit, kind):
    x, kern, gout = _inputs(shape, k, 41)
    from torch_admm_deconv_b200.eops.deconv import _tau_map
    tau, planes = _tau_map(torch.tensor(make_map(shape, kind, 43)), torch.tensor([RHO]), shape, False, torch.device("cpu"))
    a = train_tau(x, kern, gout, tau.numpy(), planes, False, maxit, ckpt=0)
    b = train_tau(x, kern, gout, tau.numpy(), planes, False, maxit, ckpt=3)
    c = train_tau(x, kern, gout, tau.numpy(), planes, False, maxit, ckpt=0)
    d = lambda u, v: float((u - v).abs().max())
    print("%s %s: output %g | checkpointed vs full %s | run to run %s" % (shape, kind, d(a[0], b[0]),
          " ".join("%g" % d(u, v) for u, v in zip(a[1], b[1])), " ".join("%g" % d(u, v) for u, v in zip(a[1], c[1]))))
    assert torch.equal(a[0], b[0])
    for ga, gb, gc in zip(a[1], b[1], c[1]):
        assert torch.equal(ga, gc)                       # run to run
        assert torch.equal(ga, gb)                       # checkpointed = full state


def test_admmdeconv_with_a_map_parameter():
    """cfg4's layer (32 x 3 x 256 x 256, no PSF, 10 iterations) with its λ replaced by a (1, 1, 256, 256) map Parameter:
    the call goes through admm_solve, and the map's gradient matches the float64 restatement."""
    from torch_admm_deconv_b200 import ADMMDeconv
    dev = _dev()
    shape, maxit = (32, 3, 256, 256), 10
    x, _, gout = _inputs(shape, 0, 51)
    layer = ADMMDeconv(None, maxit, lmbda=None, rho=RHO, iso=False).to(dev)
    lmap = make_map(shape, "shared", 53)
    layer.lmbda = torch.nn.Parameter(torch.tensor(lmap, device=dev))
    out = layer(torch.tensor(x, device=dev))
    (out * torch.tensor(gout, dtype=torch.float32, device=dev)).sum().backward()
    assert layer.lmbda.grad is not None and layer.lmbda.grad.shape == (1, 1, 256, 256)
    xs = torch.tensor(x[:4], dtype=torch.float64)
    l64 = torch.tensor(lmap, dtype=torch.float64, requires_grad=True)
    ref = restatement(xs, l64, torch.tensor(RHO, dtype=torch.float64), np.zeros((0,)), False, maxit)
    (ref * torch.tensor(gout[:4])).sum().backward()
    # the layer ran the whole batch: redo the first four images on the GPU for a like-for-like gradient
    layer.lmbda.grad = None
    out4 = layer(torch.tensor(x[:4], device=dev))
    (out4 * torch.tensor(gout[:4], dtype=torch.float32, device=dev)).sum().backward()
    e = float((layer.lmbda.grad.cpu().double() - l64.grad).norm() / l64.grad.norm())
    print("ADMMDeconv map gradient vs restatement: %.1e" % e)
    assert e < 5e-3


# e. errors before anything runs ---------------------------------------------------------------------------------------
def test_errors():
    from torch_admm_deconv_b200 import fft_admm_tv
    from torch_admm_deconv_b200.eops.deconv import admm_solve, admm_solve_tol
    dev = _dev()
    x = torch.rand(2, 3, 32, 32, device=dev)
    k = torch.empty(0, device=dev)
    rho = torch.tensor([RHO], device=dev)
    with pytest.raises(ValueError, match="broadcast"):
        fft_admm_tv(x, torch.rand(2, 3, 16, 32, device=dev), rho, k)
    with pytest.raises(ValueError, match="rho map"):
        fft_admm_tv(x, torch.rand(1, 1, 32, 32, device=dev), torch.rand(1, 1, 32, 32, device=dev), k)
    with pytest.raises(ValueError, match="iso=True"):
        fft_admm_tv(x, torch.rand(2, 3, 1, 1, device=dev), rho, k, iso=True)
    with pytest.raises(ValueError, match="scalar lmbd"):
        admm_solve_tol(x, torch.rand(1, 1, 32, 32, device=dev), rho, k, maxit=5)
    with pytest.raises(ValueError, match="one element"):
        admm_solve(x, torch.rand(1, 1, 32, 32, device=dev), torch.rand(2, device=dev), k)
