"""Checkpointed training (admm_ext.ckpt_interval = K) on the generic row kernel, odd frame heights above all.

The generic row kernel FFTs two real rows as one complex row and recomputes one halo row above and below each band.  On
an odd height the last band has an odd row count and its bottom halo wraps to row 0: the forward's v of row H-1 must be
the v that the backward rebuilds from the stored q (k_bwd_recompute_v), or every block re-run from a checkpoint starts
from a field the forward never used.  The ρ and kernel gradients, built from the regenerated v, then move in the last
bits, and on large frames the drift reaches a threshold decision and moves the λ gradient as well.

Every case checks four things: the saved buffer has the checkpointed size (no silent fall-back to full state), the
output and every requested gradient equal those of the full-state run bit for bit, and a second checkpointed run equals
the first bit for bit."""
import math

import numpy as np
import pytest
import torch

from oracle import admm_oracle as O

pytestmark = pytest.mark.gpu

RHO = 0.04
ALL = ("x", "lambda", "rho", "kernel")


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
    gout = np.random.default_rng(seed + 1).standard_normal(shape).astype(np.float32)
    return x, kern, gout


def _map(shape, kind, seed, lam=0.02):
    """λ map: "shared" (1, 1, H, W) positive, "full" (B, C, H, W) positive, "mixed" (1, 1, H, W) of both signs."""
    B, C, H, W = shape
    r = np.random.default_rng(seed)
    s = (B, C, H, W) if kind == "full" else (1, 1, H, W)
    m = lam * r.uniform(0.3, 1.7, s)
    if kind == "mixed":
        m *= np.where(r.random(s) < 0.4, -1.0, 1.0)
    return m.astype(np.float32)


def _train(x, kern, lmbd, gout, maxit, K, need):
    """One training step through admm_solve with gradients requested for the inputs named in `need`: the output, those
    gradients and the size of the saved state."""
    from torch_admm_deconv_b200.eops.deconv import admm_solve
    dev = _dev()
    xt = torch.tensor(x, device=dev, requires_grad="x" in need)
    lt = torch.tensor(lmbd, device=dev, requires_grad="lambda" in need)
    rt = torch.tensor([RHO], device=dev, requires_grad="rho" in need)
    kt = torch.tensor(kern, device=dev, requires_grad="kernel" in need and np.size(kern) > 0)
    out = admm_solve(xt, lt, rt, kt, False, maxit, ckpt_interval=K)
    nbytes = out.grad_fn.saved_tensors[4].numel()
    (out * torch.tensor(gout, device=dev)).sum().backward()
    torch.cuda.synchronize()
    grads = {n: t.grad for n, t in zip(ALL, (xt, lt, rt, kt)) if n in need and t.requires_grad}
    assert all(g is not None for g in grads.values())
    return out.detach(), grads, nbytes


def _diff(a, b):
    d = float((a - b).abs().max())
    return "max abs %.3e, rel %.3e" % (d, d / max(float(a.abs().max()), 1e-30))


def check_ckpt(shape, k, maxit, K, lam=0.02, need=ALL, lmap=None, opts=None, seed=29):
    """Full-state vs checkpointed training of one case (the four assertions of the module docstring)."""
    from torch_admm_deconv_b200 import _lib
    x, kern, gout = _inputs(shape, k, seed)
    lmbd = lmap if lmap is not None else np.array([lam], np.float32)
    run = lambda ck: _with_options(dict(opts or {}), lambda: _train(x, kern, lmbd, gout, maxit, ck, need))
    full, ck, again = run(0), run(K), run(K)
    B, C, H, W = shape
    Keff = K if K > 0 else int(math.ceil(math.sqrt(maxit - 1)))
    field = B * C * H * W * 4
    assert full[2] == (maxit - 1) * 2 * field + 256
    assert ck[2] == _lib.load().admm_query_saved_ex(B * C, H, W, k, 0, maxit, Keff)
    assert ck[2] == ((maxit - 1) // Keff) * 2 * field + 256
    assert torch.equal(full[0], ck[0]), "output: " + _diff(full[0], ck[0])
    assert sorted(full[1]) == sorted(ck[1]) == sorted(n for n in need if n != "kernel" or k)
    for n in full[1]:
        assert torch.equal(full[1][n], ck[1][n]), "%s gradient, checkpointed vs full: %s" % (n, _diff(full[1][n], ck[1][n]))
    assert torch.equal(ck[0], again[0])
    for n in ck[1]:
        assert torch.equal(ck[1][n], again[1][n]), "%s gradient, run to run" % n


def _ids(v):
    return "x".join(map(str, v)) if isinstance(v, tuple) else None


# odd heights run the generic row kernel whatever the width (the power-of-two and large-frame row kernels take even H)
ODD = [((1, 2, 33, 45), 5, 10),          # last band is one row
       ((2, 3, 31, 37), 5, 10),          # prime in both axes
       ((1, 2, 3, 64), 3, 6),            # one band holds the whole frame
       ((1, 2, 45, 256), 5, 10),         # power-of-two width, odd height: generic rows
       ((1, 1, 9, 4151), 3, 8),          # two-row bands (the width leaves room for no more)
       ((1, 1, 9, 5811), 3, 8),          # two-row bands at batch stride 2
       ((1, 2, 1079, 1920), 5, 7),
       ((1, 1, 2161, 3840), 5, 5),       # prime height, few iterations
       ((70, 1, 33, 45), 3, 8)]          # more planes than the 64 plane groups


@pytest.mark.parametrize("lam", [0.02, -0.02])
@pytest.mark.parametrize("K", [3, -1])
@pytest.mark.parametrize("shape,k,maxit", ODD, ids=_ids)
def test_odd_height(shape, k, maxit, K, lam):
    check_ckpt(shape, k, maxit, K, lam)


# even heights: the generic rows, the power-of-two rows and the large-frame rows, each with generic columns, and the
# power-of-two kernels
EVEN = [((1, 2, 48, 40), 5, 10), ((2, 2, 130, 256), 5, 9), ((1, 2, 1078, 1920), 5, 7), ((2, 2, 128, 512), 5, 9)]


@pytest.mark.parametrize("K", [3, -1])
@pytest.mark.parametrize("shape,k,maxit", EVEN, ids=_ids)
def test_even_height_control(shape, k, maxit, K):
    check_ckpt(shape, k, maxit, K)


# maxit = 10 keeps 9 slots: K = 8 re-runs a one-slot block from a checkpoint, K = 9 keeps only the last slot, K >= 10
# keeps none (one block from the start)
@pytest.mark.parametrize("maxit,K", [(10, 2), (10, 3), (10, 4), (10, 8), (10, 9), (10, 10), (10, 20), (2, 2), (3, 2)])
def test_interval_sweep(maxit, K):
    check_ckpt((1, 2, 33, 45), 5, maxit, K)


# the band height moves the odd band: on 45 rows the last band has 1, 1, 3, 13 or 45 rows
@pytest.mark.parametrize("rows", [2, 4, 6, 16, 64])
@pytest.mark.parametrize("shape", [(1, 2, 33, 45), (1, 2, 45, 63)], ids=_ids)
def test_rows_per_band(shape, rows):
    check_ckpt(shape, 5, 10, 3, opts={"rows_per_band": rows})


# without the ρ and kernel gradients the backward needs no spectrum of v and re-runs blocks in another order
@pytest.mark.parametrize("need", [("x",), ("lambda",), ("rho",), ("kernel",)], ids=lambda v: v[0])
@pytest.mark.parametrize("shape", [(1, 2, 33, 45), (1, 2, 45, 256)], ids=_ids)
def test_partial_gradients(shape, need):
    check_ckpt(shape, 5, 10, 3, need=need)


# λ maps run the generic row kernel's map mode; on 45 x 256 the restart takes the generic R2C at a power-of-two width
@pytest.mark.parametrize("kind", ["shared", "full", "mixed"])
@pytest.mark.parametrize("shape", [(1, 2, 33, 45), (2, 3, 31, 37), (1, 2, 45, 256)], ids=_ids)
def test_lambda_map(shape, kind):
    check_ckpt(shape, 5, 10, 3, lmap=_map(shape, kind, 31))


def test_admmdeconv_layer():
    """ADMMDeconv with learnable PSF, λ and ρ, ckpt_interval = -1 (K = ceil(sqrt(max_iters - 1)))."""
    from torch_admm_deconv_b200 import ADMMDeconv, _lib
    dev = _dev()
    shape, maxit = (2, 3, 33, 45), 10
    x, _, gout = _inputs(shape, 0, 37)
    torch.manual_seed(3)
    m = ADMMDeconv((5, 5), maxit, iso=False).to(dev)
    with torch.no_grad():
        m.lmbda.fill_(0.02)
        m.rho.fill_(RHO)

    def run(ck):
        m.zero_grad(set_to_none=True)
        m.ckpt_interval = ck
        xt = torch.tensor(x, device=dev, requires_grad=True)
        y = m(xt)
        nbytes = y.grad_fn.saved_tensors[4].numel()
        (y * torch.tensor(gout, device=dev)).sum().backward()
        torch.cuda.synchronize()
        return [y.detach(), xt.grad, m.w.grad.clone(), m.lmbda.grad.clone(), m.rho.grad.clone()], nbytes

    full, ck, again = run(0), run(-1), run(-1)
    field = int(np.prod(shape)) * 4
    assert full[1] == (maxit - 1) * 2 * field + 256
    assert ck[1] == _lib.load().admm_query_saved_ex(6, 33, 45, 5, 0, maxit, 3) == 3 * 2 * field + 256
    for name, a, b, c in zip(("output", "x", "kernel", "lambda", "rho"), full[0], ck[0], again[0]):
        assert torch.equal(a, b), "%s, checkpointed vs full: %s" % (name, _diff(a, b))
        assert torch.equal(b, c), "%s, run to run" % name
