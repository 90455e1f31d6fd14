"""Checkpointed training (admm_ext.ckpt_interval = K) on the large frames.

The backward re-runs each block of K iterations from its checkpoint with the forward's own kernels and layouts: with both
large-frame kernels the spectra between them are tile-major, and the large-frame row kernel restarts from a checkpoint
by forming v inside its R2C with the march's operation order.  The gradients must equal those of the run that keeps
every iteration bit for bit, and the saved buffer must have the checkpointed size (no fall-back to full state).

The host-side size queries run without a GPU; the solves are marked gpu."""
import numpy as np
import pytest
import torch

from oracle import admm_oracle as O

BIG_FRAMES = [(1080, 1920), (2160, 3840), (1024, 1024), (720, 1280), (1440, 2560), (2048, 2048)]


@pytest.mark.parametrize("H,W", BIG_FRAMES)
@pytest.mark.parametrize("planes,k,maxit,K", [(3, 63, 200, 10), (24, 15, 100, 10), (2, 0, 11, 3), (1, 5, 6, 8)])
def test_query_saved_ex_keeps_every_kth_iteration(lib, H, W, planes, k, maxit, K):
    n = lib.admm_query_saved_ex(planes, H, W, k, 0, maxit, K)
    assert n == ((maxit - 1) // K) * 2 * planes * H * W * 4 + 256
    assert lib.admm_query_saved_ex(planes, H, W, k, 0, maxit, 0) == (maxit - 1) * 2 * planes * H * W * 4 + 256


@pytest.mark.parametrize("H,W", BIG_FRAMES)
def test_query_workspace_backward_ex_accepts_k(lib, H, W):
    full = lib.admm_query_workspace_backward_ex(2, H, W, 5, 0, 20, 0)
    ck = lib.admm_query_workspace_backward_ex(2, H, W, 5, 0, 20, 4)
    # + K-1 regenerated slots, the block's A, S0, S1 and one real field
    assert full > 0 and ck > full + 3 * 2 * 2 * H * W * 4


@pytest.mark.parametrize("H,W", BIG_FRAMES[:3])
def test_iso_checkpointing_stays_unavailable(lib, H, W):
    assert lib.admm_query_saved_ex(3, H, W, 5, 1, 20, 4) == 0
    assert lib.admm_query_workspace_backward_ex(3, H, W, 5, 1, 20, 4) == 0


# ------------------------------------------------------------------------------------------------------------ GPU
def _dev():
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    return torch.device("cuda:0")


def _with_option(key, value, fn):
    from torch_admm_deconv_b200 import _lib
    old = _lib.get_option(key)
    _lib.set_option(key, value)
    try:
        return fn()
    finally:
        _lib.set_option(key, old)


def _compare(shape, k, maxit, K, lam=0.02):
    from torch_admm_deconv_b200.eops.deconv import admm_solve
    dev = _dev()
    rng = np.random.default_rng(sum(shape) + k + K)
    psf = O.make_psf("gauss", k, 1.5) if k else None
    x = O.make_blurred(shape, psf, seed=17, noise=0.02)
    gout = torch.tensor(rng.standard_normal(shape).astype(np.float32), device=dev)
    res = []
    for ck in (0, K):
        xt = torch.tensor(x, device=dev, requires_grad=True)
        lt = torch.tensor([lam], device=dev, requires_grad=True)
        rt = torch.tensor([0.04], device=dev, requires_grad=True)
        kt = torch.tensor(psf[None, None], device=dev, requires_grad=True) if k else torch.empty(0, device=dev)
        out = admm_solve(xt, lt, rt, kt, False, maxit, ckpt_interval=ck)
        nbytes = out.grad_fn.saved_tensors[4].numel()
        (out * gout).sum().backward()
        res.append((out.detach(), xt.grad, lt.grad, rt.grad, kt.grad if k else None, nbytes))
        del out, xt
    full, ck = res
    Keff = K if K > 0 else int(np.ceil(np.sqrt(maxit - 1)))
    field = int(np.prod(shape)) * 4
    assert full[5] == (maxit - 1) * 2 * field + 256
    assert ck[5] == ((maxit - 1) // Keff) * 2 * field + 256            # checkpointed: no silent fall-back to full state
    assert torch.equal(full[0], ck[0])
    for name, a, b in zip(("x", "lambda", "rho", "kernel"), full[1:5], ck[1:5]):
        if a is not None:
            assert torch.equal(a, b), (name, float((a - b).abs().max() / a.abs().max().clamp_min(1e-30)))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,k,maxit,K,lam", [
    ((1, 3, 2160, 3840), 63, 11, 3, 0.02),          # BASELINE cfg3 frame
    ((2, 3, 1080, 1920), 5, 13, -1, 0.02),
    ((1, 2, 1024, 1024), 0, 10, 3, -0.02),          # negative tau
    ((1, 1, 720, 1280), 7, 6, 8, 0.02),             # K larger than the slot count: nothing kept, one block
    ((2, 2, 1440, 2560), 3, 9, 2, 0.02),
    ((2, 2, 256, 1024), 5, 10, 3, 0.02),            # large-frame row kernel only (row-major spectra)
    ((1, 1, 64, 3840), 3, 9, 2, 0.02),
    ((1, 2, 1080, 96), 5, 9, 3, 0.02),              # large-frame column kernel only
])
def test_checkpointed_gradients_match_full_state_on_large_frames(shape, k, maxit, K, lam):
    _compare(shape, k, maxit, K, lam)


@pytest.mark.gpu
@pytest.mark.parametrize("use_big", [1, 2])
def test_checkpointed_gradients_with_one_large_kernel(use_big):
    """use_big = 1: only the large row kernel (row-major spectra); 2: only the large column kernel."""
    _with_option("use_big", use_big, lambda: _compare((1, 2, 1080, 1920), 5, 10, 3))


@pytest.mark.gpu
def test_module_checkpointed_training_on_1080p():
    from torch_admm_deconv_b200 import ADMMDeconv
    dev = _dev()
    torch.manual_seed(5)
    m = ADMMDeconv((5, 5), 12, iso=False).to(dev)
    x = torch.rand(1, 3, 1080, 1920, device=dev)
    gout = torch.randn(1, 3, 1080, 1920, device=dev)
    res = []
    for ck in (0, 4):
        m.zero_grad(set_to_none=True)
        m.ckpt_interval = ck
        y = m(x)
        nbytes = y.grad_fn.saved_tensors[4].numel()
        (y * gout).sum().backward()
        res.append((y.detach(), m.w.grad.clone(), m.lmbda.grad.clone(), m.rho.grad.clone(), nbytes))
    full, ck = res
    field = 3 * 1080 * 1920 * 4
    assert full[4] == 11 * 2 * field + 256 and ck[4] == (11 // 4) * 2 * field + 256
    for a, b in zip(full[:4], ck[:4]):
        assert torch.equal(a, b)
