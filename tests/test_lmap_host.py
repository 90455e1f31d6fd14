"""λ maps (DESIGN.md section 11), host side: argument checks of the Python layer and of the C ABI, which refuse a bad
request before anything is launched (no GPU needed)."""
import ctypes

import pytest
import torch

from torch_admm_deconv_b200 import _lib
from torch_admm_deconv_b200.eops.deconv import _tau_map

CPU = torch.device("cpu")


@pytest.mark.parametrize("lshape,planes,tshape", [((1, 1, 8, 12), 1, (1, 1, 8, 12)), ((8, 12), 1, (1, 1, 8, 12)),
                                                  ((12,), 1, (1, 1, 8, 12)), ((2, 3, 8, 12), 6, (2, 3, 8, 12)),
                                                  ((2, 3, 1, 1), 6, (2, 3, 8, 12)), ((3, 1, 1), 6, (2, 3, 8, 12)),
                                                  ((1, 1, 8, 1), 1, (1, 1, 8, 12))])
def test_tau_map_layout(lshape, planes, tshape):
    lmbd = torch.rand(lshape, dtype=torch.float64)
    tau, p = _tau_map(lmbd, torch.tensor([0.04]), (2, 3, 8, 12), False, CPU)
    assert p == planes and tuple(tau.shape) == tshape and tau.is_contiguous() and tau.dtype == torch.float32
    # divided in float32, element by element, like lmbd / rho in the reference (deconv.py:44)
    want = (lmbd.to(torch.float32) / torch.tensor(0.04, dtype=torch.float32)).expand(tshape)
    assert torch.equal(tau, want)


def test_tau_map_gradient_reaches_lmbd_and_rho():
    lmbd = torch.rand(1, 1, 8, 12, dtype=torch.float64, requires_grad=True)
    rho = torch.tensor([0.04], requires_grad=True)
    tau, _ = _tau_map(lmbd, rho, (2, 3, 8, 12), False, CPU)
    tau.sum().backward()
    assert lmbd.grad.dtype == torch.float64 and lmbd.grad.shape == lmbd.shape
    assert rho.grad is not None


@pytest.mark.parametrize("lshape", [(2, 3, 4, 12), (3, 3, 8, 12), (1, 1, 1, 8, 12), (8, 13)])
def test_tau_map_rejects_shapes_that_do_not_broadcast(lshape):
    with pytest.raises(ValueError, match="broadcast"):
        _tau_map(torch.rand(lshape), 0.04, (2, 3, 8, 12), False, CPU)


def test_tau_map_rejects_rho_maps_per_plane_iso_and_integer_maps():
    with pytest.raises(ValueError, match="rho map"):
        _tau_map(torch.rand(1, 1, 8, 12), torch.rand(1, 1, 8, 12), (2, 3, 8, 12), False, CPU)
    with pytest.raises(ValueError, match="iso=True"):
        _tau_map(torch.rand(2, 3, 1, 1), 0.04, (2, 3, 8, 12), True, CPU)
    with pytest.raises(ValueError, match="iso=True"):
        _tau_map(torch.rand(1, 3, 8, 12), 0.04, (2, 3, 8, 12), True, CPU)
    _tau_map(torch.rand(8, 12), 0.04, (2, 3, 8, 12), True, CPU)          # shared map: fine with iso
    with pytest.raises(ValueError, match="floating"):
        _tau_map(torch.ones(8, 12, dtype=torch.int32), 0.04, (2, 3, 8, 12), False, CPU)


def test_admm_solve_tol_refuses_a_map():
    from torch_admm_deconv_b200.eops.deconv import admm_solve_tol
    with pytest.raises(ValueError, match="scalar lmbd"):
        admm_solve_tol(torch.zeros(1, 1, 8, 8), torch.rand(1, 1, 8, 8), 0.04, None, maxit=5)


def test_f64_solve_refuses_a_map():
    from torch_admm_deconv_b200 import fft_admm_tv_f64
    with pytest.raises((ValueError, TypeError)):
        fft_admm_tv_f64(torch.zeros(1, 1, 8, 8, dtype=torch.float64), torch.rand(1, 1, 8, 8), 0.04, None)


# ---- C ABI: every bad map request returns ADMM_ERR_INVALID before any launch.  The pointers are never dereferenced: the
# checks run first, so placeholder addresses suffice on a machine without a GPU.
FAKE = 1 << 20


def _forward(lib, B=1, C=2, H=16, W=16, iso=0, tau_map=FAKE, planes=1, resid_every=0, rtol=0.0):
    ext = _lib.AdmmExt()
    ext.struct_size = ctypes.sizeof(_lib.AdmmExt)
    ext.tau_map = tau_map
    ext.tau_map_planes = planes
    ext.resid_every = resid_every
    ext.resid = FAKE if resid_every else None
    ext.rtol = rtol
    ext.host_flag = FAKE if rtol else None
    p = ctypes.c_void_p(FAKE)
    return lib.admm_tv_forward_ex(p, p, None, 0, None, p, None, B, C, H, W, iso, 5, p, 1 << 30, None, 0, None,
                                  ctypes.byref(ext))


@pytest.mark.parametrize("planes", [0, -1, 3, 4])
def test_abi_rejects_bad_tau_map_planes(lib, planes):
    assert _forward(lib, planes=planes) == 1
    assert b"tau_map_planes" in lib.admm_last_error()


def test_abi_rejects_misaligned_maps_per_plane_iso_and_residuals(lib):
    assert _forward(lib, tau_map=FAKE + 4) == 1
    assert b"aligned" in lib.admm_last_error()
    assert _forward(lib, iso=1, planes=2) == 1
    assert b"iso" in lib.admm_last_error()
    assert _forward(lib, resid_every=2) == 1
    assert b"residuals" in lib.admm_last_error()


def test_abi_backward_rejects_bad_maps(lib):
    p = ctypes.c_void_p(FAKE)

    def bwd(tau_map, planes, iso=0):
        return lib.admm_tv_backward_map(p, p, None, 0, tau_map, planes, p, 1, 2, 16, 16, iso, 5, p, 1 << 30, p, 1 << 30,
                                        None, None, None, None, None, 0)
    assert bwd(ctypes.c_void_p(FAKE), 3) == 1 and b"tau_map_planes" in lib.admm_last_error()
    assert bwd(None, 1) == 1 and b"NULL" in lib.admm_last_error()
    assert bwd(ctypes.c_void_p(FAKE), 2, iso=1) == 1 and b"iso" in lib.admm_last_error()


def test_abi_backward_workspace_query(lib):
    q = lib.admm_query_workspace_backward_map
    base = lib.admm_query_workspace_backward_ex(6, 16, 20, 5, 0, 6, 0)
    # the per-element tau-gradient accumulator (doubles) comes on top of the scalar backward's workspace
    assert q(6, 16, 20, 5, 0, 6, 0, 1) >= base + 6 * 16 * 20 * 8
    assert q(6, 16, 20, 5, 0, 6, 0, 6) == q(6, 16, 20, 5, 0, 6, 0, 1)
    assert q(6, 16, 20, 5, 1, 6, 0, 1) >= lib.admm_query_workspace_backward_ex(6, 16, 20, 5, 1, 6, 0) + 16 * 20 * 8
    assert q(6, 16, 20, 5, 0, 6, 0, 2) == 0          # neither 1 nor B*C
    assert q(6, 16, 20, 5, 1, 6, 0, 6) == 0          # iso takes a shared map only
    assert q(6, 16, 20, 5, 1, 6, 3, 1) == 0          # no checkpointing with iso
