"""CPU tests of the float64 solve's host side (admm_*_f64 of include/admm_b200.h): sizes of the saved state and the
workspaces, and invalid input.  No kernels are launched here."""
import pytest
import torch


@pytest.mark.parametrize("iso", [0, 1])
@pytest.mark.parametrize("planes,H,W,k,maxit", [(6, 16, 20, 5, 6), (3, 31, 37, 3, 8), (2, 512, 512, 31, 100),
                                                (1, 16, 16, 3, 1), (4, 33, 45, 0, 2)])
def test_saved_state_is_the_float32_layout_in_double(lib, planes, H, W, k, maxit, iso):
    # both queries add one 256-byte pad to the state itself
    n32 = lib.admm_query_saved(planes, H, W, k, iso, maxit)
    n64 = lib.admm_query_saved_f64(planes, H, W, k, iso, maxit)
    assert n32 > 0 and n64 > 0
    assert n64 - 256 == 2 * (n32 - 256)


@pytest.mark.parametrize("iso", [0, 1])
def test_workspaces_hold_the_double_fields(lib, iso):
    planes, H, W = 6, 64, 48
    fwd = lib.admm_query_workspace_f64(planes, H, W, 5, iso, 10)
    bwd = lib.admm_query_workspace_backward_f64(planes, H, W, 5, iso, 10)
    fields = 4 + (2 if iso else 0)                      # q ping-pong (+ x, v real fields for iso)
    spectra = 3                                         # S0, S1, A
    assert fwd >= planes * H * W * 8 * fields + planes * H * ((W + 1) // 2) * 16 * spectra
    assert bwd > fwd + planes * H * W * 8 * 2           # + vbar, xbar and the backward spectra


@pytest.mark.parametrize("query", ["admm_query_workspace_f64", "admm_query_workspace_backward_f64", "admm_query_saved_f64"])
def test_queries_return_zero_for_invalid_input(lib, query):
    q = getattr(lib, query)
    assert q(6, 16, 20, 5, 0, 6) > 0
    assert q(0, 16, 16, 3, 0, 5) == 0                  # planes < 1
    assert q(1, 1, 16, 0, 0, 5) == 0                   # H < 2
    assert q(1, 16, 1, 0, 1, 5) == 0                   # W < 2
    assert q(1, 16, 16, 17, 0, 10) == 0                # PSF larger than the image
    assert b"PSF" in lib.admm_last_error()
    assert q(1, 16, 16, -1, 0, 10) == 0                # negative PSF size


def test_version_and_float32_entry_points_unchanged(lib):
    assert lib.admm_version() == 300
    from torch_admm_deconv_b200 import fft_admm_tv, fft_admm_tv_f64, eops
    assert eops.fft_admm_tv_f64 is fft_admm_tv_f64
    lam, rho = torch.tensor([0.02]), torch.tensor([0.04])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        fft_admm_tv(torch.zeros(1, 1, 8, 8), lam, rho, torch.tensor([]))


def test_f64_input_validation_without_a_gpu():
    from torch_admm_deconv_b200 import fft_admm_tv_f64
    lam, rho = torch.tensor([0.02]), torch.tensor([0.04])
    with pytest.raises(TypeError, match="float64"):
        fft_admm_tv_f64(torch.zeros(1, 1, 8, 8), lam, rho, torch.tensor([]))            # float32
    with pytest.raises(TypeError, match="CPU"):
        fft_admm_tv_f64(torch.zeros(1, 1, 8, 8, dtype=torch.float64), lam, rho, torch.tensor([]))


def test_module_precision_attribute():
    from torch_admm_deconv_b200 import ADMMDeconv
    from torch_admm_deconv_b200.dropin import convert_admm_layer
    m = ADMMDeconv((3, 3), 4)
    assert m.precision == "float32"
    assert list(m.state_dict().keys()) == ["w", "lmbda", "rho", "b"]    # an attribute, not state
    assert convert_admm_layer(m).precision == "float32"
    m.precision = "float16"
    with pytest.raises(ValueError, match="precision"):
        m(torch.zeros(1, 1, 8, 8))
