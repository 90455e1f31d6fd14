"""CPU tests of the host side: the C-ABI library loads and exports every symbol of include/admm_b200.h,
pure-host entry points work without a GPU, and the Python mirror of the reference API behaves like the
reference (constructor, state dict, RNG order, error types).  No kernels are launched here."""
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, golden


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "admm_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(admm_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_header_symbol(lib):
    from torch_admm_deconv_b200 import _lib
    syms = header_symbols()
    assert len(syms) >= 10
    for s in syms:
        assert hasattr(lib, s), "libadmm_b200.so does not export %s" % s
        assert s in _lib.SIGNATURES, "ctypes binding missing for %s" % s
    assert lib.admm_version() >= 100


def test_query_workspace_is_pure_host(lib):
    n = lib.admm_query_workspace(192, 512, 512, 31, 0, 100)
    assert n > 3 * 192 * 512 * 512 * 4
    assert lib.admm_query_workspace(0, 512, 512, 31, 0, 100) == 0          # planes < 1
    assert lib.admm_query_workspace(1, 16, 16, 17, 0, 10) == 0            # PSF larger than the image
    assert lib.admm_query_saved(6, 16, 20, 5, 0, 6) >= 5 * 2 * 6 * 16 * 20 * 4
    assert b"PSF" in lib.admm_last_error() or b"planes" in lib.admm_last_error()


def test_options_roundtrip(lib):
    from torch_admm_deconv_b200 import _lib
    old = _lib.get_option("rows_per_band")
    _lib.set_option("rows_per_band", 8)
    assert _lib.get_option("rows_per_band") == 8
    _lib.set_option("rows_per_band", old)
    with pytest.raises(KeyError):
        _lib.set_option("no_such_option", 1)


def test_module_matches_reference_construction():
    from torch_admm_deconv_b200 import ADMMDeconv
    d = golden("module_k5_bias")
    torch.manual_seed(1234)
    m = ADMMDeconv((5, 5), max_iters=8, lmbda=None, rho=None, iso=False, bias=True)
    sd = m.state_dict()
    assert list(sd.keys()) == ["w", "lmbda", "rho", "b"]
    for k in sd:                                                   # same RNG draw order as the reference
        assert np.array_equal(sd[k].numpy(), d["init_" + k]), k
    assert [isinstance(getattr(m, n), torch.nn.Parameter) for n in ("w", "lmbda", "rho", "b")] == list(d["is_param"])
    # a reference state dict loads strictly
    ref_sd = {k: torch.from_numpy(d["sd_" + k]) for k in ("w", "lmbda", "rho", "b")}
    m.load_state_dict(ref_sd, strict=True)


def test_module_empty_kernel_and_defaults():
    from torch_admm_deconv_b200 import ADMMDeconv, identity
    d = golden("module_empty")
    m = ADMMDeconv((), max_iters=5, lmbda=0.02, rho=0.04)
    assert list(m.state_dict().keys()) == list(d["keys"])
    assert tuple(m.w.shape) == tuple(d["w_shape"]) == (0,)
    assert m.iso is True and bool(d["iso"]) is True                # module default is iso=True
    assert [isinstance(getattr(m, n), torch.nn.Parameter) for n in ("w", "lmbda", "rho", "b")] == list(d["is_param"])
    assert m.activation is identity
    # falsy lmbda / rho (None or 0) mean "learnable" (admmdeconv.py:27,36)
    m0 = ADMMDeconv((3, 3), 4, lmbda=0.0, rho=0)
    assert isinstance(m0.lmbda, torch.nn.Parameter) and isinstance(m0.rho, torch.nn.Parameter)
    # kwargs-dict construction used by the reference callers (admmfusion.py:30, deconver.py:19)
    ADMMDeconv(**{"kern_size": (3, 3), "max_iters": 2, "lmbda": 0.1, "rho": 0.2, "iso": False})
    # external clippers mutate .data in place (scripts/train.py:31-38)
    m0.lmbda.data.clamp_(1e-12, 5); m0.rho.data.clamp_(1e-12, 5); m0.w.data.clamp_(-1, 1)


def test_input_validation_no_cpu_fallback():
    from torch_admm_deconv_b200 import fft_admm_tv
    lam, rho = torch.tensor([0.02]), torch.tensor([0.04])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        fft_admm_tv(torch.zeros(1, 1, 8, 8), lam, rho, torch.tensor([]))
    with pytest.raises(ValueError):
        fft_admm_tv(torch.zeros(8, 8), lam, rho, torch.tensor([]))


def test_helper_ops_match_oracle():
    from torch_admm_deconv_b200.eops import deconv as D
    from oracle import admm_oracle as O
    rng = np.random.default_rng(0)
    x = rng.standard_normal((2, 3, 5, 7))
    xt = torch.from_numpy(x)
    assert np.allclose(D.soft_thresh(xt, 0.3).numpy(), O.soft_thresh(x, 0.3))
    assert np.allclose(D.hard_thresh(xt, 0.3).numpy(), O.hard_thresh(x, 0.3))
    assert np.allclose(D.block_thresh(xt, torch.tensor(0.3)).numpy(), O.block_thresh(x, 0.3))
    assert np.allclose(D.pixelnorm(xt).numpy(), O.pixelnorm(x))
    assert np.allclose(D.torch_abs2(xt).numpy(), O.abs2(x))
    assert D.identity(xt) is xt
    w = torch.tensor([[[[0., 0.], [-1., 1.]]]], dtype=torch.float64).repeat(3, 1, 1, 1)
    dx = D.conv_circular(xt, w, (1, 0, 1, 0), 3).numpy()
    assert np.allclose(dx, x - np.roll(x, 1, -1))


def test_activation_codes():
    from torch_admm_deconv_b200.eops.deconv import activation_code, identity
    from torch_admm_deconv_b200 import _lib
    import torch.nn.functional as F
    assert activation_code(identity) == _lib.ACT_NONE and activation_code(None) == _lib.ACT_NONE
    assert activation_code(torch.nn.Identity()) == _lib.ACT_NONE
    assert activation_code(torch.relu) == activation_code(F.relu) == activation_code(torch.nn.ReLU()) == _lib.ACT_RELU
    assert activation_code(torch.sigmoid) == activation_code(torch.nn.Sigmoid()) == _lib.ACT_SIGMOID
    assert activation_code(torch.tanh) == activation_code(torch.nn.Tanh()) == _lib.ACT_TANH
    assert activation_code(torch.nn.ReLU(inplace=True)) is None           # in-place semantics are left to Python
    assert activation_code(lambda t: t) is None and activation_code(torch.nn.GELU()) is None


def _ref_path():
    import os, sys
    ref = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "baseline", "_ref")
    if not os.path.exists(os.path.join(ref, "admmtor", "elayers", "admmdeconv.py")):
        pytest.skip("baseline/_ref not installed")
    if ref not in sys.path:
        sys.path.insert(0, ref)


def _reference_classes():
    """Stand-ins for the reference's `ADMMDeconv` (elayers/admmdeconv.py:6-64) and `MultiADMM` (modelbuild/blocks.py:252-261),
    which `use_b200_admm` meets inside reference models: a class of its own named ADMMDeconv with the reference's
    attributes, parameter-vs-buffer status, state-dict keys and RNG draw order (checked against the reference's recorded
    construction, fixture module_k5_bias), and a container holding the layers in `admms`."""
    from torch_admm_deconv_b200 import ADMMDeconv as Ours

    class ADMMDeconv(torch.nn.Module):
        def __init__(self, *args, **kwargs):
            super().__init__()
            src = Ours(*args, **kwargs)
            for name in ("w", "lmbda", "rho", "b"):
                t = getattr(src, name)
                if isinstance(t, torch.nn.Parameter):
                    self.register_parameter(name, t)
                else:
                    self.register_buffer(name, t)
            self.max_iters, self.iso, self.activation = src.max_iters, src.iso, src.activation

    class MultiADMM(torch.nn.Module):
        def __init__(self, admm_dicts):
            super().__init__()
            self.admms = torch.nn.ModuleList(ADMMDeconv(**d) for d in admm_dicts)

    d = golden("module_k5_bias")
    torch.manual_seed(1234)
    ref = ADMMDeconv((5, 5), max_iters=8, lmbda=None, rho=None, iso=False, bias=True)
    assert list(ref.state_dict().keys()) == ["w", "lmbda", "rho", "b"]
    assert all(np.array_equal(v.numpy(), d["init_" + k]) for k, v in ref.state_dict().items())
    assert [isinstance(getattr(ref, n), torch.nn.Parameter) for n in ("w", "lmbda", "rho", "b")] == list(d["is_param"])
    return MultiADMM, ADMMDeconv


def test_drop_in_conversion_shares_parameters_and_keys():
    """use_b200_admm swaps the reference's ADMMDeconv layers inside the reference's own model, keeping the very same
    Parameter objects (optimizers, clippers that reach into .lmbda/.rho/.w, checkpoints: scripts/train.py:27-38,75-78)."""
    RefMulti, RefLayer = _reference_classes()
    from torch_admm_deconv_b200 import use_b200_admm, ADMMDeconv
    cfgs = [dict(kern_size=(3, 3), max_iters=4, lmbda=None, rho=0.1, iso=False, bias=True, activation=torch.relu),
            dict(kern_size=(), max_iters=7)]
    m = RefMulti(cfgs)
    before = dict(m.state_dict())
    params = {n: p for n, p in m.named_parameters()}
    assert use_b200_admm(m) == 2 and use_b200_admm(m) == 0
    assert all(isinstance(a, ADMMDeconv) and not isinstance(a, RefLayer) for a in m.admms)
    assert list(m.state_dict().keys()) == list(before.keys())
    assert all(p is params[n] for n, p in m.named_parameters())
    assert m.admms[0].max_iters == 4 and m.admms[0].iso is False and m.admms[0].activation is torch.relu
    assert m.admms[1].iso is True and isinstance(m.admms[1].w, torch.Tensor) and m.admms[1].w.numel() == 0
    m.load_state_dict(before, strict=True)


def test_admmfusion_state_dict_matches_reference():
    _ref_path()
    from admmtor.elayers.admmfusion import ADMMFusion as RefFusion
    from torch_admm_deconv_b200 import ADMMFusion
    cfgs = [dict(kern_size=(), max_iters=3), dict(kern_size=(3, 3), max_iters=2, bias=True)]
    torch.manual_seed(0); r = RefFusion(cfgs, in_channels=3)
    torch.manual_seed(0); o = ADMMFusion(cfgs, in_channels=3)
    rs, os_ = r.state_dict(), o.state_dict()
    assert list(rs.keys()) == list(os_.keys())
    assert all(torch.equal(rs[k], os_[k]) for k in rs)                   # same RNG draw order as the reference
    o.load_state_dict(rs, strict=True)


FANOUT_CFGS = [dict(kern_size=(), max_iters=12, lmbda=0.02, rho=0.04, iso=True),
               dict(kern_size=(5, 5), max_iters=8, lmbda=None, rho=None, iso=False),
               dict(kern_size=(), max_iters=10, lmbda=None, rho=None, iso=False, bias=True)]


def keyed_module(sd):
    """A module holding zero parameters under the keys of the state dict `sd` (stands in for a block that is not part of
    this package, so that a state dict containing it loads with strict=True)."""
    root = torch.nn.Module()
    for key, v in sd.items():
        *path, leaf = key.split(".")
        m = root
        for p in path:
            if not hasattr(m, p):
                m.add_module(p, torch.nn.Module())
            m = getattr(m, p)
        m.register_parameter(leaf, torch.nn.Parameter(torch.zeros(v.shape)))
    return root


def test_admmfusion_solver_state_dict_matches_reference_fixture():
    """The solver part of ADMMFusion against the reference's ADMMFusion(FANOUT_CFGS, in_channels=3) built after
    torch.manual_seed(12) (fixture fanout_fusion; the reference then replaced the 5 x 5 `w` by a Gaussian): same keys in
    the same order, same RNG draws, and the reference state dict loads with strict=True.  The pooling block `acp` is
    reference code, given here as a module with its keys."""
    from torch_admm_deconv_b200 import ADMMFusion
    d = golden("fanout_fusion")
    sd = {k[3:]: torch.from_numpy(d[k]) for k in d.files if k.startswith("sd.")}
    acp = keyed_module({k[4:]: v for k, v in sd.items() if k.startswith("acp.")})
    torch.manual_seed(12)
    o = ADMMFusion(FANOUT_CFGS, in_channels=3, with_admms=True, acp=acp)
    os_ = o.state_dict()
    assert list(os_.keys()) == list(sd.keys())
    for k, v in sd.items():
        if k.startswith("admms.") and k != "admms.1.w":
            assert torch.equal(os_[k], v), k
    o.load_state_dict(sd, strict=True)
