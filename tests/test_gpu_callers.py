"""GPU parity tests (-m gpu) for the CALLERS of the hot path (SURVEY.md section 8f): the multi-solver containers
(MultiADMM / Deconvs / ADMMFusion), the fused activation epilogue and uint8 prologue of the layer, and the reference's
end-to-end model (DivergentRestorer) with this package's solver dropped in.  Every expected value comes from the
UNMODIFIED reference (tests/golden/make_golden_models.py, run on the CPU in the build container)."""
import os
import sys
import time

import numpy as np
import pytest
import torch

from conftest import golden, ROOT
from oracle import admm_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-4

FANOUT_CFGS = [dict(kern_size=(), max_iters=12, lmbda=0.02, rho=0.04, iso=True),
               dict(kern_size=(5, 5), max_iters=8, lmbda=None, rho=None, iso=False),
               dict(kern_size=(), max_iters=10, lmbda=None, rho=None, iso=False, bias=True)]


def _dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _sd(d, rename=None):
    sd = {k[3:]: torch.from_numpy(d[k]) for k in d.files if k.startswith("sd.")}
    return {(rename(k) if rename else k): v for k, v in sd.items()}


def _reference_package():
    """The pip-installed reference (baseline/_ref, written by baseline/install_ref.py in the build container)."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref, "admmtor", "elayers", "admmdeconv.py")):
        pytest.skip("baseline/_ref is not installed (python baseline/install_ref.py in the build container)")
    if ref not in sys.path:
        sys.path.insert(0, ref)


@pytest.mark.parametrize("concurrent", [True, False])
def test_multiadmm_and_deconvs_match_reference_fixture(concurrent):
    """reference MultiADMM (blocks.py:252-261) -> fixture; here: shared F(x), results written into channel slices, solvers
    on cached side streams.  Same state-dict keys (strict load), output within 1e-4 of the reference."""
    from torch_admm_deconv_b200 import MultiADMM, Deconvs
    d = golden("fanout_multiadmm")
    m = MultiADMM(FANOUT_CFGS, concurrent=concurrent)
    m.load_state_dict(_sd(d), strict=True)
    m = m.to(_dev())
    x = torch.from_numpy(d["x"]).to(_dev())
    with torch.inference_mode():
        y = m(x)
        seq = torch.cat([a(x) for a in m.admms], dim=1)
    e = O.rel_err(y.cpu().numpy(), d["out32"])
    print("MultiADMM concurrent=%s vs reference: %.2e" % (concurrent, e))
    assert y.shape == d["out32"].shape and e < TOL
    assert torch.equal(y, seq)                       # shared spectrum + slice output == separate calls, bit for bit
    dv = Deconvs(FANOUT_CFGS, concurrent=concurrent)
    dv.load_state_dict(_sd(d, lambda k: k.replace("admms.", "blocks.")), strict=True)
    with torch.inference_mode():
        assert torch.equal(dv.to(_dev())(x), y)


def test_fanout_training_matches_sequential_and_reference_grads():
    """Under autograd the containers give the gradients of the plain sequential composition."""
    from torch_admm_deconv_b200 import MultiADMM
    d = golden("fanout_multiadmm")
    dev = _dev()
    m = MultiADMM(FANOUT_CFGS).to(dev)
    m.load_state_dict(_sd(d), strict=True)
    x = torch.from_numpy(d["x"]).to(dev).requires_grad_(True)
    (m(x) ** 2).mean().backward()
    g1 = [x.grad.clone()] + [p.grad.clone() for p in m.parameters()]
    x.grad = None; m.zero_grad()
    (torch.cat([a(x) for a in m.admms], dim=1) ** 2).mean().backward()
    g2 = [x.grad.clone()] + [p.grad.clone() for p in m.parameters()]
    for a, b in zip(g1, g2):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-8)


def test_admmfusion_matches_reference_fixture():
    """reference ADMMFusion (admmfusion.py:9-40) with its own AttentionChannelPooling (imported from baseline/_ref, a
    plain CNN block outside the solver path) around this package's solvers: strict state-dict load, same output."""
    _reference_package()
    from torch_admm_deconv_b200 import ADMMFusion
    d = golden("fanout_fusion")
    f = ADMMFusion(FANOUT_CFGS, in_channels=3, with_admms=True)
    f.load_state_dict(_sd(d), strict=True)
    f = f.to(_dev()).eval()
    x = torch.from_numpy(d["x"]).to(_dev())
    with torch.inference_mode():
        y = f(x)
        probs = f.acp.cwa(torch.cat([a(x) for a in f.admms], dim=1))
    assert O.rel_err(probs.cpu().numpy(), d["probs"]) < 1e-3          # channel attention probabilities (top-k selection input)
    e = O.rel_err(y.cpu().numpy(), d["out32"])
    print("ADMMFusion vs reference: %.2e" % e)
    assert y.shape == d["out32"].shape and e < TOL


def test_admmfusion_solvers_match_reference_fixture():
    """The solver part of the reference ADMMFusion (fixture fanout_fusion, with_admms=True: the output ends with the
    concatenated solver results) without the reference's pooling block: the fixture's state dict loads with strict=True
    and the solver channels match the reference's within 1e-4."""
    from test_host_api import keyed_module
    from torch_admm_deconv_b200 import ADMMFusion
    d = golden("fanout_fusion")
    sd = _sd(d)

    class Pooling(torch.nn.Module):                      # keys of the reference's AttentionChannelPooling; 3 zero channels out
        def __init__(self):
            super().__init__()
            self.cwa = keyed_module({k[8:]: v for k, v in sd.items() if k.startswith("acp.cwa.")}).to(_dev())

        def forward(self, x):
            return torch.zeros_like(x[:, :3])
    f = ADMMFusion(FANOUT_CFGS, in_channels=3, with_admms=True, acp=Pooling())
    f.load_state_dict(sd, strict=True)
    f = f.to(_dev()).eval()
    x = torch.from_numpy(d["x"]).to(_dev())
    with torch.inference_mode():
        y = f(x)
    want = d["out32"][:, 3:]
    e = O.rel_err(y[:, 3:].cpu().numpy(), want)
    print("ADMMFusion solver channels vs reference: %.2e" % e)
    assert y.shape == d["out32"].shape and e < TOL


def test_fused_activation_and_uint8_input_match_reference_fixture():
    """activation(x + b) applied by the last kernel (admmdeconv.py:64) and a uint8 image read as x / 255 by the first
    (etransforms.py:29-31, dataload.py:31): against the reference's outputs, and bit-identical to the float path."""
    from torch_admm_deconv_b200 import ADMMDeconv
    d = golden("act_u8")
    dev = _dev()
    img = torch.from_numpy(d["img"]).to(dev)
    # x / 255.0 as the reference's loader computes it (CPU, IEEE division; torch's CUDA kernel multiplies by 1/255 instead)
    xs = (torch.from_numpy(d["img"]).to(torch.float32) / 255.0).to(dev)
    for name, act in (("relu", torch.relu), ("sigmoid", torch.nn.Sigmoid()), ("tanh", torch.tanh)):
        m = ADMMDeconv((3, 3), max_iters=9, lmbda=0.02, rho=0.04, iso=False, bias=True, activation=act).to(dev)
        with torch.no_grad():
            m.w.copy_(torch.from_numpy(d["w"]).to(dev)); m.b.fill_(-0.4)
        # the same layer with an unknown callable: the activation is applied after the call, in Python
        mp = ADMMDeconv((3, 3), max_iters=9, lmbda=0.02, rho=0.04, iso=False, bias=True, activation=lambda t, act=act: act(t)).to(dev)
        mp.load_state_dict(m.state_dict())
        with torch.inference_mode():
            y8, yf, yp = m(img), m(xs), mp(xs)
        e = O.rel_err(y8.cpu().numpy(), d["out_" + name])
        print("%s + uint8 input vs reference: %.2e" % (name, e))
        assert e < TOL and torch.equal(y8, yf)
        assert torch.allclose(yf, yp, rtol=1e-6, atol=1e-7)
    # gradients through a fused activation == gradients through the Python callable
    for act in (torch.relu, torch.sigmoid, torch.tanh):
        gs = []
        for fused in (True, False):
            m = ADMMDeconv((3, 3), max_iters=6, lmbda=None, rho=None, iso=False, bias=True,
                           activation=act if fused else (lambda t, act=act: act(t))).to(dev)
            with torch.no_grad():
                m.w.copy_(torch.from_numpy(d["w"]).to(dev)); m.b.fill_(-0.4); m.lmbda.fill_(0.02); m.rho.fill_(0.04)
            x = xs.clone().requires_grad_(True)
            (m(x) * torch.linspace(-1, 1, x.numel(), device=dev).reshape(x.shape)).sum().backward()
            gs.append([x.grad] + [p.grad for p in m.parameters()])
        for a, b in zip(*gs):
            assert torch.allclose(a, b, rtol=1e-4, atol=1e-6)


def test_restorer_end_to_end_with_solver_dropped_in():
    """The reference's trained architecture (DivergentRestorer built as scripts/train.py:19-24,70-73: two ADMMDeconv
    branches, kern_size=(), 100 iterations, iso=True, learnable lmbda / rho) with `use_b200_admm`: a checkpoint written by
    the REFERENCE model loads with strict=True, and the output matches the reference's CPU output."""
    _reference_package()
    from admmtor.modelbuild.denoiser import DivergentRestorer
    from torch_admm_deconv_b200 import use_b200_admm, ADMMDeconv
    d = golden("restorer_e2e")
    dev = _dev()
    cfg = lambda: [{'kern_size': (), 'max_iters': 100, 'iso': True}, {'kern_size': (), 'max_iters': 100, 'iso': True}]
    build = lambda: DivergentRestorer([2, 8, 32], 3, 3, 86, 86, 8, output_activation=torch.nn.Sigmoid(), admms=cfg())
    torch.manual_seed(int(d["seed"]))
    ref = build().eval()
    sd = ref.state_dict()
    assert list(sd.keys()) == list(d["sd_keys"])
    sums = np.array([float(v.double().sum()) for v in sd.values()])
    assert np.allclose(sums, d["sd_sums"], rtol=1e-9, atol=1e-9), "reference weights differ from the fixture's (seeded init)"
    ckpt = os.path.join("/tmp", "restorer_ckpt_%d.tar" % os.getpid())
    torch.save({"epoch": 0, "model_state_dict": sd}, ckpt)              # etrain/saver.py:47-54 format
    torch.manual_seed(99)
    model = build().eval()
    assert use_b200_admm(model) == 2
    assert all(isinstance(a, ADMMDeconv) for a in model.blocks[0].admms)
    model.load_state_dict(torch.load(ckpt, weights_only=False)["model_state_dict"], strict=True)   # scripts/train.py:75-78
    os.remove(ckpt)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
    try:
        model = model.to(dev)
        x = torch.from_numpy(d["x"]).to(dev)
        with torch.inference_mode():
            y = model(x)
            a0, a1 = (a(x) for a in model.blocks[0].admms)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(5):
                model(x)
            torch.cuda.synchronize()
            t_ours = (time.perf_counter() - t0) / 5
            ref_gpu = ref.to(dev)                                        # the reference's own eager CUDA path, same GPU
            yr = ref_gpu(x); torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(2):
                ref_gpu(x)
            torch.cuda.synchronize()
            t_ref = (time.perf_counter() - t0) / 2
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    e0, e1 = O.rel_err(a0.cpu().numpy(), d["admm0"]), O.rel_err(a1.cpu().numpy(), d["admm1"])
    e = O.rel_err(y.cpu().numpy(), d["out32"])
    e_ref = O.rel_err(yr.cpu().numpy(), d["out32"])                      # the reference's own GPU-vs-CPU deviation
    print("DivergentRestorer 2x3x64x64: ADMM branches vs reference %.2e / %.2e; model output vs reference CPU %.2e (the reference's "
          "own eager CUDA run vs its CPU run: %.2e); inference %.2f ms with the solver dropped in vs %.2f ms reference eager CUDA" %
          (e0, e1, e, e_ref, t_ours * 1e3, t_ref * 1e3))
    # the solver branches -- the part this package replaces -- are gated at the path's tolerance
    assert e0 < TOL and e1 < TOL
    # The random-weight network behind them (86-channel 1x1 / 3x3 stacks, CBAM max / lse pooling, sigmoid) amplifies a 1e-6
    # input perturbation to ~4e-3 at its output (measured with the reference itself on the CPU), so the end-to-end gate is
    # relative to the reference's own device-to-device deviation on the same weights
    assert e < max(3.0 * e_ref, 1e-3)


def test_restorer_solver_branches_match_reference_fixture():
    """The two ADMMDeconv branches of the reference's DivergentRestorer (fixture restorer_e2e: kern_size=(), 100
    iterations, iso=True, learnable lmbda / rho drawn from the seeded init) on the fixture's input, against the branch
    outputs of the reference's CPU run.  The scalar parameters are read back from the fixture's per-tensor sums."""
    from torch_admm_deconv_b200 import ADMMDeconv
    d = golden("restorer_e2e")
    dev = _dev()
    sums = dict(zip(d["sd_keys"].tolist(), d["sd_sums"].tolist()))
    x = torch.from_numpy(d["x"]).to(dev)
    for i in range(2):
        pre = "blocks.0.admms.%d." % i
        assert sums[pre + "w"] == 0.0 and sums[pre + "b"] == 0.0
        m = ADMMDeconv((), max_iters=100, iso=True).to(dev)
        with torch.no_grad():
            m.lmbda.fill_(sums[pre + "lmbda"]); m.rho.fill_(sums[pre + "rho"])
        with torch.inference_mode():
            y = m(x)
        e = O.rel_err(y.cpu().numpy(), d["admm%d" % i])
        print("DivergentRestorer ADMM branch %d vs reference: %.2e" % (i, e))
        assert e < TOL


def test_cast_shim_for_float64_inputs():
    """fp64 inputs are refused by `fft_admm_tv` (float32 kernels) and served by the explicit shim `fft_admm_tv_cast`;
    checked against the reference's own fp64 output and fp64 autograd (fixture)."""
    from torch_admm_deconv_b200 import fft_admm_tv
    from torch_admm_deconv_b200.eops.deconv import fft_admm_tv_cast
    d = golden("grad_aniso_k5_16x20_n6")
    dev = _dev()
    x = torch.tensor(d["x"], dtype=torch.float64, device=dev, requires_grad=True)
    lam = torch.tensor([float(d["lam"])], dtype=torch.float64, device=dev, requires_grad=True)
    rho = torch.tensor([float(d["rho"])], dtype=torch.float64, device=dev, requires_grad=True)
    k = torch.tensor(d["kern"], dtype=torch.float64, device=dev, requires_grad=True)
    with pytest.raises(TypeError):
        fft_admm_tv(x, lam, rho, k, False, int(d["maxit"]))
    out = fft_admm_tv_cast(x, lam, rho, k, False, int(d["maxit"]))
    assert out.dtype == torch.float64 and O.rel_err(out.detach().cpu().numpy(), d["out64"]) < TOL
    (out * torch.tensor(d["gout"], device=dev)).sum().backward()
    assert x.grad.dtype == torch.float64 and O.rel_err(x.grad.cpu().numpy(), d["gx"]) < 1e-5
    assert abs(float(lam.grad) - d["glam"][0]) < 1e-4 * abs(d["glam"][0]) and abs(float(rho.grad) - d["grho"][0]) < 1e-4 * abs(d["grho"][0])
    assert O.rel_err(k.grad.cpu().numpy(), d["gkern"]) < 1e-4


def test_concurrent_host_threads_and_streams():
    """Two host threads drive the library at the same time, each on its own stream (the C ABI keeps no per-call global
    state: atomic option reads, atomic launch counter, per-device attribute caches): results equal the serial ones."""
    import threading
    from torch_admm_deconv_b200 import fft_admm_tv, ADMMDeconv
    dev = _dev()
    psf = O.make_psf("gauss", 7, 1.5)
    kern = torch.from_numpy(psf[None, None]).to(dev)
    lam, rho = torch.tensor([0.02], device=dev), torch.tensor([0.04], device=dev)
    xs = [torch.from_numpy(O.make_blurred(s, psf, seed=i)).to(dev)
          for i, s in enumerate([(2, 3, 128, 128), (1, 2, 60, 90), (3, 1, 256, 256), (1, 1, 512, 512)])]
    want = [fft_admm_tv(x, lam, rho, kern, False, 8).clone() for x in xs]
    torch.cuda.synchronize()
    got = [[None] * len(xs) for _ in range(2)]
    errs = []

    def work(k):
        try:
            st = torch.cuda.Stream(dev)
            with torch.cuda.stream(st):
                for rep in range(6):
                    for i, x in enumerate(xs):
                        got[k][i] = fft_admm_tv(x, lam, rho, kern, False, 8)
            st.synchronize()
        except Exception as e:   # pragma: no cover
            errs.append(e)
    th = [threading.Thread(target=work, args=(k,)) for k in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    for k in range(2):
        for a, b in zip(got[k], want):
            assert torch.equal(a, b)
    # python-number parameters are uploaded once and cached (no per-call host-to-device copy)
    out = fft_admm_tv(xs[0], 0.02, 0.04, kern, False, 8)
    assert torch.equal(out, want[0])


def test_ext_abi_corner_paths():
    """C-ABI paths the Python layer does not take by default: a solver that WRITES the shared spectrum (admm_ext.yhat_out)
    and a second one that reads it; L2 plane chunks (option chunk_mb) in inference and training; uint8 input, activation
    and channel-slice output on the large-frame and generic kernels."""
    import ctypes
    from torch_admm_deconv_b200 import _lib, fft_admm_tv, ADMMDeconv
    from torch_admm_deconv_b200.eops.deconv import admm_solve
    lib = _lib.load()
    dev = _dev()
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)
    lam, rho = torch.tensor([0.02], device=dev), torch.tensor([0.04], device=dev)
    psf = O.make_psf("gauss", 5, 1.2)
    kern = torch.from_numpy(psf[None, None]).to(dev)
    # --- yhat_out then yhat_in, on the power-of-two kernels (20 planes: not the cluster path) and the generic engine
    for shape in ((10, 2, 128, 256), (2, 3, 60, 90)):
        x = torch.from_numpy(O.make_blurred(shape, psf, seed=5)).to(dev)
        B, C, H, W = shape
        want = fft_admm_tv(x, lam, rho, kern, False, 7)
        ws = torch.empty(lib.admm_query_workspace(B * C, H, W, 5, 0, 7), dtype=torch.uint8, device=dev)
        yhat = torch.empty(lib.admm_query_yhat(B * C, H, W), dtype=torch.uint8, device=dev)
        outs = []
        for mode in ("out", "in"):
            ext = _lib.AdmmExt(); ext.struct_size = ctypes.sizeof(_lib.AdmmExt)
            setattr(ext, "yhat_" + mode, yhat.data_ptr())
            o = torch.empty_like(x)
            st = lib.admm_tv_forward_ex(p(x), p(o), p(kern), 5, p(lam), p(rho), None, B, C, H, W, 0, 7, p(ws), ws.numel(), None, 0,
                                        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream), ctypes.byref(ext))
            _lib.check(st, "admm_tv_forward_ex")
            outs.append(o)
        torch.cuda.synchronize()
        assert float((outs[0] - want).abs().max()) < 2e-6 and torch.equal(outs[0], outs[1])
    # --- plane chunks: same bits in inference, same gradients in training
    x = torch.from_numpy(O.make_blurred((20, 1, 256, 256), psf, seed=6)).to(dev)
    res = []
    for mb in (0, 8):
        _lib.set_option("chunk_mb", mb)
        try:
            y = fft_admm_tv(x, lam, rho, kern, False, 9)
            xg = x.clone().requires_grad_(True); lg = lam.clone().requires_grad_(True)
            (fft_admm_tv(xg, lg, rho, kern, False, 6) ** 2).sum().backward()
            res.append((y, xg.grad, lg.grad))
        finally:
            _lib.set_option("chunk_mb", -1)
    for a, b in zip(*res):
        assert torch.equal(a, b)
    # --- uint8 input + tanh + bias + channel slice on the large-frame kernels and the generic engine
    for shape in ((1, 2, 1080, 1920), (2, 2, 45, 63)):
        img = torch.randint(0, 256, shape, dtype=torch.uint8, device=dev)
        xf = (img.cpu().to(torch.float32) / 255.0).to(dev)
        b = torch.tensor([-0.2], device=dev)
        big = torch.zeros(shape[0], 5, *shape[2:], device=dev)
        y8 = admm_solve(img, lam, rho, kern, False, 4, bias=b, activation=torch.tanh, out=big[:, 1:3])
        yf = torch.tanh(fft_admm_tv(xf, lam, rho, kern, False, 4) + b)
        assert float((y8 - yf).abs().max()) < 2e-6 and torch.equal(big[:, 1:3], y8) and float(big[:, 3:].abs().max()) == 0.0
