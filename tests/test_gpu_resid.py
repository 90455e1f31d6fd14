"""Convergence residuals and tolerance-based early stopping (admm_ext.resid*, admm_solve_tol; DESIGN.md section 10).

`residuals_reference` below restates the residual test in numpy from a list of states (the checker of the GPU values).

Host (unmarked): that restatement against the textbook form, sizes of admm_query_resid and the ABI's refusals.  GPU:
  * residual values against residuals_reference on the GPU's own saved states, on every row x column kernel family;
  * an early stop returns exactly what a fixed solve with maxit = k returns, on every route;
  * residual histories are bit-identical from run to run and without programmatic dependent launch;
  * a residual history leaves the gradients unchanged.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

from conftest import ROOT  # noqa: F401  (puts the repository on sys.path)
from oracle import admm_oracle as O

RHO = 0.04
ALIGN = 256


def _al(n):
    return (n + ALIGN - 1) // ALIGN * ALIGN


def residuals_reference(states, lmbd, rho, iso=False, nmaps=None, atol=0.0, rtol=0.0, dtype=np.float64):
    """Primal / dual residuals of the splitting Dx - z = 0 (Boyd et al. 2011, 3.3) after each state, per plane.

    states : [(q_x, q_y)] pre-threshold states of iterations 1 .. n, each (B, C, H, W); q_0 = 0
    nmaps  : iso only: [(n_x, n_y)] pixel-norm maps of the same iterations (the threshold is decided on them), or None
             to compute them from the states
    dtype  : np.float64 forms every term in double; np.float32 forms u, z and the differences in float32 with the
             expressions of the CUDA kernel (tau = float32(lmbd) / float32(rho)), the sums of squares in double
    With u_k = dual(q_k), z_k = q_k - u_k, Dx_k = q_k - u_{k-1}, returns an (n, B, C, 4) float64 array of
        r = ||u_k - u_{k-1}||,  s = rho ||D^T(z_k - z_{k-1})||,
        eps_pri = sqrt(2HW) atol + rtol max(||Dx_k||, ||z_k||),  eps_dual = sqrt(HW) atol + rtol rho ||D^T u_k||,
    norms over both fields of one plane."""
    dt = np.dtype(dtype).type
    tau = dt(lmbd) / dt(rho)
    eps = dt(1e-15)

    def dual(q, n):
        if iso:
            s = np.maximum(dt(1) - tau / (np.asarray(n, dtype=dt) + eps), dt(0))
            return ((dt(1) - s) * q).astype(dt)
        if tau < 0:
            return (np.sign(q) * tau).astype(dt)
        return np.clip(q, -tau, tau).astype(dt)

    def sq(a):
        return np.sum(np.asarray(a, dtype=np.float64) ** 2, axis=(-2, -1))

    out = []
    qp = up = None
    for k, (q_x, q_y) in enumerate(states):
        q = (np.asarray(q_x, dtype=dt), np.asarray(q_y, dtype=dt))
        if iso and nmaps is None:
            n = tuple(np.sqrt(np.sum(np.asarray(a, np.float64) ** 2, (0, 1)) + 1e-15) for a in q)
        else:
            n = nmaps[k] if iso else (None, None)
        u = (dual(q[0], n[0]), dual(q[1], n[1]))
        if qp is None:
            qp = tuple(np.zeros_like(a) for a in q)
            up = tuple(np.zeros_like(a) for a in q)
        dz = tuple((q[f] - u[f]) - (qp[f] - up[f]) for f in range(2))
        dtz = (dz[0] - np.roll(dz[0], -1, axis=-1)) + (dz[1] - np.roll(dz[1], -1, axis=-2))
        dtu = (u[0] - np.roll(u[0], -1, axis=-1)) + (u[1] - np.roll(u[1], -1, axis=-2))
        r2 = sq(u[0] - up[0]) + sq(u[1] - up[1])
        dx2 = sq(q[0] - up[0]) + sq(q[1] - up[1])
        z2 = sq(q[0] - u[0]) + sq(q[1] - u[1])
        H, W = q[0].shape[-2:]
        rh = float(dt(rho))
        res = np.stack([np.sqrt(r2), rh * np.sqrt(sq(dtz)),
                        math.sqrt(2.0 * H * W) * atol + rtol * np.maximum(np.sqrt(dx2), np.sqrt(z2)),
                        math.sqrt(float(H * W)) * atol + rtol * rh * np.sqrt(sq(dtu))], axis=-1)
        out.append(res)
        qp, up = q, u
    return np.stack(out) if out else np.zeros((0, 0, 0, 4))


# ------------------------------------------------------------------------------------------------------------- host
@pytest.mark.parametrize("iso", [False, True], ids=["aniso", "iso"])
@pytest.mark.parametrize("lam", [0.5 * RHO, -0.5 * RHO], ids=["tau+0.5", "tau-0.5"])
def test_residuals_reference_matches_textbook_form(lam, iso):
    """The reduced-state restatement against the ADMM variables written out: x from q_k = Dx_k + u_{k-1}, z_k the
    reference's soft / block threshold of q_k, r = ||Dx_k - z_k||, s = rho ||D^T(z_k - z_{k-1})||, norms as in Boyd 3.3."""
    rng = np.random.default_rng(4)
    shape, n, tau = (2, 3, 9, 11), 4, lam / RHO
    states = [tuple(rng.standard_normal(shape) for _ in range(2)) for _ in range(n)]
    got = residuals_reference(states, lam, RHO, iso, None, atol=1e-3, rtol=1e-2)
    z_prev = (np.zeros(shape), np.zeros(shape))
    u_prev = (np.zeros(shape), np.zeros(shape))
    for k, q in enumerate(states):
        z = tuple(O.block_thresh(a, tau) if iso else O.soft_thresh(a, tau) for a in q)
        u = (q[0] - z[0], q[1] - z[1])
        dx = (q[0] - u_prev[0], q[1] - u_prev[1])
        dzs = (z[0] - z_prev[0], z[1] - z_prev[1])
        plane = lambda a, b: np.sqrt(np.sum(a ** 2, (-2, -1)) + np.sum(b ** 2, (-2, -1)))
        dt = lambda a, b: (a - np.roll(a, -1, -1)) + (b - np.roll(b, -1, -2))
        HW = shape[-2] * shape[-1]
        want = np.stack([plane(dx[0] - z[0], dx[1] - z[1]),
                         RHO * np.sqrt(np.sum(dt(*dzs) ** 2, (-2, -1))),
                         math.sqrt(2 * HW) * 1e-3 + 1e-2 * np.maximum(plane(*dx), plane(*z)),
                         math.sqrt(HW) * 1e-3 + 1e-2 * RHO * np.sqrt(np.sum(dt(*u) ** 2, (-2, -1)))], axis=-1)
        assert np.allclose(got[k], want, rtol=1e-12, atol=1e-14)
        z_prev, u_prev = z, u
    # the float32 restatement (the kernel's expressions) differs from float64 by float32 rounding only
    q32 = [tuple(a.astype(np.float32) for a in q) for q in states]
    g64 = residuals_reference(q32, lam, RHO, iso, None, atol=1e-3, rtol=1e-2)
    g32 = residuals_reference(q32, lam, RHO, iso, None, atol=1e-3, rtol=1e-2, dtype=np.float32)
    assert np.max(np.abs(g32 - g64) / np.abs(g64)) < 1e-6


def test_query_resid_sizes(lib):
    P, H, W = 6, 64, 48
    spec = P * H * ((W + 1) // 2) * 8
    base = lib.admm_query_resid(P, H, W, 1, 3, 0)          # maxit <= 1: no checks, scratch only
    assert base > 0
    assert lib.admm_query_resid(P, H, W, 0, 3, 0) == base
    assert lib.admm_query_resid(P, H, W, 3, 3, 0) == base   # (3 - 1) // 3 = 0 checks
    assert lib.admm_query_resid(P, H, W, 4, 3, 0) == base + _al(P * 16)
    assert lib.admm_query_resid(P, H, W, 100, 10, 0) == base + _al(9 * P * 16)
    assert lib.admm_query_resid(P, H, W, 100, 1, 0) == base + _al(99 * P * 16)
    # the spare spectrum of an early stop appears only when asked for
    assert lib.admm_query_resid(P, H, W, 100, 10, 1) == lib.admm_query_resid(P, H, W, 100, 10, 0) + _al(spec)
    assert lib.admm_query_resid(P, H, W, 1, 10, 1) == base + _al(spec)
    # off, or invalid
    assert lib.admm_query_resid(P, H, W, 100, 0, 0) == 0
    assert lib.admm_query_resid(P, H, W, 100, -1, 1) == 0
    assert lib.admm_query_resid(0, H, W, 100, 10, 0) == 0


def _ext(**kw):
    from torch_admm_deconv_b200 import _lib
    e = _lib.AdmmExt()
    e.struct_size = ctypes.sizeof(_lib.AdmmExt)
    for k, v in kw.items():
        setattr(e, k, v)
    return e


@pytest.mark.parametrize("fields,msg", [
    (dict(resid_every=10, rtol=1e-3, saved=True), "saved must be NULL"),
    (dict(resid_every=10, atol=1e-3, saved=True), "saved must be NULL"),
    (dict(resid_every=10, rtol=1e-3), "host_flag"),
    (dict(resid_every=10, rtol=-1e-3, flag=True), ">= 0"),
    (dict(resid_every=10, atol=-1.0, flag=True), ">= 0"),
    (dict(resid_every=10, rtol=float("nan"), flag=True), ">= 0"),
    (dict(resid_every=-1), "resid_every"),
    (dict(resid_every=0, rtol=1e-3, flag=True), "resid_every"),
    (dict(resid_every=10, resid=0), "resid"),
    (dict(resid_every=10, resid=ALIGN + 4), "aligned"),
])
def test_abi_rejects_invalid_residual_requests(lib, fields, msg):
    from torch_admm_deconv_b200 import _lib
    flag = ctypes.c_int(0)
    f = dict(fields)
    saved = ctypes.c_void_p(ALIGN * 64) if f.pop("saved", False) else ctypes.c_void_p(0)
    if f.pop("flag", False):
        f["host_flag"] = ctypes.addressof(flag)
    f.setdefault("resid", ALIGN * 16)
    ext = _ext(**f)
    before = lib.admm_launch_count()
    dummy = ctypes.c_void_p(ALIGN * 8)
    st = lib.admm_tv_forward_ex(dummy, dummy, None, 0, dummy, dummy, None, 1, 1, 16, 16, 0, 10, dummy, 1 << 20,
                                saved, 1 << 20, None, ctypes.byref(ext))
    assert st == 1
    assert msg in _lib.last_error()
    assert lib.admm_launch_count() == before


# -------------------------------------------------------------------------------------------------------------- GPU
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


def _input(shape, k, seed=5, u8=False):
    psf = O.make_psf("gauss", k, 1.5) if k else None
    x = O.make_blurred(shape, psf, seed=seed, noise=0.02)
    dev = _dev()
    kern = torch.tensor(psf[None, None], device=dev) if k else torch.empty(0, device=dev)
    if u8:
        return torch.tensor(np.clip(x * 255, 0, 255).astype(np.uint8), device=dev), kern
    return torch.tensor(x, device=dev), kern


def _train_history(x, kern, lam, iso, maxit, every, ckpt=0):
    """Training forward with a residual history (rtol = atol = 0).  Returns the history and the saved states q_1 ..
    q_{maxit-1} (every ckpt-th only when ckpt >= 2) with their iso norm maps."""
    from torch_admm_deconv_b200.eops.deconv import admm_solve_tol
    dev = x.device
    lt = torch.tensor([lam], dtype=torch.float32, device=dev, requires_grad=True)
    rt = torch.tensor([RHO], dtype=torch.float32, device=dev)
    out, info = admm_solve_tol(x, lt, rt, kern, iso, maxit, rtol=0.0, atol=0.0, check_every=every, ckpt_interval=ckpt)
    assert info.iters == maxit
    saved = out.grad_fn.saved_tensors[4]
    shape = tuple(x.shape)
    n, hw = x.numel(), shape[-2] * shape[-1]
    S = (maxit - 1) // ckpt if ckpt >= 2 else maxit - 1
    flt = saved[: (S * 2 * n + (S * 2 * hw if iso else 0)) * 4].view(torch.float32).cpu().numpy()
    q = flt[: S * 2 * n].reshape(S, 2, *shape)
    states = [(q[i, 0], q[i, 1]) for i in range(S)]
    nmaps = None
    if iso:
        m = flt[S * 2 * n:].reshape(S, 2, *shape[-2:])
        nmaps = [(m[i, 0], m[i, 1]) for i in range(S)]
    return info.residuals.cpu().numpy().astype(np.float64), states, nmaps


def _rel(a, b, floor):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), floor))


SMALL = float(np.float32(1e-9))   # a tolerance no check meets: every iteration runs; eps / SMALL = the norms

RESID_CASES = [
    # (shape, psf size, maxit, use_big) -- every row x column kernel family the solver pairs
    ((2, 3, 128, 128), 5, 6, 3),
    ((1, 3, 256, 256), 7, 6, 3),
    ((1, 2, 512, 512), 7, 5, 3),
    ((1, 2, 1080, 1920), 9, 4, 3),
    ((1, 1, 2160, 3840), 9, 4, 3),        # tile-major spectra between the large kernels
    ((1, 1, 2160, 3840), 9, 3, 1),        # large rows, generic columns
    ((1, 1, 2160, 3840), 9, 3, 2),        # generic rows, large columns
    ((2, 3, 33, 45), 5, 8, 3),            # generic engine, odd
    ((2, 2, 31, 37), 3, 8, 3),            # generic engine, prime
]


def _resid_case_ids():
    return ["%s-use_big%d" % ("x".join(map(str, c[0])), c[3]) for c in RESID_CASES]


def _check_values(x, kern, lam, iso, maxit, ckpt=0):
    from torch_admm_deconv_b200.eops.deconv import admm_solve_tol
    hist, states, nmaps = _train_history(x, kern, lam, iso, maxit, 1 if ckpt < 2 else ckpt, ckpt)
    with torch.no_grad():
        out, info = admm_solve_tol(x, lam, RHO, kern, iso, maxit, rtol=SMALL, atol=0.0, check_every=1 if ckpt < 2 else ckpt)
    assert info.iters == maxit
    inf = info.residuals.cpu().numpy().astype(np.float64)
    # inference keeps q as state when it checks residuals: the same numbers as training
    assert np.array_equal(inf[..., :2], hist[..., :2])
    if ckpt >= 2:
        return hist, states
    assert hist.shape[0] == len(states) == maxit - 1
    got = np.concatenate([hist[..., :2], inf[..., 2:] / SMALL], axis=-1)
    o32 = residuals_reference(states, lam, RHO, iso, nmaps, atol=0.0, rtol=1.0, dtype=np.float32)
    o64 = residuals_reference(states, lam, RHO, iso, nmaps, atol=0.0, rtol=1.0, dtype=np.float64)
    # the terms formed in float32 exactly as the kernel forms them: only the order of the double sums differs
    e32 = _rel(got, o32, 1e-30)
    # float64 throughout: relative, with a floor of 1e-6 of the plane's eps scale (rtol = 1) for residuals near zero
    floor = np.concatenate([o64[..., 2:3], o64[..., 3:4], o64[..., 2:4]], axis=-1) * 1e-6
    e64 = _rel(got, o64, np.maximum(floor, 1e-30))
    print("resid vs oracle: fp32 terms %.2e, fp64 %.2e" % (e32, e64))
    assert e32 <= 1e-6, e32
    assert e64 <= 1e-4, e64
    return hist, states


@pytest.mark.gpu
@pytest.mark.parametrize("iso", [False, True], ids=["aniso", "iso"])
@pytest.mark.parametrize("lam", [0.5 * RHO, -0.5 * RHO], ids=["tau+0.5", "tau-0.5"])
@pytest.mark.parametrize("case", RESID_CASES, ids=_resid_case_ids())
def test_residuals_match_oracle(case, lam, iso):
    shape, k, maxit, use_big = case
    x, kern = _input(shape, k)
    _with_options({"use_big": use_big}, lambda: _check_values(x, kern, lam, iso, maxit))


@pytest.mark.gpu
def test_residuals_uint8_input():
    x, kern = _input((2, 3, 128, 128), 5, u8=True)
    _check_values(x, kern, 0.5 * RHO, False, 6)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 3, 128, 128), (1, 1, 2160, 3840), (2, 3, 33, 45)], ids=lambda s: "x".join(map(str, s)))
def test_residuals_checkpointed_training(shape):
    """ckpt_interval = 3: the residual checks at 3, 6, ... read the checkpoint slots, the others the ping-pong state."""
    x, kern = _input(shape, 5)
    maxit, K = 10, 3
    hist, states = _check_values(x, kern, 0.5 * RHO, False, maxit, ckpt=K)
    full, _, _ = _train_history(x, kern, 0.5 * RHO, False, maxit, K)
    assert np.array_equal(hist, full)
    assert hist.shape[0] == (maxit - 1) // K


# ---- early stop
def _pick_rtol(info_small):
    """From a history at rtol = SMALL (eps / SMALL = the norms): a tolerance whose first met check is clear of the others
    by at least 2 % on both sides.  Returns (rtol, index of that check)."""
    h = info_small.residuals.cpu().numpy().astype(np.float64)
    need = np.max(np.maximum(h[..., 0] / (h[..., 2] / SMALL), h[..., 1] / (h[..., 3] / SMALL)), axis=(1, 2))
    cands = []
    for c in range(len(need)):
        prev = np.min(need[:c]) if c else np.inf
        if need[c] * 1.02 < prev:
            cands.append((c, need[c] * 1.02 if c == 0 else np.sqrt(need[c] * prev)))
    assert cands, need
    c, rtol = cands[len(cands) // 2]
    return float(rtol), c


STOP_CASES = [
    # (shape, psf, iso, maxit, check_every, activation, bias)
    ((2, 3, 128, 128), 5, False, 40, 3, None, False),
    ((2, 3, 128, 128), 5, True, 30, 3, None, False),
    ((2, 3, 256, 256), 7, False, 30, 2, "relu", True),
    ((1, 2, 512, 512), 7, False, 30, 4, "sigmoid", True),
    ((1, 1, 1080, 1920), 9, False, 20, 3, None, True),
    ((1, 1, 2160, 3840), 9, False, 20, 3, "tanh", True),
    ((1, 1, 2160, 3840), 9, True, 12, 2, None, False),
    ((2, 3, 33, 45), 5, False, 40, 3, "relu", True),
    ((2, 2, 31, 37), 3, True, 30, 2, None, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", STOP_CASES, ids=["%s-%s-%s" % ("x".join(map(str, c[0])), "iso" if c[2] else "aniso", c[5])
                                                  for c in STOP_CASES])
def test_early_stop_is_exact(case):
    from torch_admm_deconv_b200.eops.deconv import admm_solve, admm_solve_tol
    shape, k, iso, maxit, every, act, has_bias = case
    x, kern = _input(shape, k, seed=11)
    dev = x.device
    activation = {None: None, "relu": torch.relu, "sigmoid": torch.sigmoid, "tanh": torch.tanh}[act]
    bias = torch.tensor([0.25], device=dev) if has_bias else None
    lam = 0.5 * RHO

    def run():
        with torch.no_grad():
            kw = dict(check_every=every, bias=bias, activation=activation)
            out_n, info_n = admm_solve_tol(x, lam, RHO, kern, iso, maxit, rtol=SMALL, **kw)
            fixed = admm_solve(x, lam, RHO, kern, iso, maxit, bias=bias, activation=activation)
            # a tolerance that is never met: every iteration, the fixed solve's output
            assert info_n.iters == maxit
            assert info_n.residuals.shape == ((maxit - 1) // every,) + tuple(shape[:2]) + (4,)
            assert torch.equal(out_n, fixed)
            rtol, c = _pick_rtol(info_n)
            kstop = (c + 1) * every
            out_t, info_t = admm_solve_tol(x, lam, RHO, kern, iso, maxit, rtol=rtol, **kw)
            assert info_t.iters == kstop, (info_t.iters, kstop, rtol)
            assert info_t.residuals.shape[0] == c + 1
            ref = admm_solve(x, lam, RHO, kern, iso, kstop, bias=bias, activation=activation)
            assert torch.equal(out_t, ref)
            # the residuals up to the stop are those of the run that went on
            assert torch.equal(info_t.residuals[..., :2], info_n.residuals[:c + 1, ..., :2])
    # the cluster-resident solver runs small batches in one launch and has no residual checks: compare on the same route
    _with_options({"use_cluster": 0}, run)


@pytest.mark.gpu
def test_layer_tolerance():
    from torch_admm_deconv_b200 import ADMMDeconv
    from torch_admm_deconv_b200.eops.deconv import admm_solve_tol
    x, _ = _input((2, 3, 128, 128), 0, seed=2)
    layer = ADMMDeconv((5, 5), max_iters=40, iso=False, bias=True, activation=torch.relu).to(x.device)
    assert layer.last_solve_info is None
    layer.tol = (1e-2, 0.0, 5)
    with torch.no_grad():
        out = layer(x)
        ref, info = admm_solve_tol(x, layer.lmbda, layer.rho, layer.w, False, 40, rtol=1e-2, atol=0.0, check_every=5,
                                   bias=layer.b, activation=torch.relu)
    assert layer.last_solve_info.iters == info.iters
    assert torch.equal(out, ref)
    # with gradients the tolerance does not apply: the fixed solve, differentiable
    layer.last_solve_info = None
    out_g = layer(x)
    assert out_g.requires_grad and layer.last_solve_info is None


@pytest.mark.gpu
def test_tolerance_refusals(monkeypatch):
    from torch_admm_deconv_b200.eops.deconv import admm_solve_tol
    x, kern = _input((1, 1, 64, 64), 3)
    lt = torch.tensor([0.02], device=x.device, requires_grad=True)
    with pytest.raises(ValueError):
        admm_solve_tol(x, lt, RHO, kern, False, 10, rtol=1e-3)
    with pytest.raises(ValueError):
        admm_solve_tol(x, 0.02, RHO, kern, False, 10, rtol=-1.0)
    with pytest.raises(ValueError):
        admm_solve_tol(x, 0.02, RHO, kern, False, 10, check_every=0)
    with monkeypatch.context() as m:                   # as during CUDA-graph capture
        m.setattr(torch.cuda, "is_current_stream_capturing", lambda: True)
        with pytest.raises(RuntimeError):
            admm_solve_tol(x, 0.02, RHO, kern, False, 10, rtol=0.0)
    # maxit 0 / 1: no check
    with torch.no_grad():
        for m in (0, 1):
            out, info = admm_solve_tol(x, 0.02, RHO, kern, False, m, rtol=1e-3, check_every=1)
            assert info.iters == m and info.residuals.shape[0] == 0


# ---- determinism
@pytest.mark.gpu
@pytest.mark.parametrize("iso", [False, True], ids=["aniso", "iso"])
@pytest.mark.parametrize("shape", [(4, 3, 256, 256), (1, 1, 2160, 3840), (2, 3, 33, 45)], ids=lambda s: "x".join(map(str, s)))
def test_residuals_are_deterministic(shape, iso):
    from torch_admm_deconv_b200.eops.deconv import admm_solve_tol
    x, kern = _input(shape, 5)

    def hist():
        with torch.no_grad():
            return admm_solve_tol(x, 0.02, RHO, kern, iso, 9, rtol=SMALL, check_every=1)[1].residuals
    a, b = hist(), hist()
    c = _with_options({"use_pdl": 0}, hist)
    assert torch.equal(a, b)
    assert torch.equal(a, c)


# ---- gradients
@pytest.mark.gpu
@pytest.mark.parametrize("shape,k,maxit", [((32, 3, 256, 256), 0, 10), ((1, 1, 2160, 3840), 9, 4)],
                         ids=["cfg4", "2160x3840"])
def test_history_leaves_gradients_unchanged(shape, k, maxit):
    from torch_admm_deconv_b200.eops.deconv import admm_solve, admm_solve_tol
    x, kern = _input(shape, k, seed=7)
    g = torch.randn(shape, generator=torch.Generator().manual_seed(3)).to(x.device)

    def step(with_history):
        xt = x.clone().requires_grad_(True)
        lt = torch.tensor([0.02], device=x.device, requires_grad=True)
        rt = torch.tensor([RHO], device=x.device, requires_grad=True)
        kt = kern.clone().requires_grad_(True) if k else kern
        if with_history:
            out, info = admm_solve_tol(xt, lt, rt, kt, False, maxit, rtol=0.0, atol=0.0, check_every=1)
            assert info.residuals.shape[0] == maxit - 1
        else:
            out = admm_solve(xt, lt, rt, kt, False, maxit)
        (out * g).sum().backward()
        return [out.detach(), xt.grad, lt.grad, rt.grad] + ([kt.grad] if k else [])
    a, b = step(False), step(True)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
