"""Every kernel route of the float32 solver, forward and backward, one iteration at a time against the fp64 oracle.

The solver picks a row kernel (generic, power-of-two for W in {128, 256, 512}, or large-frame for ten widths) and a
column kernel (generic, power-of-two for H in {128, 256, 512}, or large-frame for eight heights) per problem; the
backward adds the fused adjoint row pass (ROWS_ADJ, power-of-two rows, iso=False), the fused adjoint column pass
(k_cols_adj) and, for iso=True, divergences formed inside the R2C row pass.  `route()` mirrors those predicates and
names the route in every test id.

The gate.  A training forward saves the pre-threshold state q_k of every iteration (and, for iso=True, its two pixel
norm maps).  Iteration k+1 is a deterministic function of q_k and y, so the oracle replays it in fp64 from the saved
fp32 state (`admm_tv_replay`): every threshold decision is taken on the GPU's numbers, and what remains is one
iteration's fp32 rounding, whatever the sign of tau or the number of iterations.  Whole trajectories are not a sharp
gate for tau < 0: u(q) jumps by 2|tau| where q changes sign, and an fp32 and an fp64 run separate (tests/test_oracle.py
shows one case at 4e-4).  The adjoint is gated the same way, with the masks and norms taken from the saved state
(`admm_tv_backward(qs_override, tau_override, nmaps_override)`).  For tau > 0 the end-to-end gates of
test_gpu_parity.py apply as well (the gradient one for iso=False only, see `gate`).

The host-side route check runs without a GPU; everything else is marked gpu."""
import numpy as np
import pytest
import torch

from oracle import admm_oracle as O

STEP_TOL = 5e-6          # one-step replay: saved q_k, norm maps, output
GRAD_TOL_X = 1e-5        # x-gradient against the same-state adjoint
GRAD_TOL_P = 1e-4        # lambda, rho, kernel gradients against the same-state adjoint
GRAD_TOL_L2 = 1e-3       # end-to-end x-gradient (tau > 0), relative L2 norm
TRAJ_TOL = 1e-4          # end-to-end output (tau > 0)
STATE_TOL = 1e-5         # end-to-end saved state (tau > 0)
RHO = 0.04

ROWS_BIG_W = (3840, 1920, 1024, 2048, 4096, 2560, 1280, 768, 1536, 3072)     # rows_big_supported
COLS_BIG_H = (2160, 1080, 1024, 1440, 720, 2048, 768, 1536)                 # cols_big_supported
POW2 = (128, 256, 512)
COLS_TILE = {128: 32, 256: 16, 512: 16}      # columns per tile of the power-of-two column kernel (cols_pow2_supported)
ADJ_TILE = {128: 32, 256: 16, 512: 8}        # ... and of the fused adjoint column kernel (cols_adj_supported)


def route(H, W):
    """(rows, cols, adj): the row and column kernel families the solver picks for an H x W plane, and whether the
    backward takes the fused adjoint column pass k_cols_adj."""
    Wc = (W + 1) // 2
    if W in POW2 and H % 2 == 0:
        rows = "pow2"
    elif W in ROWS_BIG_W and H % 2 == 0 and H >= 4:
        rows = "big%d" % W
    else:
        rows = "generic"
    if H in POW2 and W % 2 == 0 and Wc % COLS_TILE[H] == 0:
        cols = "pow2"
    elif H in COLS_BIG_H and Wc % 8 == 0:
        cols = "big%d" % H
    else:
        cols = "generic"
    adj = H in POW2 and W % 2 == 0 and Wc % ADJ_TILE[H] == 0
    return rows, cols, adj


def route_name(shape):
    rows, cols, adj = route(shape[-2], shape[-1])
    return "%s-rows=%s-cols=%s%s" % ("x".join(map(str, shape)), rows, cols, "+adj" if adj and cols != "pow2" else "")


def route_id(shape, iso, lam):
    return "%s-%s-%s" % (route_name(shape), "iso" if iso else "aniso", "negtau" if lam < 0 else "postau")


@pytest.mark.parametrize("H,W", [(60, 90), (45, 63), (256, 256), (512, 512), (128, 512), (512, 256), (60, 256), (6, 512),
                                 (256, 96), (512, 48), (100, 1920), (4, 3840), (1080, 48), (720, 1280), (1080, 1920),
                                 (2160, 3840), (256, 1920), (512, 3840), (1080, 512), (720, 256), (1080, 100), (2160, 18),
                                 (1536, 16), (768, 24), (1440, 2560), (2048, 2048), (1024, 1024)])
def test_route_helper_matches_library(lib, H, W):
    """admm_query_yhat returns 0 exactly when the large-frame column kernel takes the problem."""
    assert (route(H, W)[1].startswith("big")) == (lib.admm_query_yhat(1, H, W) == 0)


# ------------------------------------------------------------------------------------------------------------ GPU
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


def _train(x, kern, gout, lam, iso, maxit, need):
    """Training forward + backward on the GPU.  Returns the output, the gradients (None where not requested), the saved
    states q_1 .. q_{maxit-1} and (iso) their norm maps."""
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    xt = torch.tensor(x, device=dev, requires_grad="x" in need)
    lt = torch.tensor([lam], dtype=torch.float32, device=dev, requires_grad="l" in need)
    rt = torch.tensor([RHO], dtype=torch.float32, device=dev, requires_grad="r" in need)
    kt = torch.tensor(np.asarray(kern, np.float32), device=dev, requires_grad="k" in need) if np.size(kern) \
        else torch.empty(0, device=dev)
    out = fft_admm_tv(xt, lt, rt, kt, iso, maxit)
    # the state the forward saved for its backward: slots 1 .. maxit-1 of [q_x, q_y] (B, C, H, W) each, then for
    # iso=True one [n_x, n_y] (H, W) pair per slot
    saved = out.grad_fn.saved_tensors[4]
    n, hw, S = x.size, x.shape[-2] * x.shape[-1], maxit - 1
    flt = saved[: (S * 2 * n + (S * 2 * hw if iso else 0)) * 4].view(torch.float32).cpu().numpy()
    q = flt[: S * 2 * n].reshape(S, 2, *x.shape)
    states = [(q[i, 0], q[i, 1]) for i in range(S)]
    nmaps = None
    if iso:
        m = flt[S * 2 * n:].reshape(S, 2, *x.shape[-2:])
        nmaps = [(m[i, 0], m[i, 1]) for i in range(S)]
    (out * torch.tensor(gout, dtype=torch.float32, device=dev)).sum().backward()
    torch.cuda.synchronize()
    g = lambda t: None if t.grad is None else t.grad.cpu().numpy().astype(np.float64)
    return out.detach().cpu().numpy(), (g(xt), g(lt), g(rt), g(kt) if np.size(kern) else None), states, nmaps


def _rel(a, b):
    return abs(float(a) - float(b)) / max(abs(float(b)), 1e-12)


def gate(shape, k, maxit, iso, lam, need="xlrk", seed=3):
    """Training forward and backward on one route against the fp64 oracle, one iteration at a time.  Returns the observed
    errors (printed as well)."""
    x, kern, gout = _inputs(shape, k, seed)
    if not np.size(kern):
        need = need.replace("k", "")
    out, (gx, gl, gr, gk), states, nmaps = _train(x, kern, gout, lam, iso, maxit, need)
    x64 = x.astype(np.float64)
    tau32 = float(np.float32(lam) / np.float32(RHO))
    preds, norms, x_out = O.admm_tv_replay(x64, lam, RHO, kern, states, iso, tau32, nmaps, workers=-1)
    e = {"step": O.pair_err(states, preds, np.abs(x_out).max()), "out": O.rel_err(out, x_out)}
    if iso:
        e["nmap"] = O.pair_err(nmaps, norms)
    sx, sl, sr, sk = O.admm_tv_backward(x64, lam, RHO, kern, gout, iso, maxit, qs_override=states, tau_override=tau32,
                                        nmaps_override=nmaps, workers=-1)
    if gx is not None:
        e["gx"] = O.rel_err(gx, sx)
    if gl is not None and maxit > 1:
        e["glam"] = _rel(gl[0], sl)
    if gr is not None:
        # rho gradient = (spectral part) - taubar * lam / rho^2: the parts can cancel, so the error is measured against the
        # larger of the result and the tau part (as in test_gpu_parity.py)
        e["grho"] = abs(float(gr[0]) - sr) / max(abs(sr), abs(sl) * abs(lam / RHO), 1e-12)
    if gk is not None:
        e["gkern"] = O.rel_err(gk, sk)
    if lam > 0 and gx is not None:
        ref, hist = O.admm_tv_spectral_form(x64, lam, RHO, kern, iso, maxit, return_state=True, workers=-1)
        e["traj"] = O.rel_err(out, ref)
        e["state"] = O.pair_err(states, hist[:-1])
        fx = O.admm_tv_backward(x64, lam, RHO, kern, gout, iso, maxit, workers=-1)[0]
        d = np.abs(gx - fx)
        e["gx_l2"] = float(np.linalg.norm(d) / np.linalg.norm(fx))
        e["flips"] = int((d > 1e-4 * np.abs(fx).max()).sum())
    print("%s k=%d N=%d need=%s: %s" % (route_id(shape, iso, lam), k, maxit, need,
                                           "  ".join("%s %.1e" % kv if kv[0] != "flips" else "flips %d" % kv[1]
                                                     for kv in e.items())))
    assert e["step"] <= STEP_TOL and e["out"] <= STEP_TOL and e.get("nmap", 0.0) <= STEP_TOL
    assert e.get("gx", 0.0) <= GRAD_TOL_X
    assert max(e.get("glam", 0.0), e.get("grho", 0.0), e.get("gkern", 0.0)) <= GRAD_TOL_P
    if "traj" in e:
        assert e["traj"] <= TRAJ_TOL and e["state"] <= STATE_TOL
        # iso=True: the block threshold's derivative jumps by tau / n^2 where a pixel's norm crosses tau, and a crossing
        # moves every plane of the pixel, so the end-to-end gradient is printed but not gated (the fp32 numpy oracle
        # itself is 1.8e-3 / 429 elements off at 1x2x1080x512, N=6); the same-state gate above is the sharp one
        if not iso:
            assert e["gx_l2"] <= GRAD_TOL_L2 and e["flips"] <= max(8, x.size // 50000)
    return e


def _cases(table, isos=(False, True), lams=(0.02, -0.02)):
    return [pytest.param(s, k, n, iso, lam, id=route_id(s, iso, lam)) for s, k, n in table for iso in isos for lam in lams]


# b. route matrix: (shape, kernel size, maxit)
ROUTES = [
    ((2, 2, 60, 90), 5, 6), ((1, 2, 45, 63), 3, 1),                                    # generic x generic (odd)
    ((1, 2, 256, 256), 7, 6), ((1, 2, 512, 512), 5, 2),                                # pow2 x pow2, square (HT, WCT)
    ((1, 2, 128, 512), 0, 6), ((2, 1, 512, 256), 3, 1),                                # pow2 x pow2
    ((2, 1, 60, 256), 5, 6), ((1, 2, 6, 512), 3, 2),                                   # pow2 rows x generic cols
    ((1, 2, 256, 96), 5, 6), ((1, 2, 512, 48), 7, 6),                                  # generic rows x pow2 cols / k_cols_adj
    ((1, 2, 100, 1920), 5, 6), ((1, 2, 4, 3840), 3, 2),                                # big rows x generic cols
    ((1, 2, 1080, 48), 5, 6),                                                          # generic rows x big cols
    ((1, 2, 720, 1280), 5, 6), ((1, 2, 1080, 1920), 3, 2),                             # big x big (tile-major)
    ((1, 2, 256, 1920), 5, 2), ((1, 2, 512, 3840), 0, 2),                              # big rows x pow2 cols
    ((1, 2, 1080, 512), 3, 6), ((1, 2, 720, 256), 7, 2),                               # pow2 rows x big cols
]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,k,maxit,iso,lam", _cases(ROUTES) + _cases([((1, 1, 2160, 3840), 7, 4)], isos=(False,)))
def test_route(shape, k, maxit, iso, lam):
    gate(shape, k, maxit, iso, lam)


# c. instantiation sweep: every compiled width / height of the row, column and adjoint kernels, on thin frames
SWEEP = ([((1, 2, 8, W), 3, 3) for W in ROWS_BIG_W] + [((1, 2, H, 16), 3, 3) for H in COLS_BIG_H]
         + [((1, 2, P, P), 3, 3) for P in POW2]                                          # square: HT = W, WCT = H/2
         + [((1, 2, 8, P), 3, 3) for P in POW2]                                          # power-of-two rows, generic columns
         + [((1, 2, 128, 64), 3, 3), ((1, 2, 256, 32), 3, 3), ((1, 2, 512, 32), 3, 3)])  # generic rows, power-of-two columns


@pytest.mark.gpu
@pytest.mark.parametrize("shape,k,maxit,iso,lam", _cases(SWEEP))
def test_instantiation(shape, k, maxit, iso, lam):
    gate(shape, k, maxit, iso, lam)


# d. reductions: more planes than plane groups (64), and the plane-group count capped by the 256 MB rule (4K: 2 groups)
@pytest.mark.gpu
@pytest.mark.parametrize("shape,k,maxit,iso,lam", _cases([((35, 2, 128, 128), 5, 3)], lams=(0.02,))
                         + _cases([((1, 3, 2160, 3840), 5, 3)], isos=(False,), lams=(0.02,)))
def test_reduction(shape, k, maxit, iso, lam):
    gate(shape, k, maxit, iso, lam)


# e. partial gradient requests: need_spec = false (only x or only lambda) and grad_y = NULL
PARTIAL = [((1, 2, 128, 256), 5, 4), ((1, 2, 720, 1280), 5, 3), ((2, 1, 60, 90), 5, 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("need", ["x", "l", "r", "k"])
@pytest.mark.parametrize("shape,k,maxit,iso,lam", _cases(PARTIAL, lams=(0.02,)))
def test_partial_gradients(shape, k, maxit, iso, lam, need):
    gate(shape, k, maxit, iso, lam, need=need)


# f. inference (ROWS_FULL_U: the clamped dual kept as state) against training (q kept, dual recomputed) on one route
INFER = [(1, 1, 256, 256), (1, 2, 128, 512), (1, 1, 100, 1920), (1, 1, 720, 1280)]


@pytest.mark.gpu
@pytest.mark.parametrize("lam", [0.02, -0.02])
@pytest.mark.parametrize("maxit", [2, 3, 8])
@pytest.mark.parametrize("shape", INFER, ids=route_name)
def test_inference_matches_training(shape, maxit, lam):
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    x, kern, _ = _inputs(shape, 5, 11)
    args = lambda rg: (torch.tensor(x, device=dev, requires_grad=rg), torch.tensor([lam], device=dev),
                       torch.tensor([RHO], device=dev), torch.tensor(kern, device=dev), False, maxit)

    def run():
        with torch.no_grad():
            a = fft_admm_tv(*args(False))
        b = fft_admm_tv(*args(True))
        assert b.grad_fn is not None
        torch.cuda.synchronize()
        return a.cpu().numpy(), b.detach().cpu().numpy()

    # the single-launch small-problem solvers (cluster, cooperative) are off: this compares the two-kernel loop's modes
    infer, train = _with_options({"use_cluster": 0, "use_coop": 0}, run)
    e = O.rel_err(infer, train)
    print("%s N=%d lam=%g: inference vs training %.1e" % (route_id(shape, False, lam), maxit, lam, e))
    assert e <= 1e-5


# g. programmatic dependent launch on and off: the same arithmetic, so the same bits
@pytest.mark.gpu
@pytest.mark.parametrize("iso", [False, True])
def test_pdl_does_not_change_results(iso):
    x, kern, gout = _inputs((1, 2, 256, 256), 5, 21)
    run = lambda: _train(x, kern, gout, 0.02, iso, 6, "xlrk")
    a = run()
    b = _with_options({"use_pdl": 0}, run)
    assert np.array_equal(a[0], b[0])
    for ga, gb in zip(a[1], b[1]):
        assert np.array_equal(ga, gb)
    for sa, sb in zip(a[2], b[2]):
        assert np.array_equal(sa[0], sb[0]) and np.array_equal(sa[1], sb[1])
