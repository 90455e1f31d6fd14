"""The generic FFT engine (fft_engine.cuh, k_rows / k_cols of admm_kernels.cu) where it changes shape: lengths with large
prime factors (the O(p^2) generic radix pass), bands and tiles at the shared-memory limit, odd and very short frames, and
the float64 solve, which runs on these kernels only.

a. Stage level: each float32 pass (row R2C and C2R, column FFT both ways, force_generic) against a numpy fp64 FFT of the
   same input.  The bar is tied to a correct fp32 FFT: the GPU error may be at most 4x that of scipy.fft in float32 on
   the same input (floor 1e-7).
b. Solver level, float32: `test_gpu_routes.gate` (one iteration at a time against the fp64 oracle, the same-state
   adjoint) on generic frames.
c. On the generic kernels, `rows_per_band`, `cols_per_tile` and `threads` only move work between threads and CTAs: rows
   always pair as (2j, 2j+1) for R2C / C2R and (2j-1, 2j) for the halo pass, the batch stride only moves data in shared
   memory, and a column FFT does not depend on its tile.  So the training results must be bit-identical.
d. Frames the generic kernels cannot hold are refused before anything is launched, and the next call works.
e. Float64, one iteration at a time: the saved double state replayed by the oracle, and the same-state adjoint.

Every test id names the frame, its largest prime factor (p) and the band height of the generic row pass (R)."""
import ctypes
import re

import numpy as np
import pytest
import scipy.fft as sf
import torch

from oracle import admm_oracle as O
from oracle import packed_layout_model as M
from test_gpu_routes import RHO, _inputs, _rel, _train, _with_options, gate

KMAX = 227 * 1024                     # shared memory of one CTA, bytes (launch_rows_generic / launch_cols_generic)
STAGE_FLOOR = 1e-7
STAGE_FACTOR = 4.0
# float64 one-step gates (e)
STEP_TOL_64 = 1e-12       # replayed state, norm maps, output
GX_TOL_64 = 1e-10         # x-gradient against the same-state adjoint
GP_TOL_64 = 1e-9          # lambda, rho, kernel gradients


def pmax(n):
    """Largest prime factor of n."""
    p, f = 1, 2
    while f * f <= n:
        while n % f == 0:
            p, n = f, n // f
        f += 1
    return max(p, n)


def band_rows(H, W, halo, cbytes=8):
    """Rows per band of the generic row pass (launch_rows_generic with the default rows_per_band), or None if even two
    rows do not fit.  halo: ROWS_FULL (iso=False, maxit >= 2); cbytes: 8 for float2, 16 for double2."""
    h = 2 if halo else 0
    smem = lambda bs: (2 * W * bs + W) * cbytes
    R = max(2, min(16, H + (H & 1))) & ~1
    while True:
        NP = (R + h + 1) // 2
        if smem(NP | 1) <= KMAX or smem(NP) <= KMAX:
            break
        if R <= 2:
            return None
        R -= 2
    while R > 4 and smem(((R + h + 1) // 2) | 1) > 100 * 1024:
        R -= 2
    return R


def regime(shape, halo, cbytes=8):
    H, W = shape[-2:]
    return "%s-p%d-R%s" % ("x".join(map(str, shape)), max(pmax(H), pmax(W)), band_rows(H, W, halo, cbytes))


def case_id(shape, iso, lam, maxit=2, cbytes=8):
    return "%s-%s-%s" % (regime(shape, not iso and maxit > 1, cbytes), "iso" if iso else "aniso",
                         "negtau" if lam < 0 else "postau")


def _dev():
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    return torch.device("cuda:0")


def _p(t):
    return ctypes.c_void_p(t.data_ptr() if t is not None else 0)


def _cerr(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


# ------------------------------------------------------------------------------------------------------- a. stages
STAGE_N = ([6, 10, 12, 18, 30, 45, 240, 720, 1000, 1200, 1600]                 # unrolled radices alone and mixed
           + [7, 49, 11, 121, 77, 143, 2310, 1147, 3024, 4032]                  # generic pass first, last, twice
           + [257, 1021, 2161, 4099, 9677]                                      # large primes
           + [9685])                                                            # stage maximum: 24 N bytes <= 227 KB


def _packed(X, W):
    """Full row DFTs (..., W) -> the packed row spectrum of packed_layout_model.rows_r2c."""
    P = X[..., :(W + 1) // 2].copy()
    P[..., 0] = X[..., 0].real + (1j * X[..., W // 2].real if W % 2 == 0 else 0)
    return P


def _half(P, W):
    """Packed row spectrum -> the W/2+1 half spectrum that irfft takes (rows_c2r of packed_layout_model)."""
    full = np.zeros(P.shape[:-1] + (W // 2 + 1,), dtype=P.dtype)
    full[..., :(W + 1) // 2] = P
    full[..., 0] = P[..., 0].real
    if W % 2 == 0:
        full[..., W // 2] = P[..., 0].imag
    return full


def _stage_gate(name, got, ref, fp32):
    e, es = _cerr(got, ref), _cerr(fp32, ref)
    bar = max(STAGE_FACTOR * es, STAGE_FLOOR)
    print("%s: gpu %.2e  scipy fp32 %.2e  gate %.2e" % (name, e, es, bar))
    return e <= bar, "%s: %.2e > %.2e" % (name, e, bar)


@pytest.mark.gpu
@pytest.mark.parametrize("axis", ["W", "H"])
@pytest.mark.parametrize("n", STAGE_N, ids=lambda n: "n%d-p%d" % (n, pmax(n)))
def test_stage_against_fp32_fft(lib, n, axis):
    """W: row R2C and C2R of length n on 3 planes of 7 rows (odd H: the last pair holds one row).  H: column FFT of
    length n, forward and inverse, on 2 planes of 10 columns (Wc = 5)."""
    from torch_admm_deconv_b200 import _lib
    dev = _dev()
    P, H, W = (3, 7, n) if axis == "W" else (2, n, 10)
    Wc = (W + 1) // 2
    rng = np.random.default_rng(n)
    ws = torch.empty(lib.admm_query_workspace(P, H, W, 0, 0, 1), dtype=torch.uint8, device=dev)
    spec_in = (rng.standard_normal((P, H, Wc)) + 1j * rng.standard_normal((P, H, Wc))).astype(np.complex64)
    st = torch.from_numpy(np.ascontiguousarray(spec_in)).to(dev)
    results = []

    def run(fn):
        try:
            _lib.set_option("force_generic", 1)
            fn()
        finally:
            _lib.set_option("force_generic", 0)
        torch.cuda.synchronize()

    if axis == "W":
        x = rng.standard_normal((P, H, W)).astype(np.float32)
        xt = torch.from_numpy(x).to(dev)
        out = torch.empty(P, H, Wc, dtype=torch.complex64, device=dev)
        run(lambda: _lib.check(lib.admm_dbg_rows_r2c(_p(xt), _p(out), P, H, W, _p(ws), ws.numel(), None), "rows_r2c"))
        results.append(_stage_gate("R2C W=%d" % W, out.cpu().numpy(), M.rows_r2c(x.astype(np.float64)),
                                   _packed(sf.fft(x, axis=-1, workers=-1), W)))
        back = torch.empty(P, H, W, dtype=torch.float32, device=dev)
        run(lambda: _lib.check(lib.admm_dbg_rows_c2r(_p(st), _p(back), P, H, W, _p(ws), ws.numel(), None), "rows_c2r"))
        results.append(_stage_gate("C2R W=%d" % W, back.cpu().numpy(), M.rows_c2r(spec_in.astype(np.complex128), W),
                                   sf.irfft(_half(spec_in, W), n=W, axis=-1, norm="forward", workers=-1)))
    else:
        s64 = spec_in.astype(np.complex128)
        for inv in (0, 1):
            out = torch.empty_like(st)
            run(lambda: _lib.check(lib.admm_dbg_cols_fft(_p(st), _p(out), P, H, W, inv, _p(ws), ws.numel(), None),
                                   "cols_fft"))
            ref = np.fft.ifft(s64, axis=-2, norm="forward") if inv else np.fft.fft(s64, axis=-2)
            fp32 = (sf.ifft(spec_in, axis=-2, norm="forward", workers=-1) if inv
                    else sf.fft(spec_in, axis=-2, workers=-1))
            results.append(_stage_gate("cols %s H=%d" % ("inv" if inv else "fwd", H), out.cpu().numpy(), ref, fp32))
    for ok, msg in results:
        assert ok, msg


# ------------------------------------------------------------------------------------------------------- b. solver
def _cases(table, isos=(False, True), lams=(0.02, -0.02), cbytes=8):
    return [pytest.param(s, k, n, iso, lam, id=case_id(s, iso, lam, n, cbytes)) for s, k, n in table for iso in isos
            for lam in lams]


REALISTIC = [((1, 2, 1079, 1920), 5, 3),          # odd height: generic rows and columns, 1079 = 13 * 83
             ((1, 2, 1000, 1000), 5, 3), ((1, 2, 1200, 1600), 5, 3)]
# a 4K crop with an odd (prime) height, and a 12 MP photo with a factor of 7 on both sides.  One plane, so for iso=True
# with tau < 0 the block threshold is u = tau q / n with n = |q|: the fp32 adjoint forms its derivative from two terms of
# size |tau| / n that cancel ((1 - s) ubar and tau sb q / n^3, iso.cu), and on 8-12 MP some |q| is small enough that x-bar
# is 6e-5 .. 1e-4 from the fp64 adjoint.  That case is a conditioning limit of the fp32 adjoint, left out here.
PHOTOS = [((1, 1, 2161, 3840), 5, 3), ((1, 1, 3024, 4032), 5, 3)]
PRIMES = [((1, 2, 1021, 1031), 5, 3), ((1, 2, 4099, 6), 5, 3), ((1, 2, 6, 4099), 5, 3)]
# the halo row pass at its band and stride edges: R >= 4 with an odd stride up to W = 4150, R = 2 with stride 2 to 5811;
# H = 9: the last band holds one row and its halo wraps to row 0, paired with zero
EDGES = [((1, 2, H, W), 3, 3) for W in (4150, 4151, 5811) for H in (8, 9)]
SHORT = [((1, 2, 3, 90), 3, 4), ((1, 2, 5, 77), 3, 4)]                          # the circular halo spans the image


@pytest.mark.gpu
@pytest.mark.parametrize("shape,k,maxit,iso,lam", _cases(REALISTIC) + _cases(PRIMES) + _cases(SHORT)
                         + _cases(PHOTOS, isos=(False,)) + _cases(PHOTOS, isos=(True,), lams=(0.02,))
                         + _cases(EDGES, isos=(False,))
                         + _cases([((1, 2, 8, 9685), 3, 3)], isos=(True,))            # R2C / C2R at their maximum
                         + _cases([((1, 2, 9685, 16), 3, 3)]))                        # columns at their maximum
def test_generic_solver_one_step(shape, k, maxit, iso, lam):
    gate(shape, k, maxit, iso, lam)


@pytest.mark.gpu
@pytest.mark.parametrize("need", ["x", "l", "r", "k"])
@pytest.mark.parametrize("shape,k,maxit,iso,lam", _cases([((2, 1, 45, 77), 5, 4)], lams=(0.02,)))
def test_generic_partial_gradients(shape, k, maxit, iso, lam, need):
    gate(shape, k, maxit, iso, lam, need=need)


# ------------------------------------------------------------------------------------------ c. schedule options
SCHEDULE = {"rows_per_band": (2, 4, 6, 16, 64), "cols_per_tile": (1, 2, 4, 16, 32), "threads": (32, 96, 256, 1024)}


def _same(a, b):
    """Output, the four gradients and the saved states (and norm maps) of two `_train` runs are bit-identical."""
    (oa, ga, sa, na), (ob, gb, sb, nb) = a, b
    pairs = [(oa, ob)] + [(x, y) for x, y in zip(ga, gb)] + [(x, y) for p, q in zip(sa, sb) for x, y in zip(p, q)]
    pairs += [(x, y) for p, q in zip(na or [], nb or []) for x, y in zip(p, q)]
    return len(sa) == len(sb) and all((x is None and y is None) or np.array_equal(x, y) for x, y in pairs)


@pytest.mark.gpu
@pytest.mark.parametrize("option", list(SCHEDULE))
@pytest.mark.parametrize("shape,k,maxit,iso,lam",
                         _cases([((2, 2, 45, 63), 5, 4), ((1, 2, 1079, 1920), 5, 3), ((1, 2, 9, 4151), 3, 3)]))
def test_schedule_options_bit_identical(shape, k, maxit, iso, lam, option):
    x, kern, gout = _inputs(shape, k, 5)
    run = lambda: _train(x, kern, gout, lam, iso, maxit, "xlrk")
    base = _with_options({"force_generic": 1}, run)
    for v in SCHEDULE[option]:
        assert _same(base, _with_options({"force_generic": 1, option: v}, run)), "%s = %d" % (option, v)


@pytest.mark.gpu
def test_schedule_check_sees_a_one_ulp_tau_change():
    """The comparison of c is not vacuous: moving lambda by one float32 ulp changes the results."""
    x, kern, gout = _inputs((1, 2, 9, 4151), 3, 5)
    lam2 = float(np.nextafter(np.float32(0.02), np.float32(1)))
    a, b = (_with_options({"force_generic": 1}, lambda: _train(x, kern, gout, l, False, 3, "xlrk")) for l in (0.02, lam2))
    assert not _same(a, b)


# ---------------------------------------------------------------------------------------------- d. size limits
def _solve32(shape, iso, maxit, grad=False):
    from torch_admm_deconv_b200 import fft_admm_tv
    dev = _dev()
    x = torch.rand(shape, device=dev, requires_grad=grad)
    return fft_admm_tv(x, torch.tensor([0.02], device=dev), torch.tensor([RHO], device=dev), torch.empty(0, device=dev),
                       iso, maxit)


def _solve64(shape, iso, maxit):
    from torch_admm_deconv_b200 import fft_admm_tv_f64
    dev = _dev()
    d = lambda v: torch.tensor([v], dtype=torch.float64, device=dev)
    return fft_admm_tv_f64(torch.rand(shape, dtype=torch.float64, device=dev), d(0.02), d(RHO),
                           torch.empty(0, dtype=torch.float64, device=dev), iso, maxit)


def _refused(fn, limit):
    from torch_admm_deconv_b200 import _lib
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with pytest.raises(RuntimeError) as e:
        fn()
    torch.cuda.synchronize()
    launched = _lib.launch_count() - n0
    print("refused (%s), %d launches: %s" % (limit, launched, e.value))
    assert launched == 0, "%d kernels were launched before the size was refused" % launched
    assert re.search("does not fit in shared memory.*%s" % limit, str(e.value)), str(e.value)


REFUSE_32 = [((1, 1, 4, 5812), False, 2, "W <= 5811"), ((1, 1, 4, 9686), True, 3, "W <= 9685"),
             ((1, 1, 4, 9686), False, 1, "W <= 9685"), ((1, 1, 9686, 4), False, 3, "H <= 9685"),
             ((1, 1, 9686, 4), True, 1, "H <= 9685")]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,iso,maxit,limit", REFUSE_32,
                         ids=["%s-%s-N%d" % ("x".join(map(str, s)), "iso" if i else "aniso", n) for s, i, n, _ in REFUSE_32])
def test_float32_size_limit_refused_before_launch(shape, iso, maxit, limit):
    _refused(lambda: _solve32(shape, iso, maxit), limit)
    gate((1, 2, 9, 90), 3, 3, iso, 0.02)                          # the next call on the same stream


@pytest.mark.gpu
@pytest.mark.parametrize("shape,limit", [((1, 1, 4, 9686), "W <= 9685"), ((1, 1, 9686, 4), "H <= 9685")],
                         ids=["1x1x4x9686", "1x1x9686x4"])
def test_float32_backward_size_limit_refused_before_launch(lib, shape, limit):
    """The backward checks too (called through the C ABI: the forward would refuse these frames first)."""
    from torch_admm_deconv_b200 import _lib
    dev = _dev()
    B, C, H, W = shape
    y, g = torch.rand(shape, device=dev), torch.rand(shape, device=dev)
    lam, rho, gx = torch.tensor([0.02], device=dev), torch.tensor([RHO], device=dev), torch.empty(shape, device=dev)
    ws = torch.empty(lib.admm_query_workspace_backward(B * C, H, W, 0, 0, 1), dtype=torch.uint8, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def call():
        _lib.check(lib.admm_tv_backward(_p(y), _p(g), None, 0, _p(lam), _p(rho), B, C, H, W, 0, 1, None, 0,
                                        _p(ws), ws.numel(), _p(gx), None, None, None, st), "admm_tv_backward")
    _refused(call, limit)
    gate((1, 2, 9, 90), 3, 3, False, 0.02)


REFUSE_64 = [((1, 1, 4, 2906), False, 2, "W <= 2905"), ((1, 1, 4, 4843), True, 3, "W <= 4842"),
             ((1, 1, 4843, 4), False, 3, "H <= 4842")]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,iso,maxit,limit", REFUSE_64,
                         ids=["%s-%s-N%d" % ("x".join(map(str, s)), "iso" if i else "aniso", n) for s, i, n, _ in REFUSE_64])
def test_float64_size_limit_refused_before_launch(shape, iso, maxit, limit):
    _refused(lambda: _solve64(shape, iso, maxit), limit)
    gate64((1, 2, 9, 90), 3, 3, iso, 0.02)


# --------------------------------------------------------------------------------------------- e. float64 one step
def gate64(shape, k, maxit, iso, lam, seed=3):
    """Training forward and backward of the float64 solve against the fp64 oracle, one iteration at a time: the saved
    double state is replayed (`admm_tv_replay`) and the adjoint is evaluated on it (`admm_tv_backward` overrides)."""
    from test_gpu_f64 import _kern, _state, _t
    from torch_admm_deconv_b200 import fft_admm_tv_f64
    x, kern, gout = _inputs(shape, k, seed)
    x64 = x.astype(np.float64)
    xt, lt, rt, kt = _t(x64, True), _t([lam], True), _t([RHO], True), _kern(kern, bool(np.size(kern)))
    out = fft_admm_tv_f64(xt, lt, rt, kt, iso, maxit)
    states, nm = _state(out, shape, maxit, iso)
    nmaps = [(nm[i, 0], nm[i, 1]) for i in range(maxit - 1)] if iso else None
    (out * _t(gout)).sum().backward()
    torch.cuda.synchronize()
    tau = lam / RHO
    preds, norms, x_out = O.admm_tv_replay(x64, lam, RHO, kern, states, iso, tau, nmaps, workers=-1)
    e = {"step": O.pair_err(states, preds, np.abs(x_out).max()), "out": O.rel_err(out.detach().cpu().numpy(), x_out)}
    if iso:
        e["nmap"] = O.pair_err(nmaps, norms)
    sx, sl, sr, sk = O.admm_tv_backward(x64, lam, RHO, kern, gout, iso, maxit, qs_override=states, tau_override=tau,
                                        nmaps_override=nmaps, workers=-1)
    e["gx"] = O.rel_err(xt.grad.cpu().numpy(), sx)
    e["glam"] = _rel(lt.grad.cpu().numpy()[0], sl)
    e["grho"] = abs(float(rt.grad.cpu().numpy()[0]) - sr) / max(abs(sr), abs(sl) * abs(tau), 1e-300)
    if np.size(kern):
        e["gkern"] = O.rel_err(kt.grad.cpu().numpy(), sk)
    print("%s k=%d N=%d float64: %s" % (case_id(shape, iso, lam, maxit, 16), k, maxit,
                                        "  ".join("%s %.1e" % kv for kv in e.items())))
    assert max(e["step"], e["out"], e.get("nmap", 0.0)) <= STEP_TOL_64
    assert e["gx"] <= GX_TOL_64
    assert max(e["glam"], e["grho"], e.get("gkern", 0.0)) <= GP_TOL_64
    return e


F64_CASES = (_cases([((1, 2, 8, 2905), 3, 3), ((1, 2, 4842, 16), 3, 3), ((1, 2, 1021, 1031), 5, 3),
                     ((1, 2, 1079, 1920), 5, 3), ((1, 2, 256, 256), 5, 3)], cbytes=16)
             + _cases([((1, 2, 8, 4842), 3, 3)], isos=(True,), cbytes=16))       # the iso=True row maximum


@pytest.mark.gpu
@pytest.mark.parametrize("shape,k,maxit,iso,lam", F64_CASES)
def test_float64_one_step(shape, k, maxit, iso, lam):
    gate64(shape, k, maxit, iso, lam)
