"""CPU oracle for the ADMM-TV deconvolution hot path  --  TEST INFRASTRUCTURE ONLY.

This file is a numpy restatement of the reference algorithm
(`/root/reference/src/admmtor/eops/deconv.py:35-117`, `fft_admm_tv`) and of the
module wrapper's epilogue (`/root/reference/src/admmtor/elayers/admmdeconv.py:63-64`).
It is the *checker* for the CUDA path: only `tests/`, `__graft_entry__.smoke()` and the
`cpu_baseline` / `--impl reference` legs of `bench.py` may import it.  The product package
(`torch_admm_deconv_b200`) never imports anything from `oracle/`.

Parity pinning: the reference ships no tests and no golden vectors (SURVEY.md section 4), so
this oracle is pinned against outputs of the *reference itself*, generated in the build
container by `tests/golden/make_golden.py` (which imports `/root/reference/src` unmodified)
and committed under `tests/golden/*.npz`.  `tests/test_oracle.py` checks every function here
against those fixtures (fp64 agreement ~1e-13, fp32 within the reference's own fp32 noise).

Two forms are provided and cross-checked:

* `admm_tv_stencil_form`  -- follows the reference statement by statement: spatial circular
  finite differences, spatial k x k circular correlation `H_t`, `z`/`u` pairs, rfft2/irfft2.
* `admm_tv_spectral_form` -- the reduced-state form the CUDA kernels mirror (SURVEY.md
  appendix A): `H_t` folded into the spectrum once, only `u_x,u_y` persist, `w = q - 2u`.

plus `admm_tv_backward` (SURVEY.md appendix B), the hand-derived adjoint that the CUDA
backward mirrors, itself pinned against reference autograd fixtures.
"""
from __future__ import annotations

import math
from concurrent.futures import ThreadPoolExecutor

import numpy as np

try:  # scipy's pocketfft front-end can use several threads; numpy's cannot.
    import scipy.fft as _sfft
except Exception:  # pragma: no cover
    _sfft = None

__all__ = [
    "soft_thresh", "block_thresh", "pixelnorm", "hard_thresh", "abs2",
    "admm_tv_stencil_form", "admm_tv_spectral_form", "admm_deconv_layer",
    "admm_tv_backward", "admm_tv_replay", "rel_err", "pair_err", "make_psf", "make_blurred",
]


# ----------------------------------------------------------------------------------------
# small operators  (deconv.py:7-24)
# ----------------------------------------------------------------------------------------
def abs2(x):
    """|x|^2  (deconv.py:7-8)."""
    return np.abs(x) ** 2


def hard_thresh(x, tau):
    """x where |x| > tau else 0  (deconv.py:11-12)."""
    return x * (np.abs(x) > tau)


def soft_thresh(x, tau):
    """sign(x) * max(|x| - tau, 0)  (deconv.py:15-16)."""
    return np.sign(x) * np.maximum(np.abs(x) - tau, 0)


def pixelnorm(x):
    """sqrt(sum over dims (0,1) of x^2 + 1e-15): one norm per pixel, shared by the whole
    batch and all channels  (deconv.py:23-24)."""
    return np.sqrt(np.sum(x ** 2, axis=(0, 1)) + x.dtype.type(1e-15))


def block_thresh(x, tau):
    """max(1 - tau / (pixelnorm + 1e-15), 0) * x  (deconv.py:19-20)."""
    return np.maximum(1 - tau / (pixelnorm(x) + x.dtype.type(1e-15)), 0).astype(x.dtype) * x


def rel_err(a, b):
    """Tolerance metric used everywhere: max|a-b| / max|b|  (SURVEY.md section 8c)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    den = np.max(np.abs(b))
    return float(np.max(np.abs(a - b)) / (den if den > 0 else 1.0))


# ----------------------------------------------------------------------------------------
# circular finite differences  (deconv.py:51-52, 69-84; closures Dx, Dy, Dx_t, Dy_t)
# ----------------------------------------------------------------------------------------
def _dx(a):     # a[i,j] - a[i,j-1]      (deconv.py:74-75 with the (1,0,1,0) circular pad)
    return a - np.roll(a, 1, axis=-1)


def _dy(a):     # a[i,j] - a[i-1,j]      (deconv.py:77-78)
    return a - np.roll(a, 1, axis=-2)


def _dxt(a):    # a[i,j] - a[i,j+1]      (deconv.py:80-81, flipped stencil, (0,1,0,1) pad)
    return a - np.roll(a, -1, axis=-1)


def _dyt(a):    # a[i,j] - a[i+1,j]      (deconv.py:83-84)
    return a - np.roll(a, -1, axis=-2)


def _rfft2(a, workers=1):
    if _sfft is not None and workers != 1:
        return _sfft.rfft2(a, axes=(-2, -1), workers=workers)
    return np.fft.rfft2(a, axes=(-2, -1))


def _irfft2(a, s, workers=1):
    if _sfft is not None and workers != 1:
        return _sfft.irfft2(a, s=s, axes=(-2, -1), workers=workers)
    return np.fft.irfft2(a, s=s, axes=(-2, -1))


def _kernel_2d(kern):
    kern = np.asarray(kern)
    if kern.size == 0:
        return None
    if kern.ndim != 4 or kern.shape[0] != 1 or kern.shape[1] != 1:
        raise ValueError("kern must have shape (1,1,k,k) or be empty")
    if kern.shape[2] != kern.shape[3]:
        # the reference builds its pads with H/W swapped (deconv.py:90-96 vs :32) and dies
        # with a shape RuntimeError for non-square kernels
        raise RuntimeError("non-square kernels are not usable in the reference (deconv.py:90-96)")
    return kern[0, 0]


def _h_t_spatial(y, k2d):
    """H_t(y)[i,j] = sum_{a,b} kern[a,b] * y[i+s-a, j+s-b] (circular), s = ceil((k-1)/2).

    Restates `htran` (deconv.py:88-101): circular pad by (floor, ceil) then cross-correlate
    with the 180-degree flipped kernel, i.e. a true convolution re-centred by s."""
    k = k2d.shape[0]
    s = int(math.ceil((k - 1) / 2))
    out = np.zeros_like(y)
    for a in range(k):
        for b in range(k):
            out += k2d[a, b] * np.roll(y, (a - s, b - s), axis=(-2, -1))
    return out


def _freq_terms(H, W, dtype):
    """|delta_dx|^2 + |delta_dy|^2 on the half spectrum  (deconv.py:51-57).

    The reference gets them from rfftn of the two 2x2 stencils zero-padded at the origin:
    |(-1 + e^{-2 pi i v/W})|^2 = 2 - 2 cos(2 pi v / W) and the same along u."""
    v = np.arange(W // 2 + 1, dtype=np.float64)
    u = np.arange(H, dtype=np.float64)
    lx = 2.0 - 2.0 * np.cos(2.0 * np.pi * v / W)
    ly = 2.0 - 2.0 * np.cos(2.0 * np.pi * u / H)
    return (ly[:, None] + lx[None, :]).astype(dtype)


# ----------------------------------------------------------------------------------------
# form 1: statement-by-statement restatement of fft_admm_tv  (deconv.py:35-117)
# ----------------------------------------------------------------------------------------
def admm_tv_stencil_form(xin, lmbd, rho, kern, iso=False, maxit=100):
    """Follows the reference line by line in `xin.dtype` precision (float32 or float64)."""
    xin = np.asarray(xin)
    dt = xin.dtype
    B, C, H, W = xin.shape                                         # deconv.py:42
    lmbd = dt.type(np.asarray(lmbd).reshape(-1)[0])
    rho = dt.type(np.asarray(rho).reshape(-1)[0])
    tau = lmbd / rho                                               # deconv.py:44
    k2d = _kernel_2d(kern)
    if k2d is None:                                                # deconv.py:46-47
        sigma = np.ones((1, 1), dtype=dt)
    else:                                                          # deconv.py:49
        pad = np.zeros((H, W), dtype=dt)
        kk = k2d.shape[0]
        if kk > H or kk > W:
            raise ValueError("kernel larger than image")
        pad[:kk, :kk] = k2d.astype(dt)
        sigma = _rfft2(pad)
    L = _freq_terms(H, W, dt)                                      # deconv.py:51-55
    freq_c = (1 / (abs2(sigma) + rho * L)).astype(dt)              # deconv.py:57
    thresh = block_thresh if iso else soft_thresh                  # deconv.py:59
    x = np.zeros_like(xin)                                         # deconv.py:61-67
    z_x = np.zeros_like(xin); z_y = np.zeros_like(xin)
    u_x = np.zeros_like(xin); u_y = np.zeros_like(xin)
    hty = xin if k2d is None else _h_t_spatial(xin, k2d.astype(dt))   # deconv.py:86-101 (loop-invariant)
    cdt = np.complex64 if dt == np.float32 else np.complex128
    for _ in range(int(maxit)):                                    # deconv.py:103
        rhs = hty + rho * (_dxt(z_x - u_x) + _dyt(z_y - u_y))      # deconv.py:104
        x = _irfft2((freq_c * _rfft2(rhs)).astype(cdt), (H, W)).astype(dt)   # deconv.py:106
        dx_k = _dx(x); dy_k = _dy(x)                               # deconv.py:108-109
        z_x = thresh(dx_k + u_x, tau).astype(dt)                   # deconv.py:111-112
        z_y = thresh(dy_k + u_y, tau).astype(dt)
        u_x = u_x + dx_k - z_x                                     # deconv.py:114-115
        u_y = u_y + dy_k - z_y
    return x                                                       # deconv.py:117


# ----------------------------------------------------------------------------------------
# form 2: reduced-state spectral form (what the CUDA kernels compute)  SURVEY.md appendix A
# ----------------------------------------------------------------------------------------
def _spectral_tables(H, W, k2d, rho, dt):
    """sigma, ph, L, den for one call  (deconv.py:46-57, 88-99)."""
    L = _freq_terms(H, W, np.float64)
    if k2d is None:
        sigma = np.ones((H, W // 2 + 1), dtype=np.complex128)
        ph = np.ones_like(sigma)
    else:
        kk = k2d.shape[0]
        if kk > H or kk > W:
            raise ValueError("kernel larger than image")
        pad = np.zeros((H, W), dtype=np.float64)
        pad[:kk, :kk] = k2d
        sigma = np.fft.rfft2(pad)
        s = int(math.ceil((kk - 1) / 2))
        u = np.arange(H, dtype=np.float64)[:, None]
        v = np.arange(W // 2 + 1, dtype=np.float64)[None, :]
        ph = np.exp(2j * np.pi * s * (u / H + v / W))
    den = np.abs(sigma) ** 2 + float(rho) * L
    return sigma, ph, L, den


def admm_tv_spectral_form(xin, lmbd, rho, kern, iso=False, maxit=100, workers=1,
                          return_state=False):
    """x = F^-1[A + Bm F(Dx^T w_x + Dy^T w_y)],  q = D x + u,  u = q - prox(q),  w = q - 2u.

    Same fixed point iteration as `admm_tv_stencil_form` with z eliminated (z = q - u,
    z - u = q - 2u) and H_t(y) moved into the spectrum: A = sigma*ph*F(y)/den, Bm = rho/den.
    Runs in xin.dtype for the fields; the shared tables are built in float64 and rounded.
    """
    xin = np.asarray(xin)
    dt = xin.dtype
    cdt = np.complex64 if dt == np.float32 else np.complex128
    B, C, H, W = xin.shape
    lam = float(np.asarray(lmbd).reshape(-1)[0]); rh = float(np.asarray(rho).reshape(-1)[0])
    tau = dt.type(dt.type(lam) / dt.type(rh))
    k2d = _kernel_2d(kern)
    k2d64 = None if k2d is None else k2d.astype(np.float64)
    sigma, ph, L, den = _spectral_tables(H, W, k2d64, rh, dt)
    with np.errstate(divide="ignore", invalid="ignore"):
        mul = (sigma * ph / den).astype(cdt)
        Bm = (rh / den).astype(dt)
    A = (mul * _rfft2(xin, workers)).astype(cdt)
    w_x = np.zeros_like(xin); w_y = np.zeros_like(xin)
    u_x = np.zeros_like(xin); u_y = np.zeros_like(xin)
    x = np.zeros_like(xin)
    hist = []
    for _ in range(int(maxit)):
        v = _dxt(w_x) + _dyt(w_y)
        x = _irfft2((A + Bm * _rfft2(v, workers)).astype(cdt), (H, W), workers).astype(dt)
        q_x = _dx(x) + u_x
        q_y = _dy(x) + u_y
        if iso:
            eps = dt.type(1e-15)
            s_x = np.maximum(1 - tau / (pixelnorm(q_x) + eps), 0).astype(dt)
            s_y = np.maximum(1 - tau / (pixelnorm(q_y) + eps), 0).astype(dt)
            u_x = (q_x - s_x * q_x).astype(dt)
            u_y = (q_y - s_y * q_y).astype(dt)
        else:
            u_x = q_x - soft_thresh(q_x, tau)          # = clip(q, -tau, tau) for tau >= 0; sign(q) tau for tau < 0
            u_y = q_y - soft_thresh(q_y, tau)
        w_x = q_x - 2 * u_x
        w_y = q_y - 2 * u_y
        if return_state:
            hist.append((q_x, q_y))
    if return_state:
        return x, hist
    return x


def _dual(q_x, q_y, iso, tau, nmap=None):
    """u = q - prox(q) of one state, in float64.  iso: s = max(1 - tau / (n + eps), 0) with n the pixel norm of q, or
    `nmap` = (n_x, n_y) when given, so the threshold is decided on those numbers."""
    if iso:
        eps = 1e-15
        if nmap is None:
            nmap = (np.sqrt(np.sum(q_x ** 2, (0, 1)) + eps), np.sqrt(np.sum(q_y ** 2, (0, 1)) + eps))
        n_x, n_y = (np.asarray(n, dtype=np.float64) for n in nmap)
        s_x = np.maximum(1 - tau / (n_x + eps), 0); s_y = np.maximum(1 - tau / (n_y + eps), 0)
        return (1 - s_x) * q_x, (1 - s_y) * q_y
    return q_x - soft_thresh(q_x, tau), q_y - soft_thresh(q_y, tau)


def admm_tv_replay(xin, lmbd, rho, kern, states, iso=False, tau=None, nmaps=None, workers=1):
    """One iteration of the reduced-state form, in float64, from each saved state of an implementation under test.

    `states` is the list of pre-threshold (q_x, q_y) after iterations 1 .. N-1 of an N-iteration solve (what a training
    forward saves).  Iteration k+1 is a deterministic function of q_k and y:
        u = q_k - prox(q_k),  v = Dx^T(q_x - 2u_x) + Dy^T(q_y - 2u_y),  x = F^-1[A + Bm F(v)],  q_{k+1} = D x + u.
    Replaying it from the saved q_k takes every threshold decision on the implementation's own numbers, so what remains
    is one iteration's rounding, whatever the sign of tau or the number of iterations (a whole fp32 trajectory with
    tau < 0 can separate from the fp64 one: u jumps by 2|tau| where q changes sign).

    `tau`: the threshold the implementation used (float32(lmbd) / float32(rho) for the float32 solver); default
    lmbd / rho.  `nmaps` (iso): the (n_x, n_y) pixel-norm maps saved with each state; when given, the block threshold
    of state k is decided from them rather than from a recomputed norm.

    Returns (preds, norms, x_out): preds[i] is the prediction of states[i] (q_1 from the zero state, q_{k+1} from
    states[k-1]); norms[i] is the fp64 pixel-norm pair of states[i] (iso; None otherwise); x_out is the output x_N
    predicted from the last state (from the zero state when `states` is empty, N = 1)."""
    x = np.asarray(xin, dtype=np.float64)
    B, C, H, W = x.shape
    lam = float(np.asarray(lmbd).reshape(-1)[0]); rh = float(np.asarray(rho).reshape(-1)[0])
    tau = lam / rh if tau is None else float(tau)
    k2d = _kernel_2d(kern)
    sigma, ph, L, den = _spectral_tables(H, W, None if k2d is None else np.asarray(k2d, dtype=np.float64), rh, np.float64)
    A = sigma * ph * _rfft2(x, workers) / den
    Bm = rh / den
    states = [tuple(np.asarray(t, dtype=np.float64) for t in s) for s in states]

    def step(k):       # x and q after the iteration that consumes states[k - 1] (k = 0: the zero state)
        if k == 0:
            xn = _irfft2(A, (H, W), workers)
            return xn, (_dx(xn), _dy(xn))
        q_x, q_y = states[k - 1]
        u_x, u_y = _dual(q_x, q_y, iso, tau, None if nmaps is None else nmaps[k - 1])
        v = _dxt(q_x - 2 * u_x) + _dyt(q_y - 2 * u_y)
        xn = _irfft2(A + Bm * _rfft2(v, workers), (H, W), workers)
        return xn, (_dx(xn) + u_x, _dy(xn) + u_y)

    preds = [step(k)[1] for k in range(len(states))]
    norms = None
    if iso:
        norms = [(pixelnorm(q_x), pixelnorm(q_y)) for q_x, q_y in states]
    return preds, norms, step(len(states))[0]


def pair_err(got, want, floor=0.0):
    """`rel_err` over a list of field pairs (states or norm maps): max|a-b| over every field / max|b| over every field;
    0 for empty lists.  `floor`: a lower bound of the denominator.  The replay gate passes max|x_N|: q = D x + u is
    formed from x, so its rounding scales with |x|, and a solve that saved only q_1 = D x_1 (max|q_1| ~ 0.4 max|x_1| on
    the test images) would otherwise grade the rounding of x against a smaller scale."""
    if not want:
        return 0.0
    num = max(float(np.max(np.abs(np.asarray(a, np.float64) - b))) for ga, wa in zip(got, want) for a, b in zip(ga, wa))
    den = max([float(floor)] + [float(np.max(np.abs(b))) for wa in want for b in wa])
    return num / (den if den > 0 else 1.0)


def admm_deconv_layer(x, w, lmbda, rho, b, iso=True, max_iters=100, activation=None,
                      form="spectral"):
    """`ADMMDeconv.forward`: activation(fft_admm_tv(x, lmbda, rho, w, iso, max_iters) + b)
    (admmdeconv.py:63-64)."""
    f = admm_tv_spectral_form if form == "spectral" else admm_tv_stencil_form
    out = f(x, lmbda, rho, w, iso, max_iters) + np.asarray(b).astype(np.asarray(x).dtype)
    return out if activation is None else activation(out)


# ----------------------------------------------------------------------------------------
# hand-derived adjoint  (SURVEY.md appendix B; replaces stock autograd over deconv.py:103-115)
# ----------------------------------------------------------------------------------------
def admm_tv_backward(xin, lmbd, rho, kern, grad_out, iso=False, maxit=100, qs_override=None, tau_override=None,
                     nmaps_override=None, workers=1):
    """Returns (grad_xin, grad_lmbd, grad_rho, grad_kern) in float64.

    Reverse sweep over the reduced-state iteration of `admm_tv_spectral_form`.  The forward
    is re-run in float64 keeping q_k; spectra F(v_k) are recomputed in the sweep.

    `qs_override`: optional list of (q_x, q_y) for iterations 1 .. len(list) -- the pre-threshold state an
    implementation under test actually saved (float32).  The soft threshold's derivative 1[|q| < tau] is
    discontinuous, and the iteration drives many q to +-tau (saturated duals in flat regions), so an fp32
    forward decides a handful of borderline masks differently from an fp64 one and each such element changes the
    gradient by O(1) locally -- for ANY fp32 implementation, the reference's included.  With the state given, the
    masks (and the recomputed v_k) are taken from it, which makes the comparison of the adjoint itself sharp;
    `tau_override` is the threshold those masks were decided with (float32(lmbd) / float32(rho)).

    `nmaps_override` (iso): optional list of the (n_x, n_y) pixel-norm maps saved with each state of `qs_override`.
    The block threshold s = max(1 - tau / (n + eps), 0) and its active set s > 0 are then decided from those maps, as
    the aniso masks are decided from the given q.  `workers`: scipy FFT threads, for large frames."""
    xin = np.asarray(xin, dtype=np.float64)
    g = np.asarray(grad_out, dtype=np.float64)
    B, C, H, W = xin.shape
    lam = float(np.asarray(lmbd).reshape(-1)[0]); rh = float(np.asarray(rho).reshape(-1)[0])
    tau = lam / rh
    k2d = _kernel_2d(kern)
    k2d64 = None if k2d is None else np.asarray(k2d, dtype=np.float64)
    sigma, ph, L, den = _spectral_tables(H, W, k2d64, rh, np.float64)
    Bm = rh / den
    Fy = _rfft2(xin, workers)
    A = sigma * ph * Fy / den
    N = int(maxit)
    if N == 0:
        gk = None if k2d is None else np.zeros((1, 1) + k2d.shape)
        return np.zeros_like(xin), 0.0, 0.0, gk
    # forward, keeping q_k and v_k (all but v_0 = 0 are replaced below when the whole state is given)
    w_x = np.zeros_like(xin); w_y = np.zeros_like(xin)
    u_x = np.zeros_like(xin); u_y = np.zeros_like(xin)
    qs = []; vs = []
    eps = 1e-15
    full_override = qs_override is not None and len(qs_override) >= N - 1
    for _ in range(1 if full_override else N):
        v = _dxt(w_x) + _dyt(w_y)
        x = _irfft2(A + Bm * _rfft2(v, workers), (H, W), workers)
        q_x = _dx(x) + u_x; q_y = _dy(x) + u_y
        if iso:
            n_x = np.sqrt(np.sum(q_x ** 2, (0, 1)) + eps); n_y = np.sqrt(np.sum(q_y ** 2, (0, 1)) + eps)
            s_x = np.maximum(1 - tau / (n_x + eps), 0); s_y = np.maximum(1 - tau / (n_y + eps), 0)
            u_x = (1 - s_x) * q_x; u_y = (1 - s_y) * q_y
        else:
            u_x = q_x - soft_thresh(q_x, tau); u_y = q_y - soft_thresh(q_y, tau)
        w_x = q_x - 2 * u_x; w_y = q_y - 2 * u_y
        qs.append((q_x, q_y)); vs.append(v)
    if tau_override is not None:
        tau = float(tau_override)
    nm = [None] * N                                             # per state: (n_x, n_y) to decide the block threshold with
    if qs_override is not None:
        if full_override:
            qs = qs[:1] + [None] * (N - 1); vs = vs[:1] + [None] * (N - 1)
        for k, (oq_x, oq_y) in enumerate(qs_override):
            qs[k] = (np.asarray(oq_x, dtype=np.float64), np.asarray(oq_y, dtype=np.float64))
        if iso and nmaps_override is not None:
            for k, (n_x, n_y) in enumerate(nmaps_override):
                nm[k] = (np.asarray(n_x, dtype=np.float64), np.asarray(n_y, dtype=np.float64))
        for k in range(1, N):                                   # v_k = D^T w(q_k) from the given state
            q_x, q_y = qs[k - 1]
            if iso:
                n_x, n_y = nm[k - 1] or (np.sqrt(np.sum(q_x ** 2, (0, 1)) + eps), np.sqrt(np.sum(q_y ** 2, (0, 1)) + eps))
                s_x = np.maximum(1 - tau / (n_x + eps), 0); s_y = np.maximum(1 - tau / (n_y + eps), 0)
                w_x = (2 * s_x - 1) * q_x; w_y = (2 * s_y - 1) * q_y
            else:
                w_x = 2 * soft_thresh(q_x, tau) - q_x; w_y = 2 * soft_thresh(q_y, tau) - q_y
            vs[k] = _dxt(w_x) + _dyt(w_y)
    # Parseval weights of the half spectrum
    cw = np.full((W // 2 + 1,), 2.0); cw[0] = 1.0
    if W % 2 == 0:
        cw[-1] = 1.0
    xb = g.copy()
    ub = [np.zeros_like(xin), np.zeros_like(xin)]
    wb = [np.zeros_like(xin), np.zeros_like(xin)]
    tau_bar = 0.0
    Gsum = np.zeros_like(A)
    GVsum = np.zeros_like(A)
    # the prox/dual state produced by iteration N is never consumed: start at the last x.
    for k in range(N - 1, -1, -1):
        if k < N - 1:
            # adjoint of (q_k -> u_k, w_k) for the state consumed by iteration k+1
            qb = []
            for f in range(2):
                q = qs[k][f]
                ut = ub[f] - 2 * wb[f]
                if iso:
                    n = nm[k][f] if nm[k] is not None else np.sqrt(np.sum(q ** 2, (0, 1)) + eps)
                    s = np.maximum(1 - tau / (n + eps), 0)
                    act = (s > 0).astype(np.float64)
                    sb = np.sum((2 * wb[f] - ub[f]) * q, (0, 1))
                    qb_f = (2 * s - 1) * wb[f] + (1 - s) * ub[f] + act * sb * tau / (n + eps) ** 2 * q / n
                    tau_bar += float(np.sum(act * sb * (-1.0 / (n + eps))))
                else:
                    m = (np.abs(q) < tau).astype(np.float64)
                    qb_f = wb[f] + m * ut
                    tau_bar += float(np.sum(ut * (1 - m) * np.sign(q)))
                qb.append(qb_f)
            xb = xb + _dxt(qb[0]) + _dyt(qb[1])
            ub = qb
        Fxb = _rfft2(xb, workers)
        G = Fxb / (H * W)                        # adjoint of irfft2 w.r.t. its half-spectrum input (weights cw applied below)
        Gsum += G
        if k > 0:                                # v_0 = 0
            GVsum += np.conj(G) * _rfft2(vs[k], workers)
        vb = _irfft2(Bm * Fxb, (H, W), workers)
        wb = [_dx(vb), _dy(vb)]
        xb = np.zeros_like(xin)
    # G above is F(xbar)/(HW); with Parseval weights cw the pairing <X, G> = sum cw Re(conj(G) X)
    wgt = cw[None, None, None, :]
    gy = _irfft2(np.conj(sigma * ph / den) * Gsum * (H * W), (H, W), workers)
    dA_drho = -A * L / den
    dBm_drho = np.abs(sigma) ** 2 / den ** 2
    rho_bar = float(np.sum(wgt * np.real(np.conj(Gsum) * dA_drho + GVsum * dBm_drho))) - tau_bar * lam / rh ** 2
    lam_bar = tau_bar / rh
    gk = None
    if k2d is not None:
        kk = k2d.shape[0]
        # d/d sigma and d/d conj(sigma) of A = sigma ph Fy / den and Bm = rho/den, den = sigma conj(sigma) + rho L
        T1 = np.conj(Gsum) * ph * Fy / den
        R = np.real((np.conj(Gsum) * A + GVsum * Bm) / den)
        S = np.sum(np.conj(T1) - 2 * R * sigma, axis=(0, 1))
        # sigma = rfft2(pad(kern)):  kbar[a,b] = sum_{u,v} cw Re( S * e^{+2 pi i (ua/H + vb/W)} )
        full = np.fft.irfft2(S * cw[None, :] / np.where(cw[None, :] == 1.0, 1.0, 2.0), s=(H, W)) * (H * W)
        gk = full[:kk, :kk][None, None]
    return gy, lam_bar, rho_bar, gk


# ----------------------------------------------------------------------------------------
# synthetic inputs pinned by SURVEY.md section 8d / BASELINE.md section 2
# ----------------------------------------------------------------------------------------
def make_psf(kind, k, sigma=None):
    """PSFs of the benchmark configs: 'gauss' (normalised Gaussian k x k) and 'motion'
    (uniform horizontal k-tap line in the middle row of a k x k window)."""
    if kind == "gauss":
        r = np.arange(k, dtype=np.float64) - (k - 1) / 2.0
        g = np.exp(-(r ** 2) / (2.0 * float(sigma) ** 2))
        p = np.outer(g, g)
        return (p / p.sum()).astype(np.float32)
    if kind == "motion":
        p = np.zeros((k, k), dtype=np.float64)
        p[k // 2, :] = 1.0 / k
        return p.astype(np.float32)
    raise ValueError(kind)


def make_blurred(shape, psf, seed=1234, noise=0.01):
    """blurred = roll(irfft2(rfft2(sharp) * rfft2(psf, s=(H,W))), (-s,-s)) + noise * randn,
    s = ceil((k-1)/2)  (numpy generator; the torch generator variant lives in bench.py)."""
    rng = np.random.default_rng(seed)
    B, C, H, W = shape
    sharp = rng.random(shape, dtype=np.float32)
    if psf is None:
        blurred = sharp
    else:
        k = psf.shape[0]
        s = int(math.ceil((k - 1) / 2))
        pad = np.zeros((H, W), dtype=np.float32); pad[:k, :k] = psf
        blurred = np.fft.irfft2(np.fft.rfft2(sharp) * np.fft.rfft2(pad), s=(H, W))
        blurred = np.roll(blurred, (-s, -s), axis=(-2, -1))
    blurred = blurred + noise * rng.standard_normal(shape)
    return blurred.astype(np.float32)
