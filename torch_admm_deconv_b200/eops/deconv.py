"""Functional layer: `fft_admm_tv` and the small helpers the reference exports beside it.

Mirror of /root/reference/src/admmtor/eops/deconv.py (same names, argument meaning and error
behaviour).  `fft_admm_tv` is the hot path; it is a `torch.autograd.Function` whose forward and
backward hand raw device pointers and the current CUDA stream to libadmm_b200.so (C ABI,
include/admm_b200.h).  PyTorch is used for memory, streams and autograd plumbing only.
"""
from __future__ import annotations

import ctypes
import math
import os
from typing import Optional, Tuple

import torch
import torch.nn.functional as F

from .. import _lib

__all__ = ["fft_admm_tv", "soft_thresh", "block_thresh", "pixelnorm", "hard_thresh", "torch_abs2", "identity",
           "conv_circular", "admm_solve", "activation_code", "shared_spectrum", "fft_admm_tv_cast", "fft_admm_tv_f64"]


# ------------------------------------------------------------------------------------------------
# helpers exported by the reference module (deconv.py:7-32); not on the hot path, kept for import
# compatibility (admmdeconv.py:3 imports `identity`)
# ------------------------------------------------------------------------------------------------
def torch_abs2(x: torch.Tensor) -> torch.Tensor:
    """|x|**2 (reference deconv.py:7-8)."""
    return x.abs().pow(2)


def hard_thresh(x: torch.Tensor, tau) -> torch.Tensor:
    """Keep entries with |x| > tau (reference deconv.py:11-12)."""
    return x * (x.abs() > tau)


def soft_thresh(x: torch.Tensor, tau) -> torch.Tensor:
    """sign(x) * max(|x| - tau, 0) (reference deconv.py:15-16)."""
    return x.sign() * (x.abs() - tau).clamp_min(0)


def pixelnorm(x: torch.Tensor) -> torch.Tensor:
    """sqrt(sum_{batch,channel} x^2 + 1e-15), one value per pixel (reference deconv.py:23-24)."""
    return (x.pow(2).sum(dim=(0, 1)) + 1e-15).sqrt()


def block_thresh(x: torch.Tensor, tau) -> torch.Tensor:
    """max(1 - tau / (pixelnorm(x) + 1e-15), 0) * x (reference deconv.py:19-20)."""
    return (1 - tau / (pixelnorm(x) + 1e-15)).clamp_min(0) * x


def identity(x: torch.Tensor) -> torch.Tensor:
    """Default activation of ADMMDeconv (reference deconv.py:27-28)."""
    return x


def conv_circular(x: torch.Tensor, w: torch.Tensor, pads: Tuple, groups: int) -> torch.Tensor:
    """Circular-padded grouped conv2d (reference deconv.py:31-32).  Not used by the CUDA path."""
    return F.conv2d(F.pad(x, pads, mode="circular"), w, groups=groups)


# ------------------------------------------------------------------------------------------------
# hot path
# ------------------------------------------------------------------------------------------------
def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


_SCALAR_CACHE = {}
_WARNED_DEVICE = set()


def _scalar_param(v, device, name):
    """lmbd / rho reach the kernels as device pointers to one float (never read on the host).  Python numbers are
    uploaded once per (value, device) and cached; a tensor that lives on another device is copied over asynchronously
    with a one-time warning (the reference would raise on the device mismatch: keep parameters on the input's device)."""
    if not torch.is_tensor(v):
        key = (float(v), device.type, device.index)
        t = _SCALAR_CACHE.get(key)
        if t is None:
            if len(_SCALAR_CACHE) > 256:
                _SCALAR_CACHE.clear()
            t = _SCALAR_CACHE[key] = torch.tensor([float(v)], dtype=torch.float32, device=device)
        return t
    if v.numel() != 1:
        raise ValueError("%s must hold exactly one element, got shape %s" % (name, tuple(v.shape)))
    if v.device != device and name not in _WARNED_DEVICE:
        _WARNED_DEVICE.add(name)
        import warnings
        warnings.warn("%s lives on %s but the input on %s: it is copied to the input's device on every call; move the "
                      "module / parameter to that device to avoid the transfer" % (name, v.device, device), stacklevel=3)
    return v


def _prep_kernel(kern: torch.Tensor):
    """Returns (ksize, contiguous fp32 (k,k) tensor or None).  Empty kernel = TV denoise (deconv.py:46,86)."""
    if kern is None or kern.numel() == 0:
        return 0
    if kern.dim() != 4 or kern.shape[0] != 1 or kern.shape[1] != 1:
        raise ValueError("kern must have shape (1, 1, k, k) or be empty, got %s" % (tuple(kern.shape),))
    if kern.shape[2] != kern.shape[3]:
        # the reference builds its circular pads with H/W swapped (deconv.py:90-96 vs :32) and raises a
        # shape RuntimeError for non-square PSFs; keep the same exception type
        raise RuntimeError("non-square PSF %s: the padded conv shapes do not match (square kernels only)"
                           % (tuple(kern.shape[2:]),))
    return int(kern.shape[2])


def _workspace(nbytes: int, device) -> torch.Tensor:
    # torch's caching allocator hands out 512-byte aligned blocks; the library borrows, never owns
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def activation_code(fn) -> Optional[int]:
    """ADMM_ACT_* code of an activation the last kernel of the solve can apply itself, or None (then the Python
    callable runs after the call, as in the reference: admmdeconv.py:64)."""
    if fn is None or fn is identity or isinstance(fn, torch.nn.Identity):
        return _lib.ACT_NONE
    if fn in (torch.relu, F.relu) or (isinstance(fn, torch.nn.ReLU) and not fn.inplace):
        return _lib.ACT_RELU
    if fn in (torch.sigmoid, F.sigmoid) or isinstance(fn, torch.nn.Sigmoid):
        return _lib.ACT_SIGMOID
    if fn in (torch.tanh, F.tanh) or isinstance(fn, torch.nn.Tanh):
        return _lib.ACT_TANH
    return None


def _act_grad(act: int, out: torch.Tensor, g: torch.Tensor) -> torch.Tensor:
    """grad wrt (x + b) from grad wrt act(x + b), using the saved output."""
    if act == _lib.ACT_RELU:
        return g * (out > 0)
    if act == _lib.ACT_SIGMOID:
        return g * out * (1 - out)
    if act == _lib.ACT_TANH:
        return g * (1 - out * out)
    return g


class _AdmmTV(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xin, lmbd, rho, kern, bias, iso, maxit, need_grad, act, out_view, yhat=None, ckpt=0):
        lib = _lib.load()
        B, C, H, W = xin.shape
        dev = xin.device
        ksize = _prep_kernel(kern)
        x = xin.contiguous()
        lam_d = lmbd.detach().to(device=dev, dtype=torch.float32, non_blocking=True).reshape(1).contiguous()
        rho_d = rho.detach().to(device=dev, dtype=torch.float32, non_blocking=True).reshape(1).contiguous()
        kern_d = kern.detach().to(device=dev, dtype=torch.float32).contiguous() if ksize else None
        bias_d = bias.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous() if bias is not None else None
        # `out_view`: a (B, C, H, W) channel slice of a wider contiguous tensor (multi-solver containers write their
        # results straight into the concatenated output); otherwise a fresh dense tensor
        out = out_view if out_view is not None else torch.empty((B, C, H, W), dtype=torch.float32, device=dev)
        ext = _lib.AdmmExt()
        ext.struct_size = ctypes.sizeof(_lib.AdmmExt)
        ext.in_dtype = _lib.IN_U8_DIV255 if x.dtype == torch.uint8 else _lib.IN_F32
        ext.activation = int(act)
        ext.out_batch_stride = int(out.stride(0))
        if yhat is not None:                           # F(y) shared by several solvers on the same input (shared_spectrum)
            ext.yhat_in = yhat.data_ptr()
        with torch.cuda.device(dev):
            ws_bytes = lib.admm_query_workspace(B * C, H, W, ksize, int(iso), maxit)
            if ws_bytes == 0:
                _lib.check(1, "admm_query_workspace")
            ws = _workspace(ws_bytes, dev)
            saved = None
            saved_bytes = 0
            if need_grad:
                if ckpt >= 2:                          # memory-saving training: keep every ckpt-th iteration's state only
                    saved_bytes = lib.admm_query_saved_ex(B * C, H, W, ksize, int(iso), maxit, ckpt)
                    if saved_bytes == 0:               # not available for this problem (iso=True)
                        ckpt = 0
                if ckpt < 2:
                    ckpt = 0
                    saved_bytes = lib.admm_query_saved(B * C, H, W, ksize, int(iso), maxit)
                saved = _workspace(saved_bytes, dev)
                ext.ckpt_interval = ckpt
            stream = torch.cuda.current_stream(dev).cuda_stream
            st = lib.admm_tv_forward_ex(_ptr(x), _ptr(out), _ptr(kern_d), ksize, _ptr(lam_d), _ptr(rho_d), _ptr(bias_d),
                                        B, C, H, W, int(iso), maxit, _ptr(ws), ws.numel(),
                                        _ptr(saved), saved_bytes, ctypes.c_void_p(stream), ctypes.byref(ext))
            _lib.check(st, "admm_tv_forward_ex")
        if need_grad:
            ctx.save_for_backward(x, lam_d, rho_d, kern_d if kern_d is not None else x.new_empty(0, dtype=torch.float32), saved,
                                  out if act != _lib.ACT_NONE else x.new_empty(0, dtype=torch.float32))
            ctx.cfg = (ksize, bool(iso), int(maxit), bias is not None,
                       tuple(kern.shape) if kern is not None else (0,), tuple(lmbd.shape), tuple(rho.shape),
                       tuple(bias.shape) if bias is not None else None, int(act), int(ckpt))
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        lib = _lib.load()
        x, lam_d, rho_d, kern_d, saved, out_saved = ctx.saved_tensors
        ksize, iso, maxit, has_bias, kshape, lshape, rshape, bshape, act, ckpt = ctx.cfg
        B, C, H, W = x.shape
        dev = x.device
        g = grad_out.to(torch.float32)
        if act != _lib.ACT_NONE:                       # fused activation: chain rule with the saved output
            g = _act_grad(act, out_saved, g)
        g = g.contiguous()
        need_x, need_l, need_r, need_k, need_b = ctx.needs_input_grad[:5]
        need_x = need_x and x.dtype == torch.float32
        gx = torch.empty_like(x) if need_x else None
        gl = torch.zeros(1, dtype=torch.float32, device=dev) if need_l else None
        gr = torch.zeros(1, dtype=torch.float32, device=dev) if need_r else None
        gk = torch.zeros(ksize, ksize, dtype=torch.float32, device=dev) if (need_k and ksize) else None
        y = x if x.dtype == torch.float32 else x.to(torch.float32) / 255.0
        with torch.cuda.device(dev):
            ws_bytes = lib.admm_query_workspace_backward_ex(B * C, H, W, ksize, int(iso), maxit, ckpt)
            ws = _workspace(ws_bytes, dev)
            stream = torch.cuda.current_stream(dev).cuda_stream
            st = lib.admm_tv_backward_ex(_ptr(y), _ptr(g), _ptr(kern_d if ksize else None), ksize, _ptr(lam_d), _ptr(rho_d),
                                         B, C, H, W, int(iso), maxit, _ptr(saved), saved.numel(),
                                         _ptr(ws), ws.numel(), _ptr(gx), _ptr(gk), _ptr(gl), _ptr(gr),
                                         ctypes.c_void_p(stream), ckpt)
            _lib.check(st, "admm_tv_backward_ex")
        gb = g.sum().reshape(bshape) if (has_bias and need_b) else None
        return (gx,
                gl.reshape(lshape) if gl is not None else None,
                gr.reshape(rshape) if gr is not None else None,
                gk.reshape(kshape) if gk is not None else None,
                gb, None, None, None, None, None, None, None)


def shared_spectrum(xin: torch.Tensor) -> Optional[torch.Tensor]:
    """F(xin) in the library's packed layout, computed once for several solvers that take the same input
    (`admm_solve(..., yhat=...)`): each of them then skips its own row R2C and column FFT of the input.
    Returns None where the library has no shared-spectrum path (the large-frame column kernels)."""
    lib = _lib.load()
    B, C, H, W = xin.shape
    n = lib.admm_query_yhat(B * C, H, W)
    if n == 0:
        return None
    x = xin.contiguous()
    dev = x.device
    with torch.cuda.device(dev):
        yhat = _workspace(n, dev)
        ws = _workspace(lib.admm_query_workspace(B * C, H, W, 0, 0, 1), dev)
        st = lib.admm_spectrum_forward(_ptr(x), _lib.IN_U8_DIV255 if x.dtype == torch.uint8 else _lib.IN_F32, _ptr(yhat),
                                       B * C, H, W, _ptr(ws), ws.numel(), ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        _lib.check(st, "admm_spectrum_forward")
    return yhat


# Two-stream split of large inference batches.  For iso=False the planes are independent, so the two halves of a batch
# can be solved on two streams: the tail of one half's kernel (a partly filled last wave: cfg2's column pass is 10.4
# waves) and the launch gap behind it are filled by the other half's kernels.  Bit-identical results (each plane's
# arithmetic is unchanged); measured +4.5 % on cfg2 (profiles/README.md).  SPLIT_STREAMS = 1 switches it off.
SPLIT_STREAMS = int(os.environ.get("ADMM_B200_SPLIT_STREAMS", "2"))
SPLIT_MIN_ELEMENTS = 1 << 23          # below ~8 M elements a half no longer fills a few waves
_SIDE_STREAMS = {}


def _side_streams(dev: torch.device, n: int):
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    pool = _SIDE_STREAMS.setdefault(key, [])
    while len(pool) < n:
        pool.append(torch.cuda.Stream(dev))
    return pool[:n]


def _solve_split(xin, lmbd, rho, kern, bias, iso, maxit, code, out):
    """Inference, iso=False: SPLIT_STREAMS contiguous parts of the batch, one on the current stream, the others on cached
    side streams."""
    B, C, H, W = xin.shape
    dev = xin.device
    x = xin.contiguous()
    res = out if out is not None else torch.empty((B, C, H, W), dtype=torch.float32, device=dev)
    n = min(SPLIT_STREAMS, B)
    bounds = [(B * i) // n for i in range(n + 1)]
    cur = torch.cuda.current_stream(dev)
    sides = _side_streams(dev, n - 1)
    for i, side in enumerate(sides, start=1):
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            _AdmmTV.apply(x[bounds[i]:bounds[i + 1]], lmbd, rho, kern, bias, bool(iso), maxit, False, code,
                          res[bounds[i]:bounds[i + 1]], None, 0)
    _AdmmTV.apply(x[:bounds[1]], lmbd, rho, kern, bias, bool(iso), maxit, False, code, res[:bounds[1]], None, 0)
    for side in sides:
        cur.wait_stream(side)
        for t in (x, res, lmbd, rho, kern, bias):
            if torch.is_tensor(t) and t.is_cuda:
                t.record_stream(side)
    return res


def admm_solve(xin: torch.Tensor, lmbd, rho, kern, iso: bool = False, maxit: int = 100,
               bias: Optional[torch.Tensor] = None, activation=None, out: Optional[torch.Tensor] = None,
               yhat: Optional[torch.Tensor] = None, ckpt_interval: int = 0) -> torch.Tensor:
    """`fft_admm_tv` plus the fused pieces of the layer around it: the scalar bias and (for identity / relu / sigmoid /
    tanh) the activation of `ADMMDeconv.forward` (admmdeconv.py:64) are applied by the last kernel of the solve; a uint8
    `xin` is read as `xin / 255.0` (eprocessing/etransforms.py:29-31) by the first kernel; `out`, when given, is a
    (B, C, H, W) float32 channel slice of a wider contiguous tensor that receives the result (containers that
    concatenate several solvers, modelbuild/blocks.py:261).  Any other activation is applied afterwards in Python.

    `ckpt_interval` (training, iso=False): K >= 2 keeps the per-iteration state of every K-th iteration only and lets the
    backward re-run each block of K iterations from its checkpoint (about one extra forward): saved memory drops from
    maxit-1 to (maxit-1)//K + K-1 fields pairs -- 99 -> 19 for 100 iterations at K = 10 (cfg2: 38 GB -> 7.6 GB).
    -1 picks K = ceil(sqrt(maxit - 1)).  0 keeps every iteration (stock-autograd-like memory, fastest backward)."""
    ckpt_interval = int(ckpt_interval)
    if ckpt_interval < 0:
        ckpt_interval = int(math.ceil(math.sqrt(max(int(maxit) - 1, 1))))
    if not torch.is_tensor(xin):
        raise TypeError("xin must be a torch.Tensor")
    if xin.dim() != 4:
        # the reference unpacks `B, C, H_im, W_im = xin.shape` (deconv.py:42) -> ValueError
        raise ValueError("xin must be 4-D (B, C, H, W), got %d-D" % xin.dim())
    if not xin.is_cuda:
        raise RuntimeError("torch_admm_deconv_b200 runs on CUDA (sm_100a) tensors only; there is no CPU fallback")
    if xin.dtype not in (torch.float32, torch.uint8):
        raise TypeError("float32 inputs (or uint8 images, read as x / 255) are supported by the sm_100a kernels (got %s); "
                        "fft_admm_tv_cast is the explicit float32 shim for other floating dtypes" % xin.dtype)
    maxit = int(maxit)
    lmbd = _scalar_param(lmbd, xin.device, "lmbd")
    rho = _scalar_param(rho, xin.device, "rho")
    if kern is None:
        kern = xin.new_empty(0, dtype=torch.float32)
    act = activation_code(activation)
    if out is not None:
        B, C, H, W = xin.shape
        if (out.shape != xin.shape or out.dtype != torch.float32 or out.device != xin.device
                or out.stride()[1:] != (H * W, W, 1) or out.stride(0) < C * H * W):
            raise ValueError("out must be a float32 (B, C, H, W) view with dense images (a channel slice of a contiguous tensor)")
    # decided here because grad mode is always off inside Function.forward
    need_grad = torch.is_grad_enabled() and any(
        torch.is_tensor(t) and t.requires_grad for t in (xin, lmbd, rho, kern, bias))
    code = act if act is not None else _lib.ACT_NONE
    if (SPLIT_STREAMS >= 2 and not need_grad and not iso and act is not None and yhat is None and xin.shape[0] >= 2
            and xin.numel() >= SPLIT_MIN_ELEMENTS and maxit >= 2 and not torch.cuda.is_current_stream_capturing()):
        return _solve_split(xin, lmbd, rho, kern, bias, iso, maxit, code, out)
    if out is not None and (need_grad or act is None):
        # training, or an activation the kernels do not know: solve into a fresh tensor and let autograd track the copy
        # into the slice (plain torch semantics); inference with a known activation writes the slice directly
        res = _AdmmTV.apply(xin, lmbd, rho, kern, bias, bool(iso), maxit, need_grad, code, None, yhat, ckpt_interval)
        out.copy_(res if act is not None else activation(res))
        return out
    res = _AdmmTV.apply(xin, lmbd, rho, kern, bias, bool(iso), maxit, need_grad, code, out, yhat, ckpt_interval)
    return res if act is not None else activation(res)


def fft_admm_tv_cast(xin: torch.Tensor, lmbd, rho, kern, iso: bool = False, maxit: int = 100) -> torch.Tensor:
    """Shim for callers that feed float64 / float16 / bfloat16 tensors (the reference computes in `xin.dtype`,
    deconv.py:50-67): the sm_100a kernels compute in float32, so the input is cast to float32, solved, and the result
    cast back to `xin.dtype`; gradients flow through the casts.  The result then carries float32 accuracy (~1e-6
    relative to a float64 run of the reference), which is why this is an explicit opt-in and `fft_admm_tv` itself
    raises TypeError for other dtypes (INTEGRATION.md, "dtypes").  `fft_admm_tv_f64` solves float64 in double."""
    dt = xin.dtype
    f = lambda t: t.to(torch.float32) if torch.is_tensor(t) and t.is_floating_point() else t
    return fft_admm_tv(f(xin), f(lmbd), f(rho), f(kern), iso, maxit).to(dt)


def fft_admm_tv(xin: torch.Tensor,
                lmbd: torch.Tensor,
                rho: torch.Tensor,
                kern: torch.Tensor,
                iso: bool = False,
                maxit: int = 100) -> torch.Tensor:
    """ADMM total-variation deconvolution / denoising, drop-in for reference deconv.py:35-117.

    xin   (B, C, H, W) float32 CUDA tensor (blurred / noisy image batch)
    lmbd  (1,) tensor, TV weight          rho (1,) tensor, ADMM penalty          tau = lmbd / rho
    kern  (1, 1, k, k) square PSF, or an empty tensor for pure TV denoising (deconv.py:46-47, 86-87)
    iso   False: anisotropic soft threshold; True: block threshold over (batch, channel) (deconv.py:19-24)
    maxit number of ADMM iterations; 0 returns zeros (deconv.py:61, 103, 117)

    Returns the last x iterate, same shape / dtype / device as xin.  Differentiable w.r.t. xin, lmbd,
    rho and kern through a hand-written backward (no autograd graph over the iterations is kept).
    """
    return admm_solve(xin, lmbd, rho, kern, iso, maxit, None)


# ------------------------------------------------------------------------------------------------
# float64 solve (admm_*_f64 of include/admm_b200.h: the generic kernels instantiated for double)
# ------------------------------------------------------------------------------------------------
class _AdmmTV64(torch.autograd.Function):
    """float64 `fft_admm_tv`; every tensor argument is a float64 tensor on xin's device (fft_admm_tv_f64 casts)."""

    @staticmethod
    def forward(ctx, xin, lmbd, rho, kern, iso, maxit, need_grad):
        lib = _lib.load()
        B, C, H, W = xin.shape
        dev = xin.device
        ksize = int(kern.shape[2]) if kern.numel() else 0
        x = xin.contiguous()
        lam_d = lmbd.detach().reshape(1).contiguous()
        rho_d = rho.detach().reshape(1).contiguous()
        kern_d = kern.detach().reshape(ksize, ksize).contiguous() if ksize else None
        out = torch.empty((B, C, H, W), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            ws_bytes = lib.admm_query_workspace_f64(B * C, H, W, ksize, int(iso), maxit)
            if ws_bytes == 0:
                _lib.check(1, "admm_query_workspace_f64")
            ws = _workspace(ws_bytes, dev)
            saved = None
            saved_bytes = 0
            if need_grad:
                saved_bytes = lib.admm_query_saved_f64(B * C, H, W, ksize, int(iso), maxit)
                saved = _workspace(saved_bytes, dev)
            stream = torch.cuda.current_stream(dev).cuda_stream
            st = lib.admm_tv_forward_f64(_ptr(x), _ptr(out), _ptr(kern_d), ksize, _ptr(lam_d), _ptr(rho_d),
                                         B, C, H, W, int(iso), maxit, _ptr(ws), ws.numel(), _ptr(saved), saved_bytes,
                                         ctypes.c_void_p(stream))
            _lib.check(st, "admm_tv_forward_f64")
        if need_grad:
            ctx.save_for_backward(x, lam_d, rho_d, kern_d if kern_d is not None else x.new_empty(0), saved)
            ctx.cfg = (ksize, bool(iso), int(maxit), tuple(kern.shape), tuple(lmbd.shape), tuple(rho.shape))
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        lib = _lib.load()
        x, lam_d, rho_d, kern_d, saved = ctx.saved_tensors
        ksize, iso, maxit, kshape, lshape, rshape = ctx.cfg
        B, C, H, W = x.shape
        dev = x.device
        g = grad_out.to(torch.float64).contiguous()
        need_x, need_l, need_r, need_k = ctx.needs_input_grad[:4]
        gx = torch.empty_like(x) if need_x else None
        gl = torch.zeros(1, dtype=torch.float64, device=dev) if need_l else None
        gr = torch.zeros(1, dtype=torch.float64, device=dev) if need_r else None
        gk = torch.zeros(ksize, ksize, dtype=torch.float64, device=dev) if (need_k and ksize) else None
        with torch.cuda.device(dev):
            ws = _workspace(lib.admm_query_workspace_backward_f64(B * C, H, W, ksize, int(iso), maxit), dev)
            stream = torch.cuda.current_stream(dev).cuda_stream
            st = lib.admm_tv_backward_f64(_ptr(x), _ptr(g), _ptr(kern_d if ksize else None), ksize, _ptr(lam_d), _ptr(rho_d),
                                          B, C, H, W, int(iso), maxit, _ptr(saved), saved.numel(), _ptr(ws), ws.numel(),
                                          _ptr(gx), _ptr(gk), _ptr(gl), _ptr(gr), ctypes.c_void_p(stream))
            _lib.check(st, "admm_tv_backward_f64")
        return (gx,
                gl.reshape(lshape) if gl is not None else None,
                gr.reshape(rshape) if gr is not None else None,
                gk.reshape(kshape) if gk is not None else None,
                None, None, None)


def _f64_scalar(v, device, name):
    if not torch.is_tensor(v):
        return torch.tensor([float(v)], dtype=torch.float64, device=device)
    if v.numel() != 1:
        raise ValueError("%s must hold exactly one element, got shape %s" % (name, tuple(v.shape)))
    return v.to(device=device, dtype=torch.float64)


def fft_admm_tv_f64(xin: torch.Tensor, lmbd, rho, kern, iso: bool = False, maxit: int = 100) -> torch.Tensor:
    """`fft_admm_tv` in float64: the reference's semantics for a float64 `xin` (it computes in xin.dtype,
    deconv.py:50-67), solved in double by the generic sm_100a kernels instantiated for double.

    xin   (B, C, H, W) float64 CUDA tensor (anything else raises TypeError)
    lmbd, rho, kern   as for `fft_admm_tv`, any floating dtype: they are cast to float64 here, so autograd returns their
          gradients in their own dtype
    Differentiable w.r.t. xin, lmbd, rho and kern (hand-written adjoint in double).  Work is enqueued on the current
    stream without a host sync.  Size limits (shared memory of the generic kernels): H <= 4842, and W <= 2905 for
    iso=False (W <= 4842 for iso=True); larger frames raise RuntimeError.  No fused bias / activation / uint8 input."""
    if not torch.is_tensor(xin) or xin.dtype != torch.float64:
        raise TypeError("fft_admm_tv_f64 takes a float64 tensor (got %s); fft_admm_tv is the float32 entry point"
                        % (xin.dtype if torch.is_tensor(xin) else type(xin).__name__))
    if not xin.is_cuda:
        raise TypeError("fft_admm_tv_f64 takes a CUDA tensor: there is no CPU fallback")
    if xin.dim() != 4:
        raise ValueError("xin must be 4-D (B, C, H, W), got %d-D" % xin.dim())
    dev = xin.device
    maxit = int(maxit)
    lmbd = _f64_scalar(lmbd, dev, "lmbd")
    rho = _f64_scalar(rho, dev, "rho")
    if kern is None or kern.numel() == 0:
        kern = xin.new_empty(0)
    else:
        _prep_kernel(kern)                             # shape checks: (1, 1, k, k), square
        kern = kern.to(device=dev, dtype=torch.float64)
    need_grad = torch.is_grad_enabled() and any(t.requires_grad for t in (xin, lmbd, rho, kern))
    return _AdmmTV64.apply(xin, lmbd, rho, kern, bool(iso), maxit, need_grad)
