"""`ADMMDeconv` -- nn.Module wrapper, drop-in for /root/reference/src/admmtor/elayers/admmdeconv.py:6-64.

Same constructor arguments, attribute names, parameter-vs-buffer status, state-dict keys (`w`, `lmbda`,
`rho`, `b`) and RNG draw order (w, lmbda, rho, b) as the reference, so reference checkpoints load with
`strict=True` and code that reaches into `.w/.lmbda/.rho` (scripts/train.py:27-38,
modelbuild/eregularizers.py:5-32) keeps working.
"""
from __future__ import annotations

from typing import Callable, Tuple

import torch

from ..eops.deconv import admm_solve, admm_solve_tol, fft_admm_tv_f64, identity

__all__ = ["ADMMDeconv"]


class ADMMDeconv(torch.nn.Module):
    def __init__(self,
                 kern_size: Tuple[int, int],
                 max_iters: int,
                 lmbda: float = None,
                 rho: float = None,
                 iso: bool = True,
                 bias: bool = False,
                 activation: Callable = identity):
        super().__init__()
        # creation order fixes the RNG stream: w -> lmbda -> rho -> b   (admmdeconv.py:17-23)
        if kern_size:                                                # admmdeconv.py:44-51
            self.w = torch.nn.Parameter(torch.empty((1, 1, *kern_size)))
            torch.nn.init.xavier_uniform_(self.w)
        else:
            self.register_buffer("w", torch.tensor([], dtype=torch.float32))
        self.max_iters = max_iters
        self._scalar("lmbda", lmbda)                                 # admmdeconv.py:35-41
        self._scalar("rho", rho)                                     # admmdeconv.py:26-32
        self.iso = iso
        if bias:                                                     # admmdeconv.py:54-60
            self.b = torch.nn.Parameter(torch.empty(1))
            torch.nn.init.uniform_(self.b, a=0.0, b=1.0)
        else:
            self.register_buffer("b", torch.tensor([0], dtype=torch.float32))
        self.activation = activation
        # not a constructor argument of the reference: set `layer.ckpt_interval = K` (or -1 for sqrt(max_iters)) to train
        # with checkpointed state (see admm_solve); 0 keeps the state of every iteration
        self.ckpt_interval = 0
        # not a constructor argument either: `layer.tol = (rtol, atol, check_every)` makes a forward that needs no gradient
        # stop at the first residual check where every plane has converged (admm_solve_tol); the solve's SolveInfo
        # (iterations, residual history) is then kept in `last_solve_info`.  None (default): fixed max_iters
        self.tol = None
        self.last_solve_info = None
        # not a constructor argument either: "float64" solves in double (fft_admm_tv_f64) for a model converted with
        # `.double()`, like the reference does for float64 inputs; "float32" (default) is the fused float32 path
        self.precision = "float32"

    def _scalar(self, name: str, value):
        """Falsy (None or 0) -> learnable U(0,1) Parameter of shape (1,); else a fixed fp32 buffer."""
        if not value:
            p = torch.nn.Parameter(torch.empty(1))
            torch.nn.init.uniform_(p, a=0.0, b=1.0)
            setattr(self, name, p)
        else:
            self.register_buffer(name, torch.tensor([value], dtype=torch.float32))

    def forward(self, x: torch.Tensor, out: torch.Tensor = None, yhat: torch.Tensor = None) -> torch.Tensor:
        precision = getattr(self, "precision", "float32")
        if precision == "float64":
            # admmdeconv.py:63-64 in double: the bias and the activation run in torch (the float64 solve fuses neither)
            if out is not None or yhat is not None:
                raise ValueError("out / yhat are float32-path options; not available with precision = 'float64'")
            return self.activation(fft_admm_tv_f64(x, self.lmbda, self.rho, self.w, self.iso, self.max_iters) + self.b)
        if precision != "float32":
            raise ValueError("ADMMDeconv.precision must be 'float32' or 'float64', got %r" % (precision,))
        # activation(fft_admm_tv(x, lmbda, rho, w, iso, max_iters) + b)   (admmdeconv.py:63-64): the scalar bias and an
        # identity / relu / sigmoid / tanh activation are applied by the last kernel of the solve; any other callable
        # runs afterwards.  A uint8 image batch is read as x / 255 by the first kernel (etransforms.py:29-31).
        tol = getattr(self, "tol", None)
        if tol is not None and out is None and yhat is None and not (torch.is_grad_enabled() and any(
                t.requires_grad for t in (x, self.lmbda, self.rho, self.w, self.b))):
            rtol, atol, check_every = tol
            res, self.last_solve_info = admm_solve_tol(x, self.lmbda, self.rho, self.w, self.iso, self.max_iters, rtol=rtol,
                                                       atol=atol, check_every=check_every, bias=self.b,
                                                       activation=self.activation)
            return res
        return admm_solve(x, self.lmbda, self.rho, self.w, self.iso, self.max_iters, bias=self.b,
                          activation=self.activation, out=out, yhat=yhat, ckpt_interval=getattr(self, "ckpt_interval", 0))

    def extra_repr(self) -> str:
        k = tuple(self.w.shape[2:]) if self.w.numel() else ()
        return "kern_size=%s, max_iters=%s, iso=%s" % (k, self.max_iters, self.iso)
