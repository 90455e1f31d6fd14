"""Drop the sm_100a solver into an existing model built from the reference's classes.

`use_b200_admm(model)` walks a `torch.nn.Module` tree (e.g. the reference's `DivergentRestorer`,
/root/reference/src/admmtor/modelbuild/denoiser.py:7-63, whose level-0 `DivergentAttention` owns two `ADMMDeconv`
layers, modelbuild/blocks.py:187-196) and replaces every reference `ADMMDeconv` (recognised by its class name and the
attributes `w, lmbda, rho, b, iso, max_iters, activation`, elayers/admmdeconv.py:6-64) by this package's `ADMMDeconv`
SHARING the same Parameter / buffer objects: state-dict keys, optimizer references and checkpoints keep working, and
the rest of the model is untouched.  Containers that only loop over solvers (`MultiADMM`, `Deconvs`, `ADMMFusion`) keep
their own forward; swap them for the classes in `elayers.multiadmm` to also get the shared-spectrum fan-out.
"""
from __future__ import annotations

import torch

from .elayers.admmdeconv import ADMMDeconv

__all__ = ["use_b200_admm", "convert_admm_layer"]

_ATTRS = ("w", "lmbda", "rho", "b", "iso", "max_iters", "activation")


def _is_reference_layer(m: torch.nn.Module) -> bool:
    return (type(m).__name__ == "ADMMDeconv" and not isinstance(m, ADMMDeconv)
            and all(hasattr(m, a) for a in _ATTRS))


def convert_admm_layer(ref: torch.nn.Module) -> ADMMDeconv:
    """This package's `ADMMDeconv` with the SAME parameter / buffer tensors as the reference layer `ref`."""
    new = ADMMDeconv.__new__(ADMMDeconv)
    torch.nn.Module.__init__(new)
    for name in ("w", "lmbda", "rho", "b"):
        t = getattr(ref, name)
        if isinstance(t, torch.nn.Parameter):
            new.register_parameter(name, t)
        else:
            new.register_buffer(name, t)
    new.max_iters = ref.max_iters
    new.iso = ref.iso
    new.activation = ref.activation
    new.ckpt_interval = 0
    new.precision = "float32"
    new.train(ref.training)
    return new


def use_b200_admm(model: torch.nn.Module) -> int:
    """Replace, in place, every reference `ADMMDeconv` below `model`.  Returns the number of layers replaced."""
    n = 0
    for parent in list(model.modules()):
        for name, child in list(parent.named_children()):
            if _is_reference_layer(child):
                setattr(parent, name, convert_admm_layer(child))       # ModuleList / ModuleDict support setattr by key
                n += 1
    return n
