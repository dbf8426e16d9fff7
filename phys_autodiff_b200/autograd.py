"""A deep network of the library as a ``torch.nn.Module``: losses written in PyTorch train it with ``torch.optim``.

``DeepMLP(ctx, H, hidden_layers)`` holds the parameters ``W1 [H, 4]``, ``b1 [H]``, ``Wh [L-1, H, H]``, ``bh [L-1, H]``,
``W2 [4, H]`` and ``b2 [4]`` (fp32, on the context's device, in ``Context.set_weights_deep``'s layouts).  ``forward(x)``
returns ``y [B, 4]`` and ``forward(x, jacobian=True)`` returns ``(y, J)`` with ``J[i, o, k] = dy_o / dc_k``.  The network,
its Jacobian and the weight gradient run in the library's CUDA kernels:

* forward: ``Context.mlp_forward_deep`` or ``Context.mlp_jacobian_deep``;
* backward: ``Context.mlp_vjp_deep`` when ``J`` received no gradient, else ``Context.mlp_jacobian_vjp_deep``.

PyTorch only evaluates the caller's loss on the B x 20 floats of ``(y, J)``.  Gradients with respect to ``x`` and double
backward are not provided: ``x.requires_grad`` raises.

Weight sync: the kernels read the network the context holds, which ``set_weights_deep`` fills from host arrays.  Before a
forward (and in the backward) the module uploads its parameters unless the context holds exactly this module's current
values, tracked by ``Context.weights_owner`` = (the module's serial number, the parameters' ``_version``s).  So the upload
is one device-to-host copy of the parameters plus host repacking once per optimizer step, and again only when another
module has used the context in between.  The parameters are saved for backward, so an in-place update between forward
and backward (an optimizer step) raises torch's usual error instead of giving a wrong gradient.

``DeepMLP.add_flat_grad(g)`` adds a gradient in the library's flat layout (dW1 | db1 | dWh | dbh | dW2 | db2) from any
fused call (``deep_tangent_points_loss_grad``, ``deep_data_loss_grad``, ...) to the parameters' ``.grad``, so fused terms
and terms written in PyTorch share one optimizer step.
"""
from __future__ import annotations

import itertools

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from .capi import MLPConfig

_SERIAL = itertools.count(1)


class _DeepMLPFunction(torch.autograd.Function):
    """forward: the library's forward (or Jacobian) of the module's network; backward: the matching VJP."""

    @staticmethod
    def forward(fctx, module, jacobian, x, *params):
        module._sync(params)
        c = module.ctx
        fctx.save_for_backward(x, *params)
        fctx.module, fctx.jacobian = module, jacobian
        fctx.set_materialize_grads(False)
        if jacobian:
            return c.mlp_jacobian_deep(x)
        return c.mlp_forward_deep(x)

    @staticmethod
    @once_differentiable
    def backward(fctx, gy, gJ=None):
        x, *params = fctx.saved_tensors   # raises if a parameter was changed in place since the forward
        module = fctx.module
        module._sync(params)
        gy = torch.zeros_like(x) if gy is None else gy.to(torch.float32)
        if fctx.jacobian and gJ is not None:
            g = module.ctx.mlp_jacobian_vjp_deep(x, gy, gJ.to(torch.float32))
        else:
            g = module.ctx.mlp_vjp_deep(x, gy)
        return (None, None, None, *module._split(g))


class DeepMLP(torch.nn.Module):
    """4 -> H -> ... -> H -> 4 (``hidden_layers`` hidden layers, ReLU) evaluated and differentiated by the library.

    ctx: an ``ops.Context``; H: 32, 64 or 128; weights: None (uniform in +-1/sqrt(fan_in), as ``torch.nn.Linear``, from
    torch's generator) or (W1, b1, Wh, bh, W2, b2) in ``set_weights_deep``'s layouts (Wh flat or [L-1, H, H]).
    minus_one_to_one: the coordinate normalisation recorded with the network for the grid calls of the context."""

    def __init__(self, ctx, H: int, hidden_layers: int, weights=None, minus_one_to_one: bool = True):
        super().__init__()
        assert H in (32, 64, 128) and hidden_layers >= 1
        self.ctx, self.H, self.hidden_layers = ctx, H, hidden_layers
        self.cfg = MLPConfig(4, H, 4, minus_one_to_one)
        self._serial = next(_SERIAL)
        nl = hidden_layers - 1
        shapes = [(H, 4), (H,), (nl, H, H), (nl, H), (4, H), (4,)]
        dev = torch.device("cuda", torch.cuda.current_device())
        if weights is None:
            fan = [4, 4, H, H, H, H]
            vals = [(torch.rand(s) * 2 - 1) / np.sqrt(f) for s, f in zip(shapes, fan)]
        else:
            vals = [torch.as_tensor(np.asarray(w if w is not None else np.zeros(0), np.float32)).reshape(s)
                    for w, s in zip(weights, shapes)]
        names = ("W1", "b1", "Wh", "bh", "W2", "b2")
        for n, v in zip(names, vals):
            setattr(self, n, torch.nn.Parameter(v.to(device=dev, dtype=torch.float32).contiguous()))
        self._sizes = [int(np.prod(s)) for s in shapes]
        self._shapes = shapes

    def _params(self):
        return (self.W1, self.b1, self.Wh, self.bh, self.W2, self.b2)

    def _sync(self, params):
        """Upload `params` (this module's parameters) unless the context already holds exactly these values."""
        token = (self._serial, tuple(p._version for p in params))
        if self.ctx.weights_owner == token:
            return
        W1, b1, Wh, bh, W2, b2 = (p.detach().cpu().numpy().reshape(-1) for p in params)
        self.ctx.set_weights_deep(self.cfg, self.hidden_layers, W1, b1, Wh if Wh.size else None, bh if bh.size else None,
                                  W2, b2)
        self.ctx.weights_owner = token

    def _split(self, g):
        """The flat float64 gradient [P] as six fp32 tensors in the parameters' shapes."""
        g = torch.as_tensor(g, device=self.W1.device).to(torch.float32)
        assert g.numel() == sum(self._sizes), (g.numel(), sum(self._sizes))
        return [t.reshape(s) for t, s in zip(torch.split(g, self._sizes), self._shapes)]

    def forward(self, x, jacobian: bool = False):
        """y [B, 4] (jacobian=False) or (y [B, 4], J [B, 4, 4]) at the network inputs x (float32 CUDA tensor [B, 4])."""
        if x.requires_grad:
            raise RuntimeError("DeepMLP: gradients with respect to the inputs x are not provided; pass x without "
                               "requires_grad")
        assert x.dtype == torch.float32 and x.is_cuda and x.shape[-1] == 4, (x.dtype, x.device, x.shape)
        return _DeepMLPFunction.apply(self, bool(jacobian), x.reshape(-1, 4).contiguous(), *self._params())

    def add_flat_grad(self, g) -> None:
        """Add a gradient in the library's flat layout (float64 device tensor or ndarray [P], e.g. the grad of
        Context.deep_tangent_points_loss_grad or deep_data_loss_grad_acc(...)[1:]) to the parameters' .grad."""
        for p, t in zip(self._params(), self._split(g)):
            if p.grad is None:
                p.grad = t.clone()
            else:
                p.grad.add_(t)

    def flat_parameters(self) -> np.ndarray:
        """The parameters in the flat layout of the gradients, float32 on the host."""
        return np.concatenate([p.detach().cpu().numpy().ravel() for p in self._params()])
