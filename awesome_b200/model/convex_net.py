"""Drop-in for ``awesome.model.convex_net.ConvexNextNet`` / ``ConvexNet`` (input-convex MLP).

Same constructor arguments, ``state_dict`` keys/shapes and initial weights for a given
seed as the reference (``awesome/model/convex_net.py:10-40,134-220``); the arithmetic runs
in ``libawb.so``.

``second_order=True`` (not a reference argument; it changes neither the state_dict nor the initial weights) makes the
coordinate gradient differentiable: ``g = grad(prior(x).sum(), x, create_graph=True)`` followed by a loss on ``g`` (a
gradient penalty) trains the prior, as with the reference's plain-torch module.  Differentiating the parameter gradients
still raises.  With the default, a double backward raises."""
from __future__ import annotations

import math

import torch
from torch import nn

from .. import _lib as L
from ..core import Prior
from .base import _PRECISIONS, Affine, ArenaPriorModule


def _linear_init(out_f: int, in_f: int, bias: bool = True):
    """Consumes the RNG exactly like ``nn.Linear(in_f, out_f, bias)`` does."""
    lin = nn.Linear(in_f, out_f, bias=bias)
    return lin.weight.detach().clone(), (lin.bias.detach().clone() if bias else None)


def _weights_init_uniform(aff: Affine, activation: str) -> None:
    """``weights_init_uniform`` (reference ``awesome/model/real_nvp/resnet_1d.py:24-36``)."""
    with torch.no_grad():
        nn.init.kaiming_uniform_(aff.weight, mode="fan_in", nonlinearity=activation)
        gain = nn.init.calculate_gain(activation, 0)
        fan = nn.init._calculate_correct_fan(aff.weight, "fan_in")
        std = gain / math.sqrt(fan)
        if aff.bias is not None:
            aff.bias.data.uniform_(-std, std)


class SkipBlock(nn.Module):
    """Parameter holder for ``relu(ln(z) + skp(x))`` (``convex_net.py:134-155``)."""

    def __init__(self, in_features=130, out_features=130, in_skip_features=2, **kwargs):
        super().__init__()
        self.ln = Affine(*_linear_init(out_features, in_features, True))
        self.skp = Affine(*_linear_init(out_features, in_skip_features, False))
        self._act = "relu"

    def reset_parameters(self) -> None:
        _weights_init_uniform(self.ln, self._act)
        _weights_init_uniform(self.skp, self._act)


class OutBlock(SkipBlock):
    """``ln(z) + skp(x)`` (``convex_net.py:158-175``)."""

    def __init__(self, in_features=130, out_features=1, in_skip_features=2, **kwargs):
        super().__init__(in_features=in_features, out_features=out_features, in_skip_features=in_skip_features)
        self._act = "linear"


class ConvexNextNet(ArenaPriorModule):
    def __init__(self, n_hidden: int = 130, in_features: int = 2, out_features: int = 1,
                 n_hidden_layers: int = 1, precision: str = "fp32", second_order: bool = False, **kwargs):
        super().__init__(precision=precision, second_order=second_order)
        if out_features != 1:
            raise ValueError("the fused prior supports out_features == 1 (as every reference config)")
        self.n_hidden, self.in_features, self.n_hidden_layers = n_hidden, in_features, n_hidden_layers
        self.input = Affine(*_linear_init(n_hidden, in_features, True))
        self.skip = nn.ModuleList([SkipBlock(in_features=n_hidden, out_features=n_hidden,
                                             in_skip_features=in_features) for _ in range(n_hidden_layers)])
        self.out = OutBlock(in_features=n_hidden, out_features=out_features, in_skip_features=in_features)
        self._flatten_()

    def _make_prior(self, device) -> Prior:
        return Prior(L.AWB_KIND_ICNN, self.in_features, self.n_hidden, self.n_hidden_layers,
                     precision=_PRECISIONS[self.precision])

    def reset_parameters(self) -> bool:
        _weights_init_uniform(self.input, "linear")
        for blk in self.skip:
            blk.reset_parameters()
        self.out.reset_parameters()
        return True

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self._forward_any(x, self.in_features)


class ConvexNet(ArenaPriorModule):
    """Older naming (``convex_net.py:10-40``): same network as ``ConvexNextNet(n_hidden_layers=1)``
    with keys ``W0y, W1z, W2z, W1y, W2y``; clamps ``W1z.weight`` and ``W2z.weight``."""

    def __init__(self, n_hidden: int = 130, in_channels: int = 2, precision: str = "fp32", second_order: bool = False,
                 **kwargs):
        super().__init__(precision=precision, second_order=second_order)
        in_features, out_features = in_channels, 1
        self.n_hidden, self.in_features = n_hidden, in_features
        # reference registration order: W0y, W1z, W2z, W1y, W2y
        self.W0y = Affine(*_linear_init(n_hidden, in_features, True))
        self.W1z = Affine(*_linear_init(n_hidden, n_hidden, True))
        self.W2z = Affine(*_linear_init(out_features, n_hidden, True))
        self.W1y = Affine(*_linear_init(n_hidden, in_features, False))
        self.W2y = Affine(*_linear_init(out_features, in_features, False))
        self._flatten_()

    def _arena_params(self):
        # arena order must be the ICNN order of libawb: input, ln, ln.bias, skp, out.ln, out.bias, out.skp
        return [self.W0y.weight, self.W0y.bias, self.W1z.weight, self.W1z.bias, self.W1y.weight,
                self.W2z.weight, self.W2z.bias, self.W2y.weight]

    def _make_prior(self, device) -> Prior:
        return Prior(L.AWB_KIND_ICNN, self.in_features, self.n_hidden, 1, precision=_PRECISIONS[self.precision])

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self._forward_any(x, self.in_features)
