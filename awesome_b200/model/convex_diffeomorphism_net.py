"""Drop-in for the older diffeomorphism prior ``ConvexDiffeomorphismNet`` (SURVEY a6;
``awesome/model/convex_diffeomorphism_net.py:130-188``): ``nn.Linear(C, C)`` on the coordinates ->
``NormalizingFlow1D`` (alternating two-variable couplings with weight-normalised backbones,
``awesome/model/diffeomorphism_net.py:83-104,208-300``) -> ``ConvexNextNet``.  Same constructor arguments,
``state_dict`` keys / shapes (``diffeo_net.{s,t}.{i}.linear{1,2}.linear.{bias,weight_g,weight_v}``,
``diffeo_net.scale.{i}.{weight,scale.bias,scale.weight_g,scale.weight_v}``) and seed-for-seed initial weights; the
modules below only hold parameters, the arithmetic runs in ``libawb.so`` (``awb_diffeo.cu``)."""
from __future__ import annotations

from typing import Any, Dict, Optional

import numpy as np
import torch
from torch import nn

from .. import _lib as L
from ..core import GridSpecHost, Prior
from .base import _PRECISIONS, ArenaPriorModule, reject_second_order
from .convex_net import ConvexNextNet


class _WN(nn.Module):
    """Holder with the parameters of ``weight_norm(nn.Linear(i, o), dim)``: ``bias, weight_g, weight_v``."""

    def __init__(self, i: int, o: int, dim):
        super().__init__()
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            lin = nn.utils.weight_norm(nn.Linear(i, o), dim=dim)      # same RNG use and (g, v) split as the reference
        self.bias = nn.Parameter(lin.bias.detach().clone())
        self.weight_g = nn.Parameter(lin.weight_g.detach().clone())
        self.weight_v = nn.Parameter(lin.weight_v.detach().clone())


class _WNLinear(nn.Module):
    def __init__(self, i: int, o: int):
        super().__init__()
        self.linear = _WN(i, o, dim=None)


class _SimpleBackbone(nn.Module):
    def __init__(self, in_channels: int = 1, network_width: int = 10):
        super().__init__()
        self.linear1 = _WNLinear(in_channels, network_width)
        self.linear2 = _WNLinear(network_width, in_channels)


class _WNScale(nn.Module):
    def __init__(self):
        super().__init__()
        scale = _WN(1, 1, dim=0)
        torch.empty(1, 1).normal_(0.0, 1.0)        # weights_init_normal writes the derived .weight: RNG only
        with torch.no_grad():
            scale.bias.fill_(0)
        w = torch.tensor([1.0 + 0.01 * torch.randn((1,))])
        self.weight = nn.Parameter(w)               # registered before `scale`, like the reference's state_dict order
        self.scale = scale


class NormalizingFlow1D(nn.Module):
    def __init__(self, num_coupling: int = 4, width: int = 130, in_features: int = 2, backbone: str = "default", **kw):
        super().__init__()
        if backbone != "default":
            raise ValueError("the fused flow implements backbone='default' (SimpleBackbone), as every reference config")
        if num_coupling % in_features != 0:
            raise ValueError(f"Number of coupling layers should be divisible by in_features ({in_features})")
        self.num_coupling, self.width, self.in_features = num_coupling, width, in_features
        self.s = nn.ModuleList([_SimpleBackbone(1, width) for _ in range(num_coupling)])
        self.t = nn.ModuleList([_SimpleBackbone(1, width) for _ in range(num_coupling)])
        self.scale = nn.ModuleList([_WNScale() for _ in range(num_coupling)])


class _Linear(nn.Module):
    def __init__(self, n: int):
        super().__init__()
        lin = nn.Linear(n, n)
        lin.weight.data.normal_(0.0, 1 / np.sqrt(n))
        lin.bias.data.fill_(0)
        self.weight = nn.Parameter(lin.weight.detach().clone())
        self.bias = nn.Parameter(lin.bias.detach().clone())


class ConvexDiffeomorphismNet(ArenaPriorModule):
    def __init__(self, n_hidden: int = 130, n_hidden_layers: int = 1, nf_layers: int = 4, nf_hidden: int = 70,
                 in_features: int = 2, diffeo_args: Optional[Dict[str, Any]] = None, precision: str = "fp32", **kwargs):
        super().__init__(precision=precision)
        reject_second_order("ConvexDiffeomorphismNet", kwargs)
        if in_features != 2:
            raise ValueError("NormalizingFlow1D couples two variables: in_features must be 2")
        self.in_features = self.in_channels = in_features
        self.convex_net = ConvexNextNet(n_hidden=n_hidden, in_features=in_features, n_hidden_layers=n_hidden_layers,
                                        precision=precision)
        da = dict(diffeo_args or {})
        da.setdefault("num_coupling", nf_layers)
        da.setdefault("width", nf_hidden)
        da.setdefault("in_features", in_features)
        self.diffeo_net = NormalizingFlow1D(**da)
        self.linear = _Linear(in_features)
        self._flatten_()

    def _optimizer_group_ids(self):
        """convex_net -> 1, flow -> 0 with the weight-norm gains in their own group 3, linear -> 2."""
        flow = [3 if k.endswith("weight_g") else 0 for k, _ in self.diffeo_net.named_parameters()]
        return [1] * len(list(self.convex_net.parameters())) + flow + [2] * len(list(self.linear.parameters()))

    # ---- affine re-positioning of the prior (convex_diffeomorphism_net.py:43-128)
    def translate(self, from_points: torch.Tensor, to_points: torch.Tensor) -> None:
        """Refit ``linear`` so that ``to_points`` map where ``from_points`` used to (least squares on the affine map)."""
        if from_points.shape != to_points.shape:
            raise ValueError("From and to points must have the same shape.")
        w, b = self.linear.weight, self.linear.bias
        if from_points.shape[0] < w.shape[0]:
            raise ValueError(f"Not enough points to sample from. Need at least {w.shape[0]} points, got {from_points.shape[0]}.")
        to_points = to_points.to(dtype=w.dtype, device=w.device)
        from_points = from_points.to(dtype=w.dtype, device=w.device)
        with torch.no_grad():
            from_transf = from_points @ w.T + b
            X = torch.cat((to_points, torch.ones((to_points.shape[0], 1), device=w.device, dtype=w.dtype)), dim=1)
            theta = torch.linalg.inv(X.T @ X) @ (X.T @ from_transf)
            w.copy_(theta[:-1, :].T)          # in place: the parameters are views into the arena
            b.copy_(theta[-1, :])

    def translate_only_point(self, from_point: torch.Tensor, to_point: torch.Tensor, grid: torch.Tensor) -> None:
        """Shift (no rotation / scale): ``to_point`` (pixel x, y) takes the place of ``from_point`` (``:43-79``)."""
        n = self.in_features
        rf = torch.zeros((n + 1, n), device=from_point.device, dtype=from_point.dtype)
        rt = torch.zeros((n + 1, n), device=to_point.device, dtype=to_point.dtype)
        rf[0], rt[0] = from_point, to_point
        for i in range(n):
            v = torch.zeros(n, device=from_point.device, dtype=from_point.dtype)
            v[i] += 3
            rf[i + 1], rt[i + 1] = rf[0] + v, rt[0] + v
        grid = grid.squeeze()
        rf = grid[..., rf[:, 1].long(), rf[:, 0].long()].T
        rt = grid[..., rt[:, 1].long(), rt[:, 0].long()].T
        self.translate(rf, rt)

    def pretrain(self, *args, **kwargs):
        """``ConvexDiffeomorphismNet.pretrain`` (``:190-475``): per-frame fits with Adam (lr 3e-3), BCE on the
        sigmoid, L2 only on the weight-norm gains, warm start + centre-of-mass re-translation (``:341-348``)."""
        from .. import pretrain as P
        from ..fit import LossConfig
        kwargs.setdefault("lr", 0.003)
        kwargs.setdefault("criterion", LossConfig("bce"))
        kwargs.setdefault("optimizer", "adam")
        kwargs.setdefault("weight_decay_on_weight_g", 5e-5)
        kwargs.setdefault("flow_weight_decay", 0.0)
        state = {"com": None}

        def hook(model, un, spec):
            fg = (un.reshape(spec.H, spec.W) <= 0.5)
            if not bool(fg.any()):
                return
            com = (torch.argwhere(fg).sum(dim=0) / fg.sum()).long()           # (row, col), like the reference's helper
            if state["com"] is not None:
                model.translate_only_point(state["com"].flip(dims=(-1,)), com.flip(dims=(-1,)),
                                           grid=spec.materialize(2, un.device).squeeze())
            state["com"] = com
        kwargs["_warm_start_hook"] = hook
        return P.pretrain(self, *args, **kwargs)

    def pretrain_load_state(self, *args, **kwargs):
        from .. import pretrain as P
        return P.pretrain_load_state(self, *args, **kwargs)

    def _make_prior(self, device) -> Prior:
        d = self.diffeo_net
        return Prior(L.AWB_KIND_DIFFEO_ICNN, self.in_features, self.convex_net.n_hidden, self.convex_net.n_hidden_layers,
                     n_flows=d.num_coupling, flow_hidden=d.width, precision=_PRECISIONS[self.precision])

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self._forward_any(x, self.in_features)

    def get_deformation(self, x: torch.Tensor) -> torch.Tensor:
        """``convex_diffeomorphism_net.py:180-185``: linear -> flow.  ``[B,2,H,W] -> [B,2,H,W]``.  Differentiable w.r.t.
        the parameters (flow and linear; the ICNN's gradients are 0) and ``x``, first order only."""
        squeeze = x.dim() == 3
        if squeeze:
            x = x.unsqueeze(0)
        rows = self._deformation_rows(x)
        B, C_, H, W = x.shape
        out = rows.reshape(B, H, W, C_).permute(0, 3, 1, 2).contiguous()
        return out[0] if squeeze else out
