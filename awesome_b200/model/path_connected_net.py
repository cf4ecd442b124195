"""Drop-in for the reference's path-connectedness prior: ``PathConnectedNet`` (RealNVP flow o ICNN),
its building blocks (``init_realnvp``, ``PixelizeNet``, ``MinMax``/``get_norm``, ``NormNet``) and the factory
``real_nvp_path_connected_net`` -- same constructor arguments, attributes (``convex_net``, ``flow_net``,
``linear``), ``state_dict`` keys/shapes and seed-for-seed initial weights as
``awesome/model/path_connected_net.py:53-85``, ``awesome/model/net_factory.py:70-176``,
``awesome/model/norm_net.py``, ``awesome/model/pixelize_net.py``, ``awesome/transforms/min_max.py``.
The building blocks only hold parameters; all arithmetic runs in ``libawb.so``."""
from __future__ import annotations

import ctypes as C
from typing import Any, Dict, Literal, Optional, Tuple

import torch
from torch import nn

from .. import _lib as L
from ..core import GridSpecHost, Prior
from .base import _PRECISIONS, Affine, ArenaPriorModule, _InverseFunction, reject_second_order
from .convex_net import ConvexNextNet


# --------------------------------------------------------------------------- flow building blocks
class _MLP(nn.Module):
    """Parameter holder with the keys of normflows ``nets.MLP([C,m,C])``: ``net.0.*``, ``net.2.*``."""

    def __init__(self, channels: int, hidden: int, init_zeros: bool = True, output_scale: Optional[float] = None):
        super().__init__()
        l0 = nn.Linear(channels, hidden)
        l2 = nn.Linear(hidden, channels)
        if init_zeros:
            nn.init.zeros_(l2.weight)
            nn.init.zeros_(l2.bias)
        self.net = nn.ModuleDict({"0": Affine(l0.weight.detach().clone(), l0.bias.detach().clone()),
                                  "2": Affine(l2.weight.detach().clone(), l2.bias.detach().clone())})
        if output_scale is not None:          # normflows ConstScaleLayer behind Linear, LeakyReLU, Linear, Tanh: key ``net.4.scale``
            self.net["4"] = _ConstScale(output_scale)


class _ConstScale(nn.Module):
    def __init__(self, scale: float):
        super().__init__()
        self.register_buffer("scale", torch.tensor(float(scale)))


class _MaskedAffineFlow(nn.Module):
    def __init__(self, b: torch.Tensor, t: _MLP, s: _MLP):
        super().__init__()
        self.register_buffer("b", b.view(1, -1))
        self.s = s          # registration order of normflows: s, then t
        self.t = t


class _ActNorm(nn.Module):
    def __init__(self, channels: int):
        super().__init__()
        self.s = nn.Parameter(torch.zeros(1, channels))
        self.t = nn.Parameter(torch.zeros(1, channels))
        self.register_buffer("data_dep_init_done", torch.tensor(0.0))


class RealNVP(nn.Module):
    """Holder for ``nf.NormalizingFlow(q0, flows, q0)`` built by ``init_realnvp``."""

    def __init__(self, channels: int, hidden_units: int, n_flows: int, output_fn: Optional[str],
                 output_scale: Optional[float] = None):
        super().__init__()
        if output_fn not in (None, "tanh"):
            raise ValueError("the fused flow supports output_fn in (None, 'tanh')")
        if output_scale is not None and not (float(output_scale) > 0):
            raise ValueError("output_scale must be positive")
        self.channels, self.hidden_units, self.n_flows, self.output_fn = channels, hidden_units, n_flows, output_fn
        # normflows nets.MLP appends ConstScaleLayer(output_scale) behind the output_fn (and only when there is one)
        self.output_scale = float(output_scale) if (output_scale is not None and output_fn is not None) else None
        masks = realnvp_masks(channels, n_flows)
        flows = []
        for i in range(n_flows):
            s = _MLP(channels, hidden_units, output_scale=self.output_scale)
            t = _MLP(channels, hidden_units, output_scale=self.output_scale)
            flows += [_MaskedAffineFlow(masks[i], t, s), _ActNorm(channels)]
        self.flows = nn.ModuleList(flows)


def realnvp_masks(channels: int, n_flows: int) -> torch.Tensor:
    """Binary-counting coupling masks (``net_factory.py:86-99``), uint8 ``[n_flows, C]``."""
    vals = torch.arange(1, 2 ** channels - 1)
    bits = 2 ** torch.arange(channels)
    base = (vals.unsqueeze(-1).bitwise_and(bits) != 0).to(torch.uint8)
    n = base.shape[0]
    rep, crop = divmod(n_flows, n)
    masks = torch.zeros((n_flows, channels), dtype=torch.uint8)
    if rep > 0:
        masks[:rep * n] = base.repeat((rep, 1))
    masks[rep * n:] = base[:crop]
    return masks


def init_realnvp(channels: int, height: int = 0, width: int = 0, hidden_units: int = 8, n_flows: int = 6,
                 output_fn: Optional[str] = None, output_scale: Optional[float] = None) -> RealNVP:
    """Same signature as ``net_factory.init_realnvp`` (``net_factory.py:70-114``)."""
    return RealNVP(channels, hidden_units, n_flows, output_fn, output_scale)


class PixelizeNet(nn.Module):
    def __init__(self, network: nn.Module, max_batch_size: Optional[int] = None):
        super().__init__()
        self.network = network
        self.max_batch_size = max_batch_size


class MinMax(nn.Module):
    """``awesome/transforms/min_max.py:21-58``: buffers ``min, max, new_min, new_max``."""

    def __init__(self, new_min=-1, new_max=1, dim=None):
        super().__init__()
        self.register_buffer("min", torch.zeros(1))
        self.register_buffer("max", torch.ones(1))
        self.register_buffer("new_min", torch.tensor(new_min))
        self.register_buffer("new_max", torch.tensor(new_max))
        self.dim = dim
        self.fitted = False

    def fit(self, x: torch.Tensor) -> None:
        self.fitted = True
        mn, mx = x, x
        dims = self.dim if self.dim is not None else tuple(range(x.dim()))
        if isinstance(dims, int):
            dims = (dims,)
        for d in dims:
            mn = mn.min(dim=d, keepdim=True).values
            mx = mx.max(dim=d, keepdim=True).values
        self.min, self.max = mn, mx


class MeanStd(nn.Module):
    """``awesome/transforms/mean_std.py``: buffers ``mean, std``; ``(x - mean) / std`` and back.  The kernels evaluate it as
    the MinMax map from [mean, mean + std] onto [0, 1] (same formula, ``(mean + std) - mean`` instead of ``std``: 1 ulp)."""

    def __init__(self, dim=None):
        super().__init__()
        self.register_buffer("mean", torch.zeros(1))
        self.register_buffer("std", torch.ones(1))
        self.dim = dim
        self.fitted = False

    def fit(self, x: torch.Tensor) -> None:
        self.fitted = True
        self.mean = x.mean(dim=self.dim, keepdim=True)
        self.std = x.std(dim=self.dim, keepdim=True)


def get_norm(norm: Literal["minmax", "meanstd"], **kwargs):
    """``net_factory.get_norm`` (``net_factory.py:116-122``)."""
    if norm == "minmax":
        return MinMax(**kwargs)
    if norm == "meanstd":
        return MeanStd(**kwargs)
    raise ValueError("Invalid norm")


class NormNet(nn.Module):
    def __init__(self, net: nn.Module, norm: nn.Module):
        super().__init__()
        self.net = net
        self.norm = norm


# --------------------------------------------------------------------------- the prior
class _Conv1x1(nn.Module):
    """Holder for ``nn.Conv2d(C, C, 1, groups=C)``: ``weight [C,1,1,1]``, ``bias [C]``, init w=1, b=0."""

    def __init__(self, channels: int):
        super().__init__()
        nn.Conv2d(channels, channels, 1, groups=channels)     # consume the RNG like the reference does
        self.weight = nn.Parameter(torch.ones(channels, 1, 1, 1))
        self.bias = nn.Parameter(torch.zeros(channels))


class PathConnectedNet(ArenaPriorModule):
    def __init__(self, convex_net: ConvexNextNet, flow_net: NormNet, in_channels: int = 2,
                 precision: Optional[str] = None, **kwargs):
        super().__init__(precision=precision or getattr(convex_net, "precision", "fp32"))
        if not isinstance(convex_net, ConvexNextNet):
            raise TypeError("convex_net must be an awesome_b200 ConvexNextNet")
        reject_second_order("PathConnectedNet", {"second_order": kwargs.get("second_order") or convex_net.second_order})
        if not isinstance(flow_net, NormNet) or not isinstance(flow_net.net, PixelizeNet) \
                or not isinstance(flow_net.net.network, RealNVP) or not isinstance(flow_net.norm, (MinMax, MeanStd)):
            raise TypeError("flow_net must be NormNet(PixelizeNet(init_realnvp(...)), MinMax | MeanStd)")
        if convex_net.in_features != in_channels or flow_net.net.network.channels != in_channels:
            raise ValueError("channel mismatch between convex_net, flow_net and in_channels")
        self.in_channels = in_channels
        self.convex_net = convex_net
        self.flow_net = flow_net
        self.linear = _Conv1x1(in_channels)
        self._flatten_()

    def _optimizer_group_ids(self):
        """Arena order is convex_net, flow_net, linear (registration order) -> native groups 1, 0, 2
        (the reference's per-frame optimizer groups: ``path_connected_net.py:923-929``)."""
        return ([1] * len(list(self.convex_net.parameters())) + [0] * len(list(self.flow_net.parameters()))
                + [2] * len(list(self.linear.parameters())))

    # ---- native handle
    @property
    def _rnvp(self) -> RealNVP:
        return self.flow_net.net.network

    def _make_prior(self, device) -> Prior:
        r = self._rnvp
        prior = Prior(L.AWB_KIND_FLOW_ICNN, self.in_channels, self.convex_net.n_hidden,
                      self.convex_net.n_hidden_layers, n_flows=r.n_flows, flow_hidden=r.hidden_units,
                      flow_tanh=(r.output_fn == "tanh"), precision=_PRECISIONS[self.precision])
        self._push_consts(prior)
        return prior

    def _push_consts(self, prior: Prior) -> None:
        norm = self.flow_net.norm
        C_ = self.in_channels
        if isinstance(norm, MeanStd):       # (x - mean) / std  ==  MinMax from [mean, mean + std] onto [0, 1]
            mn = norm.mean.detach().float().reshape(-1).cpu()
            sd = norm.std.detach().float().reshape(-1).cpu()
            mn = mn.expand(C_) if mn.numel() == 1 else mn
            mx = mn + (sd.expand(C_) if sd.numel() == 1 else sd)
            new_min, new_max = 0.0, 1.0
        else:
            mn = norm.min.detach().float().reshape(-1).cpu()
            mx = norm.max.detach().float().reshape(-1).cpu()
            mn = mn.expand(C_) if mn.numel() == 1 else mn
            mx = mx.expand(C_) if mx.numel() == 1 else mx
            new_min, new_max = float(norm.new_min), float(norm.new_max)
        masks = torch.stack([self._rnvp.flows[2 * f].b.reshape(-1) for f in range(self._rnvp.n_flows)])
        prior.set_flow_consts(mn.tolist(), mx.tolist(), new_min, new_max,
                              masks.reshape(-1).to(torch.uint8).cpu().tolist())
        if self._rnvp.output_scale is not None:
            L.check(prior.lib.awb_prior_set_flow_output_scale(prior.handle, self._rnvp.output_scale))
        prior.set_flow_eval(int(getattr(self, "flow_eval", 0)))     # 0 auto / 1 unit loops / 2 segment tables (awb.h)

    def load_state_dict(self, state_dict, *args, **kwargs):
        out = super().load_state_dict(state_dict, *args, **kwargs)
        if self._prior is not None:
            self._push_consts(self._prior)      # MinMax buffers may have changed
        return out

    # ---- reference API
    def reset_parameters(self) -> None:
        self.convex_net.reset_parameters()
        r = self._rnvp
        with torch.no_grad():
            for f in range(r.n_flows):
                fl, an = r.flows[2 * f], r.flows[2 * f + 1]
                for mlp in (fl.s, fl.t):
                    l0 = nn.Linear(r.channels, r.hidden_units)
                    mlp.net["0"].weight.copy_(l0.weight)
                    mlp.net["0"].bias.copy_(l0.bias)
                    mlp.net["2"].weight.zero_()
                    mlp.net["2"].bias.zero_()
                an.s.zero_()
                an.t.zero_()
                an.data_dep_init_done.fill_(0.0)
            self.linear.weight.fill_(1)
            self.linear.bias.fill_(0)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        self._maybe_actnorm_init(x)
        return self._forward_any(x, self.in_channels)

    def enforce_convexity(self) -> None:
        super().enforce_convexity()

    def make_fitter(self, grid, target, loss=None, optim=None, **kw):
        """Fused fit loop on this prior; un-initialised ActNorms get their data-dependent init from ``grid`` first, as the
        reference's first training forward would do (normflows ``ActNorm.forward``)."""
        if isinstance(grid, torch.Tensor):
            grid = GridSpecHost.from_tensor(grid)
        self._ensure_flat()
        r = self._rnvp
        if not all(float(r.flows[2 * f + 1].data_dep_init_done) > 0 for f in range(r.n_flows)):
            self.actnorm_init(grid, use_linear=True)
        return super().make_fitter(grid, target, loss, optim, **kw)

    def get_deformation(self, x: torch.Tensor) -> torch.Tensor:
        """``path_connected_net.py:125-129``: 1x1 conv -> NormNet(flow).  ``[B,C,H,W] -> [B,C,H,W]``.  Differentiable
        w.r.t. the parameters (flow and 1x1 conv; the ICNN's gradients are 0) and ``x``, first order only."""
        squeeze = x.dim() == 3
        if squeeze:
            x = x.unsqueeze(0)
        self._maybe_actnorm_init(x)
        rows = self._deformation_rows(x)
        B, C_, H, W = x.shape
        out = rows.reshape(B, H, W, C_).permute(0, 3, 1, 2).contiguous()
        return out[0] if squeeze else out

    def inverse(self, x: torch.Tensor, *args, **kwargs) -> torch.Tensor:
        """``path_connected_net.py:107-122``: inverse of ``get_deformation``.  ``[B,C,H,W] -> [B,C,H,W]``.  With grad
        mode on and ``x`` or a parameter requiring grad it is differentiable w.r.t. the parameters (flow and 1x1 conv; the
        ICNN's gradients are 0) and ``x``, first order only; otherwise the result carries no autograd graph."""
        squeeze = x.dim() == 3
        if squeeze:
            x = x.unsqueeze(0)
        arena = self._ensure_flat()
        prior = self._prior_for(arena.device)
        x = x.to(arena.device)
        spec = GridSpecHost.from_tensor(x)
        B, C_, H, W = x.shape
        params = self._arena_params()
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params)):
            with torch.cuda.device(arena.device):
                out = _InverseFunction.apply(self, spec, x if x.requires_grad else None, *params)
        else:
            gs = spec.to_c()
            out = torch.empty((spec.n_pixels, C_), dtype=torch.float32, device=arena.device)
            with torch.no_grad(), torch.cuda.device(arena.device):
                L.check(prior.lib.awb_prior_flow_inverse(prior.handle, arena.data_ptr(), C.byref(gs), out.data_ptr(),
                                                         L.stream_ptr()))
        out = out.reshape(B, H, W, C_).permute(0, 3, 1, 2).contiguous()
        return out[0] if squeeze else out

    def _maybe_actnorm_init(self, x: torch.Tensor) -> None:
        """normflows ``ActNorm.forward`` initialises ``s,t`` from the first batch it sees; the same
        happens here the first time the full prior runs with un-initialised ActNorms."""
        r = self._rnvp
        if all(float(r.flows[2 * f + 1].data_dep_init_done) > 0 for f in range(r.n_flows)):
            return
        if x.dim() == 3:
            x = x.unsqueeze(0)
        elif x.dim() == 2:                    # pixel rows [N, C], as forward takes them
            x = x.detach().t().reshape(1, x.shape[1], 1, x.shape[0])
        self.actnorm_init(GridSpecHost.from_tensor(x), use_linear=True)

    def actnorm_init(self, grid: GridSpecHost, use_linear: bool = True) -> None:
        arena = self._ensure_flat()
        prior = self._prior_for(arena.device)
        if not use_linear:
            saved = (self.linear.weight.detach().clone(), self.linear.bias.detach().clone())
            with torch.no_grad():
                self.linear.weight.fill_(1)
                self.linear.bias.fill_(0)
        gs = grid.to_c()
        with torch.no_grad(), torch.cuda.device(arena.device):
            ws = prior.cached_workspace(grid.n_pixels, L.AWB_WS_INFERENCE, arena.device)
            L.check(prior.lib.awb_prior_actnorm_init(prior.handle, arena.data_ptr(), C.byref(gs), ws.data_ptr(),
                                                     ws.numel(), L.stream_ptr()))
            if not use_linear:
                self.linear.weight.copy_(saved[0])
                self.linear.bias.copy_(saved[1])
            for f in range(self._rnvp.n_flows):
                self._rnvp.flows[2 * f + 1].data_dep_init_done.fill_(1.0)

    def learn_flow_identity(self, x: torch.Tensor, lr: float = 1e-2, weight_decay: float = 1e-5,
                            max_iter: int = 1000, device: Optional[torch.device] = None, zoo: Any = None,
                            use_progress_bar: bool = True, batch_size: int = 1) -> torch.Tensor:
        """``path_connected_net.py:155-250``: regress the NormNet-wrapped flow onto its own input with SE("mean") and
        Adamax(lr, weight_decay).  Like the reference, ``max_iter`` passes over a shuffled ``DataLoader`` of the frames of
        ``x`` with ``batch_size`` frames per optimizer step (the frame order comes from the same sampler, hence the same
        global-RNG stream); ``loss_hist[i]`` is the loss of the last batch of pass ``i``.  One frame (every per-frame
        config) or one batch per pass: the whole fit is replayed from CUDA graphs."""
        from ..fit import OptimConfig, FlowIdentityFitter
        if x.dim() == 3:
            x = x.unsqueeze(0)
        if device is not None and self._ensure_flat().device != torch.device(device):
            self.to(device)
        arena = self._ensure_flat()
        x = x.to(arena.device)
        T = x.shape[0]
        bs = max(1, int(batch_size))
        r = self._rnvp
        cfg = OptimConfig("adamax", lr=lr, weight_decay=[weight_decay, 0.0, 0.0, 0.0])
        if T <= bs:                                       # a single batch per pass: frame order inside it is immaterial
            grid = GridSpecHost.from_tensor(x)
            if not all(float(r.flows[2 * f + 1].data_dep_init_done) > 0 for f in range(r.n_flows)):
                self.actnorm_init(grid, use_linear=False)
            fitter = FlowIdentityFitter(self._prior_for(arena.device), arena, grid, cfg)
            hist = fitter.run(max_iter)
            fitter.raise_if_nonfinite()
            return hist.reshape(-1)
        from torch.utils.data import DataLoader, TensorDataset
        loader = DataLoader(TensorDataset(torch.arange(T)), batch_size=bs, shuffle=True)
        prior = self._prior_for(arena.device)
        fitters, stage = {}, {}
        hist = torch.full((max_iter,), float("nan"), device=arena.device)
        for i in range(max_iter):
            for (idx,) in loader:
                nb = int(idx.numel())
                if nb not in fitters:
                    stage[nb] = torch.empty((nb,) + tuple(x.shape[1:]), dtype=torch.float32, device=arena.device)
                    fitters[nb] = FlowIdentityFitter(prior, arena, GridSpecHost.from_tensor(stage[nb]), cfg, use_graph=False)
                    if len(fitters) > 1:                  # every batch size steps the same optimizer
                        fitters[nb].opt_state = next(iter(fitters.values())).opt_state
                torch.index_select(x, 0, idx.to(arena.device), out=stage[nb])
                if not all(float(r.flows[2 * f + 1].data_dep_init_done) > 0 for f in range(r.n_flows)):
                    self.actnorm_init(GridSpecHost.from_tensor(stage[nb]), use_linear=False)   # first batch the flow ever sees
                hist[i] = fitters[nb].run(1)[0, 0]
        next(iter(fitters.values())).raise_if_nonfinite()
        return hist

    def learn_convex_net(self, x: torch.Tensor, unaries: torch.Tensor, mode: Literal["circle", "unaries"] = "unaries",
                         use_deformed_grid: bool = True, lr: float = 1e-3, weight_decay: float = 0,
                         max_iter: int = 1000, device: Optional[torch.device] = None,
                         use_progress_bar: bool = True) -> torch.Tensor:
        """``path_connected_net.py:307-390``: fit the ICNN alone (Adam, SE) on the deformed grid."""
        from ..fit import LossConfig, OptimConfig
        if mode not in ("circle", "unaries"):
            raise ValueError("Mode must be either 'circle' or 'unaries'!")
        if x.dim() == 3:
            x = x.unsqueeze(0)
        if unaries.dim() != 4:
            unaries = unaries.unsqueeze(0)
        arena = self._ensure_flat()
        x = x.to(arena.device)
        if use_deformed_grid:
            with torch.no_grad():                 # a fixed input grid of the ICNN fit: no graph, no training workspace
                x = self.get_deformation(x)
        if mode == "circle":
            unaries = 1 - self.get_unary_circle_approximation(1 - unaries[0])[None, ...].float()
        fitter = self.convex_net.make_fitter(x, unaries.to(arena.device), LossConfig("mse"),
                                             OptimConfig("adam", lr=lr, weight_decay=weight_decay))
        hist = fitter.run(max_iter)
        fitter.raise_if_nonfinite()
        return hist.reshape(-1)

    def create_circle(self, grid_shape: Tuple[int, ...], radius: float, center) -> torch.Tensor:
        """``path_connected_net.py:298-305``, as written there: ``create_coordinate_grid`` returns (x, y) planes and the
        reference unpacks them as ``yy, xx`` -- the centre's row is compared with the column plane.  Kept bit for bit."""
        grid = PathConnectedNet.create_coordinate_grid(grid_shape)
        yy, xx = grid
        return ((yy - center[0]) ** 2 + (xx - center[1]) ** 2) <= radius ** 2

    def get_unary_circle_approximation(self, unaries: torch.Tensor) -> torch.Tensor:
        """``path_connected_net.py:143-152``: disc of the mask's area around its centre of mass."""
        import math
        area = unaries.sum()
        com = torch.argwhere(unaries.squeeze() > 0.).to(dtype=torch.float32).mean(dim=0).cpu()
        radius = math.sqrt(float(area) / math.pi)
        circle = self.create_circle(tuple(unaries.shape[-2:]), radius, com).to(unaries.device)
        if unaries.dim() == 3:
            circle = circle.unsqueeze(0)
        return circle

    def save_state(self, path: str) -> None:
        import os
        os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
        torch.save(self.state_dict(), path)

    def load_state(self, path: str) -> None:
        self.load_state_dict(torch.load(path))

    def pretrain(self, *args, **kwargs):
        """``PretrainableModule.pretrain`` (``path_connected_net.py:472-509``), see ``awesome_b200/pretrain.py``."""
        from .. import pretrain as P
        return P.pretrain(self, *args, **kwargs)

    def pretrain_load_state(self, *args, **kwargs):
        from .. import pretrain as P
        return P.pretrain_load_state(self, *args, **kwargs)

    @classmethod
    def create_coordinate_grid(cls, grid_shape: Tuple[int, ...]) -> torch.Tensor:
        """``path_connected_net.py:252-271``."""
        ar = [torch.arange(s).float() for s in grid_shape]
        grid = torch.stack(torch.meshgrid(*ar, indexing="ij")[::-1])
        if grid.dim() == 4:
            grid = grid.swapaxes(0, 1)
        return grid

    @classmethod
    def create_normalized_grid(cls, grid_shape: Tuple[int, ...]) -> torch.Tensor:
        """``path_connected_net.py:273-296``: per-channel min-max of the integer grid to [0,1]."""
        grid = cls.create_coordinate_grid(grid_shape)
        if grid.dim() == 3:
            grid = grid.unsqueeze(0)
        mn = grid.amin(dim=(0, 2, 3), keepdim=True)
        mx = grid.amax(dim=(0, 2, 3), keepdim=True)
        return (grid - mn) / (mx - mn) * (1.0 - 0.0) + 0.0


class NoisyPathConnectedNet(PathConnectedNet):
    """``awesome/model/noisy_path_connected_net.py``: the spatio-temporal fit with a fraction of the frames' unaries
    replaced by noise (``pretrain_args["noisy_percentage"]``, default 1/3) -- robustness experiment of the paper."""

    def pretrain(self, *args, **kwargs):
        kwargs.setdefault("noisy_percentage", 0.333)
        return super().pretrain(*args, **kwargs)


def real_nvp_path_connected_net(channels: int = 2, hidden_units: int = 130, flow_n_flows: int = 6,
                                flow_output_fn: Optional[str] = None, flow_output_scale: Optional[float] = None,
                                norm: Literal["minmax", "meanstd"] = "minmax", spatial_shape: tuple = (1000, 1000),
                                convex_net_hidden_units: int = 130, convex_net_hidden_layers: int = 2,
                                dtype: torch.dtype = torch.float32, network_type: Optional[type] = None,
                                network_args: Optional[Dict[str, Any]] = None, precision: str = "fp32",
                                **kwargs) -> PathConnectedNet:
    """Same signature and construction order (hence the same RNG stream) as
    ``net_factory.real_nvp_path_connected_net`` (``net_factory.py:124-176``).  The MinMax fit on a
    [0,1] coordinate grid is min=0, max=1 per channel (SURVEY 7.2 item 6), so the 1.2 GB grid the
    reference materialises for C=3 is never built."""
    reject_second_order("real_nvp_path_connected_net", kwargs)
    network_type = network_type or PathConnectedNet
    network_args = network_args or {}
    flow = init_realnvp(channels=channels, hidden_units=hidden_units, output_fn=flow_output_fn,
                        output_scale=flow_output_scale, n_flows=flow_n_flows,
                        height=spatial_shape[0], width=spatial_shape[1])
    nrm = get_norm(norm, dim=(0, 2, 3))
    if isinstance(nrm, MeanStd):
        # fitted like the reference on the normalised coordinate grid of ``spatial_shape`` (net_factory.py:159-165); the grid
        # factorises per axis, so mean / unbiased std per channel follow from the 1-D coordinate vectors (fp64, then fp32)
        dims = tuple(spatial_shape)[::-1][:channels] if channels == 2 else (spatial_shape[-1], spatial_shape[-2], spatial_shape[0])
        total = 1
        for d_ in spatial_shape:
            total *= int(d_)
        means, stds = [], []
        for n_c in dims:
            v = torch.arange(int(n_c), dtype=torch.float64) / max(1, int(n_c) - 1)
            mu = v.mean()
            var = ((v - mu) ** 2).mean() * total / max(1, total - 1)
            means.append(float(mu)); stds.append(float(var.sqrt()))
        nrm.fitted = True
        nrm.mean = torch.tensor(means, dtype=torch.float32).view(1, channels, 1, 1)
        nrm.std = torch.tensor(stds, dtype=torch.float32).view(1, channels, 1, 1)
    else:
        nrm.fitted = True
        nrm.min = torch.zeros(1, channels, 1, 1)
        nrm.max = torch.ones(1, channels, 1, 1)
    norm_flow = NormNet(net=PixelizeNet(flow), norm=nrm)
    return network_type(convex_net=ConvexNextNet(n_hidden=convex_net_hidden_units,
                                                 n_hidden_layers=convex_net_hidden_layers,
                                                 in_features=channels, precision=precision),
                        flow_net=norm_flow, in_channels=channels, **network_args)
