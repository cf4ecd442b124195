"""Star-shape prior (SURVEY a16): drop-in for the notebook class ``myNet``
(``notebooks/icml_teaser_code/star_shaped/star.ipynb`` cell 2) -- same constructor argument, parameter names
(``offset, W0, W1, W2, W1_r, W2_r``), initial weights for a given seed and ``forward(x[n,2]) -> [n,1]`` -- with the
training loop of cell 3 as fused native steps (``StarFitter``).  It also takes ``[B,2,H,W]`` grids and fits whole frames
with ``make_fitter(grid, target, loss, optim)`` (``PriorFitter``; weight maps, ignore label, ``fit_frames``).

``forward`` is differentiable w.r.t. the parameters and the points (``awb_star_forward`` / ``awb_star_backward``), so
the notebook's own loop (``loss = mse(sigmoid(net(x)), t); loss.backward(); optimizer.step()``), a custom loss or a
gradient w.r.t. ``x`` work as with the plain-torch class.  First order only: a double backward raises.  A point at
exactly ``-offset`` gets ``dx = 0`` (torch's ``sqrt`` backward gives NaN there; see ``include/awb.h``)."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
from torch import nn

from .. import _lib as L
from ..core import GridSpecHost, Prior
from .base import Affine, ArenaPriorModule, _first_order_only, _split_grads, reject_second_order


def _lin(i: int, o: int) -> Affine:
    l = nn.Linear(i, o)
    return Affine(l.weight.detach().clone(), l.bias.detach().clone())


class _StarFunction(torch.autograd.Function):
    """``apply(module, x, *params)``: the parameters are inputs so that autograd routes their gradients.  The forward is
    ``awb_star_forward`` whether or not a graph is built (same bits); the backward is ``awb_star_backward``."""

    @staticmethod
    def forward(ctx, module, x, *params):
        prior = module._prior_for(x.device)
        arena = module._arena
        xs = x.detach().contiguous().float()
        out = torch.empty(xs.shape[0], dtype=torch.float32, device=x.device)
        L.check(prior.lib.awb_star_forward(prior.handle, arena.data_ptr(), xs.data_ptr(), xs.shape[0], out.data_ptr(),
                                           L.stream_ptr()))
        ctx.module, ctx.prior, ctx.x_dtype = module, prior, x.dtype
        ctx.shapes = [p.shape for p in params]
        ctx.save_for_backward(xs, *params)    # params: autograd refuses a backward after they were modified in place
        return out.reshape(-1, 1)

    @staticmethod
    @_first_order_only
    def backward(ctx, dy):
        xs = ctx.saved_tensors[0]
        prior, arena, n = ctx.prior, ctx.module._arena, xs.shape[0]
        dy = dy.detach().reshape(-1).contiguous().float()
        grads = torch.empty(arena.numel(), dtype=torch.float32, device=xs.device)
        dx = torch.empty_like(xs) if ctx.needs_input_grad[1] else None
        ws = torch.empty(int(prior.lib.awb_star_backward_workspace_bytes(prior.handle, n)), dtype=torch.uint8,
                         device=xs.device)
        L.check(prior.lib.awb_star_backward(prior.handle, arena.data_ptr(), xs.data_ptr(), n, dy.data_ptr(),
                                            grads.data_ptr(), dx.data_ptr() if dx is not None else None, ws.data_ptr(),
                                            ws.numel(), L.stream_ptr()))
        pgrads = tuple(g if need else None for g, need in zip(_split_grads(grads, ctx.shapes), ctx.needs_input_grad[2:]))
        return (None, dx.to(ctx.x_dtype) if dx is not None else None) + pgrads


class StarShapedNet(ArenaPriorModule):
    def __init__(self, n_hidden: int = 150, **kwargs):
        super().__init__(precision="fp32")
        reject_second_order("StarShapedNet", kwargs)
        self.n_hidden = n_hidden
        self.offset = nn.Parameter(torch.zeros(1, 2))
        self.offset.requires_grad = False            # the notebook unfreezes it at epoch 1000
        self.W0 = _lin(2, n_hidden)
        self.W1 = _lin(n_hidden, n_hidden)
        self.W2 = _lin(n_hidden, 1)
        self.W1_r = _lin(1, n_hidden)
        self.W2_r = _lin(n_hidden, 1)
        self._flatten_()

    def _make_prior(self, device) -> Prior:
        return Prior(L.AWB_KIND_STAR, 2, self.n_hidden, 0)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """Native forward, differentiable w.r.t. the parameters and ``x``: points ``[n,2]`` -> ``[n,1]``, a grid
        ``[B,2,H,W]`` -> ``[B,1,H,W]`` or ``[2,H,W]`` -> ``[1,H,W]`` (pixel rows in ``(b, h, w)`` order through the same
        kernels: a grid and its rows give the same bits).  ``make_fitter`` runs fused fit steps."""
        if x.dim() == 2:
            if x.shape[1] != 2:
                raise ValueError(f"expected [n,2] points, got {tuple(x.shape)}")
            return self._points(x)
        squeeze = x.dim() == 3
        g = x.unsqueeze(0) if squeeze else x
        if g.dim() != 4 or g.shape[1] != 2:
            raise ValueError(f"expected [n,2] points or a [B,2,H,W] grid, got {tuple(x.shape)}")
        B, _, H, W = g.shape
        y = self._points(g.permute(0, 2, 3, 1).reshape(-1, 2)).reshape(B, H, W, 1).permute(0, 3, 1, 2)
        return y[0] if squeeze else y

    def _points(self, x: torch.Tensor) -> torch.Tensor:
        if not x.is_cuda:
            raise L.AwbLibraryError("awesome_b200 priors run on CUDA only (no CPU fallback)")
        self._ensure_flat()
        with torch.cuda.device(x.device):
            return _StarFunction.apply(self, x, *self._arena_params())

    @staticmethod
    def create_grid(H: int, W: int, B: int = 1, device=None) -> torch.Tensor:
        """``[B,2,H,W]`` coordinates of an ``H x W`` likelihood image as ``fit_likelihood`` samples them (the notebook's
        cell 3): channel 0 = ``i / (H - 1) - 0.5`` (row), channel 1 = ``j / (W - 1) - 0.5`` (column)."""
        if H < 2 or W < 2:
            raise ValueError(f"the notebook's coordinates need H, W >= 2, got {H}x{W}")
        i = torch.arange(H, device=device) / (H - 1) - 0.5
        j = torch.arange(W, device=device) / (W - 1) - 0.5
        ii, jj = torch.meshgrid(i, j, indexing="ij")
        return torch.stack([ii, jj], 0).float().unsqueeze(0).expand(B, 2, H, W).contiguous()

    def reset_parameters(self) -> None:
        """Draw the weights again as the constructor does (``nn.Linear`` init, same order), in place in the arena; the
        offset goes back to 0 and keeps its ``requires_grad``.  ``fit_frames`` calls it before a retry."""
        self._ensure_flat()
        h = self.n_hidden
        fresh = [_lin(2, h), _lin(h, h), _lin(h, 1), _lin(1, h), _lin(h, 1)]
        with torch.no_grad():
            self.offset.zero_()
            for mod, new in zip((self.W0, self.W1, self.W2, self.W1_r, self.W2_r), fresh):
                mod.weight.copy_(new.weight)
                mod.bias.copy_(new.bias)

    def enforce_convexity(self) -> None:
        """The notebook's projection: ``W2_r.weight <- relu(W2_r.weight)`` (cell 3)."""
        with torch.no_grad():
            self.W2_r.weight.clamp_(min=0)

    def make_fitter(self, grid=None, target=None, loss=None, optim=None, **kw):
        """With a ``grid`` (``[B,2,H,W]`` tensor or ``GridSpecHost``; a generated one is materialised) and its
        ``target``: a ``PriorFitter`` of fused whole-frame steps (``awb_prior_fit_step`` on the star handle), taking
        weight maps and an ignore label like the other priors; ``kw`` goes to ``PriorFitter``.  The offset is trained iff
        ``offset.requires_grad`` when the fitter is built.  Without a grid: the notebook's sampled-point ``StarFitter``
        (``make_fitter()``, ``make_fitter(optim=..., loss=...)``)."""
        if grid is None:
            return StarFitter(self, optim, loss)
        from ..fit import LossConfig, OptimConfig, PriorFitter
        arena = self._ensure_flat()
        prior = self._prior_for(arena.device)
        if isinstance(grid, torch.Tensor):
            grid = GridSpecHost.from_tensor(grid.to(arena.device))
        elif grid.mode != "explicit":
            grid = GridSpecHost.from_tensor(grid.materialize(2, arena.device))
        if target is None:
            raise ValueError("a grid fit needs its target")
        groups = 0b110 if self.offset.requires_grad else 0b010      # 1: the network's weights, 2: the offset
        return PriorFitter(prior, arena, grid, target, loss or LossConfig("mse"), optim or OptimConfig(),
                           active_groups=groups, **kw)


class StarFitter:
    """``step(x, t)``: one iteration of cell 3 on the sampled points ``x [n,2]`` with labels ``t [n]``;
    ``train_offset`` mirrors ``net.offset.requires_grad = True`` (set at epoch 1000 in the notebook)."""

    def __init__(self, model: StarShapedNet, optim=None, loss=None):
        from ..fit import LossConfig, OptimConfig
        self.model = model
        self.arena = model._ensure_flat()
        self.device = self.arena.device
        self.prior = model._prior_for(self.device)
        self.lib = self.prior.lib
        self.optim = optim or OptimConfig("adam", lr=1e-2)
        self.loss = loss or LossConfig("mse")
        self.train_offset = bool(model.offset.requires_grad)
        self._ws = None
        self._n = -1
        with torch.cuda.device(self.device):
            self.opt_state = torch.empty(self.prior.opt_state_bytes(), dtype=torch.uint8, device=self.device)
            lrs = (C.c_double * L.AWB_MAX_GROUPS)(*self.optim.lrs())
            L.check(self.lib.awb_opt_state_init(self.prior.handle, self.opt_state.data_ptr(), lrs, L.stream_ptr()))
        self._loss_out = torch.zeros(1, dtype=torch.float32, device=self.device)

    def step(self, x: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
        x = x.detach().to(self.device).contiguous().float()
        t = t.detach().to(self.device).contiguous().float().reshape(-1)
        n = x.shape[0]
        if t.numel() != n:
            raise ValueError("one label per point")
        with torch.cuda.device(self.device):
            if n != self._n:
                self._ws = torch.empty(int(self.lib.awb_star_workspace_bytes(self.prior.handle, n)), dtype=torch.uint8,
                                       device=self.device)
                self._n = n
            spec = self.loss.to_specs(t.reshape(1, -1))[0]
            hy = self.optim.to_c()
            hy.active_groups = 0b110 if self.train_offset else 0b010
            L.check(self.lib.awb_star_fit_step(self.prior.handle, self.arena.data_ptr(), self.opt_state.data_ptr(),
                                               x.data_ptr(), t.data_ptr(), n, C.byref(spec), C.byref(hy),
                                               self._loss_out.data_ptr(), self._ws.data_ptr(), self._ws.numel(),
                                               L.stream_ptr()))
        return self._loss_out.clone()

    def fit_likelihood(self, likelihood: torch.Tensor, steps: int = 10000, number: int = 500,
                       unfreeze_offset_at: int = 1000, generator: Optional[torch.Generator] = None) -> torch.Tensor:
        """The whole of cell 3: ``number`` background (likelihood < 0.5) and ``number`` foreground pixels per step,
        coordinates ``idx / (size - 1) - 0.5``, labels ``1 - likelihood``."""
        lk = likelihood.to(self.device).float()
        nx, ny = lk.shape
        def info(mask):
            idx = torch.nonzero(mask)
            pix = torch.stack([idx[:, 0] / (nx - 1) - 0.5, idx[:, 1] / (ny - 1) - 0.5], dim=1).float()
            return pix, 1 - lk[mask]
        pb, lb = info(lk < 0.5)
        pf, lf = info(lk > 0.5)
        hist = []
        for epoch in range(steps):
            ib = torch.randperm(pb.shape[0], device=self.device, generator=generator)[:number]
            jf = torch.randperm(pf.shape[0], device=self.device, generator=generator)[:number]
            if epoch == unfreeze_offset_at:
                self.train_offset = True
            hist.append(self.step(torch.cat([pb[ib], pf[jf]]), torch.cat([lb[ib], lf[jf]])))
        return torch.cat(hist)
