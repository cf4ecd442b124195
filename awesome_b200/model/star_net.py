"""Star-shape prior (SURVEY a16): drop-in for the notebook class ``myNet``
(``notebooks/icml_teaser_code/star_shaped/star.ipynb`` cell 2) -- same constructor argument, parameter names
(``offset, W0, W1, W2, W1_r, W2_r``), initial weights for a given seed and ``forward(x[n,2]) -> [n,1]`` -- with the
training loop of cell 3 as fused native steps (``StarFitter``)."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
from torch import nn

from .. import _lib as L
from ..core import Prior
from .base import Affine, ArenaPriorModule, reject_second_order


def _lin(i: int, o: int) -> Affine:
    l = nn.Linear(i, o)
    return Affine(l.weight.detach().clone(), l.bias.detach().clone())


class _StarFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, x):
        prior = module._prior_for(x.device)
        arena = module._ensure_flat()
        xs = x.detach().contiguous().float()
        out = torch.empty(xs.shape[0], dtype=torch.float32, device=x.device)
        L.check(prior.lib.awb_star_forward(prior.handle, arena.data_ptr(), xs.data_ptr(), xs.shape[0], out.data_ptr(),
                                           L.stream_ptr()))
        return out.reshape(-1, 1)


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
        """Inference forward (native).  Training goes through ``make_fitter`` (the notebook's loop, fused)."""
        if x.dim() != 2 or x.shape[1] != 2:
            raise ValueError(f"expected [n,2] points, got {tuple(x.shape)}")
        if not x.is_cuda:
            raise L.AwbLibraryError("awesome_b200 priors run on CUDA only (no CPU fallback)")
        with torch.cuda.device(x.device):
            return _StarFunction.apply(self, x)

    def enforce_convexity(self) -> None:
        """The notebook's projection: ``W2_r.weight <- relu(W2_r.weight)`` (cell 3)."""
        with torch.no_grad():
            self.W2_r.weight.clamp_(min=0)

    def make_fitter(self, optim=None, loss=None, **kw) -> "StarFitter":
        return StarFitter(self, optim, loss)


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
