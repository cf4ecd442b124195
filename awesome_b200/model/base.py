"""Shared machinery of the drop-in prior modules: one flat fp32 parameter arena per module
(state-dict tensors are views into it), lazy creation of the native handle, and the
autograd bridges to ``awb_prior_forward`` / ``awb_prior_backward``, to ``awb_prior_deformation`` /
``awb_prior_deformation_backward`` and to ``awb_prior_inverse`` / ``awb_prior_inverse_backward``.  The backwards are
first-order only: a double backward raises.  The exception is an
ICNN prior built with ``second_order=True``: under ``create_graph`` its coordinate gradient is differentiable
(``_GridGradFunction``, ``awb_prior_grid_grad_backward``)."""
from __future__ import annotations

import functools
from typing import List, Optional, Tuple

import torch
from torch import nn
from torch.autograd.function import once_differentiable

from .. import _lib as L
from ..core import GridSpecHost, Prior

_PRECISIONS = {"fp32": L.AWB_PREC_FP32, "f16": L.AWB_PREC_F16}


class Affine(nn.Module):
    """Parameter holder with the key names of ``nn.Linear`` (``weight`` [, ``bias``])."""

    def __init__(self, weight: torch.Tensor, bias: Optional[torch.Tensor] = None):
        super().__init__()
        self.weight = nn.Parameter(weight)
        if bias is not None:
            self.bias = nn.Parameter(bias)
        else:
            self.register_parameter("bias", None)

    @property
    def in_features(self):
        return self.weight.shape[1]

    @property
    def out_features(self):
        return self.weight.shape[0]

    def extra_repr(self):
        return f"weight={tuple(self.weight.shape)}, bias={self.bias is not None}"


def _first_order_only(backward):
    """``once_differentiable`` for a backward whose upstream gradient may be a constant.  torch's decorator arms its
    double-backward error only when the incoming gradient requires grad; for ``grad(y.sum(), x, create_graph=True)`` it does
    not, and a gradient penalty built on the result would silently lose its second-order term.  Under ``create_graph``
    (grad mode on during the backward) the incoming gradients are passed as aliases that require grad, so every result
    carries a grad_fn that raises when it is differentiated."""
    inner = once_differentiable(backward)

    @functools.wraps(backward)
    def wrapper(ctx, *grads):
        if torch.is_grad_enabled():
            grads = tuple(g.detach().requires_grad_() if isinstance(g, torch.Tensor) and not g.requires_grad else g
                          for g in grads)
        return inner(ctx, *grads)
    return wrapper


def reject_second_order(kind: str, kwargs) -> None:
    """Second derivatives are provided for the ICNN priors only: any other prior refuses the flag instead of ignoring it."""
    if kwargs.get("second_order"):
        raise ValueError(f"{kind} has no second-order backward (second_order=True is provided for ConvexNextNet and "
                         "ConvexNet: the flows' couplings have non-zero second derivatives in the coordinates)")


def _split_grads(flat: torch.Tensor, shapes) -> Tuple[torch.Tensor, ...]:
    """Views of the arena-ordered gradient vector in the shapes of the module's parameters."""
    outs, off = [], 0
    flat = flat.reshape(-1)
    for shp in shapes:
        n = 1
        for s in shp:
            n *= s
        outs.append(flat[off:off + n].view(shp))
        off += n
    return tuple(outs)


def _prior_backward(ctx, dlogits):
    module, spec, prior = ctx.module, ctx.spec, ctx.prior
    if ctx.ws is None:
        raise RuntimeError("backward through an awesome_b200 prior needs a forward that ran with grad enabled")
    want_dgrid = ctx.needs_input_grad[3]
    grads, dgrid = prior.backward(module._arena, spec, dlogits.contiguous().float(), ctx.ws, want_dgrid)
    if dgrid is not None and ctx.rows_input:      # pixel rows [N,C] went in as [1,C,1,N]: hand their gradient back as [N,C]
        dgrid = dgrid.reshape(dgrid.shape[1], -1).t().contiguous()
    if not ctx.second_order:    # second order: a retained graph may come back through here after the second-order pass
        ctx.ws = None
    return (None, None, None, dgrid) + _split_grads(grads, ctx.shapes)


_prior_backward_first_order = _first_order_only(_prior_backward)


class _GridGradFunction(torch.autograd.Function):
    """The first backward of an ICNN prior as a differentiable function of its upstream gradient ``w`` and the
    parameters.  Forward: ``awb_prior_backward`` (dgrid and the parameter gradients, the bits of the first-order path).
    Backward: ``awb_prior_grid_grad_backward`` turns the gradient ``u`` on dgrid into ``J u`` for ``w`` and
    ``sum_n w_n d(J_n u_n) / d params`` for the parameters; the grid gets nothing (the ICNN is piecewise linear in it).
    Differentiating the parameter-gradient outputs raises."""

    @staticmethod
    def forward(ctx, module, spec, prior, ws, rows_input, dlogits, *params):
        ctx.set_materialize_grads(False)
        w = dlogits.contiguous().float()
        grads, dgrid = prior.backward(module._arena, spec, w, ws, True)
        if rows_input:
            dgrid = dgrid.reshape(dgrid.shape[1], -1).t().contiguous()
        ctx.module, ctx.spec, ctx.prior, ctx.ws, ctx.rows_input = module, spec, prior, ws, rows_input
        ctx.shapes = [p.shape for p in params]
        ctx.save_for_backward(w)
        return (dgrid,) + tuple(g.clone() for g in _split_grads(grads, ctx.shapes))

    @staticmethod
    @_first_order_only
    def backward(ctx, d_dgrid, *d_grads):
        if any(g is not None for g in d_grads):
            raise RuntimeError("awesome_b200 priors do not differentiate their parameter gradients: with "
                               "second_order=True only the coordinate gradient of an ICNN prior (a penalty on d prior / "
                               "d grid) has a second derivative")
        if d_dgrid is None:
            return (None,) * (6 + len(ctx.shapes))
        (w,) = ctx.saved_tensors
        module, spec, prior = ctx.module, ctx.spec, ctx.prior
        u = (d_dgrid.t() if ctx.rows_input else d_dgrid).contiguous().float()    # planar [B,C,H,W] ([1,C,1,N] for rows)
        u = u.reshape(spec.B, -1, spec.H, spec.W)
        ws = ctx.ws
        if module.precision == "f16":
            # the first order ran on the tensor path, which keeps no activations: an exact fp32 forward provides them
            ws = prior.new_workspace(spec.n_pixels, L.AWB_WS_SECOND_ORDER, w.device)
            prior.forward(module._arena, spec, L.AWB_FWD_EXACT_TRAINING, ws)
        d_w, grads = prior.grid_grad_backward(module._arena, spec, w, u, ws)
        return (None, None, None, None, None, d_w) + _split_grads(grads, ctx.shapes)


class _PriorFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, spec, needs_grad, grid_tensor, *params):
        """``needs_grad`` is decided by the caller (grad mode is always off inside ``Function.forward`` and
        ``ctx.needs_input_grad`` ignores ``torch.no_grad()``): a forward under ``no_grad`` takes the exact fp32 inference
        path (``AWB_FWD_EXACT``) on the cached workspace, whatever ``requires_grad`` says."""
        prior = module._prior_for(params[0].device)
        arena = module._arena
        second_order = needs_grad and module.second_order
        if needs_grad:
            # private: several forwards may precede backward.  An exact second-order module also keeps room for the
            # tangent rows of the second-order pass (the training layout is a prefix of that one).
            layout = L.AWB_WS_SECOND_ORDER if second_order and module.precision == "fp32" else L.AWB_WS_TRAINING
            ws = prior.new_workspace(spec.n_pixels, layout, arena.device)
            # training forward of a tensor-path module: logits from the fused tcgen05 kernel; backward re-runs it with
            # the upstream gradient
            mode = L.AWB_FWD_TC_TRAINING if module.precision == "f16" else L.AWB_FWD_EXACT_TRAINING
        else:   # inference (no grad) always takes the exact fp32 path
            ws = prior.cached_workspace(spec.n_pixels, L.AWB_WS_INFERENCE, arena.device)
            mode = L.AWB_FWD_EXACT
        logits, _ = prior.forward(arena, spec, mode, ws)
        ctx.module, ctx.spec, ctx.ws, ctx.prior = module, spec, (ws if needs_grad else None), prior
        ctx.shapes = [p.shape for p in params]
        ctx.rows_input = grid_tensor is not None and grid_tensor.dim() == 2
        ctx.second_order = second_order
        if second_order:
            ctx.save_for_backward(*params)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        # a backward that builds a graph (create_graph) and returns dgrid: differentiable on second-order modules
        if ctx.second_order and torch.is_grad_enabled() and ctx.needs_input_grad[3]:
            if ctx.ws is None:
                raise RuntimeError("backward through an awesome_b200 prior needs a forward that ran with grad enabled")
            # the graph built here comes back through this forward when w depends on the logits
            outs = _GridGradFunction.apply(ctx.module, ctx.spec, ctx.prior, ctx.ws, ctx.rows_input, dlogits,
                                           *ctx.saved_tensors)
            return (None, None, None) + tuple(outs)
        return _prior_backward_first_order(ctx, dlogits)


class _DeformationFunction(torch.autograd.Function):
    """``get_deformation`` of a flow prior with autograd: pixel rows ``[N, C]`` of the deformed coordinates.  The forward keeps
    the coupling records in a private deformation-only workspace; the backward returns the flow and linear gradients (the
    ICNN's are 0) and, when the grid requires grad, ``dgrid``."""

    @staticmethod
    def forward(ctx, module, spec, grid_tensor, *params):
        prior = module._prior_for(params[0].device)
        arena = module._arena
        ws = prior.new_workspace(spec.n_pixels, L.AWB_WS_DEFORMATION, arena.device)
        rows = prior.deformation(arena, spec, True, ws)
        ctx.module, ctx.spec, ctx.ws, ctx.prior = module, spec, ws, prior
        ctx.shapes = [p.shape for p in params]
        return rows

    @staticmethod
    @_first_order_only
    def backward(ctx, d_rows):
        if ctx.ws is None:
            raise RuntimeError("get_deformation's backward runs once per forward (its workspace is released after it)")
        grads, dgrid = ctx.prior.deformation_backward(ctx.module._arena, ctx.spec, d_rows.contiguous().float(), ctx.ws,
                                                      ctx.needs_input_grad[2])
        ctx.ws = None
        return (None, None, dgrid) + _split_grads(grads, ctx.shapes)


class _InverseFunction(torch.autograd.Function):
    """``PathConnectedNet.inverse`` with autograd: pixel rows ``[N, C]`` of the points mapped back through the flow.  The
    forward keeps the coupling records in a private deformation-only workspace; the backward returns the flow and 1x1-conv
    gradients (the ICNN's are 0) and, when ``x`` requires grad, ``dgrid``."""

    @staticmethod
    def forward(ctx, module, spec, x, *params):
        prior = module._prior_for(params[0].device)
        arena = module._arena
        ws = prior.new_workspace(spec.n_pixels, L.AWB_WS_DEFORMATION, arena.device)
        rows = prior.inverse(arena, spec, True, ws)
        ctx.module, ctx.spec, ctx.ws, ctx.prior = module, spec, ws, prior
        ctx.shapes = [p.shape for p in params]
        return rows

    @staticmethod
    @_first_order_only
    def backward(ctx, d_rows):
        if ctx.ws is None:
            raise RuntimeError("inverse's backward runs once per forward (its workspace is released after it)")
        grads, dgrid = ctx.prior.inverse_backward(ctx.module._arena, ctx.spec, d_rows.contiguous().float(), ctx.ws,
                                                  ctx.needs_input_grad[2])
        ctx.ws = None
        return (None, None, dgrid) + _split_grads(grads, ctx.shapes)


class ArenaPriorModule(nn.Module):
    """Base class: subclasses register their parameters (in state_dict order == arena order)
    and implement ``_make_prior(device)``."""

    def __init__(self, precision: str = "fp32", second_order: bool = False):
        super().__init__()
        if precision not in _PRECISIONS:
            raise ValueError(f"precision must be one of {list(_PRECISIONS)}, got {precision!r}")
        self.precision = precision
        self.second_order = bool(second_order)
        self._arena: Optional[torch.Tensor] = None
        self._prior: Optional[Prior] = None
        self._prior_device = None
        from ..optim import _ARENA_MODULES
        _ARENA_MODULES.add(self)
        from ..reference_bridge import integrate_with_reference
        integrate_with_reference()

    def _optimizer_group_ids(self) -> List[int]:
        """Native optimizer group of every arena parameter (0 flow_net, 1 convex_net, 2 linear), in arena order."""
        return [1] * len(self._arena_params())

    # ---- arena
    def _arena_params(self) -> List[nn.Parameter]:
        return [p for p in self.parameters()]

    def _flatten_(self) -> None:
        params = self._arena_params()
        if not params:
            return
        dev = params[0].device
        n = sum(p.numel() for p in params)
        arena = torch.empty(n, dtype=torch.float32, device=dev)
        off = 0
        with torch.no_grad():
            for p in params:
                k = p.numel()
                arena[off:off + k].copy_(p.detach().reshape(-1).float())
                p.data = arena[off:off + k].view(p.shape)
                off += k
        self._arena = arena

    def _ensure_flat(self) -> torch.Tensor:
        """The parameters as one contiguous fp32 vector.  When they already sit back to back in
        memory (e.g. this module's tensors are views into a parent module's arena) the arena is
        re-derived as a view; otherwise they are copied into a fresh arena and re-pointed."""
        params = self._arena_params()
        first = params[0]
        off, ok = first.data_ptr(), first.dtype == torch.float32
        for p in params:
            if p.data_ptr() != off or p.device != first.device or p.dtype != torch.float32:
                ok = False
                break
            off += p.numel() * 4
        n = sum(p.numel() for p in params)
        if ok:
            try:
                if first.untyped_storage().nbytes() - first.storage_offset() * 4 < n * 4:
                    ok = False
            except Exception:
                ok = False
        if ok:
            a = self._arena
            if a is None or a.data_ptr() != first.data_ptr() or a.numel() != n:
                self._arena = torch.as_strided(first.detach(), (n,), (1,), first.storage_offset())
        else:
            self._flatten_()
        return self._arena

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self._flatten_()
        return out

    def load_state_dict(self, state_dict, *args, **kwargs):
        out = super().load_state_dict(state_dict, *args, **kwargs)
        self._ensure_flat()
        return out

    # ---- native handle
    def _make_prior(self, device) -> Prior:
        raise NotImplementedError

    def _prior_for(self, device) -> Prior:
        if device.type != "cuda":
            raise L.AwbLibraryError("awesome_b200 priors run on CUDA only (no CPU fallback); move the module "
                                    "and its inputs to a cuda device.")
        if self._prior is None or self._prior_device != device:
            with torch.cuda.device(device):
                self._prior = self._make_prior(device)
            self._prior_device = device
        return self._prior

    # ---- forward through the native library
    def _logits(self, spec: GridSpecHost, grid_tensor: Optional[torch.Tensor]) -> torch.Tensor:
        self._ensure_flat()
        params = self._arena_params()
        self._prior_for(self._arena.device)       # raises loudly on a non-CUDA device
        needs_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in params)
                                                  or (grid_tensor is not None and grid_tensor.requires_grad))
        with torch.cuda.device(self._arena.device):
            return _PriorFunction.apply(self, spec, needs_grad, grid_tensor, *params)

    def _forward_any(self, x: torch.Tensor, n_channels: int) -> torch.Tensor:
        """Accepts ``[B,C,H,W]`` (-> ``[B,1,H,W]``), ``[C,H,W]`` (-> ``[1,H,W]``) or pixel rows ``[N,C]``
        (-> ``[N,1]``), like the reference's ``@pixelize`` / ``@batcherize`` decorators."""
        if x.dim() == 2:
            if x.shape[1] != n_channels:
                raise ValueError(f"expected [N,{n_channels}] pixel rows, got {tuple(x.shape)}")
            g = x.t().reshape(1, n_channels, 1, x.shape[0])
            spec = GridSpecHost.from_tensor(g)
            return self._logits(spec, x if x.requires_grad else None).reshape(-1, 1)
        squeeze = x.dim() == 3
        if squeeze:
            x = x.unsqueeze(0)
        if x.dim() != 4 or x.shape[1] != n_channels:
            raise ValueError(f"expected a [B,{n_channels},H,W] grid, got {tuple(x.shape)}")
        spec = GridSpecHost.from_tensor(x)
        out = self._logits(spec, x if x.requires_grad else None).reshape(x.shape[0], 1, x.shape[2], x.shape[3])
        return out[0] if squeeze else out

    def _deformation_rows(self, x: torch.Tensor) -> torch.Tensor:
        """``get_deformation`` of ``x`` (``[B,C,H,W]``) as pixel rows ``[N, C]``.  With grad mode on and a parameter or ``x``
        requiring grad it runs through ``_DeformationFunction`` (differentiable w.r.t. the parameters and ``x``); otherwise
        through the inference forward on the cached workspace, as it always has."""
        arena = self._ensure_flat()
        params = self._arena_params()
        prior = self._prior_for(arena.device)
        spec = GridSpecHost.from_tensor(x)
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params)):
            with torch.cuda.device(arena.device):
                return _DeformationFunction.apply(self, spec, x if x.requires_grad else None, *params)
        with torch.no_grad(), torch.cuda.device(arena.device):
            ws = prior.cached_workspace(spec.n_pixels, L.AWB_WS_INFERENCE, arena.device)
            _, deformed = prior.forward(arena, spec, L.AWB_FWD_EXACT, ws, want_deformed=True)
        return deformed[0]

    def make_fitter(self, grid, target, loss=None, optim=None, **kw):
        """A ``PriorFitter`` running fused fit steps in place on this module's parameters."""
        from ..fit import LossConfig, OptimConfig, PriorFitter
        arena = self._ensure_flat()
        prior = self._prior_for(arena.device)
        if isinstance(grid, torch.Tensor):
            grid = GridSpecHost.from_tensor(grid)
        return PriorFitter(prior, arena, grid, target, loss or LossConfig(), optim or OptimConfig(), **kw)

    def enforce_convexity(self) -> None:
        """``W <- max(W, 0)`` on every ``skip.i.ln.weight`` and ``out.ln.weight`` in one pass
        (reference ``awesome/model/convex_net.py:151-154,216-220``)."""
        arena = self._ensure_flat()
        with torch.no_grad(), torch.cuda.device(arena.device):
            self._prior_for(arena.device).enforce_convexity(arena)
