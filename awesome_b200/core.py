"""Thin host-side objects over the C-ABI: prior handle, grid specs, workspaces."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple, Union

import torch

from . import _lib as L

GridLike = Union[torch.Tensor, "GridSpecHost"]


class GridSpecHost:
    """Host description of the coordinate grid of a fit (SURVEY a1).

    ``mode``: "explicit" (a ``[B,C,H,W]`` fp32 CUDA tensor, reference layout), "linspace"
    (``Transformator.get_positional_matrices``, reference ``awesome/dataset/transformator.py:25-61``)
    or "index" (how-to notebooks' ``create_grid``).  Generated modes never touch HBM for the grid.
    """

    def __init__(self, mode: str, B: int, H: int, W: int, grid: Optional[torch.Tensor] = None,
                 t0: float = 0.0, t_step: float = 0.0):
        self.mode, self.B, self.H, self.W = mode, int(B), int(H), int(W)
        self.grid, self.t0, self.t_step = grid, float(t0), float(t_step)

    @property
    def n_pixels(self) -> int:
        return self.B * self.H * self.W

    @staticmethod
    def from_tensor(grid: torch.Tensor) -> "GridSpecHost":
        if grid.dim() == 3:
            grid = grid.unsqueeze(0)
        if grid.dim() != 4:
            raise ValueError(f"expected a [B,C,H,W] grid, got shape {tuple(grid.shape)}")
        g = grid.detach()
        if g.dtype != torch.float32 or not g.is_contiguous():
            g = g.contiguous().float()
        return GridSpecHost("explicit", g.shape[0], g.shape[2], g.shape[3], grid=g)

    def to_c(self) -> L.GridSpec:
        mode = {"explicit": L.AWB_GRID_EXPLICIT, "linspace": L.AWB_GRID_LINSPACE, "index": L.AWB_GRID_INDEX}[self.mode]
        ptr = self.grid.data_ptr() if self.grid is not None else None
        return L.GridSpec(mode, self.B, self.H, self.W, self.t0, self.t_step, ptr)

    def materialize(self, C_: int, device) -> torch.Tensor:
        """The grid as the reference would build it (for callers that want the tensor)."""
        if self.mode == "explicit":
            return self.grid
        if self.mode == "linspace":
            y = torch.linspace(0, 1, self.H, device=device)
            x = torch.linspace(0, 1, self.W, device=device)
        else:
            y = torch.arange(self.H, device=device).float() / self.H
            x = torch.arange(self.W, device=device).float() / self.W
        yy, xx = torch.meshgrid(y, x, indexing="ij")
        frames = []
        for b in range(self.B):
            ch = [xx, yy]
            if C_ == 3:
                ch.append(torch.full_like(xx, self.t0 + b * self.t_step))
            frames.append(torch.stack(ch, 0))
        return torch.stack(frames, 0).float()


class Prior:
    """Owns an ``awb_handle``; all device memory stays owned by torch."""

    def __init__(self, kind: int, C_: int, h: int, n_layers: int, n_flows: int = 0, flow_hidden: int = 0,
                 flow_tanh: bool = True, n_objects: int = 1, precision: int = L.AWB_PREC_FP32):
        L.require_cuda()
        self.lib = L.load()
        self.desc = L.Desc(kind, C_, h, n_layers, n_flows, flow_hidden, int(flow_tanh), n_objects, precision)
        self._h = C.c_void_p()
        L.check(self.lib.awb_prior_create(C.byref(self.desc), C.byref(self._h)))
        self.n_params = int(self.lib.awb_prior_param_count(self._h))
        self.n_objects = n_objects
        self.C = C_
        self._ws_cache = {}

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and self._h.value:
                self.lib.awb_prior_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def workspace_bytes(self, n_pixels: int, layout: int) -> int:
        """Bytes of a workspace of ``layout`` (``L.AWB_WS_*``, see ``awb_prior_workspace_bytes``)."""
        b = int(self.lib.awb_prior_workspace_bytes(self._h, n_pixels, layout))
        if b < 0:
            raise L.AwbError(b, "workspace size query failed")
        return b

    def new_workspace(self, n_pixels: int, layout: int, device) -> torch.Tensor:
        return torch.empty(self.workspace_bytes(n_pixels, layout), dtype=torch.uint8, device=device)

    def cached_workspace(self, n_pixels: int, layout: int, device) -> torch.Tensor:
        key = (n_pixels, layout, str(device))
        ws = self._ws_cache.get(key)
        if ws is None:
            self._ws_cache.clear()
            ws = self.new_workspace(n_pixels, layout, device)
            self._ws_cache[key] = ws
        return ws

    def opt_state_bytes(self) -> int:
        return int(self.lib.awb_opt_state_bytes(self._h))

    def set_flow_consts(self, nmin: Sequence[float], nmax: Sequence[float], new_min: float, new_max: float,
                        masks: Sequence[int]) -> None:
        a = (C.c_float * len(nmin))(*nmin)
        b = (C.c_float * len(nmax))(*nmax)
        m = (C.c_uint8 * len(masks))(*masks)
        L.check(self.lib.awb_prior_set_flow_consts(self._h, a, b, new_min, new_max, m))

    def set_flow_eval(self, mode: int) -> None:
        """RealNVP coupling MLPs: 0 auto, 1 unit loops (reference order of operations), 2 segment tables (C = 2);
        see ``awb_prior_set_flow_eval`` in ``include/awb.h``."""
        L.check(self.lib.awb_prior_set_flow_eval(self._h, int(mode)))

    # ---- kernels
    def forward(self, params: torch.Tensor, grid: GridSpecHost, mode: int, ws: torch.Tensor,
                want_deformed: bool = False) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        """``mode``: ``L.AWB_FWD_*``; ``ws`` of the workspace layout ``awb_prior_forward`` names for it."""
        N = grid.n_pixels
        logits = torch.empty((self.n_objects, N), dtype=torch.float32, device=params.device)
        deformed = torch.empty((self.n_objects, N, self.C), dtype=torch.float32, device=params.device) \
            if want_deformed else None
        gs = grid.to_c()
        L.check(self.lib.awb_prior_forward(self._h, params.data_ptr(), C.byref(gs), logits.data_ptr(),
                                           deformed.data_ptr() if deformed is not None else None,
                                           mode, ws.data_ptr(), ws.numel(), L.stream_ptr()))
        return logits, deformed

    def backward(self, params: torch.Tensor, grid: GridSpecHost, dlogits: torch.Tensor, ws: torch.Tensor,
                 want_dgrid: bool) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        grads = torch.empty((self.n_objects, self.n_params), dtype=torch.float32, device=params.device)
        dgrid = torch.empty((grid.B, self.C, grid.H, grid.W), dtype=torch.float32, device=params.device) \
            if want_dgrid else None
        gs = grid.to_c()
        L.check(self.lib.awb_prior_backward(self._h, params.data_ptr(), C.byref(gs), dlogits.data_ptr(),
                                            grads.data_ptr(), dgrid.data_ptr() if dgrid is not None else None,
                                            ws.data_ptr(), ws.numel(), L.stream_ptr()))
        return grads, dgrid

    def grid_grad_backward(self, params: torch.Tensor, grid: GridSpecHost, dlogits: torch.Tensor, d_dgrid: torch.Tensor,
                           ws: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """Double backward of ``backward``'s dgrid (``awb_prior_grid_grad_backward``, single-object ICNN): ``dlogits``
        (``[1, N]``) is the first backward's, ``d_dgrid`` (``[B, C, H, W]`` fp32, contiguous) the gradient on its dgrid.
        Returns ``d_dlogits [1, N]`` and ``grads [1, P]``.  ``ws``: layout ``AWB_WS_SECOND_ORDER``, after
        ``forward(AWB_FWD_EXACT_TRAINING)`` on it."""
        d_dlogits = torch.empty((self.n_objects, grid.n_pixels), dtype=torch.float32, device=params.device)
        grads = torch.empty((self.n_objects, self.n_params), dtype=torch.float32, device=params.device)
        gs = grid.to_c()
        L.check(self.lib.awb_prior_grid_grad_backward(self._h, params.data_ptr(), C.byref(gs), dlogits.data_ptr(),
                                                      d_dgrid.data_ptr(), d_dlogits.data_ptr(), grads.data_ptr(),
                                                      ws.data_ptr(), ws.numel(), L.stream_ptr()))
        return d_dlogits, grads

    def deformation(self, params: torch.Tensor, grid: GridSpecHost, training: bool, ws: torch.Tensor) -> torch.Tensor:
        """``get_deformation`` alone (1x1 conv / linear and flow, no ICNN): pixel rows ``[N, C]``.  ``ws``:
        layout ``AWB_WS_DEFORMATION``; ``training`` keeps the coupling records for ``deformation_backward``."""
        out = torch.empty((grid.n_pixels, self.C), dtype=torch.float32, device=params.device)
        gs = grid.to_c()
        L.check(self.lib.awb_prior_deformation(self._h, params.data_ptr(), C.byref(gs), out.data_ptr(), int(bool(training)),
                                               ws.data_ptr(), ws.numel(), L.stream_ptr()))
        return out

    def deformation_backward(self, params: torch.Tensor, grid: GridSpecHost, d_deformed: torch.Tensor, ws: torch.Tensor,
                             want_dgrid: bool) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        """Gradients of ``deformation(training=True)`` on the same ``ws`` for the upstream ``d_deformed`` (``[N, C]``
        fp32, contiguous): ``grads [P]`` (ICNN entries 0) and, when asked, ``dgrid [B, C, H, W]``."""
        grads = torch.empty(self.n_params, dtype=torch.float32, device=params.device)
        dgrid = torch.empty((grid.B, self.C, grid.H, grid.W), dtype=torch.float32, device=params.device) \
            if want_dgrid else None
        gs = grid.to_c()
        L.check(self.lib.awb_prior_deformation_backward(self._h, params.data_ptr(), C.byref(gs), d_deformed.data_ptr(),
                                                        grads.data_ptr(), dgrid.data_ptr() if dgrid is not None else None,
                                                        ws.data_ptr(), ws.numel(), L.stream_ptr()))
        return grads, dgrid

    def inverse(self, params: torch.Tensor, grid: GridSpecHost, training: bool, ws: torch.Tensor) -> torch.Tensor:
        """``PathConnectedNet.inverse`` of the explicit ``grid``: pixel rows ``[N, C]``.  ``ws``: layout
        ``AWB_WS_DEFORMATION``; ``training`` keeps the coupling records for ``inverse_backward``."""
        out = torch.empty((grid.n_pixels, self.C), dtype=torch.float32, device=params.device)
        gs = grid.to_c()
        L.check(self.lib.awb_prior_inverse(self._h, params.data_ptr(), C.byref(gs), out.data_ptr(), int(bool(training)),
                                           ws.data_ptr(), ws.numel(), L.stream_ptr()))
        return out

    def inverse_backward(self, params: torch.Tensor, grid: GridSpecHost, d_out: torch.Tensor, ws: torch.Tensor,
                         want_dgrid: bool) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        """Gradients of ``inverse(training=True)`` on the same ``ws`` for the upstream ``d_out`` (``[N, C]`` fp32,
        contiguous): ``grads [P]`` (ICNN entries 0) and, when asked, ``dgrid [B, C, H, W]``."""
        grads = torch.empty(self.n_params, dtype=torch.float32, device=params.device)
        dgrid = torch.empty((grid.B, self.C, grid.H, grid.W), dtype=torch.float32, device=params.device) \
            if want_dgrid else None
        gs = grid.to_c()
        L.check(self.lib.awb_prior_inverse_backward(self._h, params.data_ptr(), C.byref(gs), d_out.data_ptr(),
                                                    grads.data_ptr(), dgrid.data_ptr() if dgrid is not None else None,
                                                    ws.data_ptr(), ws.numel(), L.stream_ptr()))
        return grads, dgrid

    def enforce_convexity(self, params: torch.Tensor) -> None:
        L.check(self.lib.awb_prior_enforce_convexity(self._h, params.data_ptr(), L.stream_ptr()))

    # ---- pixel-sliced fit step (awb_prior_slice_grads / awb_prior_rows_opt_step)
    @property
    def grad_row_floats(self) -> int:
        """``P + 1``: a slice's gradient in state_dict order, then its loss sum."""
        return int(self.lib.awb_prior_grad_row_floats(self._h))

    def slice_grads(self, params: torch.Tensor, grid: GridSpecHost, row_begin: int, row_end: int, target: torch.Tensor,
                    loss, grad_row: torch.Tensor, ws: torch.Tensor, reuse_packed: bool = False) -> None:
        """Gradient row of pixel rows ``[row_begin, row_end)`` of the batch into ``grad_row`` (``[P + 1]`` fp32, device).
        ``target`` is the FULL batch ``[N]``; ``loss`` the ``LossSpec`` of the full batch (its weight map, when set, too
        covers the full batch and is read at the global rows).  ``ws``:
        layout ``AWB_WS_FIT_STEP`` for ``row_end - row_begin`` pixels.  ``reuse_packed``: the previous call on ``ws`` was
        a slice of the same parameters."""
        gs = grid.to_c()
        L.check(self.lib.awb_prior_slice_grads(self._h, params.data_ptr(), C.byref(gs), int(row_begin), int(row_end),
                                               target.data_ptr(), C.byref(loss), grad_row.data_ptr(), ws.data_ptr(),
                                               ws.numel(), L.AWB_FIT_REUSE_PACKED if reuse_packed else 0,
                                               L.stream_ptr()))

    def rows_opt_step(self, params: torch.Tensor, opt_state: torch.Tensor, rows: torch.Tensor, hyper,
                      loss_out: Optional[torch.Tensor] = None) -> None:
        """Sum of the gradient rows ``rows`` (``[S, P + 1]`` fp32, device) in a fixed order, then the optimizer step of
        the fused fit step.  ``loss_out`` (optional, one device float) receives the summed loss."""
        if rows.dim() != 2 or rows.shape[1] != self.grad_row_floats or not rows.is_contiguous():
            raise ValueError(f"rows must be a contiguous [S, {self.grad_row_floats}] tensor, got {tuple(rows.shape)}")
        L.check(self.lib.awb_prior_rows_opt_step(self._h, params.data_ptr(), opt_state.data_ptr(), rows.data_ptr(),
                                                 rows.shape[0], C.byref(hyper),
                                                 loss_out.data_ptr() if loss_out is not None else None, None, 0,
                                                 L.stream_ptr()))


def iou_counts(pred: torch.Tensor, target: torch.Tensor, pred_is_logit: bool, n_objects: int = 1) -> torch.Tensor:
    """``[O,4]`` int64 counts {intersection, pred_fg, target_fg, n}; fg = value <= 0.5.
    Inputs hold ``n_objects`` masks back to back (any shape)."""
    L.require_cuda()
    lib = L.load()
    O = n_objects
    p = pred.detach().reshape(O, -1).contiguous().float()
    t = target.detach().reshape(O, -1).contiguous().float()
    counts = torch.empty((O, 4), dtype=torch.int64, device=p.device)
    L.check(lib.awb_mask_iou_counts(p.data_ptr(), t.data_ptr(), p.shape[1], O, int(pred_is_logit),
                                    counts.data_ptr(), L.stream_ptr()))
    return counts


def target_counts(target: torch.Tensor, cls_rule: int, n_objects: int = 1,
                  ignore_value: Optional[float] = None) -> torch.Tensor:
    """``[O,2]`` int64 counts {fg, bg} of the target under ``cls_rule`` (``n_objects`` targets back to back).
    ``ignore_value``: pixels whose target equals it count in neither class (``awb_target_counts_ignore``)."""
    L.require_cuda()
    lib = L.load()
    t = target.detach()
    O = n_objects
    t = t.reshape(O, -1).contiguous().float()
    counts = torch.empty((O, 2), dtype=torch.int64, device=t.device)
    if ignore_value is None:
        L.check(lib.awb_target_counts(t.data_ptr(), t.shape[1], O, cls_rule, counts.data_ptr(), L.stream_ptr()))
    else:
        L.check(lib.awb_target_counts_ignore(t.data_ptr(), t.shape[1], O, cls_rule, 1, float(ignore_value),
                                             counts.data_ptr(), L.stream_ptr()))
    return counts
