"""The fused fit loop: the body of the reference's per-frame hot loops
(``awesome/model/path_connected_net.py:939-953``, ``:364-379``; how-to notebooks cell 9)
as one native call per step, replayed through CUDA graphs so the host never touches a step.

``forward -> sigmoid -> loss -> backward -> optimizer.step -> enforce_convexity ->
lr_scheduler.step(loss)`` all happen inside ``awb_prior_fit_step``; the loss history stays on
the device and is read back once per fit (the reference syncs three times per step)."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Union

import torch

from . import _lib as L
from .core import GridSpecHost, Prior, target_counts


@dataclass
class LossConfig:
    """Which per-pixel loss the fit minimises (SURVEY a10).

    kind "mse": ``UnariesWeightedLoss(SE("mean"), mode=...)`` on ``sigmoid(y)``
    (``path_connected_net.py:768``; modes of ``unaries_weighted_loss.py:35-69``).
    kind "fgbg_se" / "fgbg_bce_logits": the how-to notebooks' fg/bg-weighted means.
    """
    kind: str = "mse"
    mode: str = "none"        # none | ratio | sssdms | equal   (kind == "mse")
    ratio: float = 1.0
    fg_weight: float = 0.4    # fgbg_* kinds

    @classmethod
    def from_reference(cls, criterion) -> "LossConfig":
        """Map a reference loss object onto the fused per-pixel loss (duck-typed by class name / attributes):
        ``UnariesWeightedLoss(SE, mode=...)`` (``awesome/measures/unaries_weighted_loss.py:35-69``),
        ``SE`` (``se.py``), ``torch.nn.MSELoss`` -> "mse"; ``BCEWithLogitsLoss`` -> fg/bg BCE with equal weights."""
        name = type(criterion).__name__
        if name == "UnariesWeightedLoss" and type(getattr(criterion, "criterion", None)).__name__ == "BCELoss":
            if (getattr(criterion, "mode", "none") or "none") != "none":
                raise ValueError("weighted BCE fits are not fused; use mode='none'")
            return cls("bce")
        if name == "UnariesWeightedLoss":
            return cls("mse", mode=getattr(criterion, "mode", "none") or "none", ratio=float(getattr(criterion, "ratio", 1.0) or 1.0))
        if name in ("SE", "MSELoss"):
            return cls("mse")
        raise ValueError(f"criterion {name} has no fused equivalent; pass an awesome_b200.LossConfig")

    def to_specs(self, target: torch.Tensor) -> List[L.LossSpec]:
        """target ``[O,N]``.  Folds 1/N, class weights and fg/bg means into two coefficients per object."""
        O, N = target.shape
        specs = []
        if self.kind == "mse":
            if self.mode == "none":
                return [L.LossSpec(L.AWB_LOSS_SE_SIGMOID, L.AWB_CLS_UNARY_LT_HALF, 1.0 / N, 1.0 / N) for _ in range(O)]
            cnt = target_counts(target, L.AWB_CLS_UNARY_LT_HALF, O).cpu()
            for o in range(O):
                fg, bg = float(cnt[o, 0]), float(cnt[o, 1])
                cc = torch.tensor(bg, dtype=torch.float32) / torch.tensor(fg, dtype=torch.float32)
                if self.mode == "ratio":
                    w = (cc - 1) * self.ratio + 1
                elif self.mode == "sssdms":
                    w = torch.round(cc / 10) + 1
                elif self.mode == "equal":
                    w = cc
                else:
                    raise ValueError(f"Mode {self.mode} is not supported")
                specs.append(L.LossSpec(L.AWB_LOSS_SE_SIGMOID, L.AWB_CLS_UNARY_LT_HALF, float(w) / N, 1.0 / N))
            return specs
        if self.kind == "bce":     # UnariesWeightedLoss(nn.BCELoss(), mode="none") on sigmoid(y), soft targets allowed
            return [L.LossSpec(L.AWB_LOSS_BCE_LOGITS, L.AWB_CLS_UNARY_LT_HALF, 1.0 / N, 1.0 / N) for _ in range(O)]
        if self.kind in ("fgbg_se", "fgbg_bce_logits"):
            cnt = target_counts(target, L.AWB_CLS_NOT_ONE, O).cpu()
            k = L.AWB_LOSS_SE_SIGMOID if self.kind == "fgbg_se" else L.AWB_LOSS_BCE_LOGITS
            for o in range(O):
                fg, bg = float(cnt[o, 0]), float(cnt[o, 1])
                specs.append(L.LossSpec(k, L.AWB_CLS_NOT_ONE, self.fg_weight / max(fg, 1.0),
                                        (1.0 - self.fg_weight) / max(bg, 1.0)))
            return specs
        raise ValueError(f"unknown loss kind {self.kind!r}")


@dataclass
class OptimConfig:
    """``torch.optim.Adam`` / ``Adamax`` hyper-parameters with the reference's parameter groups
    (0 flow_net, 1 convex_net, 2 linear; ``path_connected_net.py:923-929``) and the optional
    ``ReduceLROnPlateau(patience=200, factor=0.5)`` stepped on the loss every iteration (``:932-953``)."""
    kind: str = "adam"
    lr: Union[float, Sequence[float]] = 1e-3
    betas: Sequence[float] = (0.9, 0.999)
    eps: float = 1e-8
    weight_decay: Union[float, Sequence[float]] = 0.0
    plateau: bool = False
    patience: int = 200
    factor: float = 0.5
    threshold: float = 1e-4
    min_lr: float = 0.0
    plateau_eps: float = 1e-8

    def _per_group(self, v) -> List[float]:
        if isinstance(v, (int, float)):
            return [float(v)] * L.AWB_MAX_GROUPS
        v = list(v) + [0.0] * L.AWB_MAX_GROUPS
        return [float(x) for x in v[:L.AWB_MAX_GROUPS]]

    def lrs(self) -> List[float]:
        return self._per_group(self.lr)

    def to_c(self) -> L.OptHyper:
        kind = {"adam": L.AWB_OPT_ADAM, "adamax": L.AWB_OPT_ADAMAX}[self.kind.lower()]
        wd = (C.c_float * L.AWB_MAX_GROUPS)(*self._per_group(self.weight_decay))
        return L.OptHyper(kind, self.betas[0], self.betas[1], self.eps, wd, int(self.plateau), self.patience,
                          self.factor, self.threshold, self.min_lr, self.plateau_eps, 0)


class PriorFitter:
    """Fits ``prior`` (a native handle) to ``target`` on ``grid`` in place on ``params``.

    params ``[O,P]`` fp32 CUDA (the module's arena), target ``[O,N]`` fp32 CUDA.
    ``run(steps)`` replays CUDA graphs of ``steps_per_graph`` fused steps.
    """

    def __init__(self, prior: Prior, params: torch.Tensor, grid: GridSpecHost, target: torch.Tensor,
                 loss: LossConfig, optim: OptimConfig, steps_per_graph: int = 25, use_graph: bool = True):
        L.require_cuda()
        self.prior, self.params, self.grid = prior, params, grid
        self.device = params.device
        O = prior.n_objects
        self.target = target.detach().reshape(O, -1).contiguous().float()
        if self.target.shape[1] != grid.n_pixels:
            raise ValueError(f"target has {self.target.shape[1]} pixels per object, grid has {grid.n_pixels}")
        if params.numel() != O * prior.n_params or params.dtype != torch.float32 or not params.is_contiguous():
            raise ValueError("params must be a contiguous fp32 [O,P] arena")
        self.lib = prior.lib
        with torch.cuda.device(self.device):
            self.ws = prior.new_workspace(grid.n_pixels, L.AWB_WS_FIT_STEP, self.device)
            self.opt_state = torch.empty(prior.opt_state_bytes(), dtype=torch.uint8, device=self.device)
            self._specs_list = loss.to_specs(self.target)
        self._specs = (L.LossSpec * O)(*self._specs_list)
        self._hyper = optim.to_c()
        self._gs = grid.to_c()
        self.optim = optim
        self.K = max(1, int(steps_per_graph))
        self.use_graph = use_graph
        self._ring = torch.zeros((self.K, O), dtype=torch.float32, device=self.device)
        self._graph = None
        self._pool = None
        self._run_pos = 0
        self.steps_done = 0
        self.reset_optimizer()

    def reset_optimizer(self) -> None:
        """Fresh optimizer + scheduler, as the reference creates per frame (``path_connected_net.py:923-933``)."""
        lrs = (C.c_double * L.AWB_MAX_GROUPS)(*self.optim.lrs())
        with torch.cuda.device(self.device):
            L.check(self.lib.awb_opt_state_init(self.prior.handle, self.opt_state.data_ptr(), lrs, L.stream_ptr()))
        self.steps_done = 0

    def set_target(self, target: torch.Tensor, loss: Optional[LossConfig] = None) -> None:
        """New unaries for the same shapes (next frame): reuses workspace, graph and state buffers."""
        self.target.copy_(target.detach().reshape(self.target.shape))
        if loss is not None:
            with torch.cuda.device(self.device):
                specs = loss.to_specs(self.target)
            changed = any((a.kind, a.cls_rule, a.coef_fg, a.coef_bg) != (b.kind, b.cls_rule, b.coef_fg, b.coef_bg)
                          for a, b in zip(specs, self._specs_list))
            if changed:
                self._specs_list = specs
                self._specs = (L.LossSpec * len(specs))(*specs)
                self._graph = None      # coefficients are baked into the captured launches

    def _step(self, k: int, reuse: bool = False) -> None:
        """One fused step.  ``reuse``: this call directly follows another ``_step`` of this fitter inside the
        same loop (nobody else can have written the parameters), so the packed weights may be reused."""
        loss_ptr = self._ring.data_ptr() + 4 * k * self.prior.n_objects
        L.check(self.lib.awb_prior_fit_step(self.prior.handle, self.params.data_ptr(), self.opt_state.data_ptr(),
                                            C.byref(self._gs), self._target_ptr(k), self._specs,
                                            C.byref(self._hyper), loss_ptr, self.ws.data_ptr(), self.ws.numel(),
                                            L.AWB_FIT_REUSE_PACKED if reuse else 0, L.stream_ptr()))

    def set_target_pool(self, pool: Optional[torch.Tensor]) -> None:
        """Fit against a rotating pool of targets ``[F,O,N]``: step ``s`` uses frame ``s % F`` (multi-frame fitting of
        one prior; also what ``bench.py`` uses to keep the per-step input out of the L2 cache)."""
        if pool is not None:
            if pool.dim() != 3 or pool.shape[1:] != self.target.shape or pool.dtype != torch.float32 \
                    or not pool.is_contiguous() or pool.device != self.device:
                raise ValueError("target pool must be a contiguous fp32 [F,O,N] tensor on the fitter's device")
        self._pool = pool
        self._graph = None

    def _target_ptr(self, k: int) -> int:
        pool = getattr(self, "_pool", None)
        if pool is None:
            return self.target.data_ptr()
        f = (self.steps_done + self._run_pos + k) % pool.shape[0]
        return pool.data_ptr() + 4 * f * pool.shape[1] * pool.shape[2]

    def _capture(self, n_steps: Optional[int] = None) -> None:
        n = self.K if n_steps is None else int(n_steps)
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            self._step(0)          # warm-up outside capture (module load, lazy init)
        torch.cuda.current_stream(self.device).wait_stream(s)
        torch.cuda.synchronize(self.device)
        # the warm-up step must not count: restore by re-running from a snapshot
        with torch.cuda.graph(g, stream=s):
            for k in range(n):
                self._step(k, reuse=k > 0)
        self._graph = g
        self._graph_steps = n

    def run(self, steps: int, record: bool = True) -> Optional[torch.Tensor]:
        """Run ``steps`` fused fit steps.  Returns the device loss history ``[steps,O]`` (no sync)."""
        hist = torch.empty((steps, self.prior.n_objects), dtype=torch.float32, device=self.device) if record else None
        done = 0
        self._run_pos = 0
        if self._pool is not None and not record:
            return self._run_pool_native(steps)
        use_graph = self.use_graph and self._pool is None     # a captured graph bakes the target pointer
        with torch.cuda.device(self.device):
            if use_graph and steps >= self.K and self._graph is None:
                snap_p, snap_o = self.params.clone(), self.opt_state.clone()
                self._capture()
                self.params.copy_(snap_p)
                self.opt_state.copy_(snap_o)
            while use_graph and self._graph is not None and steps - done >= self.K:
                self._graph.replay()
                if record:
                    hist[done:done + self.K].copy_(self._ring)
                done += self.K
            first = True
            while done < steps:
                self._run_pos = done
                self._step(0, reuse=not first)
                first = False
                if record:
                    hist[done].copy_(self._ring[0])
                done += 1
        self._run_pos = 0
        self.steps_done += steps
        return hist

    def _run_pool_native(self, steps: int) -> None:
        """Target pool, no history: ONE native call runs all ``steps`` fused steps with the rotating device targets
        (``awb_prior_fit_steps``) -- no Python / ctypes round trip per step.  (Replaying a captured CUDA graph of a pool
        rotation was measured 26 % slower than host launches on B200: the programmatic-dependent-launch overlap between the
        two kernels of a step does not survive capture.)"""
        F = int(self._pool.shape[0])
        stride = 4 * self._pool.shape[1] * self._pool.shape[2]
        ptrs = (C.c_void_p * F)(*[self._pool.data_ptr() + f * stride for f in range(F)])
        with torch.cuda.device(self.device):
            L.check(self.lib.awb_prior_fit_steps(self.prior.handle, self.params.data_ptr(), self.opt_state.data_ptr(),
                                                 C.byref(self._gs), ptrs, F, self.steps_done % F, int(steps), self._specs,
                                                 C.byref(self._hyper), None, self.ws.data_ptr(), self.ws.numel(), 0,
                                                 L.stream_ptr()))
        self.steps_done += steps
        return None

    def run_host_frames(self, host_frames: Sequence[torch.Tensor], steps: Optional[int] = None) -> torch.Tensor:
        """``steps`` fused fit steps whose unaries arrive from HOST memory: step ``s`` fits
        ``host_frames[s % len(host_frames)]`` (each ``[O,N]`` fp32; pinned memory makes the copy overlap).  One native
        call (``awb_prior_fit_host_frames``): the host->device copy of the next frame runs on a copy stream into a
        double-buffered staging area while the current step computes, and the optimizer kernel stores every step's
        loss straight into pinned host memory.  Returns that pinned ``[steps,O]`` tensor; it is valid after the
        current stream is synchronised (this method does not block)."""
        O, N = self.target.shape
        frames = [f.detach().reshape(O, N) for f in host_frames]
        for f in frames:
            if f.device.type != "cpu" or f.dtype != torch.float32 or not f.is_contiguous():
                raise ValueError("host frames must be contiguous fp32 CPU tensors of the fitter's [O,N] shape")
        steps = len(frames) if steps is None else int(steps)
        losses = torch.empty((max(steps, 1), O), dtype=torch.float32).pin_memory()
        if getattr(self, "_staging", None) is None:
            self._staging = torch.empty((2, O, N), dtype=torch.float32, device=self.device)
        ptrs = (C.c_void_p * len(frames))(*[f.data_ptr() for f in frames])
        with torch.cuda.device(self.device):
            L.check(self.lib.awb_prior_fit_host_frames(
                self.prior.handle, self.params.data_ptr(), self.opt_state.data_ptr(), C.byref(self._gs), ptrs, len(frames),
                steps, self._specs, C.byref(self._hyper), losses.data_ptr(), self._staging.data_ptr(), self.ws.data_ptr(),
                self.ws.numel(), 0, L.stream_ptr()))
        self._host_keepalive = (frames, losses)     # the copies are still in flight when this returns
        self.steps_done += steps
        return losses[:steps]

    def scalars(self, obj: int = 0) -> L.OptScalars:
        """Synchronises and returns step / lr / plateau / non-finite flag of one object."""
        out = L.OptScalars()
        with torch.cuda.device(self.device):
            L.check(self.lib.awb_opt_read_scalars(self.prior.handle, self.opt_state.data_ptr(), obj, C.byref(out),
                                                  L.stream_ptr()))
        return out

    def raise_if_nonfinite(self) -> None:
        """Reference behaviour: ``ValueError("Loss is nan or inf!")`` (``path_connected_net.py:232,374,456,702``)."""
        for o in range(self.prior.n_objects):
            if self.scalars(o).nonfinite:
                raise ValueError("Loss is nan or inf!")


class FlowIdentityFitter(PriorFitter):
    """``PathConnectedNet.learn_flow_identity`` (``path_connected_net.py:155-250``) as fused steps:
    flow-only forward (no 1x1 conv), SE("mean") against the input grid, Adamax on the flow group."""

    def __init__(self, prior: Prior, params: torch.Tensor, grid: GridSpecHost, optim: OptimConfig,
                 steps_per_graph: int = 25, use_graph: bool = True):
        L.require_cuda()
        self.prior, self.params, self.grid = prior, params, grid
        self.device = params.device
        self.lib = prior.lib
        with torch.cuda.device(self.device):
            self.ws = prior.new_workspace(grid.n_pixels, L.AWB_WS_TRAINING, self.device)
            self.opt_state = torch.empty(prior.opt_state_bytes(), dtype=torch.uint8, device=self.device)
        self._hyper = optim.to_c()
        self._gs = grid.to_c()
        self.optim = optim
        self.K = max(1, int(steps_per_graph))
        self.use_graph = use_graph
        self._ring = torch.zeros((self.K, prior.n_objects), dtype=torch.float32, device=self.device)
        self._graph = None
        self._pool = None
        self._run_pos = 0
        self.steps_done = 0
        self.reset_optimizer()

    def _step(self, k: int, reuse: bool = False) -> None:
        loss_ptr = self._ring.data_ptr() + 4 * k * self.prior.n_objects
        L.check(self.lib.awb_flow_identity_step(self.prior.handle, self.params.data_ptr(), self.opt_state.data_ptr(),
                                                C.byref(self._gs), C.byref(self._hyper), loss_ptr,
                                                self.ws.data_ptr(), self.ws.numel(), L.stream_ptr()))


# ------------------------------------------------------------------ pixel-sliced fit step (one prior on several GPUs)
SLICE_ALIGN = 128     # one tile of the tensor path


def slice_plan(n_rows: int, n_slices: int) -> List[tuple]:
    """Cut the pixel rows ``[0, n_rows)`` of a step's batch into ``n_slices`` contiguous ``(begin, end)`` slices.

    Boundaries lie on multiples of 128 rows (except ``n_rows`` itself) and slice sizes differ by at most 128: slice ``k``
    gets tiles ``[k T // S, (k + 1) T // S)`` of the ``T = ceil(n_rows / 128)`` tiles, so the last slice, which holds
    the partial tile, is one of the larger ones.  With fewer tiles than slices some slices are empty (``begin == end``);
    their gradient row is zero.  The plan depends on ``n_rows`` and ``n_slices`` only, never on the number of ranks."""
    if n_slices < 1:
        raise ValueError(f"n_slices must be >= 1, got {n_slices}")
    if n_rows < 1:
        raise ValueError(f"n_rows must be >= 1, got {n_rows}")
    tiles = (n_rows + SLICE_ALIGN - 1) // SLICE_ALIGN
    cuts = [min(n_rows, (k * tiles // n_slices) * SLICE_ALIGN) for k in range(n_slices + 1)]
    return [(cuts[k], cuts[k + 1]) for k in range(n_slices)]


def rank_slices(n_slices: int, rank: int, world: int) -> range:
    """The slices rank ``rank`` of ``world`` computes: ``[rank S / world, (rank + 1) S / world)``."""
    if world < 1 or not 0 <= rank < world:
        raise ValueError(f"bad rank {rank} of world {world}")
    if n_slices % world:
        raise ValueError(f"the number of slices ({n_slices}) must be a multiple of the number of ranks ({world})")
    per = n_slices // world
    return range(rank * per, (rank + 1) * per)


def gather_slice_rows(mine: Sequence[int], local: torch.Tensor, rows: torch.Tensor, produce, group=None) -> torch.Tensor:
    """One sliced step up to the optimizer: ``produce(k, local[j], j)`` writes the row of this rank's ``j``-th slice ``k``
    into ``local``, then ``all_gather_into_tensor`` gives every rank all ``[S, R]`` rows in slice order (a copy: every rank
    holds the same bits).  ``local`` may be ``rows`` itself (one rank: no collective)."""
    for j, k in enumerate(mine):
        produce(k, local[j], j)
    if local.data_ptr() != rows.data_ptr() or local.shape != rows.shape:
        import torch.distributed as dist
        dist.all_gather_into_tensor(rows, local, group=group)
    return rows


class SlicedFitter:
    """The fused fit step of ``PriorFitter`` computed in pixel slices, for fitting ONE prior on several GPUs.

    The batch's pixel rows are cut into ``n_slices`` slices (``slice_plan``); this rank computes the gradient rows of its
    slices (``rank_slices``), the rows of all ranks are gathered in slice order over ``group`` and every rank runs the same
    optimizer kernel on the same rows.  The parameters after any number of steps are therefore bit-identical for every
    ``world`` dividing ``n_slices``, and on every rank; a one-rank run computes all slices one after the other.

    The loss is the full batch's (coefficients from ``loss.to_specs`` on the whole target), so the rows add up to the
    fused step's gradient and loss up to summation order.  Single-object ICNN and RealNVP o ICNN priors."""

    def __init__(self, prior: Prior, params: torch.Tensor, grid: GridSpecHost, target: torch.Tensor,
                 loss: LossConfig, optim: OptimConfig, n_slices: int = 8, group=None):
        L.require_cuda()
        if prior.n_objects != 1:
            raise ValueError("sliced fits take single-object priors")
        if group is not None:
            import torch.distributed as dist
            rank, world = dist.get_rank(group), dist.get_world_size(group)
        else:
            rank, world = 0, 1
        self.mine = rank_slices(int(n_slices), rank, world)        # raises unless world divides n_slices
        self.prior, self.params, self.group = prior, params, group
        self.n_slices = int(n_slices)
        self.device = params.device
        self.lib = prior.lib
        self.target = target.detach().reshape(1, -1).contiguous().float()
        if self.target.shape[1] != grid.n_pixels:
            raise ValueError(f"target has {self.target.shape[1]} pixels, grid has {grid.n_pixels}")
        if params.numel() != prior.n_params or params.dtype != torch.float32 or not params.is_contiguous():
            raise ValueError("params must be a contiguous fp32 [1,P] arena")
        self.grid = grid
        self.plan = slice_plan(grid.n_pixels, self.n_slices)
        R = prior.grad_row_floats
        biggest = max(e - b for b, e in self.plan)
        with torch.cuda.device(self.device):
            self.ws = prior.new_workspace(biggest, L.AWB_WS_FIT_STEP, self.device)   # one slice after the other
            self.opt_state = torch.empty(prior.opt_state_bytes(), dtype=torch.uint8, device=self.device)
            self.rows = torch.zeros((self.n_slices, R), dtype=torch.float32, device=self.device)   # empty slices stay 0
            self.local = self.rows if world == 1 else torch.zeros((len(self.mine), R), dtype=torch.float32,
                                                                   device=self.device)
            self._spec = loss.to_specs(self.target)[0]
        self._hyper = optim.to_c()
        self.optim = optim
        self.steps_done = 0
        self.reset_optimizer()

    def reset_optimizer(self) -> None:
        lrs = (C.c_double * L.AWB_MAX_GROUPS)(*self.optim.lrs())
        with torch.cuda.device(self.device):
            L.check(self.lib.awb_opt_state_init(self.prior.handle, self.opt_state.data_ptr(), lrs, L.stream_ptr()))
        self.steps_done = 0

    def set_target(self, target: torch.Tensor) -> None:
        """New unaries for the same grid shape; the loss coefficients are kept (as ``PriorFitter.set_target``)."""
        self.target.copy_(target.detach().reshape(self.target.shape))

    def _produce(self, k: int, row: torch.Tensor, j: int) -> None:
        b, e = self.plan[k]
        if j == 0:
            self._packed = 0            # the parameters have changed since the last slice
        if b == e:
            row.zero_()
            return
        # the weight image sits at an offset of the workspace that depends on the window's row count
        self.prior.slice_grads(self.params, self.grid, b, e, self.target, self._spec, row, self.ws,
                               reuse_packed=self._packed == e - b)
        self._packed = e - b

    def step(self, loss_out: Optional[torch.Tensor] = None) -> None:
        """One sliced step; ``loss_out`` (optional, one device float) receives the step's loss.  No host sync."""
        with torch.cuda.device(self.device):
            rows = gather_slice_rows(self.mine, self.local, self.rows, self._produce, self.group)
            self.prior.rows_opt_step(self.params, self.opt_state, rows, self._hyper, loss_out)
        self.steps_done += 1

    def run(self, steps: int) -> torch.Tensor:
        """``steps`` sliced steps.  Returns the device loss history ``[steps, 1]`` (written by the optimizer kernel)."""
        hist = torch.empty((steps, 1), dtype=torch.float32, device=self.device)
        for s in range(steps):
            self.step(hist[s])
        return hist

    def scalars(self, obj: int = 0) -> L.OptScalars:
        out = L.OptScalars()
        with torch.cuda.device(self.device):
            L.check(self.lib.awb_opt_read_scalars(self.prior.handle, self.opt_state.data_ptr(), obj, C.byref(out),
                                                  L.stream_ptr()))
        return out

    def raise_if_nonfinite(self) -> None:
        if self.scalars(0).nonfinite:
            raise ValueError("Loss is nan or inf!")
