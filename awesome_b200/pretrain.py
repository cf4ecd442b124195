"""The reference's per-frame / per-sequence pretrain loops as fused fits (SURVEY a12):

* ``fit_frames``  -- ``PathConnectedNet._prior_based_pretrain`` (``awesome/model/path_connected_net.py:730-1007``):
  one prior state per frame, optional warm start from the previous frame (``reuse_state``), optional prefits
  (``learn_flow_identity`` / ``learn_convex_net``), the main Adamax + ReduceLROnPlateau fit, the "proper prior fit"
  IoU check with retry after ``reset_parameters`` (``:964-982``), the no-foreground skip (``:848-855``).
* ``fit_sequence`` -- ``_non_prior_based_pretrain`` (``:511-728``): ONE (x, y, t) prior for all frames, batches of
  ``batch_size`` frames per step, ``num_epochs`` passes.

Every inner loop is ``PriorFitter.run`` (one native call per step, replayed from CUDA graphs); the host only sees a
frame once per fit, not once per step.  ``pretrain`` / ``pretrain_load_state`` glue these into the reference's
``PretrainableModule`` protocol (``awesome/model/pretrainable_module.py:16-82``) by duck-typing the agent, dataset
and wrapper module the reference hands in."""
from __future__ import annotations

import logging
from dataclasses import dataclass, field
from typing import Any, Callable, Dict, Iterable, List, Optional, Sequence

import torch

from . import _lib as L
from .core import GridSpecHost, iou_counts, target_counts
from .fit import LossConfig, OptimConfig, PriorFitter, SlicedFitter


@dataclass
class FitSchedule:
    """The recognised ``pretrain_args`` (``path_connected_net.py:536-560,756-786``) with the reference defaults."""
    num_epochs: int = 2000
    lr: float = 1e-3
    flow_weight_decay: float = 1e-5
    reuse_state: bool = True
    reuse_state_epochs: int = 200
    batch_size: int = 1
    dataloader_shuffle: bool = False     # spatio-temporal loop: shuffled frame batches per epoch (:550, :654)
    noisy_percentage: float = 0.0        # NoisyPathConnectedNet (noisy_path_connected_net.py:87): frames with noise unaries
    unet_batch_size: int = 8             # N1: frames per frozen-UNet inference call when collecting the unaries
    prefit_flow_net_identity: bool = False
    prefit_flow_net_identity_lr: float = 1e-2
    prefit_flow_net_identity_weight_decay: float = 1e-5
    prefit_flow_net_identity_num_epochs: int = 100
    prefit_convex_net: bool = False
    prefit_convex_net_lr: float = 1e-3
    prefit_convex_net_weight_decay: float = 0.0
    prefit_convex_net_num_epochs: int = 200
    proper_prior_fit_threshold: float = 0.5
    proper_prior_fit_retrys: int = 1
    criterion: LossConfig = field(default_factory=lambda: LossConfig("mse"))
    weight_decay_on_weight_g: float = 0.0    # ConvexDiffeomorphismNet.pretrain decays only the weight-norm gains
    optimizer: str = "adamax"            # the pretrain loops use Adamax + plateau(200, 0.5) (:929-933)
    plateau: bool = True
    plateau_patience: int = 200          # ReduceLROnPlateau(patience=200, factor=0.5) in every pretrain loop (:644, :932)
    plateau_factor: float = 0.5
    plateau_threshold: float = 1e-4      # torch default (rel)
    steps_per_graph: int = 50
    sequence_slices: int = 0             # spatio-temporal loop: pixel slices per step across the ranks of torch.distributed
                                         # (0 = off; used by pretrain() when a process group is initialised)

    @classmethod
    def from_pretrain_args(cls, kwargs: Dict[str, Any]) -> "FitSchedule":
        known = {f for f in cls.__dataclass_fields__}
        vals = {k: v for k, v in kwargs.items() if k in known and k != "criterion"}
        s = cls(**vals)
        crit = kwargs.get("criterion")
        if crit is not None:
            s.criterion = crit if isinstance(crit, LossConfig) else LossConfig.from_reference(crit)
        return s

    def optim(self, has_flow: bool) -> OptimConfig:
        wd = [self.flow_weight_decay if has_flow else 0.0, 0.0, 0.0, self.weight_decay_on_weight_g]
        return OptimConfig(self.optimizer, lr=self.lr, weight_decay=wd, plateau=self.plateau, patience=self.plateau_patience,
                           factor=self.plateau_factor, threshold=self.plateau_threshold)


@dataclass
class FrameResult:
    index: int
    skipped: bool = False
    iou: float = -1.0
    proper_fit: bool = False
    retries: int = 0
    steps: int = 0
    final_loss: float = float("nan")
    state: Optional[torch.Tensor] = None      # the fitted arena (device), one row
    mask_fg: Optional[torch.Tensor] = None    # fitted foreground mask (bool, device, flat), when ``keep_masks``


def _as_grid(grid, device) -> GridSpecHost:
    if isinstance(grid, GridSpecHost):
        return grid
    g = grid.to(device)
    return GridSpecHost.from_tensor(g)


def mask_iou(pred_prob: torch.Tensor, target_prob: torch.Tensor) -> float:
    """``MIOU(average="binary", invert=True)`` on masks thresholded at 0.5 (``awesome/measures/miou.py:29-48``):
    Jaccard of the foreground (value <= 0.5); 0 when the target has no foreground.  Exact integer counts on device."""
    c = iou_counts(pred_prob, target_prob, pred_is_logit=False).cpu()[0]
    inter, pf, tf = int(c[0]), int(c[1]), int(c[2])
    if tf == 0:
        return 0.0
    return inter / float(pf + tf - inter)


def fit_frames(model, grids: Sequence, unaries: Sequence[torch.Tensor], schedule: Optional[FitSchedule] = None,
               on_frame: Optional[Callable[[FrameResult], None]] = None, frame_indices: Optional[Sequence[int]] = None,
               warm_start_hook: Optional[Callable[[Any, torch.Tensor, Any], None]] = None,
               keep_masks: bool = False, initial_previous: Optional[torch.Tensor] = None) -> List[FrameResult]:
    """Fit ``model`` (ConvexNextNet or PathConnectedNet drop-in) to every frame in turn.  ``grids[i]`` is a
    ``[1,C,H,W]`` tensor or ``GridSpecHost``; ``unaries[i]`` the frame's soft segmentation (any shape with H*W
    elements; convention fg = 0, bg = 1 like the reference).  The model ends holding the last proper state."""
    s = schedule or FitSchedule()
    arena = model._ensure_flat()
    dev = arena.device
    has_flow = hasattr(model, "flow_net")
    flow_group = has_flow or hasattr(model, "diffeo_net")
    results: List[FrameResult] = []
    previous: Optional[torch.Tensor] = initial_previous      # a proper state carried in from an earlier call / a checkpoint
    fitter: Optional[PriorFitter] = None
    fitter_key = None
    for k, (grid, un) in enumerate(zip(grids, unaries)):
        idx = frame_indices[k] if frame_indices is not None else k
        res = FrameResult(index=idx)
        un = un.detach().to(dev).float().reshape(1, -1)
        spec = _as_grid(grid, dev)
        cnt = target_counts(un, L.AWB_CLS_UNARY_LT_HALF).cpu()[0]
        if int(cnt[0]) == 0 or int(cnt[1]) == 0:       # torch.unique(unaries >= 0.5) has one value (:848-855)
            logging.warning("Unaries of segmentation model contain no foreground. Skipping image. %s", idx)
            res.skipped = True
            results.append(res)
            if on_frame:
                on_frame(res)
            continue
        warm = s.reuse_state and previous is not None
        if warm:
            with torch.no_grad():
                arena.copy_(previous)
            if warm_start_hook is not None:
                warm_start_hook(model, un, spec)         # e.g. centre-of-mass re-translation of the diffeomorphism prior
        else:
            if has_flow and s.prefit_flow_net_identity:
                model.learn_flow_identity(spec.materialize(model.in_channels, dev), lr=s.prefit_flow_net_identity_lr,
                                          weight_decay=s.prefit_flow_net_identity_weight_decay,
                                          max_iter=s.prefit_flow_net_identity_num_epochs, use_progress_bar=False)
            if has_flow and s.prefit_convex_net:
                model.learn_convex_net(spec.materialize(model.in_channels, dev), un.reshape(spec.B, 1, spec.H, spec.W),
                                       lr=s.prefit_convex_net_lr, weight_decay=s.prefit_convex_net_weight_decay,
                                       max_iter=s.prefit_convex_net_num_epochs, use_progress_bar=False)
        if has_flow:
            model._maybe_actnorm_init(spec.materialize(model.in_channels, dev))
        key = (spec.mode, spec.B, spec.H, spec.W, spec.t0, spec.t_step, id(spec.grid))
        if fitter is None or fitter_key != key:
            fitter = model.make_fitter(spec, un, s.criterion, s.optim(flow_group), steps_per_graph=s.steps_per_graph)
            fitter_key = key
        else:
            fitter.set_target(un, s.criterion)
        proper = False
        while not proper and res.retries <= s.proper_prior_fit_retrys:
            epochs = s.reuse_state_epochs if (warm and res.retries == 0) else s.num_epochs
            fitter.reset_optimizer()                   # fresh optimizer + scheduler per attempt (:923-933)
            hist = fitter.run(epochs)
            fitter.raise_if_nonfinite()
            res.steps += epochs
            res.final_loss = float(hist[-1, 0]) if epochs > 0 else float("nan")
            with torch.no_grad():
                prob = torch.sigmoid(model(spec.materialize(getattr(model, "in_channels", getattr(model, "in_features", 2)), dev)))
            res.iou = mask_iou(prob.reshape(1, -1), un)
            if keep_masks:
                res.mask_fg = (prob.reshape(-1) <= 0.5)
            proper = res.iou >= s.proper_prior_fit_threshold
            if not proper and res.retries < s.proper_prior_fit_retrys:
                logging.info("Prior fit not proper on image index: %s. Retrying. Metric: %s", idx, res.iou)
                model.reset_parameters()
                model._ensure_flat()
                if has_flow:
                    model._maybe_actnorm_init(spec.materialize(model.in_channels, dev))
            res.retries += 1
        res.retries -= 1
        res.proper_fit = proper
        res.state = model._ensure_flat().detach().clone()
        if s.reuse_state and proper:
            previous = res.state
        results.append(res)
        if on_frame:
            on_frame(res)
    return results


def fit_frames_grouped(multi, grid, unaries: Sequence[torch.Tensor], schedule: Optional[FitSchedule] = None,
                       on_frame: Optional[Callable[[FrameResult], None]] = None,
                       frame_indices: Optional[Sequence[int]] = None, keep_masks: bool = False) -> List[FrameResult]:
    """``fit_frames`` for frames that are fitted WITHOUT chaining inside a group: ``multi`` (a
    ``NumberBasedMultiPriorModule`` of G equal priors) takes G frames per fused launch, one prior per frame -- the
    execution that ``bench.py`` measures (G = 4: one wave of 37 persistent CTAs per frame, see DESIGN 3h).

    Semantics relative to the reference's loop (``path_connected_net.py:730-1007``): the reference carries the module
    state from frame to frame (explicitly with ``reuse_state``, implicitly otherwise).  Here every frame of a group starts
    from the state the group was entered with -- the last proper state of the previous group under ``reuse_state`` (then
    ``reuse_state_epochs`` steps), else the state of ``multi.priors[0]`` at the call (``num_epochs`` steps) -- exactly the
    cut that sharding frames over GPUs makes at shard boundaries.  The no-foreground skip, the "proper prior fit" IoU check
    and its retry after ``reset_parameters`` (per frame, through the one-frame path) are the reference's.  All frames
    share ``grid`` (a ``GridSpecHost`` or ``[1,C,H,W]`` tensor).  Priors with a flow need their prefits per frame and are
    not grouped here."""
    s = schedule or FitSchedule()
    G = len(multi.priors)
    if G < 1:
        raise ValueError("the container holds no priors")
    if any(hasattr(p, "flow_net") or hasattr(p, "diffeo_net") for p in multi.priors):
        raise NotImplementedError("grouped frame fits are for priors without a flow (use fit_frames)")
    big = multi._group_arena()
    dev = big.device
    spec = _as_grid(grid, dev)
    entry = big[0].detach().clone()
    previous: Optional[torch.Tensor] = None
    results: List[FrameResult] = []
    todo: List[tuple] = []
    for k, un in enumerate(unaries):
        idx = frame_indices[k] if frame_indices is not None else k
        un = un.detach().to(dev).float().reshape(1, -1)
        cnt = target_counts(un, L.AWB_CLS_UNARY_LT_HALF).cpu()[0]
        if int(cnt[0]) == 0 or int(cnt[1]) == 0:       # torch.unique(unaries >= 0.5) has one value (:848-855)
            logging.warning("Unaries of segmentation model contain no foreground. Skipping image. %s", idx)
            results.append(FrameResult(index=idx, skipped=True))
            if on_frame:
                on_frame(results[-1])
        else:
            todo.append((idx, un))
    # the fitter (workspace, optimizer state, captured CUDA graphs) is kept on the container between calls: a rank that
    # fits one segment of the sequence after the other pays for the capture once
    fkey = tuple(getattr(spec, a, None) for a in ("mode", "B", "H", "W", "t0", "t_step")) + (
        id(getattr(spec, "grid", None)), big.data_ptr(), s.optimizer, s.lr, s.plateau, s.steps_per_graph, s.criterion.kind,
        s.criterion.mode)
    cached = getattr(multi, "_grouped_fitter", None)
    fitter: Optional[PriorFitter] = cached[1] if cached is not None and cached[0] == fkey else None
    C_in = getattr(multi.priors[0], "in_channels", getattr(multi.priors[0], "in_features", 2))
    for g0 in range(0, len(todo), G):
        chunk = todo[g0:g0 + G]
        n_real = len(chunk)
        chunk = chunk + [chunk[-1]] * (G - n_real)          # a short last group repeats its last frame (result ignored)
        tg = torch.cat([u for _, u in chunk], dim=0)
        warm = s.reuse_state and previous is not None
        with torch.no_grad():
            big.copy_((previous if warm else entry).unsqueeze(0).expand_as(big))
        if fitter is None:
            fitter = multi.make_fitter(spec, tg, s.criterion, s.optim(False), steps_per_graph=s.steps_per_graph)
            multi._grouped_fitter = (fkey, fitter)
        else:
            fitter.set_target(tg, s.criterion)
        epochs = s.reuse_state_epochs if warm else s.num_epochs
        fitter.reset_optimizer()                           # fresh optimizer + scheduler per frame (:923-933)
        hist = fitter.run(epochs)
        fitter.raise_if_nonfinite()
        with torch.no_grad():
            logits = multi(spec.materialize(C_in, dev), num_priors=G)           # [1,G,1,H,W]
        cnts = iou_counts(logits.reshape(G, -1), tg, pred_is_logit=True, n_objects=G).cpu()
        for k in range(n_real):
            idx, un = chunk[k]
            res = FrameResult(index=idx, steps=epochs, final_loss=float(hist[-1, k]) if epochs > 0 else float("nan"))
            inter, pf, tf = int(cnts[k, 0]), int(cnts[k, 1]), int(cnts[k, 2])
            res.iou = 0.0 if tf == 0 else inter / float(pf + tf - inter)
            res.proper_fit = res.iou >= s.proper_prior_fit_threshold
            if keep_masks:
                res.mask_fg = logits.reshape(G, -1)[k] <= 0
            if not res.proper_fit and s.proper_prior_fit_retrys > 0:
                # the reference's retry: reset_parameters, full schedule -- per frame, through the one-frame path
                logging.info("Prior fit not proper on image index: %s. Retrying. Metric: %s", idx, res.iou)
                pk = multi.priors[k]
                pk.reset_parameters()
                pk._ensure_flat()
                import dataclasses
                again = fit_frames(pk, [spec], [un], dataclasses.replace(s, reuse_state=False,
                                                                         proper_prior_fit_retrys=s.proper_prior_fit_retrys - 1),
                                   frame_indices=[idx], keep_masks=keep_masks)[0]
                multi._arena_all = None                       # the one-frame path may have re-pointed the prior's arena
                big = multi._group_arena()
                fitter = None
                multi._grouped_fitter = None
                res.mask_fg = again.mask_fg
                res.retries = 1 + again.retries
                res.steps += again.steps
                res.iou, res.proper_fit, res.final_loss = again.iou, again.proper_fit, again.final_loss
            res.state = big[k].detach().clone()
            if s.reuse_state and res.proper_fit:
                previous = res.state
            results.append(res)
            if on_frame:
                on_frame(res)
    order = {(frame_indices[k] if frame_indices is not None else k): k for k in range(len(unaries))}
    results.sort(key=lambda r: order[r.index])
    return results


def noisy_unaries(unaries: torch.Tensor, noisy_percentage: float, seed: Optional[int] = None):
    """``NoisyPathConnectedNet._non_prior_based_pretrain`` (``awesome/model/noisy_path_connected_net.py:179-228``):
    a fraction of the frames (never the first or the last) gets its unaries replaced ONCE by
    ``clamp(randn + 0.5, 0, 1)``; the replacement is kept for every later epoch.  Returns (unaries, noisy indices)."""
    import numpy as np
    T = unaries.shape[0]
    rng = np.random.RandomState(seed) if seed is not None else np.random
    candidates = np.arange(1, T - 1)
    k = min(int(round(T * noisy_percentage)), len(candidates))
    idx = sorted(rng.choice(candidates, size=k, replace=False).tolist()) if k > 0 else []
    out = unaries.clone()
    g = torch.Generator(device=unaries.device)
    if seed is not None:
        g.manual_seed(seed)
    for i in idx:
        out[i] = torch.clamp(torch.randn(out[i].shape, device=out.device, generator=g) + 0.5, 0.0, 1.0)
    return out, idx


def _plateau_hyper(s: FitSchedule, has_flow: bool):
    o = s.optim(has_flow)
    o.plateau = True
    return o.to_c()


def fit_sequence(model, n_frames: int, H: int, W: int, unaries: torch.Tensor, schedule: Optional[FitSchedule] = None,
                 grid_mode: str = "linspace", first_last_unaries: Optional[torch.Tensor] = None,
                 lr_trace: Optional[list] = None, n_slices: Optional[int] = None, group=None) -> torch.Tensor:
    """Spatio-temporal fit (``_non_prior_based_pretrain``, ``path_connected_net.py:511-728``): ONE (x, y, t) prior for all
    frames.  ``unaries`` ``[T,H,W]``; frame ``i`` has ``t = i / (T - 1)`` (``awesome/dataset/transformator.py:54-60``).

    * prefits (``:577-631``): ``learn_flow_identity`` on the normalised ``(T, 3, H, W)`` grid in shuffled batches of
      ``batch_size`` frames, then ``learn_convex_net`` on the first and the last frame stacked (their unaries:
      ``first_last_unaries`` ``[2,H,W]``, default ``unaries[[0, -1]]``);
    * main loop (``:633-719``): ONE optimizer (Adamax, flow weight decay) for all epochs, ``num_epochs`` passes over the
      ``ceil(T / batch_size)`` frame batches (in order, or shuffled with ``dataloader_shuffle``), one fused fit step per
      batch; ``ReduceLROnPlateau.step`` ONCE PER EPOCH on the epoch-mean loss (``:719``) -- the batch steps run with the
      scheduler off and the epoch end calls ``awb_opt_plateau_step``.

    ``n_slices``: the main loop runs pixel-sliced (``SlicedFitter``): the pixel rows of every batch are cut into
    ``n_slices`` slices, spread over the ranks of ``group`` (a ``torch.distributed`` process group, ``None`` = this
    process alone), whose gradient rows are gathered and summed in slice order before the optimizer step.  The batches,
    their order and the number of optimizer steps are the reference's; only the summation order of a step's gradient
    differs from the unsliced loop, and the result is bit-identical for every number of ranks dividing ``n_slices``.  The
    prefits and the ActNorm init are not sliced: every rank runs them, and rank 0's result (arena and, with
    ``noisy_percentage``, the unaries) is then broadcast, so all ranks start the main loop from the same bits even when
    their random number generators differ.  With ``dataloader_shuffle`` rank 0 draws each epoch's permutation from the
    global RNG exactly as a one-rank run does and broadcasts it.  ``None`` keeps the unsliced fused loop.
    Returns the per-step loss history ``[num_epochs * n_batches]`` (device)."""
    import ctypes as C
    import dataclasses
    s = schedule or FitSchedule()
    arena = model._ensure_flat()
    dev = arena.device
    T, bs = int(n_frames), max(1, int(s.batch_size))
    t_step = 1.0 / (T - 1) if T > 1 else 0.0
    un = unaries.detach().to(dev).float().reshape(T, H * W)
    if s.noisy_percentage > 0:
        un, _ = noisy_unaries(un, s.noisy_percentage)
    sliced = n_slices is not None
    multi_rank = sliced and group is not None
    if multi_rank:
        import torch.distributed as dist
        src = dist.get_global_rank(group, 0)
        if s.noisy_percentage > 0:
            un = un.contiguous()
            dist.broadcast(un, src, group=group)
    has_flow = hasattr(model, "flow_net")
    C_in = getattr(model, "in_channels", getattr(model, "in_features", 2))
    full = GridSpecHost(grid_mode, T, H, W, t0=0.0, t_step=t_step)
    if has_flow and s.prefit_flow_net_identity:
        model.learn_flow_identity(full.materialize(C_in, dev), lr=s.prefit_flow_net_identity_lr,
                                  weight_decay=s.prefit_flow_net_identity_weight_decay,
                                  max_iter=s.prefit_flow_net_identity_num_epochs, use_progress_bar=False, batch_size=bs)
    if has_flow and s.prefit_convex_net:
        fl = first_last_unaries if first_last_unaries is not None else un[[0, T - 1]]
        g2 = torch.stack([GridSpecHost(grid_mode, 1, H, W, t0=0.0).materialize(C_in, dev)[0],
                          GridSpecHost(grid_mode, 1, H, W, t0=(T - 1) * t_step).materialize(C_in, dev)[0]])
        model.learn_convex_net(g2, fl.detach().to(dev).float().reshape(2, 1, H, W), mode="unaries", use_deformed_grid=True,
                               lr=s.prefit_convex_net_lr, weight_decay=s.prefit_convex_net_weight_decay,
                               max_iter=s.prefit_convex_net_num_epochs, use_progress_bar=False)
    if has_flow:
        model._maybe_actnorm_init(full.materialize(C_in, dev)[:min(bs, T)])     # first batch the full prior ever sees
    if multi_rank:
        arena = model._ensure_flat()
        dist.broadcast(arena.data, src, group=group)
    # batch steps never advance the scheduler; the epoch end does
    step_optim = dataclasses.replace(s.optim(has_flow), plateau=False)
    plateau_hy = _plateau_hyper(s, has_flow)
    n_batches = (T + bs - 1) // bs
    hist: List[torch.Tensor] = []
    first: Optional[PriorFitter] = None

    def share(f: PriorFitter) -> PriorFitter:
        nonlocal first
        if first is None:
            first = f
        else:                       # the reference builds the optimizer once, outside the loops (:633-645)
            f.opt_state = first.opt_state
            if f.ws.numel() == first.ws.numel():
                f.ws = first.ws     # batches run one after the other: one scratch area
            if sliced:              # ... and one row buffer
                f.rows, f.local = first.rows, (first.rows if first.local is first.rows else first.local)
        return f

    def make(spec: GridSpecHost, target: torch.Tensor):
        if not sliced:
            return share(model.make_fitter(spec, target, s.criterion, step_optim, use_graph=False))
        prior = model._prior_for(model._ensure_flat().device)
        return share(SlicedFitter(prior, model._ensure_flat(), spec, target, s.criterion, step_optim, n_slices=n_slices,
                                  group=group))

    def epoch_batches() -> List[torch.Tensor]:
        """The reference's DataLoader(shuffle=True) batches of this epoch (same sampler, same global-RNG stream); with
        several ranks rank 0 draws them and broadcasts the permutation."""
        from torch.utils.data import DataLoader, TensorDataset
        if not multi_rank:
            return [idx for (idx,) in DataLoader(TensorDataset(torch.arange(T)), batch_size=bs, shuffle=True)]
        perm = torch.empty(T, dtype=torch.int64, device=dev)
        if dist.get_rank(group) == 0:
            perm.copy_(torch.cat([idx for (idx,) in DataLoader(TensorDataset(torch.arange(T)), batch_size=bs, shuffle=True)]))
        dist.broadcast(perm, src, group=group)
        return list(perm.cpu().split(bs))

    def end_of_epoch(losses: List[torch.Tensor]) -> None:
        if not s.plateau:
            return
        mean = torch.stack(losses).mean().reshape(1)
        L.check(first.lib.awb_opt_plateau_step(first.prior.handle, first.opt_state.data_ptr(), mean.data_ptr(), 0,
                                               C.byref(plateau_hy), L.stream_ptr()))
        first._keep = mean          # the kernel reads it asynchronously
        if lr_trace is not None:    # diagnostics / tests: the learning rates after this epoch's scheduler step (synchronises)
            lr_trace.append(list(first.scalars(0).lr))

    if not s.dataloader_shuffle:
        fitters = []
        for b0 in range(0, T, bs):
            nb = min(bs, T - b0)
            spec = GridSpecHost(grid_mode, nb, H, W, t0=b0 * t_step, t_step=t_step)
            fitters.append(make(spec, un[b0:b0 + nb].reshape(1, -1)))
        for _ in range(s.num_epochs):
            ep = [f.run(1)[0, 0] for f in fitters]
            hist += ep
            end_of_epoch(ep)
    else:
        # shuffled batches (the reference's DataLoader(shuffle=True): same sampler, same global-RNG stream): the frames of a
        # batch are not equidistant in t, so the batch grid is gathered into a staging tensor
        gfull = full.materialize(C_in, dev)
        stage_g, stage_u, fitters_by = {}, {}, {}
        for _ in range(s.num_epochs):
            ep = []
            for idx in epoch_batches():
                nb = int(idx.numel())
                if nb not in fitters_by:
                    stage_g[nb] = torch.empty((nb, C_in, H, W), dtype=torch.float32, device=dev)
                    stage_u[nb] = torch.empty((1, nb * H * W), dtype=torch.float32, device=dev)
                    fitters_by[nb] = make(GridSpecHost.from_tensor(stage_g[nb]), stage_u[nb])
                di = idx.to(dev)
                torch.index_select(gfull, 0, di, out=stage_g[nb])
                fitters_by[nb].set_target(torch.index_select(un, 0, di).reshape(1, -1))
                ep.append(fitters_by[nb].run(1)[0, 0])
            hist += ep
            end_of_epoch(ep)
    if first is not None:
        first.raise_if_nonfinite()
    return torch.stack(hist) if hist else torch.empty(0, device=dev)


# ------------------------------------------------------------------ pretrain checkpoints (reference format)
def save_pretrain_checkpoint(model, path: str) -> bool:
    """``path_connected_net.py:45-51``: ``torch.save(model.state_dict(), path)``."""
    try:
        torch.save({k: v.detach().cpu() for k, v in model.state_dict().items()}, path)
        return True
    except Exception as e:          # the reference logs and carries on
        logging.error("Could not save pretrain checkpoint to %s. Error: %s", path, e)
        return False


def load_pretrain_checkpoint(model, path: str, device=None) -> bool:
    """``path_connected_net.py:33-43``: ``model.load_state_dict(torch.load(path, map_location=device))``."""
    try:
        model.load_state_dict(torch.load(path, map_location=device))
        return True
    except Exception as e:
        logging.error("Could not load pretrain checkpoint from %s. Error: %s", path, e)
        return False


# ------------------------------------------------------------------ N1: unaries of the frozen segmentation net, batched
def _cat_inputs(items: Sequence[Any]):
    """Stack the per-frame inputs (each a tensor or a list / tuple of tensors with leading batch dimension 1)."""
    first = items[0]
    if torch.is_tensor(first):
        return [torch.cat(list(items), dim=0)]
    return [torch.cat([it[j] for it in items], dim=0) if torch.is_tensor(first[j]) else first[j] for j in range(len(first))]


def _segmentation_unaries(wrapper_module, batch):
    """Unaries ``[k,1,H,W]`` of ``k`` stacked frames.  The reference ``WrapperModule.forward`` loops over the batch items and
    calls the segmentation net once per image (``wrapper_module.py:196-239``); for a real reference wrapper the net is called
    ONCE on the stacked frames with the wrapper's own argument selection and output processing
    (``get_segmentation_module_args`` ``:141-155``, ``process_segmentation_output`` ``:248-262``: sigmoid, inversion -- both
    elementwise).  Duck-typed wrappers are simply called."""
    seg = getattr(wrapper_module, "segmentation_module", None)
    if seg is None or not hasattr(wrapper_module, "get_segmentation_module_args") or not hasattr(wrapper_module, "process_segmentation_output"):
        return wrapper_module(*batch)
    primary, args, kwargs = wrapper_module.get_segmentation_module_args(batch[0], tuple(batch[1:]), {}, targets=None)
    out = seg(primary, *args, **kwargs)
    k = out.shape[0]
    u = wrapper_module.process_segmentation_output(out)
    if k == 1 and u.dim() == out.dim() - 1:        # the wrapper drops a batch dimension of one
        u = u[None]
    return u


def collect_unaries(wrapper_module, agent, train_set, device, unet_batch_size: int = 8):
    """The UNet side of the pretrain loops (``path_connected_net.py:672-676, 832-836``): the reference evaluates the frozen
    segmentation net once per frame and loop iteration (per EPOCH in the spatio-temporal loop).  Here every frame is
    evaluated once, ``unet_batch_size`` frames per call (the net is in eval mode: BatchNorm uses its running statistics, so a
    frame's unaries do not depend on its batch mates), and the unaries stay on the device for all epochs.
    Returns (inputs per frame, grids ``[1,C,H,W]`` per frame, unaries ``[1,1,H,W]`` per frame, prior keys)."""
    from torch.utils.data import DataLoader
    loader = DataLoader(train_set, batch_size=1, shuffle=False)
    dec = [agent._decompose_training_item(item) for item in loader]
    ins = [d[0] if isinstance(d[0], (list, tuple)) else [d[0]] for d in dec]
    keys = [int(d[3][0]) if d[3] is not None else i for i, d in enumerate(dec)]
    grids, uns, dev_ins = [], [], []
    old = getattr(wrapper_module, "evaluate_prior", True)
    wrapper_module.evaluate_prior = False
    try:
        bs = max(1, int(unet_batch_size))
        for b0 in range(0, len(ins), bs):
            chunk = ins[b0:b0 + bs]
            batch = [x.to(device) if torch.is_tensor(x) else x for x in _cat_inputs(chunk)]
            with torch.no_grad():
                u = _segmentation_unaries(wrapper_module, batch)
            for k in range(len(chunk)):
                one = [x[k:k + 1] if torch.is_tensor(x) else x for x in batch]
                pa, _ = wrapper_module.get_prior_args(one[0], *one[1:], segm=u[k])
                g = pa[0].detach()
                grids.append(g if g.dim() == 4 else g.unsqueeze(0))
                uns.append(u[k:k + 1].detach())
                dev_ins.append(one)
    finally:
        wrapper_module.evaluate_prior = old
    return dev_ins, grids, uns, keys


def evaluate_frames(wrapper_module, agent, dataset, device, prior_cache=None, unet_batch_size: int = 8) -> List[torch.Tensor]:
    """Evaluation path of ``get_result`` (``awesome/run/functions.py:2111-2151``) over a whole dataset: segmentation net
    batched over frames, the prior evaluated per frame with that frame's weights swapped in from ``prior_cache``
    (``PriorManager``, ``awesome/dataset/prior_dataset.py:70-110``).  Returns per frame ``cat([sigmoid(seg), sigmoid(prior)], 1)``
    on the host -- what ``WrapperModule.forward`` returns for ``evaluate_prior=True`` (``wrapper_module.py:157-228``)."""
    was = wrapper_module.training
    wrapper_module.eval()
    try:
        _, grids, uns, keys = collect_unaries(wrapper_module, agent, dataset, device, unet_batch_size)
        prior = wrapper_module.prior_module
        out = []
        with torch.no_grad():
            for g, u, key in zip(grids, uns, keys):
                if prior_cache is not None and hasattr(prior_cache, "load_into"):
                    prior_cache.load_into(prior, key)
                elif prior_cache is not None:
                    prior.load_state_dict(prior_cache[key])
                p = prior(g.to(device))
                p = torch.sigmoid(p) if getattr(wrapper_module, "use_prior_sigmoid", True) else p
                out.append(torch.cat([u, p.reshape(u.shape)], dim=1).cpu())
        return out
    finally:
        wrapper_module.train(was)


# ------------------------------------------------------------------ PretrainableModule protocol (duck-typed)
def pretrain(self, train_set, test_set=None, device=None, agent=None, use_progress_bar: bool = True,
             do_pretrain_checkpoints: bool = False, use_pretrain_checkpoints: bool = False,
             pretrain_checkpoint_dir: Optional[str] = None, wrapper_module=None, **kwargs) -> Any:
    """``PathConnectedNet.pretrain`` (``path_connected_net.py:472-509``) with the reference's arguments.  The agent,
    dataset and wrapper module are the reference's objects (this module is plugged into ``scripts/run.py``):
    ``agent._decompose_training_item`` splits a dataset item, ``wrapper_module(...)`` with ``evaluate_prior=False``
    yields the UNet unaries, ``wrapper_module.get_prior_args`` the coordinate grid.

    Per-frame mode (dataset with a prior cache): ``fit_frames`` per frame; ``pretrain_checkpoint_{i}.pth`` (the frame's
    ``state_dict``, ``torch.save``) is written after every fitted frame with ``do_pretrain_checkpoints`` and, with
    ``use_pretrain_checkpoints``, an existing file is loaded instead of fitting -- the loaded state counts as a proper fit
    and becomes the warm start of the next frame (``:857-870, 996-998``).  Otherwise the spatio-temporal ``fit_sequence``."""
    import os
    if wrapper_module is None:
        raise ValueError("Wrapper model must be provided for pretraining.")
    if do_pretrain_checkpoints:
        if pretrain_checkpoint_dir is None:
            raise ValueError("Pretrain checkpoint dir must be provided.")
        os.makedirs(pretrain_checkpoint_dir, exist_ok=True)
    sched = FitSchedule.from_pretrain_args(kwargs)
    device = torch.device(device) if device is not None else self._ensure_flat().device
    ds = getattr(agent, "training_dataset", None)
    cache = getattr(ds, "__prior_cache__", None)
    per_frame = cache is not None and bool(getattr(ds, "has_prior", getattr(ds, "__has_prior__", False)))
    was_training = wrapper_module.training
    wrapper_module.eval()
    try:
        _, grids, uns, keys = collect_unaries(wrapper_module, agent, train_set, device, sched.unet_batch_size)
        if per_frame:
            def keep(res: FrameResult):
                if res.skipped:
                    return
                if hasattr(cache, "store_from"):
                    cache.store_from(self, res.index)
                else:
                    cache[res.index] = {k: v.detach().clone() for k, v in self.state_dict().items()}

            pos_of = {k: i for i, k in enumerate(keys)}
            run: List[int] = []            # consecutive frames without a checkpoint: one fit_frames call (keeps the chain)
            previous_from_ckpt = [None]

            def flush():
                if not run:
                    return
                def on_frame(res: FrameResult):
                    keep(res)
                    if do_pretrain_checkpoints and not res.skipped:
                        # on_frame runs right after the frame's fit: the module holds exactly this frame's state (:996-998)
                        save_pretrain_checkpoint(self, os.path.join(pretrain_checkpoint_dir,
                                                                    f"pretrain_checkpoint_{pos_of[res.index]}.pth"))
                if previous_from_ckpt[0] is not None:
                    self.load_state_dict(previous_from_ckpt[0])
                fit_frames(self, [grids[i] for i in run], [uns[i] for i in run], sched, on_frame=on_frame,
                           frame_indices=[keys[i] for i in run], warm_start_hook=kwargs.get("_warm_start_hook"),
                           initial_previous=self._ensure_flat().detach().clone() if previous_from_ckpt[0] is not None else None)
                previous_from_ckpt[0] = {k: v.detach().clone() for k, v in self.state_dict().items()}
                run.clear()

            for i in range(len(grids)):
                path = os.path.join(pretrain_checkpoint_dir, f"pretrain_checkpoint_{i}.pth") if pretrain_checkpoint_dir else None
                if use_pretrain_checkpoints and path and os.path.exists(path):
                    flush()
                    if load_pretrain_checkpoint(self, path, device=device):
                        logging.info("Loaded pretrain checkpoint from %s. Continuing with next image.", path)
                        keep(FrameResult(index=keys[i], proper_fit=True))
                        previous_from_ckpt[0] = {k: v.detach().clone() for k, v in self.state_dict().items()}
                        continue
                run.append(i)
            flush()
            return cache.get_state()
        T = len(grids)
        H, W = grids[0].shape[-2:]
        import torch.distributed as dist
        sliced = sched.sequence_slices > 0 and dist.is_available() and dist.is_initialized()
        fit_sequence(self, T, H, W, torch.stack([u.reshape(H, W) for u in uns]), sched,
                     n_slices=sched.sequence_slices if sliced else None, group=dist.group.WORLD if sliced else None)
        return {k: v.detach().cpu().clone() for k, v in self.state_dict().items()}
    finally:
        wrapper_module.train(was_training)


def pretrain_load_state(self, train_set, test_set, device, agent, state, use_progress_bar: bool = True,
                        wrapper_module=None, **kwargs):
    """``path_connected_net.py:1010-1019``: the per-frame states go back into the dataset's prior cache."""
    cache = getattr(getattr(agent, "training_dataset", None), "__prior_cache__", None)
    if cache is not None and isinstance(state, dict) and "cache" in state:
        cache.set_state(state)
    elif isinstance(state, dict):
        self.load_state_dict(state)
