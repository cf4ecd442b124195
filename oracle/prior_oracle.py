"""CPU oracle for AWESOME's shape-prior fitting hot path.

TEST INFRASTRUCTURE ONLY.  Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import this file.
The product path (``awesome_b200/``) never does; it fails loudly when its CUDA
library is missing.

This is a functional restatement (plain fp32 torch-on-CPU tensor arithmetic, no
``nn.Module``; autograd is used only to obtain reference gradients) of the
reference's algorithm.  Every function cites the reference ``file:line`` it
follows (paths relative to the reference checkout).  Parameters are plain dicts
keyed by the reference's ``state_dict`` names, so checkpoints are interchangeable.

PINNING: the reference ships no tests or golden vectors (SURVEY.md section 4), so
the oracle is pinned against outputs of the reference's own modules, generated in
the build container by ``tests/golden/make_golden.py`` and committed under
``tests/golden/*.pt`` (checked by ``tests/test_oracle_golden.py``).  The RealNVP
arithmetic lives in the third-party ``normflows==1.7.3`` (absent offline); the
golden flow vectors come from the reference's ``net_factory`` running on top of
``oracle/normflows_restated.py``, therefore the flow boundary is "parity
unpinned" with respect to the real wheel.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

Params = Dict[str, torch.Tensor]


# --------------------------------------------------------------------------- a1
def grid_linspace(H: int, W: int, t: Optional[float] = None,
                  t_max: Optional[float] = None) -> torch.Tensor:
    """FBMS coordinate grid ``[C,H,W]``, channels (x, y[, t]).

    Follows ``awesome/dataset/transformator.py:25-61``: ``x=linspace(0,1,W)``,
    ``y=linspace(0,1,H)``, ``t`` channel is the constant ``t/t_max``.
    """
    y = torch.linspace(0, 1, H)
    x = torch.linspace(0, 1, W)
    yy, xx = torch.meshgrid(y, x, indexing="ij")
    if t is None:
        return torch.stack((xx, yy), dim=0).float()
    if t_max is None:
        raise ValueError("t_max must be set if t is set")
    return torch.stack((xx, yy, torch.ones_like(xx) * t / t_max), dim=0).float()


def grid_index(H: int, W: int) -> torch.Tensor:
    """How-to notebook grid ``[1,2,H,W]``: ``x=j/W``, ``y=i/H``.

    Follows ``notebooks/how_to/convexity.ipynb`` cell 7 (``create_grid``).
    """
    x = torch.arange(0, W)
    y = torch.arange(0, H)
    xx, yy = torch.meshgrid(x, y, indexing="xy")
    grid = torch.stack((xx, yy), dim=0)
    return grid.unsqueeze(0).float() / torch.tensor([W, H]).float().unsqueeze(-1).unsqueeze(-1)


def grid_normalized(shape: Sequence[int]) -> torch.Tensor:
    """``PathConnectedNet.create_normalized_grid`` (``path_connected_net.py:252-296``):
    integer meshgrid, channel order (x, y[, z]), min-max scaled to [0,1] per channel."""
    ar = [torch.arange(s).float() for s in shape]
    grid = torch.stack(torch.meshgrid(*ar, indexing="ij")[::-1])
    if grid.dim() == 4:
        grid = grid.swapaxes(0, 1)
    else:
        grid = grid.unsqueeze(0)
    mn = grid.amin(dim=(0, 2, 3), keepdim=True)
    mx = grid.amax(dim=(0, 2, 3), keepdim=True)
    return (grid - mn) / (mx - mn) * (1.0 - 0.0) + 0.0


# --------------------------------------------------------------------------- a4
def pixelize(x: torch.Tensor) -> torch.Tensor:
    """``[B,C,H,W] -> [B*H*W, C]`` rows in (b,h,w) order (``awesome/util/pixelize.py:30-32``)."""
    return x.permute(0, 2, 3, 1).reshape(-1, x.shape[1])


def unpixelize(x: torch.Tensor, B: int, H: int, W: int) -> torch.Tensor:
    """Inverse layout (``awesome/util/pixelize.py:34-36``)."""
    return x.reshape(B, H, W, -1).permute(0, 3, 1, 2)


# --------------------------------------------------------------------------- a7
def icnn_num_layers(p: Params, prefix: str = "") -> int:
    n = 0
    while f"{prefix}skip.{n}.ln.weight" in p:
        n += 1
    return n


def icnn_forward(p: Params, x: torch.Tensor, prefix: str = "") -> torch.Tensor:
    """ConvexNextNet on pixel rows ``x[N,C] -> logits[N,1]``.

    ``awesome/model/convex_net.py:205-214`` (forward), ``:144-145`` (SkipBlock:
    ``relu(ln(z) + skp(x))``), ``:170-171`` (OutBlock: ``ln(z) + skp(x)``).
    """
    z = F.relu(x @ p[prefix + "input.weight"].T + p[prefix + "input.bias"])
    for i in range(icnn_num_layers(p, prefix)):
        z = F.relu(z @ p[f"{prefix}skip.{i}.ln.weight"].T + p[f"{prefix}skip.{i}.ln.bias"]
                   + x @ p[f"{prefix}skip.{i}.skp.weight"].T)
    return (z @ p[prefix + "out.ln.weight"].T + p[prefix + "out.ln.bias"]
            + x @ p[prefix + "out.skp.weight"].T)


def convexnet_forward(p: Params, x: torch.Tensor) -> torch.Tensor:
    """Older ``ConvexNet`` (``awesome/model/convex_net.py:27-35``), == L=1 ICNN with
    keys ``W0y, W1z, W2z, W1y, W2y``."""
    z = F.relu(x @ p["W0y.weight"].T + p["W0y.bias"])
    z = F.relu(z @ p["W1z.weight"].T + p["W1z.bias"] + x @ p["W1y.weight"].T)
    return z @ p["W2z.weight"].T + p["W2z.bias"] + x @ p["W2y.weight"].T


# --------------------------------------------------------------------------- a8
def icnn_clamp_keys(p: Params, prefix: str = "") -> List[str]:
    """Names of the tensors ``enforce_convexity`` clamps: every ``skip.i.ln.weight``
    and ``out.ln.weight``; not ``input.*``, ``*.skp.weight`` or biases
    (``awesome/model/convex_net.py:151-154,216-220``)."""
    return [f"{prefix}skip.{i}.ln.weight" for i in range(icnn_num_layers(p, prefix))] + \
           [prefix + "out.ln.weight"]


def icnn_enforce_convexity(p: Params, prefix: str = "") -> None:
    with torch.no_grad():
        for k in icnn_clamp_keys(p, prefix):
            p[k].copy_(F.relu(p[k]))


# --------------------------------------------------------------------------- a3
def minmax(v, v_min, v_max, new_min, new_max):
    """``awesome/transforms/min_max.py:9-19``."""
    return (v - v_min) / (v_max - v_min) * (new_max - new_min) + new_min


# --------------------------------------------------------------------------- a5
def realnvp_masks(channels: int, n_flows: int) -> torch.Tensor:
    """Coupling masks ``[n_flows, C]`` (uint8): binary counting 1 .. 2^C-2, LSB first,
    repeated and truncated (``awesome/model/net_factory.py:86-99``)."""
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


def flow_num(p: Params, prefix: str) -> int:
    n = 0
    while f"{prefix}flows.{2 * n}.b" in p:
        n += 1
    return n


def _mlp(p: Params, pre: str, zm: torch.Tensor, output_fn: Optional[str]) -> torch.Tensor:
    """normflows ``nets.MLP([C,m,C])``: Linear, LeakyReLU(0.0), Linear[, Tanh]."""
    hdn = F.leaky_relu(zm @ p[pre + "net.0.weight"].T + p[pre + "net.0.bias"], 0.0)
    o = hdn @ p[pre + "net.2.weight"].T + p[pre + "net.2.bias"]
    if output_fn == "tanh":
        o = torch.tanh(o)
    elif output_fn is not None:
        raise NotImplementedError(output_fn)
    return o


def flow_forward(p: Params, z: torch.Tensor, prefix: str, output_fn: Optional[str] = "tanh",
                 actnorm_init: bool = False) -> torch.Tensor:
    """RealNVP stack on pixel rows ``[N,C] -> [N,C]`` (normflows semantics, built at
    ``awesome/model/net_factory.py:101-113``): per flow f a ``MaskedAffineFlow`` then
    an ``ActNorm``.  With ``actnorm_init`` the ActNorm parameters whose
    ``data_dep_init_done`` buffer is 0 are set from the batch statistics (first
    forward call) and written back into ``p``."""
    nan = torch.tensor(float("nan"), dtype=z.dtype, device=z.device)
    for f in range(flow_num(p, prefix)):
        a, n = f"{prefix}flows.{2 * f}.", f"{prefix}flows.{2 * f + 1}."
        b = p[a + "b"].to(z.dtype)
        zm = b * z
        s = _mlp(p, a + "s.", zm, output_fn)
        s = torch.where(torch.isfinite(s), s, nan)
        t = _mlp(p, a + "t.", zm, output_fn)
        t = torch.where(torch.isfinite(t), t, nan)
        z = zm + (1 - b) * (z * torch.exp(s) + t)
        if actnorm_init and not bool(p[n + "data_dep_init_done"] > 0):
            with torch.no_grad():
                s_init = -torch.log(z.std(dim=0, keepdim=True) + 1e-6)
                p[n + "s"].copy_(s_init)
                p[n + "t"].copy_(-z.mean(dim=0, keepdim=True) * torch.exp(s_init))
                p[n + "data_dep_init_done"].fill_(1.0)
        z = z * torch.exp(p[n + "s"]) + p[n + "t"]
    return z


def flow_inverse(p: Params, x: torch.Tensor, prefix: str,
                 output_fn: Optional[str] = "tanh") -> torch.Tensor:
    """Reverse walk: ActNorm inverse ``(x-t)*exp(-s)`` then coupling inverse
    ``zm + (1-b)*(x-t(zm))*exp(-s(zm))``."""
    for f in range(flow_num(p, prefix) - 1, -1, -1):
        a, n = f"{prefix}flows.{2 * f}.", f"{prefix}flows.{2 * f + 1}."
        x = (x - p[n + "t"]) * torch.exp(-p[n + "s"])
        b = p[a + "b"].to(x.dtype)
        xm = b * x
        s = _mlp(p, a + "s.", xm, output_fn)
        t = _mlp(p, a + "t.", xm, output_fn)
        x = xm + (1 - b) * (x - t) * torch.exp(-s)
    return x


# ------------------------------------------------------------------- a2 + a3..a7
FLOW_PREFIX = "flow_net.net.network."


def pathconnected_deformation(p: Params, grid: torch.Tensor,
                              output_fn: Optional[str] = "tanh",
                              actnorm_init: bool = False) -> torch.Tensor:
    """``PathConnectedNet.get_deformation`` (``path_connected_net.py:125-129``):
    grouped 1x1 conv (``:65,82``) -> NormNet(min-max to [-1,1], flow, inverse min-max)
    (``norm_net.py:17-27``, ``pixelize_net.py:14-18``).  ``grid`` is ``[B,C,H,W]``;
    returns pixel rows ``[N,C]``."""
    B, C, H, W = grid.shape
    w = p["linear.weight"].reshape(1, C, 1, 1)
    x = grid * w + p["linear.bias"].reshape(1, C, 1, 1)
    mn, mx = p["flow_net.norm.min"], p["flow_net.norm.max"]
    nmn, nmx = p["flow_net.norm.new_min"], p["flow_net.norm.new_max"]
    x = minmax(x, mn, mx, nmn, nmx)
    z = flow_forward(p, pixelize(x), FLOW_PREFIX, output_fn, actnorm_init)
    z = unpixelize(z, B, H, W)
    z = minmax(z, nmn, nmx, mn, mx)
    return pixelize(z)


def pathconnected_forward(p: Params, grid: torch.Tensor, output_fn: Optional[str] = "tanh",
                          actnorm_init: bool = False) -> torch.Tensor:
    """``PathConnectedNet.forward`` (``path_connected_net.py:79-85``) -> ``[B,1,H,W]``."""
    B, C, H, W = grid.shape
    xd = pathconnected_deformation(p, grid, output_fn, actnorm_init)
    y = icnn_forward(p, xd, "convex_net.")
    return unpixelize(y, B, H, W)


# --------------------------------------------------------------------------- a6
def wn_linear(p: Params, pre: str, x: torch.Tensor) -> torch.Tensor:
    """``WNLinear`` = ``weight_norm(nn.Linear, dim=None)``: ``W = g * v / ||v||_F``
    (``awesome/model/real_nvp/resnet_1d.py:39-63``)."""
    v = p[pre + "linear.weight_v"]
    w = p[pre + "linear.weight_g"] * v / v.norm()
    return x @ w.T + p[pre + "linear.bias"]


def _simple_backbone(p: Params, pre: str, x: torch.Tensor) -> torch.Tensor:
    """``SimpleBackbone`` (``awesome/model/diffeomorphism_net.py:83-104``)."""
    return torch.tanh(wn_linear(p, pre + "linear2.", F.relu(wn_linear(p, pre + "linear1.", x))))


def _wn_scale(p: Params, pre: str, x: torch.Tensor) -> torch.Tensor:
    """``WNScale`` (``awesome/model/diffeomorphism_net.py:208-232``): ``forward()`` ignores its input and returns
    the scalar ``scale(weight)`` with ``scale = weight_norm(nn.Linear(1, 1))`` (default ``dim=0``); the coupling
    multiplies the backbone output by it (``:291,294``)."""
    v = p[pre + "scale.weight_v"]
    w = p[pre + "scale.weight_g"] * v / v.norm(dim=1, keepdim=True)
    c = p[pre + "weight"] @ w.T + p[pre + "scale.bias"]
    return c * x


def flow1d_num(p: Params, prefix: str) -> int:
    n = 0
    while f"{prefix}s.{n}.linear1.linear.bias" in p:
        n += 1
    return n


def flow1d_forward(p: Params, x: torch.Tensor, prefix: str = "diffeo_net.") -> torch.Tensor:
    """``NormalizingFlow1D.forward`` (``awesome/model/diffeomorphism_net.py:286-300``):
    alternating two-variable affine couplings."""
    x1, x2 = x[:, 0:1], x[:, 1:2]
    for i in range(flow1d_num(p, prefix)):
        if i % 2 == 0:
            x2 = torch.exp(_wn_scale(p, f"{prefix}scale.{i}.", _simple_backbone(p, f"{prefix}s.{i}.", x1))) * x2 \
                + _simple_backbone(p, f"{prefix}t.{i}.", x1)
        else:
            x1 = torch.exp(_wn_scale(p, f"{prefix}scale.{i}.", _simple_backbone(p, f"{prefix}s.{i}.", x2))) * x1 \
                + _simple_backbone(p, f"{prefix}t.{i}.", x2)
    return torch.cat([x1, x2], dim=1)


# -------------------------------------------------------------------------- a16
def star_forward(p: Params, x: torch.Tensor) -> torch.Tensor:
    """Star-shape prior ``myNet`` (``notebooks/icml_teaser_code/star_shaped/star.ipynb``
    cell 2): ``x+=offset; r=||x||; u=x/(0.01+r); a=relu(W0 u); b=relu(W1 a + W1r r);
    y = r*(W2 a + W2r b) - 1`` (every Linear carries its bias)."""
    x = x + p["offset"]
    r = torch.sqrt(torch.sum(x ** 2, dim=1, keepdim=True))
    u = x / (0.01 + r)
    a = F.relu(u @ p["W0.weight"].T + p["W0.bias"])
    b = F.relu(a @ p["W1.weight"].T + p["W1.bias"] + r @ p["W1_r.weight"].T + p["W1_r.bias"])
    return r * (a @ p["W2.weight"].T + p["W2.bias"] + b @ p["W2_r.weight"].T + p["W2_r.bias"]) - 1


# --------------------------------------------------------------------------- a9/a10
LOSS_MSE, LOSS_FGBG_SE, LOSS_FGBG_BCE_LOGITS, LOSS_BCE = "mse", "fgbg_se", "fgbg_bce_logits", "bce"


def unaries_weight(target: torch.Tensor, mode: str, ratio: float = 1.0) -> torch.Tensor:
    """``UnariesWeightedLoss._compute_weight`` (``unaries_weighted_loss.py:35-69``).
    fg = pixels with ``target < 0.5``; weight on fg pixels by mode."""
    if mode == "none":
        return torch.ones_like(target)
    fg = (target < 0.5)
    fg_count = fg.sum().to(torch.float32)
    bg_count = (~fg).sum().to(torch.float32)
    cc = bg_count / fg_count
    if mode == "ratio":
        wv = (cc - 1) * ratio + 1
    elif mode == "sssdms":
        wv = torch.round(cc / 10) + 1
    elif mode == "equal":
        wv = cc
    else:
        raise ValueError(f"Mode {mode} is not supported")
    w = torch.ones_like(target)
    w[fg] = wv
    return w


def loss_unaries_weighted_se(logits: torch.Tensor, target: torch.Tensor, mode: str = "none",
                             ratio: float = 1.0) -> torch.Tensor:
    """Default pretrain criterion ``UnariesWeightedLoss(SE("mean"))`` on ``sigmoid(y)``
    (``path_connected_net.py:768,944-948``; ``weighted_loss.py:67-92``; ``se.py:21-23``)."""
    o = torch.sigmoid(logits).reshape(-1)
    t = target.reshape(-1)
    se = (t - o) ** 2
    if mode != "none":
        se = se * unaries_weight(t, mode, ratio)
    return se.mean()


def loss_fgbg_se(logits: torch.Tensor, unaries: torch.Tensor, fg_weight: float) -> torch.Tensor:
    """Convexity how-to loss (``notebooks/how_to/convexity.ipynb`` cell 9):
    ``(1-w)*mean_bg(SE) + w*mean_fg(SE)`` on ``sigmoid(y)``; bg = ``unaries == 1``."""
    o = torch.sigmoid(logits).reshape(-1)
    t = unaries.reshape(-1)
    bg = t == 1.0
    se = (t - o) ** 2
    return (1 - fg_weight) * (se[bg].sum() / bg.sum()) + fg_weight * (se[~bg].sum() / (~bg).sum())


def loss_fgbg_bce_logits(logits: torch.Tensor, unaries: torch.Tensor, fg_weight: float) -> torch.Tensor:
    """Path-connectedness how-to loss (``notebooks/how_to/path-connectedness.ipynb`` cell 9)."""
    y = logits.reshape(-1)
    t = unaries.reshape(-1)
    bg = t == 1.0
    l = F.binary_cross_entropy_with_logits(y, t, reduction="none")
    return ((1 - fg_weight) * l[bg]).sum() / bg.sum() + (fg_weight * l[~bg]).sum() / (~bg).sum()


def loss_weighted_bce_sssdms(prob: torch.Tensor, target: torch.Tensor,
                             noneclass: Optional[float] = 2.0) -> torch.Tensor:
    """``WeightedLoss(BCELoss, mode="sssdms", noneclass=2)`` (``weighted_loss.py:41-92``):
    drop none-class pixels, weight on ``target == 0`` pixels = ``round(bg/fg/10)+1``."""
    o, t = prob.reshape(-1), target.reshape(-1)
    if noneclass is not None:
        keep = t != noneclass
        o, t = o[keep], t[keep]
    l = F.binary_cross_entropy(o, t, reduction="none")
    fg = (t == 0).sum().float()
    bg = (t == 1).sum().float()
    w = torch.ones_like(t)
    w[t == 0] = torch.round(bg / fg / 10) + 1
    return (l * w).mean()


def loss_fbms_joint(seg_prob: torch.Tensor, prior_prob: torch.Tensor, target: torch.Tensor,
                    alpha: float = 1.0, beta: float = 1.0, clip_penalty: bool = True,
                    noneclass: Optional[float] = 2.0) -> torch.Tensor:
    """``FBMSJointLoss`` (``awesome/measures/fbms_joint_loss.py:35-59``):
    ``alpha*wBCE(seg,target) + beta*MSE(prior,seg)`` with the penalty soft-clipped to the
    segmentation loss through a detached ratio."""
    seg = alpha * loss_weighted_bce_sssdms(seg_prob, target, noneclass)
    pen = beta * ((seg_prob - prior_prob) ** 2).mean()
    if clip_penalty and bool(pen > seg):
        pen = pen * (seg / pen).detach()
    return seg + pen


# --------------------------------------------------------------------------- a11
def adam_step(p, g, m, v, step: int, lr: float, beta1=0.9, beta2=0.999, eps=1e-8,
              weight_decay=0.0) -> None:
    """``torch.optim.Adam`` single-tensor path (torch ``optim/adam.py``
    ``_single_tensor_adam``), L2 decay folded into the gradient.  ``step`` is 1-based."""
    with torch.no_grad():
        if weight_decay != 0:
            g = g + weight_decay * p
        m.lerp_(g, 1 - beta1)
        v.mul_(beta2).addcmul_(g, g, value=1 - beta2)
        bc1 = 1 - beta1 ** step
        bc2 = 1 - beta2 ** step
        step_size = lr / bc1
        denom = (v.sqrt() / math.sqrt(bc2)).add_(eps)
        p.addcdiv_(m, denom, value=-step_size)


def adamax_step(p, g, m, u, step: int, lr: float, beta1=0.9, beta2=0.999, eps=1e-8,
                weight_decay=0.0) -> None:
    """``torch.optim.Adamax`` single-tensor path (torch ``optim/adamax.py``
    ``_single_tensor_adamax``): ``u = max(beta2*u, |g|+eps)``; ``p -= lr/(1-beta1^t) * m/u``."""
    with torch.no_grad():
        if weight_decay != 0:
            g = g + weight_decay * p
        m.lerp_(g, 1 - beta1)
        torch.maximum(u * beta2, g.abs() + eps, out=u)
        p.addcdiv_(m, u, value=-(lr / (1 - beta1 ** step)))


class Plateau:
    """``ReduceLROnPlateau(mode="min", factor, patience, threshold=1e-4 rel,
    cooldown=0, min_lr=0, eps=1e-8)`` stepped on the loss every iteration
    (``path_connected_net.py:932-933,953``; torch ``lr_scheduler.py``)."""

    def __init__(self, lrs: Sequence[float], patience=200, factor=0.5, threshold=1e-4,
                 min_lr=0.0, eps=1e-8):
        self.lrs = list(lrs)
        self.patience, self.factor, self.threshold = patience, factor, threshold
        self.min_lr, self.eps = min_lr, eps
        self.best = float("inf")
        self.num_bad = 0

    def step(self, metric: float) -> None:
        if metric < self.best * (1.0 - self.threshold):
            self.best = metric
            self.num_bad = 0
        else:
            self.num_bad += 1
        if self.num_bad > self.patience:
            for i, lr in enumerate(self.lrs):
                new = max(lr * self.factor, self.min_lr)
                if lr - new > self.eps:
                    self.lrs[i] = new
            self.num_bad = 0


# --------------------------------------------------------------------------- a15
def miou_binary_inverted(output_mask: torch.Tensor, target_mask: torch.Tensor) -> float:
    """``MIOU(average="binary", invert=True)`` (``awesome/measures/miou.py:29-48``):
    Jaccard of the foreground (``1 - mask``); 0 when the target has no foreground."""
    o = (1.0 - output_mask.reshape(-1).float()) > 0.5
    t = (1.0 - target_mask.reshape(-1).float()) > 0.5
    if not bool(t.any()):
        return 0.0
    inter = (o & t).sum().item()
    union = (o | t).sum().item()
    return float(inter) / float(union) if union > 0 else 0.0


# --------------------------------------------------------------------------- a12
def leaves(p: Params, keys: Sequence[str]) -> List[torch.Tensor]:
    return [p[k] for k in keys]


def clone_params(p: Params, requires_grad: bool = False) -> Params:
    out = {}
    for k, v in p.items():
        t = v.detach().clone()
        if requires_grad and t.dtype.is_floating_point:
            t.requires_grad_(True)
        out[k] = t
    return out


def icnn_param_keys(p: Params, prefix: str = "") -> List[str]:
    """Trainable tensors in ``state_dict`` order."""
    keys = [prefix + "input.weight", prefix + "input.bias"]
    for i in range(icnn_num_layers(p, prefix)):
        keys += [f"{prefix}skip.{i}.ln.weight", f"{prefix}skip.{i}.ln.bias", f"{prefix}skip.{i}.skp.weight"]
    keys += [prefix + "out.ln.weight", prefix + "out.ln.bias", prefix + "out.skp.weight"]
    return keys


def fit_icnn(p: Params, x_rows: torch.Tensor, target: torch.Tensor, steps: int, loss: str = LOSS_MSE,
             optimizer: str = "adam", lr: float = 1e-3, fg_weight: float = 0.4,
             weight_mode: str = "none", plateau: bool = False, record: Optional[list] = None) -> Params:
    """The convexity fit loop (``notebooks/how_to/convexity.ipynb`` cell 9 for
    ``fgbg_se``; ``path_connected_net.py:364-379`` / ``:939-953`` for ``mse``):
    ``sigmoid(model(grid))`` -> loss -> backward -> optimizer step -> enforce_convexity
    [-> plateau scheduler step on the loss].  In-place on ``p``; returns ``p``."""
    keys = icnn_param_keys(p)
    for k in keys:
        p[k].requires_grad_(True)
    ms = {k: torch.zeros_like(p[k]) for k in keys}
    vs = {k: torch.zeros_like(p[k]) for k in keys}
    sched = Plateau([lr]) if plateau else None
    for step in range(1, steps + 1):
        y = icnn_forward(p, x_rows)
        if loss == LOSS_MSE:
            l = loss_unaries_weighted_se(y, target, weight_mode)
        elif loss == LOSS_FGBG_SE:
            l = loss_fgbg_se(y, target, fg_weight)
        elif loss == LOSS_FGBG_BCE_LOGITS:
            l = loss_fgbg_bce_logits(y, target, fg_weight)
        else:
            raise ValueError(loss)
        if not math.isfinite(float(l.detach())):
            raise ValueError("Loss is nan or inf!")
        grads = torch.autograd.grad(l, leaves(p, keys))
        cur_lr = sched.lrs[0] if sched else lr
        for k, g in zip(keys, grads):
            if optimizer == "adam":
                adam_step(p[k], g, ms[k], vs[k], step, cur_lr)
            else:
                adamax_step(p[k], g, ms[k], vs[k], step, cur_lr)
        icnn_enforce_convexity(p)
        if sched:
            sched.step(float(l.detach()))
        if record is not None:
            record.append(float(l.detach()))
    for k in keys:
        p[k].requires_grad_(False)
    return p
