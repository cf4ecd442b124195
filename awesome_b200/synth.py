"""Synthetic FBMS-shaped inputs of the BASELINE configs (SURVEY 8d): seeded, CPU-generated, dataset-free.

Shared by ``bench.py``, ``tests/`` and ``tests/golden/make_golden_full.py`` so that the reference-side fits
(golden fixtures) and the device fits start from the same unaries.  Everything is plain ``torch`` on the CPU with an
explicit ``torch.Generator`` (mt19937): the hard masks are reproducible bit for bit, the soft unaries up to the last
ulp of the host's ``sigmoid`` (irrelevant for the mask-level comparisons they are used in).

Convention of the reference: **foreground = 0, background = 1** (``awesome/run/awesome_config.py:114-116``)."""
from __future__ import annotations

import math

import torch


def _grid01(H: int, W: int):
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    return xx, yy


def convex_polygon_mask(H: int, W: int, seed: int = 0) -> torch.Tensor:
    """Filled random convex polygon: 8-12 vertices on a jittered ellipse (sorted by angle, radii jittered by at most
    +-8 % so the polygon stays convex).  Returns a ``[H,W]`` float mask, 1 inside."""
    g = torch.Generator().manual_seed(seed)
    n = int(torch.randint(8, 13, (1,), generator=g))
    ang = torch.sort(torch.rand(n, generator=g) * 2 * math.pi).values
    # spread the angles so that no gap exceeds ~pi/2 (keeps the hull well conditioned)
    ang = 0.5 * ang + 0.5 * torch.arange(n) * (2 * math.pi / n)
    rx, ry = 0.30, 0.24
    jit = 1.0 + 0.08 * (2 * torch.rand(n, generator=g) - 1)
    vx, vy = 0.5 + rx * jit * torch.cos(ang), 0.5 + ry * jit * torch.sin(ang)
    xx, yy = _grid01(H, W)
    inside = torch.ones(H, W, dtype=torch.bool)
    for i in range(n):          # intersection of the half planes of the hull of the (angle-sorted) vertices
        j = (i + 1) % n
        ex, ey = vx[j] - vx[i], vy[j] - vy[i]
        cross = ex * (yy - vy[i]) - ey * (xx - vx[i])
        inside &= cross >= 0
    return inside.float()


def c1_unaries(H: int = 256, W: int = 256, seed: int = 0) -> torch.Tensor:
    """Config 1 (how_to/convexity): convex polygon, 5 % of the pixels flipped, 3 random occluding discs;
    unaries = 1 - mask in {0, 1} (like the notebook's thresholded likelihood)."""
    g = torch.Generator().manual_seed(seed + 1000)
    mask = convex_polygon_mask(H, W, seed)
    xx, yy = _grid01(H, W)
    for _ in range(3):
        cx, cy = 0.25 + 0.5 * torch.rand(1, generator=g), 0.25 + 0.5 * torch.rand(1, generator=g)
        r = 0.03 + 0.03 * torch.rand(1, generator=g)
        mask = torch.where((xx - cx) ** 2 + (yy - cy) ** 2 < r * r, torch.zeros_like(mask), mask)
    flip = torch.rand(H, W, generator=g) < 0.05
    mask = torch.where(flip, 1 - mask, mask)
    return (1 - mask).float()


def c1_clean_mask(H: int = 256, W: int = 256, seed: int = 0) -> torch.Tensor:
    """The noise-free convex polygon of ``c1_unaries`` as a fg = 0 mask (the shape the convex prior should recover)."""
    return (1 - convex_polygon_mask(H, W, seed)).float()


def c2_unaries(H: int = 480, W: int = 640, seed: int = 42, t: float = 0.0, tau: float = 0.08) -> torch.Tensor:
    """Config 2: soft UNet-like unaries in (0,1): elliptic blob on a Lissajous path with breathing axes,
    ``sigmoid((sdf + noise) / tau)``."""
    g = torch.Generator().manual_seed(seed)
    xx, yy = _grid01(H, W)
    cx, cy = 0.5 + 0.2 * math.sin(2.0 * t), 0.5 + 0.15 * math.sin(3.0 * t + 0.5)
    rx, ry = 0.22 * (1 + 0.2 * math.sin(5.0 * t)), 0.28 * (1 + 0.2 * math.cos(4.0 * t))
    sdf = torch.sqrt(((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2) - 1
    return torch.sigmoid((sdf + 0.05 * torch.randn(H, W, generator=g)) / tau).float()


def c3_unaries(H: int = 480, W: int = 640, seed: int = 42, t: float = 0.0, tau: float = 0.08, hard: bool = False) -> torch.Tensor:
    """Config 3: a non-convex (C-shaped) blob: an ellipse minus an off-centre bite; soft like ``c2_unaries`` or a hard
    {0,1} mask (the notebook variant)."""
    g = torch.Generator().manual_seed(seed)
    xx, yy = _grid01(H, W)
    cx, cy = 0.5 + 0.1 * math.sin(2.0 * t), 0.5 + 0.08 * math.sin(3.0 * t + 0.5)
    outer = torch.sqrt(((xx - cx) / 0.30) ** 2 + ((yy - cy) / 0.32) ** 2) - 1
    bite = torch.sqrt(((xx - cx - 0.16) / 0.17) ** 2 + ((yy - cy) / 0.15) ** 2) - 1
    sdf = torch.maximum(outer, -bite)            # inside the ellipse and outside the bite
    if hard:
        return (sdf > 0).float()
    return torch.sigmoid((sdf + 0.05 * torch.randn(H, W, generator=g)) / tau).float()


def star_unaries(H: int = 480, W: int = 640, seed: int = 42, r0: float = 0.25, a: float = 0.3, k: int = 5,
                 tau: float = 0.08, noise: float = 0.05) -> torch.Tensor:
    """A non-convex star-shaped blob for the star prior: boundary ``r(theta) = r0 (1 + a cos(k theta))`` around a
    seeded centre near the middle, soft like ``c2_unaries`` (fg = 0 inside).  ``noise = 0``: the clean blob."""
    g = torch.Generator().manual_seed(seed)
    xx, yy = _grid01(H, W)
    c = 0.5 + 0.04 * (torch.rand(2, generator=g) - 0.5)
    phase = float(torch.rand(1, generator=g)) * 2 * math.pi
    dx, dy = xx - float(c[0]), yy - float(c[1])
    rho = torch.sqrt(dx ** 2 + dy ** 2)
    r = r0 * (1 + a * torch.cos(k * torch.atan2(dy, dx) + phase))
    sdf = rho / r - 1
    return torch.sigmoid((sdf + noise * torch.randn(H, W, generator=g)) / tau).float()


def multi_object_unaries(H: int = 480, W: int = 640, n_objects: int = 8, seed: int = 42, tau: float = 0.08) -> torch.Tensor:
    """Config 4: ``[1, O+1, H, W]`` -- channel 0 background, channel k+1 the soft unaries of object k (fg = 0): O disjoint
    elliptic blobs on a 4 x 2 lattice (``multiple_object_aware_path_connected_net.py:186-192``)."""
    g = torch.Generator().manual_seed(seed)
    xx, yy = _grid01(H, W)
    cols = 4
    rows = (n_objects + cols - 1) // cols
    chans = []
    for k in range(n_objects):
        cx = (k % cols + 0.5) / cols + 0.02 * float(torch.randn(1, generator=g))
        cy = (k // cols + 0.5) / rows + 0.02 * float(torch.randn(1, generator=g))
        rx = 0.08 * (1 + 0.2 * float(torch.rand(1, generator=g)))
        ry = 0.5 / rows * 0.6 * (1 + 0.2 * float(torch.rand(1, generator=g)))
        sdf = torch.sqrt(((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2) - 1
        chans.append(torch.sigmoid((sdf + 0.05 * torch.randn(H, W, generator=g)) / tau))
    obj = torch.stack(chans)
    bg = 1 - torch.clamp((1 - obj).sum(0), 0, 1)
    return torch.cat([bg[None], obj])[None].float()


def pack_mask(mask: torch.Tensor) -> torch.Tensor:
    """Bool / {0,1} mask -> uint8 bit-packed (row-major, 8 pixels per byte, MSB first)."""
    import numpy as np
    return torch.from_numpy(np.packbits(mask.detach().cpu().reshape(-1).numpy().astype(bool)))


def unpack_mask(packed: torch.Tensor, H: int, W: int) -> torch.Tensor:
    import numpy as np
    bits = np.unpackbits(packed.cpu().numpy())[:H * W]
    return torch.from_numpy(bits.astype(bool)).reshape(H, W)


def fg_iou(pred_fg: torch.Tensor, target_fg: torch.Tensor) -> float:
    """``MIOU(average="binary", invert=True)`` on boolean foreground masks (``awesome/measures/miou.py:29-48``):
    Jaccard of the foreground; 0 when the target has none."""
    p, t = pred_fg.reshape(-1).bool(), target_fg.reshape(-1).bool()
    if int(t.sum()) == 0:
        return 0.0
    inter = int((p & t).sum())
    union = int((p | t).sum())
    return inter / union if union else 0.0


def stock_unet(in_chn: int = 4, out_chn: int = 1):
    """A plain PyTorch U-Net of the reference segmentation net's size (``awesome/model/unet.py``: widths 64-128-256-512-512,
    two 3x3 conv + BatchNorm + ReLU per level, 2x max-pool down, bilinear 2x up + skip concatenation, 1x1 output conv;
    13 395 905 parameters for ``in_chn=4``) -- the frozen / jointly trained segmentation side of BASELINE configs[4].  Stock
    cuDNN work and NOT part of the prior path: it exists so that the joint step and its gradient all-reduce are measured at
    the reference's message size (53.6 MB)."""
    import torch.nn as nn
    import torch.nn.functional as F

    def double(i, o):
        return nn.Sequential(nn.Conv2d(i, o, 3, padding=1), nn.BatchNorm2d(o), nn.ReLU(inplace=True),
                             nn.Conv2d(o, o, 3, padding=1), nn.BatchNorm2d(o), nn.ReLU(inplace=True))

    class UNet(nn.Module):
        def __init__(self):
            super().__init__()
            w = (64, 128, 256, 512, 512)
            self.enc = nn.ModuleList([double(in_chn, w[0])] + [double(w[i], w[i + 1]) for i in range(4)])
            self.dec = nn.ModuleList([double(w[4] + w[3], 256), double(256 + w[2], 128), double(128 + w[1], 64),
                                      double(64 + w[0], 64)])
            self.head = nn.Conv2d(64, out_chn, 1)

        def forward(self, x):
            skips = []
            for i, e in enumerate(self.enc):
                x = e(x if i == 0 else F.max_pool2d(x, 2))
                skips.append(x)
            x = skips.pop()
            for d in self.dec:
                s = skips.pop()
                x = F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True)
                dy, dx = s.shape[2] - x.shape[2], s.shape[3] - x.shape[3]
                if dy or dx:
                    x = F.pad(x, (dx // 2, dx - dx // 2, dy // 2, dy - dy // 2))
                x = d(torch.cat([s, x], dim=1))
            return self.head(x)
    return UNet()
