"""Cost of a gradient penalty trained through an ICNN prior (``second_order=True``).

    python scripts/second_order_cost.py [--steps K] [--warmup W] [--rounds R] [--out FILE]

On one 640x480 frame with ``ConvexNextNet(n_hidden_layers=2, second_order=True)``, fp32 and f16, times from device events
  - a first-order autograd step: ``mse(sigmoid(y), target).backward()``;
  - a penalised step: ``g = grad(y.sum(), grid, create_graph=True)``, then
    ``(mse(sigmoid(y), target) + lam * mean((|g| - 1)^2)).backward()``, which runs the second-order pass
    (``awb_prior_grid_grad_backward``) once.
The two steps alternate R times, each block of K steps after W warm steps; the median block counts.  libawb's per-class
timing of the penalised step follows in a separate pass (profile mode brackets every launch with events).  Prints and
appends one JSON line per precision; GPU name and power limit are read in the same call."""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.dont_write_bytecode = True

import awesome_b200 as A  # noqa: E402
from awesome_b200 import _lib  # noqa: E402
from coord_grad_cost import power_limit, timed  # noqa: E402

LAM = 0.1


def per_class(lib, fn, steps):
    n_cls = lib.awb_profile_classes()
    lib.awb_profile_enable(1)
    for _ in range(steps):
        fn()
    tot, cnt = (C.c_double * n_cls)(), (C.c_int32 * n_cls)()
    _lib.check(lib.awb_profile_read(tot, cnt))
    lib.awb_profile_enable(0)
    names = [lib.awb_profile_class_name(i).decode() for i in range(n_cls)]
    return {names[i]: {"ms_per_step": tot[i] / steps, "launches_per_step": cnt[i] / steps}
            for i in range(n_cls) if cnt[i] > 0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("second_order_cost.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    H, W = 480, 640
    hw = {"gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit(0)}
    grid = A.GridSpecHost("linspace", 1, H, W).materialize(2, dev)
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H, device=dev), torch.linspace(0, 1, W, device=dev), indexing="ij")
    target = (((xx - 0.5) / 0.3) ** 2 + ((yy - 0.5) / 0.25) ** 2 < 1).float().reshape(1, 1, H, W)
    lines = []
    for prec in ("fp32", "f16"):
        torch.manual_seed(0)
        m = A.ConvexNextNet(n_hidden_layers=2, precision=prec, second_order=True).to(dev)
        lib = m._prior_for(dev).lib

        def first_order():
            y = m(grid)
            torch.nn.functional.mse_loss(torch.sigmoid(y), target).backward()

        def penalised():
            x = grid.detach().requires_grad_(True)
            y = m(x)
            g = torch.autograd.grad(y.sum(), x, create_graph=True)[0]
            pen = ((g.pow(2).sum(1) + 1e-12).sqrt() - 1).pow(2).mean()
            (torch.nn.functional.mse_loss(torch.sigmoid(y), target) + LAM * pen).backward()

        modes = {"first_order": first_order, "penalised": penalised}
        for fn in modes.values():
            for _ in range(args.warmup):
                fn()
        blocks = {k: [] for k in modes}
        for _ in range(args.rounds):
            for k, fn in modes.items():
                blocks[k].append(timed(fn, args.steps))
        rec = {"case": "icnn_L2_640x480", "precision": prec, "pixels": H * W, "steps_per_block": args.steps,
               "rounds": args.rounds, **hw}
        rec.update({f"ms_{k}": statistics.median(v) for k, v in blocks.items()})
        rec.update({f"ms_{k}_blocks": v for k, v in blocks.items()})
        rec["delta_ms"] = rec["ms_penalised"] - rec["ms_first_order"]
        rec["penalised_per_class"] = per_class(lib, penalised, args.steps)
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))
        del m
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
