"""Cost of autograd through the star-shape prior (``awb_star_backward``, ``k_star_bwd``).

    python scripts/star_backward_cost.py [--steps K] [--warmup W] [--rounds R] [--out FILE]

For ``StarShapedNet(150)`` at n = 1 000 points (the notebook's sample) and n = 307 200 (a 640x480 likelihood image),
times from CUDA events, each mode in blocks of K calls after W warm calls, the modes alternating R times (median block):
  - ``native``: ``y = net(x); (w * y).sum().backward()`` on the drop-in (forward + backward, parameter gradients);
  - ``native_dx``: the same with ``x.requires_grad`` (also the point gradients);
  - ``eager``: the same loss through ``oracle.prior_oracle.star_forward`` in fp32 torch autograd on the same GPU;
  - ``fused_step``: one ``StarFitter.step`` (the per-point ``k_star<true>`` kernel, its reduction and Adam).
libawb's per-class timing follows in a separate pass: ``star_bwd`` is ``k_star_bwd``'s kernel time, ``misc`` in the
native modes is the forward ``k_star<false>`` and in the fused step ``k_star<true>``.  Prints and appends one JSON line
per size; the GPU's name and power limit are read in the same call."""
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
from oracle import prior_oracle as O  # noqa: E402


def per_class(lib, fn, steps):
    n_cls = lib.awb_profile_classes()
    lib.awb_profile_enable(1)
    for _ in range(steps):
        fn()
    tot, cnt = (C.c_double * n_cls)(), (C.c_int32 * n_cls)()
    _lib.check(lib.awb_profile_read(tot, cnt))
    lib.awb_profile_enable(0)
    names = [lib.awb_profile_class_name(i).decode() for i in range(n_cls)]
    return {names[i]: {"ms_per_call": tot[i] / steps, "launches_per_call": cnt[i] / steps}
            for i in range(n_cls) if cnt[i] > 0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("star_backward_cost.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    hw = {"gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit(0)}
    lines = []
    for n in (1000, 640 * 480):
        torch.manual_seed(0)
        m = A.StarShapedNet(150).to(dev)
        m.offset.requires_grad_(True)
        lib = m._prior_for(dev).lib
        g = torch.Generator(device=dev).manual_seed(n)
        x = torch.rand(n, 2, device=dev, generator=g) - 0.5
        w = torch.randn(n, device=dev, generator=g)
        t = (torch.rand(n, device=dev, generator=g) > 0.5).float()
        p32 = {k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
        fitter = A.StarShapedNet(150).to(dev).make_fitter(optim=A.OptimConfig("adam", lr=1e-2))
        fitter.train_offset = True

        def native():
            (w * m(x).reshape(-1)).sum().backward()

        def native_dx():
            xr = x.detach().requires_grad_(True)
            (w * m(xr).reshape(-1)).sum().backward()

        def eager():
            (w * O.star_forward(p32, x).reshape(-1)).sum().backward()

        def fused_step():
            fitter.step(x, t)

        modes = {"native": native, "native_dx": native_dx, "eager": eager, "fused_step": fused_step}
        for fn in modes.values():
            for _ in range(args.warmup):
                fn()
        blocks = {k: [] for k in modes}
        for _ in range(args.rounds):
            for k, fn in modes.items():
                blocks[k].append(timed(fn, args.steps))
        rec = {"case": "star_h150", "points": n, "calls_per_block": args.steps, "rounds": args.rounds, **hw}
        rec.update({f"ms_{k}": statistics.median(v) for k, v in blocks.items()})
        rec.update({f"ms_{k}_blocks": v for k, v in blocks.items()})
        rec["native_per_class"] = per_class(lib, native, args.steps)
        rec["fused_step_per_class"] = per_class(lib, fused_step, args.steps)
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))
        del m, fitter
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
