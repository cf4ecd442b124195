"""Cost of autograd through ``PathConnectedNet.inverse`` (``awb_prior_inverse``, ``awb_prior_inverse_backward``).

    python scripts/inverse_grad_cost.py [--steps K] [--warmup W] [--rounds R] [--out FILE]

Two cases with m = 32 tanh couplings on the exact fp32 handle: one 640x480 frame at C = 2, F = 12, and two 640x480
frames at C = 3, F = 18 (the spatio-temporal prior; its backward keeps the running gradient in the workspace).  Times
from CUDA events, each mode in blocks of K calls after W warm calls, the modes alternating R times (median block):
  - ``inverse``: ``awb_prior_inverse(training = 0)`` (``k_flow_inv``, what the no-grad module call runs);
  - ``inverse_training``: ``awb_prior_inverse(training = 1)`` (``k_flow_inv_rec``, which also keeps the records);
  - ``inverse_backward``: ``awb_prior_inverse_backward`` with dgrid (``k_flow_inv_bwd`` and the gradient reduction);
  - ``autograd``: ``(w * m.inverse(x)).sum().backward()`` with ``x.requires_grad``;
  - ``deformation_backward``: ``awb_prior_deformation_backward`` with dgrid (the unit-loop ``k_flow_bwd``), for scale.
libawb's per-class timing follows in a separate pass: ``flow_fwd`` / ``flow_bwd`` are the kernel times of the inverse and
of its backward.  Prints and appends one JSON line per case; the GPU's name and power limit are read in the same call."""
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
from star_backward_cost import per_class  # noqa: E402


def make(C_, F, dev):
    torch.manual_seed(0)
    m = A.real_nvp_path_connected_net(channels=C_, hidden_units=32, flow_n_flows=F, flow_output_fn="tanh",
                                      convex_net_hidden_units=130, convex_net_hidden_layers=2)
    sd = m.state_dict()
    for k in sd:
        if ".net.2." in k:
            sd[k] = 0.05 * torch.randn_like(sd[k])
        elif k.endswith((".s", ".t")) and ".flows." in k:
            sd[k] = 0.1 * torch.randn_like(sd[k])
        elif k.endswith("data_dep_init_done"):
            sd[k] = torch.ones_like(sd[k])
    m.load_state_dict(sd)
    return m.to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("inverse_grad_cost.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    hw = {"gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit(0)}
    lines = []
    for C_, F, B in ((2, 12, 1), (3, 18, 2)):
        H, W = 480, 640
        m = make(C_, F, dev)
        arena = m._ensure_flat()
        prior = m._prior_for(dev)
        lib = prior.lib
        yy, xx = torch.meshgrid(torch.linspace(0, 1, H, device=dev), torch.linspace(0, 1, W, device=dev), indexing="ij")
        ch = [xx.expand(B, H, W), yy.expand(B, H, W)] + ([torch.full((B, H, W), 0.25, device=dev)] if C_ == 3 else [])
        grid = torch.stack(ch, 1).contiguous()
        with torch.no_grad():
            xd = m.get_deformation(grid).contiguous()
        spec = A.GridSpecHost.from_tensor(xd)
        gspec = A.GridSpecHost.from_tensor(grid)
        n = spec.n_pixels
        ws = prior.new_workspace(n, _lib.AWB_WS_DEFORMATION, dev)
        ws_def = prior.new_workspace(n, _lib.AWB_WS_DEFORMATION, dev)
        g = torch.Generator(device=dev).manual_seed(n)
        d_out = torch.randn(n, C_, device=dev, generator=g)
        w = torch.randn(B, C_, H, W, device=dev, generator=g)
        prior.inverse(arena, spec, True, ws)
        prior.deformation(arena, gspec, True, ws_def)

        def inverse():
            prior.inverse(arena, spec, False, ws)

        def inverse_training():
            prior.inverse(arena, spec, True, ws)

        def inverse_backward():
            prior.inverse_backward(arena, spec, d_out, ws, True)

        def autograd():
            x = xd.detach().requires_grad_(True)
            (w * m.inverse(x)).sum().backward()

        def deformation_backward():
            prior.deformation_backward(arena, gspec, d_out, ws_def, True)

        modes = {"inverse": inverse, "inverse_training": inverse_training, "inverse_backward": inverse_backward,
                 "autograd": autograd, "deformation_backward": deformation_backward}
        for fn in modes.values():
            for _ in range(args.warmup):
                fn()
        blocks = {k: [] for k in modes}
        for _ in range(args.rounds):
            for k, fn in modes.items():
                blocks[k].append(timed(fn, args.steps))
        rec = {"case": f"inverse_c{C_}_f{F}_m32", "B": B, "H": H, "W": W, "pixels": n, "calls_per_block": args.steps,
               "rounds": args.rounds, **hw}
        rec.update({f"ms_{k}": statistics.median(v) for k, v in blocks.items()})
        rec.update({f"ms_{k}_blocks": v for k, v in blocks.items()})
        for k in ("inverse", "inverse_training", "inverse_backward", "deformation_backward"):
            rec[f"{k}_per_class"] = per_class(lib, modes[k], args.steps)
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))
        del m, ws, ws_def
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
