"""Cost of the coordinate gradient (d / d grid) of the flow priors, and of a differentiable get_deformation.

    python scripts/coord_grad_cost.py [--steps K] [--warmup W] [--rounds R] [--out FILE]

Times, from device events, one autograd ``forward + backward`` of ``sum(w * prior(grid))`` with and without
``grid.requires_grad`` (the two modes alternate R times, each block of K steps after W warm steps; the median block
counts) for:
  - the path-connectedness prior of bench.py's c2 leg (C = 2, F = 12, 1 x 480 x 640), f16 (segment tables) and fp32;
  - the spatio-temporal prior of its c4 leg (C = 3, F = 18, 2 x 480 x 640), f16;
  - a ConvexDiffeomorphismNet (4 couplings of width 70, ICNN 130 x 1) at 640x480, f16 and fp32;
and ``get_deformation`` forward + backward of the two RealNVP priors, with and without the grid gradient.  The flow
backward's kernel time per step (libawb's per-class timing, in a separate pass) isolates the store of dgrid.  Prints and
appends one JSON line per case; GPU name and power limit are read in the same call."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.dont_write_bytecode = True

import awesome_b200 as A  # noqa: E402
from awesome_b200 import _lib  # noqa: E402


def power_limit(index: int) -> str:
    try:
        r = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or "unknown"
    except Exception:
        return "unknown"


def timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def flow_bwd_ms(lib, fn, steps):
    n_cls = lib.awb_profile_classes()
    lib.awb_profile_enable(1)
    for _ in range(steps):
        fn()
    tot, cnt = (C.c_double * n_cls)(), (C.c_int32 * n_cls)()
    _lib.check(lib.awb_profile_read(tot, cnt))
    lib.awb_profile_enable(0)
    names = [lib.awb_profile_class_name(i).decode() for i in range(n_cls)]
    return tot[names.index("flow_bwd")] / steps


def realnvp(dev, C_, F, precision):
    torch.manual_seed(0)
    m = A.real_nvp_path_connected_net(channels=C_, hidden_units=32, flow_n_flows=F, flow_output_fn="tanh", norm="minmax",
                                      convex_net_hidden_units=130, convex_net_hidden_layers=2, precision=precision).to(dev)
    sd = m.state_dict()
    for k in sd:                      # non-trivial couplings and 1x1 conv, initialised ActNorms
        if ".net.2." in k:
            sd[k] = 0.05 * torch.randn_like(sd[k])
        elif k.endswith((".s", ".t")) and ".flows." in k:
            sd[k] = 0.1 * torch.randn_like(sd[k])
        elif k.endswith("data_dep_init_done"):
            sd[k] = torch.ones_like(sd[k])
        elif k == "linear.weight":
            sd[k] = 1.0 + 0.3 * torch.randn_like(sd[k])
    m.load_state_dict(sd)
    return m


def diffeo(dev, precision):
    torch.manual_seed(0)
    return A.ConvexDiffeomorphismNet(n_hidden=130, n_hidden_layers=1, nf_layers=4, nf_hidden=70, precision=precision).to(dev)


def measure(m, grid, w, what, steps, warmup, rounds, lib):
    def step(want):
        x = grid.detach().requires_grad_(want)
        y = m.get_deformation(x) if what == "get_deformation" else m(x)
        (w * y).sum().backward()

    modes = {"without_dgrid": False, "with_dgrid": True}
    for want in modes.values():
        for _ in range(warmup):
            step(want)
    blocks = {k: [] for k in modes}
    for _ in range(rounds):
        for k, want in modes.items():
            blocks[k].append(timed(lambda: step(want), steps))
    out = {f"ms_{k}": statistics.median(v) for k, v in blocks.items()}
    out.update({f"ms_{k}_blocks": v for k, v in blocks.items()})
    out["delta_ms"] = out["ms_with_dgrid"] - out["ms_without_dgrid"]
    out.update({f"flow_bwd_kernel_ms_{k}": flow_bwd_ms(lib, lambda: step(want), steps) for k, want in modes.items()})
    out["flow_bwd_kernel_delta_ms"] = out["flow_bwd_kernel_ms_with_dgrid"] - out["flow_bwd_kernel_ms_without_dgrid"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("coord_grad_cost.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    H, W = 480, 640
    hw = {"gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit(0)}
    g2 = A.GridSpecHost("linspace", 1, H, W).materialize(2, dev)
    g3 = A.GridSpecHost("linspace", 2, H, W, t0=0.2, t_step=0.005).materialize(3, dev)
    cases = [
        ("c2_path_connected_640x480", "forward", lambda: realnvp(dev, 2, 12, "f16"), g2, "f16"),
        ("c2_path_connected_640x480", "forward", lambda: realnvp(dev, 2, 12, "fp32"), g2, "fp32"),
        ("c4_spatio_temporal_prior_2x640x480", "forward", lambda: realnvp(dev, 3, 18, "f16"), g3, "f16"),
        ("convex_diffeomorphism_640x480", "forward", lambda: diffeo(dev, "f16"), g2, "f16"),
        ("convex_diffeomorphism_640x480", "forward", lambda: diffeo(dev, "fp32"), g2, "fp32"),
        ("c2_path_connected_640x480", "get_deformation", lambda: realnvp(dev, 2, 12, "f16"), g2, "f16"),
        ("c4_spatio_temporal_prior_2x640x480", "get_deformation", lambda: realnvp(dev, 3, 18, "f16"), g3, "f16"),
    ]
    lines = []
    for name, what, make, grid, prec in cases:
        m = make()
        lib = m._prior_for(dev).lib
        torch.manual_seed(1)
        w = torch.randn((grid.shape[0], 1 if what == "forward" else grid.shape[1]) + tuple(grid.shape[2:]), device=dev)
        rec = {"case": name, "what": f"{what} + backward, autograd", "precision": prec, "pixels": grid.numel() // grid.shape[1],
               "steps_per_block": args.steps, "rounds": args.rounds, **hw}
        rec.update(measure(m, grid, w, what, args.steps, args.warmup, args.rounds, lib))
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
