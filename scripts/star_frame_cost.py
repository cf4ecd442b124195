"""Cost of the star prior's whole-frame fit step (``awb_prior_fit_step`` on a star handle, ``k_star_bwd`` in its fit
mode) against the notebook's per-point step (``awb_star_fit_step``, ``k_star<true>``), on the same points.

    python scripts/star_frame_cost.py [--steps K] [--rounds R] [--out FILE]

Sizes: n = 1000 (grid [1,2,1,1000], the notebook's sampled points), 640x480 and two 640x480 frames.  Every shape is
warmed up; then the two steps alternate in blocks of K steps (at least 200), timed with CUDA events, R rounds each; the
median per-step time is reported.  A separate pass reads the kernel time per step from libawb's profile classes
(``star_fit`` for the grid step, ``misc`` = ``k_star<true>`` for the per-point step, ``reduce_opt`` for both).  Prints
and appends one JSON line per size, with the card's name and power limit, to ``--out``."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import awesome_b200 as A  # noqa: E402
from awesome_b200 import _lib as L  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    name, pl = (q[0].split(", ") + ["?"])[:2] if q else (torch.cuda.get_device_name(0), "?")
    return {"gpu": name, "power_limit": pl}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="profiles/r11_star_frames.jsonl")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("star_frame_cost.py measures on a CUDA device; none is visible")
    K = max(200, a.steps)
    dev = torch.device("cuda:0")
    lib = L.load()
    hw = card()
    sizes = [("n1000", 1, 1, 1000), ("640x480", 1, 480, 640), ("2x640x480", 2, 480, 640)]
    for name, B, H, W in sizes:
        N = B * H * W
        torch.manual_seed(0)
        m = A.StarShapedNet(150).to(dev)
        g = torch.Generator(device=dev).manual_seed(1)
        rows = torch.rand((N, 2), device=dev, generator=g) - 0.5
        t = torch.rand(N, device=dev, generator=g)
        grid = rows.reshape(B, H, W, 2).permute(0, 3, 1, 2).contiguous()
        loss = A.LossConfig("mse")
        opt = A.OptimConfig("adam", lr=1e-5)
        fg = m.make_fitter(grid, t, loss, opt, use_graph=False)
        fp = m.make_fitter(optim=opt, loss=loss)
        step_grid = lambda: fg._step(0)
        step_pts = lambda: fp.step(rows, t)
        for f in (step_grid, step_pts):
            for _ in range(10):
                f()
        torch.cuda.synchronize()
        times = {"grid": [], "points": []}
        for _ in range(a.rounds):
            for key, f in (("grid", step_grid), ("points", step_pts)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(K):
                    f()
                e1.record()
                e1.synchronize()
                times[key].append(e0.elapsed_time(e1) / K)
        kern = {}
        n_cls = lib.awb_profile_classes()
        for key, f in (("grid", step_grid), ("points", step_pts)):
            tot = (C.c_double * n_cls)()
            cnt = (C.c_int32 * n_cls)()
            lib.awb_profile_read(tot, cnt)          # clears what earlier passes left
            lib.awb_profile_enable(1)
            for _ in range(50):
                f()
            lib.awb_profile_read(tot, cnt)
            lib.awb_profile_enable(0)
            kern[key] = {lib.awb_profile_class_name(c).decode(): round(tot[c] / 50, 4) for c in range(n_cls) if cnt[c]}
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        rec = {"case": f"star_h150_{name}", "points": N, "steps_per_block": K, "rounds": a.rounds, **hw,
               "grid_step_ms": round(med["grid"], 4), "point_step_ms": round(med["points"], 4),
               "speedup": round(med["points"] / med["grid"], 2),
               "grid_step_ms_rounds": [round(x, 4) for x in times["grid"]],
               "point_step_ms_rounds": [round(x, 4) for x in times["points"]],
               "kernel_ms_per_step": kern}
        print(json.dumps(rec), flush=True)
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "a") as fh:
            fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
