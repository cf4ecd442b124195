"""Step time of the fused fit with and without per-pixel loss weights and an ignore label, in alternating blocks.

    python scripts/loss_weights_cost.py --out OUT.jsonl [--steps 200] [--blocks 4]

Configurations: configs[1] (4 grouped ConvexNextNet(h=130, L=2) priors on one 640x480 frame each, tensor path, Adam 1e-3)
and the c3 flow prior of configs[4] ((x, y, t) RealNVP(18 flows, m=32) o ICNN(L=2) on 2 frames of 640x480, Adamax +
plateau), fp32 and f16.  Weighted: a weight map uniform in [0, 2] and 30 % of the pixels at the ignore label 2; the
unweighted fit uses the same targets with the ignored pixels set to 1.  Each block times ``steps`` host-launched steps
(``awb_prior_fit_steps`` over a pool of two targets, no history) with CUDA events, unweighted then weighted; every line
carries the GPU name and its power limit."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import awesome_b200 as A  # noqa: E402

H, W = 480, 640
IGN = 2.0


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in q.split(","))
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def targets(n_frames, O_):
    g = torch.Generator().manual_seed(0)
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    un = torch.sigmoid((torch.sqrt(((xx - 0.52) / 0.27) ** 2 + ((yy - 0.47) / 0.31) ** 2) - 1) / 0.08)
    t = torch.stack([torch.roll(un, shifts=(3 * k, 5 * k), dims=(0, 1)) for k in range(n_frames * O_)])
    t = t.reshape(O_, -1)
    ign = torch.rand(t.shape, generator=g) < 0.3
    weak = torch.where(ign, torch.full_like(t, IGN), t)
    plain = torch.where(ign, torch.ones_like(t), t)
    w = 2.0 * torch.rand(t.shape, generator=g)
    return plain.cuda(), weak.cuda(), w.cuda()


def make(cfg, weighted):
    torch.manual_seed(0)
    if cfg == "configs1":
        O_, n_frames = 4, 1
        multi = A.NumberBasedMultiPriorModule(prior_type=A.ConvexNextNet, prior_args=dict(n_hidden_layers=2, precision="f16"),
                                              min_priors=O_).cuda()
        grid, opt = A.GridSpecHost("linspace", 1, H, W), A.OptimConfig("adam", lr=1e-3)
        plain, weak, w = targets(n_frames, O_)
        make_fitter = multi.make_fitter
    else:
        prec = "f16" if cfg.endswith("f16") else "fp32"
        O_, n_frames = 1, 2
        m = A.real_nvp_path_connected_net(channels=3, hidden_units=32, flow_n_flows=18, flow_output_fn="tanh", norm="minmax",
                                          convex_net_hidden_units=130, convex_net_hidden_layers=2, precision=prec).cuda()
        grid = A.GridSpecHost("linspace", 2, H, W, t0=0.0, t_step=1.0 / 199)
        opt = A.OptimConfig("adamax", lr=1e-3, weight_decay=[1e-5, 0.0, 0.0, 0.0], plateau=True)
        plain, weak, w = targets(n_frames, O_)
        make_fitter = m.make_fitter
    tg = weak if weighted else plain
    loss = A.LossConfig("mse", weight=w, ignore_value=IGN) if weighted else A.LossConfig("mse")
    f = make_fitter(grid, tg, loss, opt, use_graph=False)
    f.set_target_pool(torch.stack([tg, torch.roll(tg, 7, dims=1)]).contiguous())
    return f


def time_steps(f, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    f.run(steps, record=False)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--blocks", type=int, default=4)
    a = ap.parse_args()
    name, power = gpu_info()
    with open(a.out, "a") as fh:
        for cfg in ("configs1", "c3flow_fp32", "c3flow_f16"):
            fits = {False: make(cfg, False), True: make(cfg, True)}
            for f in fits.values():
                f.run(20, record=False)                        # warm-up: module load, first launches
            torch.cuda.synchronize()
            ms = {False: [], True: []}
            for _ in range(a.blocks):                          # alternating blocks: unweighted, weighted
                for wt in (False, True):
                    ms[wt].append(time_steps(fits[wt], a.steps))
            for f in fits.values():
                f.raise_if_nonfinite()
            r = dict(config=cfg, steps_per_block=a.steps, blocks=a.blocks, unweighted_ms=ms[False], weighted_ms=ms[True],
                     unweighted_ms_median=sorted(ms[False])[len(ms[False]) // 2],
                     weighted_ms_median=sorted(ms[True])[len(ms[True]) // 2], gpu=name, power_limit=power)
            r["weighted_over_unweighted"] = r["weighted_ms_median"] / r["unweighted_ms_median"]
            line = json.dumps(r)
            print(line, flush=True)
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
