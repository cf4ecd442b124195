"""Device time of the fused optimizer kernel (profile class PK_OPT: ``k_reduce_opt_aug`` on these fits) per fit step of
the BASELINE configs[1] and configs[4] priors, and the whole step with the profiler off.

    python scripts/opt_kernel_cost.py --out OUT.jsonl [--label NAME]

``AWB_LIB_PATH`` selects the library build (A/B comparisons: run the script once per build, alternating, in one job).
Each line: GPU name and power limit, config, PK_OPT ms per launch (CUDA events around each launch, in a window of its
own; one launch per step) and ms per step of an unprofiled window (CUDA events around ``steps`` host-launched steps)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import awesome_b200 as A  # noqa: E402
from awesome_b200 import _lib  # noqa: E402

H, W = 480, 640


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in q.split(","))
    except Exception:       # the numbers stand without it; the line says so
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def unaries():
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    return torch.sigmoid((torch.sqrt(((xx - 0.52) / 0.27) ** 2 + ((yy - 0.47) / 0.31) ** 2) - 1) / 0.08).cuda()


def make(cfg):
    torch.manual_seed(0)
    un = unaries()
    if cfg == "configs1":     # ConvexNextNet(h=130, L=2, C=2), tensor path, one 640x480 frame, Adam 1e-3
        m = A.ConvexNextNet(n_hidden=130, in_features=2, n_hidden_layers=2, precision="f16").cuda()
        return m.make_fitter(A.GridSpecHost("linspace", 1, H, W), un, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3),
                             use_graph=False)
    # configs[4] prior: (x, y, t) RealNVP(18 flows, m=32) o ICNN(L=2) on 2 frames, Adamax + plateau, flow wd 1e-5
    m = A.real_nvp_path_connected_net(channels=3, hidden_units=32, flow_n_flows=18, flow_output_fn="tanh", norm="minmax",
                                      convex_net_hidden_units=130, convex_net_hidden_layers=2, precision="f16").cuda()
    tg = torch.stack([un, torch.roll(un, shifts=(5, 9), dims=(0, 1))])
    opt = A.OptimConfig("adamax", lr=1e-3, weight_decay=[1e-5, 0.0, 0.0, 0.0], plateau=True)
    return m.make_fitter(A.GridSpecHost("linspace", 2, H, W, t0=0.0, t_step=1.0 / 199), tg, A.LossConfig("mse"), opt,
                         use_graph=False)


def measure(cfg, steps):
    lib = _lib.load()
    f = make(cfg)
    f.run(20, record=False)                                   # warm-up: module load, first launches
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    f.run(steps, record=False)
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / steps
    n = lib.awb_profile_classes()
    names = [lib.awb_profile_class_name(i).decode() for i in range(n)]
    tot, cnt = (C.c_double * n)(), (C.c_int32 * n)()
    lib.awb_profile_enable(1)                                 # resets the per-class records (at most 256 per class)
    f.run(steps, record=False)
    _lib.check(lib.awb_profile_read(tot, cnt))
    lib.awb_profile_enable(0)
    k = names.index("reduce_opt")
    return dict(opt_ms_per_launch=tot[k] / max(cnt[k], 1), opt_launches_timed=cnt[k], step_ms_unprofiled=step_ms,
                steps=steps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--label", default=os.environ.get("AWB_LIB_PATH", "in-tree build"))
    ap.add_argument("--steps", type=int, default=200)
    a = ap.parse_args()
    name, power = gpu_info()
    with open(a.out, "a") as fh:
        for cfg in ("configs1", "configs4"):
            r = measure(cfg, a.steps)
            r.update(config=cfg, label=a.label, gpu=name, power_limit=power)
            line = json.dumps(r)
            print(line, flush=True)
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
