"""Scaling of the pixel-sliced spatio-temporal fit step (SlicedFitter, DESIGN 6) over the ranks of one box.

    torchrun --nproc-per-node N --master-addr 127.0.0.1 scripts/sequence_slices_scaling.py [--out FILE]

Workload: the BASELINE configs[4] prior (RealNVP, C = 3, 18 flows of width 32, ICNN 130 x 2, precision f16) on batches of
2 x 640x480 frames of a T = 200 sequence, S = 8 slices.  Prints one JSON line (rank 0): ms per sliced step from device
events over --steps warm steps (the slowest rank), the per-kernel-class split of a sliced step, the time of the row
gather alone, the SHA-256 of the parameters after --digest-steps sliced steps from the seeded start (equal for every N),
and, in the same call, the unsliced fused step of today's fit_sequence loop on one GPU.  GPU name and power limit are
read in the same call."""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.dont_write_bytecode = True

import awesome_b200 as A  # noqa: E402
from awesome_b200 import _lib  # noqa: E402

T, B, H, W = 200, 2, 480, 640


def power_limit(index: int) -> str:
    try:
        r = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or "unknown"
    except Exception:
        return "unknown"


def make_case(dev):
    torch.manual_seed(0)
    m = A.real_nvp_path_connected_net(channels=3, hidden_units=32, flow_n_flows=18, flow_output_fn="tanh",
                                      convex_net_hidden_units=130, convex_net_hidden_layers=2, precision="f16").to(dev)
    t_step = 1.0 / (T - 1)
    b0 = 40                                                           # batch of frames 40, 41
    grid = A.GridSpecHost("linspace", B, H, W, t0=b0 * t_step, t_step=t_step)
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    un = torch.stack([torch.sigmoid((torch.sqrt(((xx - 0.45 - 0.01 * b) / 0.2) ** 2 + ((yy - 0.5) / 0.25) ** 2) - 1) / 0.08)
                      for b in range(B)])
    return m, grid, un.reshape(1, -1).to(dev)


def timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def profile_split(lib, fn, steps=20):
    n_cls = lib.awb_profile_classes()
    lib.awb_profile_enable(1)
    for _ in range(steps):
        fn()
    tot, cnt = (C.c_double * n_cls)(), (C.c_int32 * n_cls)()
    _lib.check(lib.awb_profile_read(tot, cnt))
    lib.awb_profile_enable(0)
    return {lib.awb_profile_class_name(i).decode(): {"ms_per_step": tot[i] / steps, "launches_per_step": cnt[i] / steps}
            for i in range(n_cls) if cnt[i] > 0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--digest-steps", type=int, default=200)
    ap.add_argument("--slices", type=int, default=8)
    ap.add_argument("--out", default=None, help="append the JSON line to this file (rank 0)")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    try:
        m, grid, target = make_case(dev)
        arena = m._ensure_flat()
        prior = m._prior_for(dev)
        lib = prior.lib
        init = arena.detach().clone()
        opt = A.OptimConfig("adamax", lr=1e-3, weight_decay=[1e-5, 0.0, 0.0, 0.0])
        f = A.SlicedFitter(prior, arena, grid, target, A.LossConfig("mse"), opt, n_slices=args.slices, group=group)
        # digest: fixed number of sliced steps from the seeded start
        loss = f.run(args.digest_steps)
        torch.cuda.synchronize()
        digest = hashlib.sha256(arena.detach().cpu().numpy().tobytes()).hexdigest()
        final_loss = float(loss[-1, 0])
        # timing: warm steps, then the timed window; the slowest rank's time counts
        for _ in range(args.warmup):
            f.step()
        if group is not None:
            dist.barrier()
        ms = timed(f.step, args.steps)
        if group is not None:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        split = profile_split(lib, f.step)
        gather_ms = 0.0
        if group is not None:
            for _ in range(20):
                dist.all_gather_into_tensor(f.rows, f.local, group=group)
            gather_ms = timed(lambda: dist.all_gather_into_tensor(f.rows, f.local, group=group), 500)
        # today's unsliced loop: one fused awb_prior_fit_step per batch (fit_sequence without n_slices), on rank 0's GPU
        fused = None
        if rank == 0:
            with torch.no_grad():
                arena.copy_(init)
            pf = A.PriorFitter(prior, arena, grid, target, A.LossConfig("mse"), opt, use_graph=False)
            for _ in range(args.warmup):
                pf.run(1)
            fused_ms = timed(lambda: pf.run(1), args.steps)
            fused = {"ms_per_step": fused_ms, "per_class": profile_split(lib, lambda: pf.run(1))}
        if rank == 0:
            out = {"workload": "spatio-temporal prior step, BASELINE configs[4] prior, 2 x 640x480 frames, T = 200",
                   "n_gpus": world, "n_slices": args.slices, "slices_per_rank": args.slices // world,
                   "params": prior.n_params, "grad_row_bytes": 4 * prior.grad_row_floats,
                   "sliced_ms_per_step": ms, "timed_steps": args.steps, "sliced_per_class": split,
                   "gather_ms": gather_ms, "digest_steps": args.digest_steps, "params_sha256": digest,
                   "loss_after_digest_steps": final_loss, "unsliced_fused": fused,
                   "speedup_vs_unsliced": (fused["ms_per_step"] / ms) if fused else None,
                   "gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit(local)}
            line = json.dumps(out)
            print(line, flush=True)
            if args.out:
                os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
                with open(args.out, "a") as fh:
                    fh.write(line + "\n")
    finally:
        if group is not None:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
