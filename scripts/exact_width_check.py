"""A/B check of the exact fp32 ICNN path between two builds of libawb: outputs bit for bit, and the fp32 fit step's time.

    python scripts/exact_width_check.py --lib parent=PATH --lib new=PATH [--rounds R] [--steps K] [--warmup W]
                                        [--dump-dir DIR] [--out FILE]

Each build runs in its own process (``AWB_LIB_PATH`` names it; the library is loaded once per process).  The first process
of each build dumps, for a fixed seeded set of shapes whose augmented rows fit one k_gemm tile (ld <= 144), the logits,
autograd parameter gradients and dgrid, the parameters, moments and loss after one fused Adam step, and the second-order
pass of a gradient penalty, to ``DIR/<label>.npz`` (a temporary directory by default); the dumps of all builds must be
equal bit for bit.  Then R rounds alternate the builds, each timing K fused fp32 fit steps (after W warm steps, device
events) of one 640x480 frame at h = 130, L = 2 (the default width) and at h = 256, L = 2 (ld = 264, two column tiles).  Prints one JSON line with the
per-build medians and every round, and the GPU name and power limit read in the same call; ``--out`` appends it to FILE."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")

# (C, h, L, O, B, H, W): ld = round_up(h + C + 1, 8) <= 144 throughout
DUMP_SHAPES = [(2, 8, 1, 1, 1, 1, 257), (3, 37, 0, 1, 3, 17, 29), (3, 37, 3, 1, 3, 17, 29), (2, 130, 2, 1, 1, 480, 640),
               (3, 130, 8, 1, 3, 17, 29), (2, 141, 2, 1, 3, 17, 29), (3, 140, 1, 4, 3, 17, 29)]
TIME_SHAPES = [(2, 130, 2), (2, 256, 2)]      # (C, h, L) on one 640x480 frame


def child(args):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    sys.dont_write_bytecode = True
    import awesome_b200 as A
    from awesome_b200 import _lib as L
    dev = torch.device("cuda", 0)

    def target_of(O, B, H, W):
        yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
        return torch.stack([torch.sigmoid((torch.sqrt(((xx - 0.4 - 0.02 * o) / 0.22) ** 2 + ((yy - 0.5) / 0.27) ** 2) - 1)
                                          / 0.08).expand(B, H, W).reshape(-1) for o in range(O)]).contiguous().to(dev)

    def setup(C_, h, L_, O, B, H, W, seed):
        models = []
        for o in range(O):
            torch.manual_seed(seed + 17 * o)
            models.append(A.ConvexNextNet(n_hidden=h, in_features=C_, n_hidden_layers=L_).to(dev))
        prior = A.Prior(L.AWB_KIND_ICNN, C_, h, L_, n_objects=O)
        params = torch.stack([m._ensure_flat().detach() for m in models]).contiguous()
        return prior, params, A.GridSpecHost("linspace", B, H, W, t0=0.1, t_step=0.3), target_of(O, B, H, W)

    if args.dump:
        out = {}
        for i, (C_, h, L_, O, B, H, W) in enumerate(DUMP_SHAPES):
            key = f"c{C_}_h{h}_L{L_}_o{O}_{B}x{H}x{W}"
            prior, params, spec, target = setup(C_, h, L_, O, B, H, W, seed=i)
            N = spec.n_pixels
            ws = prior.new_workspace(N, L.AWB_WS_TRAINING, dev)
            logits, _ = prior.forward(params, spec, L.AWB_FWD_EXACT_TRAINING, ws)
            s = torch.sigmoid(logits)
            dlog = (2.0 * (s - target) * s * (1 - s) / N).contiguous()
            grads, dgrid = prior.backward(params, spec, dlog, ws, O == 1)     # dgrid: single-object handles
            f = A.PriorFitter(prior, params.clone(), spec, target, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3),
                              use_graph=False)
            loss = f.run(1)
            out.update({f"{key}/logits": logits, f"{key}/grads": grads, f"{key}/step_loss": loss,
                        f"{key}/step_params": f.params, f"{key}/step_opt_state": f.opt_state})
            if O == 1:   # dgrid, and the second-order pass with a random cotangent on it
                out[f"{key}/dgrid"] = dgrid
                ws2 = prior.new_workspace(N, L.AWB_WS_SECOND_ORDER, dev)
                prior.forward(params, spec, L.AWB_FWD_EXACT_TRAINING, ws2)
                d_dgrid = torch.randn(dgrid.shape, device=dev, generator=torch.Generator(device=dev).manual_seed(i))
                d_dlogits, g2 = prior.grid_grad_backward(params, spec, dlog, d_dgrid, ws2)
                out.update({f"{key}/tangent_dlogits": d_dlogits, f"{key}/tangent_grads": g2})
        torch.cuda.synchronize()
        np.savez(args.dump, **{k: v.detach().cpu().numpy() for k, v in out.items()})

    rec = {}
    for C_, h, L_ in TIME_SHAPES:
        prior, params, spec, target = setup(C_, h, L_, 1, 1, 480, 640, seed=0)
        f = A.PriorFitter(prior, params.clone(), spec, target, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3))
        f.run(args.warmup)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        f.run(args.steps)
        e1.record()
        torch.cuda.synchronize()
        rec[f"c{C_}_h{h}_L{L_}_640x480"] = e0.elapsed_time(e1) / args.steps
        del f, prior, params
        torch.cuda.empty_cache()
    print("RESULT " + json.dumps(rec), flush=True)


def gpu_info():
    import torch
    r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30)
    return {"gpu": torch.cuda.get_device_name(0), "power_limit": r.stdout.strip() or "unknown"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="LABEL=PATH of a libawb.so build (two or more)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=25)
    ap.add_argument("--dump-dir", default=None, help="where the .npz dumps go (default: a temporary directory)")
    ap.add_argument("--out", default=None, help="append the JSON line to this file")
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        return child(args)
    libs = dict(s.split("=", 1) for s in args.lib)
    if len(libs) < 2:
        raise SystemExit("name two or more builds with --lib LABEL=PATH")
    dump_dir = args.dump_dir or tempfile.mkdtemp(prefix="exact_width_")
    os.makedirs(dump_dir, exist_ok=True)
    times = {k: [] for k in libs}
    for r in range(args.rounds):
        order = list(libs) if r % 2 == 0 else list(libs)[::-1]
        for label in order:
            cmd = [sys.executable, os.path.abspath(__file__), "--child", "--steps", str(args.steps), "--warmup",
                   str(args.warmup)]
            if r == 0:
                cmd += ["--dump", os.path.join(dump_dir, f"{label}.npz")]
            res = subprocess.run(cmd, env=dict(os.environ, AWB_LIB_PATH=os.path.abspath(libs[label])), capture_output=True,
                                 text=True)
            if res.returncode != 0:
                sys.stderr.write(res.stdout + res.stderr)
                raise SystemExit(f"{label}: child failed ({res.returncode})")
            times[label].append(json.loads(res.stdout.split("RESULT ", 1)[1]))
    import numpy as np
    dumps = {k: np.load(os.path.join(dump_dir, f"{k}.npz")) for k in libs}
    first = next(iter(libs))
    differ = sorted({f"{k}:{n}" for k in libs for n in set(dumps[k].files) | set(dumps[first].files)
                     if n not in dumps[k].files or n not in dumps[first].files
                     or dumps[k][n].tobytes() != dumps[first][n].tobytes()})
    shapes = list(times[first][0])
    rec = {"check": "exact_width", **gpu_info(), "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
           "arrays": len(dumps[first].files), "bit_identical": not differ, "differ": differ,
           "ms_per_step_median": {k: {s: statistics.median(t[s] for t in times[k]) for s in shapes} for k in libs},
           "ms_per_step_rounds": {k: {s: [t[s] for t in times[k]] for s in shapes} for k in libs}}
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")
    if differ:
        raise SystemExit(f"outputs differ between builds: {differ}")


if __name__ == "__main__":
    main()
