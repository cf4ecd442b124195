#!/usr/bin/env python
"""Benchmark of the prior-fit hot path (BASELINE.json metric: prior-fit pixel-samples/sec, fwd+bwd+step).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision fp32|f16] [--dump-outputs DIR]

Workload (config.workload): BASELINE configs[1] -- the convexity prior ``ConvexNextNet(h=130, L=2, C=2)``
fitted per frame on a synthetic FBMS-shaped 640x480 frame (unaries = soft UNet-like blob), loss
``UnariesWeightedLoss(SE)`` = MSE(sigmoid(y), unaries), Adam lr 1e-3, enforce_convexity every step.
One "step" = one fused fit step (forward + loss + backward + gradient reduction + Adam + clamp) over a group of
G = --frames-per-step (default 4) independent frames of the rank's share of the sequence, one prior per frame,
= G x 307 200 pixel-samples per GPU.  With N GPUs every rank fits its own frames (frames are independent: no
data-path collective; weak scaling); value = N * G * 307200 * K / max-over-ranks time.

Prints ONE JSON line (see the task contract): value (inputs resident in HBM, device-timed with CUDA
events), e2e (same metric through the public fit API with the step's unaries coming from pinned host
memory and the step's loss read back, copies inside the timed region), roofline (dominant kernel,
timed live with CUDA events on the launch stream), cpu_baseline (the oracle port on the host cores,
rank 0, bounded sample), clocks, gpu_launches.

``--dump-outputs DIR`` writes what the K timed steps computed (rank 0): ``params.npy`` = the fitted parameters of the
G priors after the last timed step [G,P] (float32, each row in ``parameters()`` order), ``loss.npy`` = the loss of that
step per frame [G] (float64).  The inputs depend on the arguments only, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import atexit
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the benchmark may run from a read-only tree: it writes nothing into it

H, W = 480, 640
N_PIX = H * W
POOL_FRAMES = 112          # 112 x 1.2288 MB = 137.6 MB of unaries > 126 MB L2
HID, LAYERS, CH = 130, 2, 2
MAC_FWD = CH * HID + LAYERS * (HID * HID + CH * HID) + HID + CH        # 34 712
FLOP_PER_PX_STEP = 6 * MAC_FWD                                          # 208 272 (SURVEY 8d)
GEMM_FLOP_PER_PX_LAUNCH = 2 * HID * (HID + CH + 1)                      # one hidden-layer contraction launch
WORKLOAD = "convexity ICNN prior fit per frame, synthetic FBMS-shaped 640x480 frames (BASELINE configs[1])"


def synth_unaries(seed: int, t: float = 0.0):
    """Soft UNet-like unaries in (0,1): blob on a Lissajous path with breathing axes (SURVEY 8d, C2)."""
    from awesome_b200 import synth
    return synth.c2_unaries(H, W, seed=seed, t=t)


def workload_config(G: int, precision: str) -> dict:
    """The ``config`` object of the JSON line -- ONE definition for both arms (``--impl ours`` and ``--impl reference``
    describe the same workload; what differs between them is reported outside ``config``)."""
    n_groups = (POOL_FRAMES + G - 1) // G
    return {"workload": WORKLOAD, "prior": f"ConvexNextNet(h={HID},L={LAYERS},C={CH})",
            "loss": "MSE(sigmoid(y), unaries)", "optimizer": "Adam lr=1e-3 + enforce_convexity",
            "frame": f"{W}x{H}", "pixels_per_frame": N_PIX, "frames_per_step_per_gpu": G,
            "pixels_per_step_per_gpu": G * N_PIX, "precision": precision,
            "grouping": f"{G} independent frames of the rank's share of the sequence per fused launch "
                        "(one prior, optimizer state and loss per frame)",
            "l2": f"each step reads its unaries from a rotating pool of {n_groups * G} distinct frames "
                  f"({n_groups * G * N_PIX * 4 / 1e6:.0f} MB > 126 MB L2); no explicit flush"}


_JSON_OUT = None


def emit(line: dict) -> None:
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    QUERY = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            atexit.register(self._kill)          # no sampler outlives the benchmark, also when it fails before stop()
        except Exception:
            self.proc = None

    def _kill(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.kill()
            self.proc.wait()

    @staticmethod
    def _epoch(ts: str) -> float:
        import datetime
        return datetime.datetime.strptime(ts.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()

    def stop(self, t0: float = None, t1: float = None):
        """Summary of the samples taken between wall-clock t0 and t1 (the timed regions); nvidia-smi needs a few
        hundred ms to deliver its first sample on an 8-GPU box, so it is started well before them."""
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    if t0 is not None and not (t0 - 0.02 <= self._epoch(f[0]) <= t1 + 0.02):
                        continue
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                    try:
                        pw.append(float(f[3]))
                    except ValueError:
                        pass
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm),
                       power_w=statistics.median(pw) if pw else None)
        return out


REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def _reference_fit_step():
    """One fit step of the BASELINE configs[1] workload with the UNMODIFIED reference package installed in
    ``baseline/_ref`` (``baseline/install_reference.py``): ``awesome.model.convex_net.ConvexNextNet``,
    ``UnariesWeightedLoss(SE("mean"))``, ``torch.optim.Adam`` and ``enforce_convexity`` exactly as the reference's per-frame
    loop runs them (``awesome/model/path_connected_net.py:939-953``).  Returns (step(rows) -> loss, kind)."""
    import torch
    if not os.path.isdir(os.path.join(REF_DIR, "awesome")) and os.path.isdir("/root/reference/awesome"):
        import subprocess as sp                                     # build container: install it now
        sp.run([sys.executable, os.path.join(ROOT, "baseline", "install_reference.py")], stdout=sp.DEVNULL, stderr=sp.DEVNULL)
    if os.path.isdir(os.path.join(REF_DIR, "awesome")):
        from oracle import ref_shim                                 # stubs for the non-numeric packages missing offline
        ref_shim.REFERENCE_ROOT = REF_DIR
        ref_shim.install()
        from awesome.dataset.transformator import Transformator
        from awesome.measures.se import SE
        from awesome.measures.unaries_weighted_loss import UnariesWeightedLoss
        from awesome.model.convex_net import ConvexNextNet
        from awesome.run.runner import seed_all
        seed_all(42)
        model = ConvexNextNet(n_hidden=HID, in_features=CH, n_hidden_layers=LAYERS)
        model.train()
        x_full = Transformator.get_positional_matrices(W, H)[None]
        un_full = synth_unaries(42)[None, None]
        crit = UnariesWeightedLoss(SE("mean"))
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)

        def step(n_rows: int) -> float:
            h = n_rows // W                                         # a horizontal band of the frame (h == H: the full frame)
            x, un = x_full[:, :, :h], un_full[:, :, :h]
            opt.zero_grad()
            loss = crit(torch.sigmoid(model(x)), un)
            loss.backward()
            opt.step()
            model.enforce_convexity()
            return float(loss.detach())
        return step, "reference"
    # no installed reference: the oracle port (same ATen op sequence)
    from oracle import prior_oracle as O
    torch.manual_seed(42)
    lin = torch.nn.Linear
    p = {}
    l = lin(CH, HID); p["input.weight"], p["input.bias"] = l.weight.detach(), l.bias.detach()
    for i in range(LAYERS):
        l = lin(HID, HID); p[f"skip.{i}.ln.weight"], p[f"skip.{i}.ln.bias"] = l.weight.detach(), l.bias.detach()
        p[f"skip.{i}.skp.weight"] = lin(CH, HID, bias=False).weight.detach()
    l = lin(HID, 1); p["out.ln.weight"], p["out.ln.bias"] = l.weight.detach(), l.bias.detach()
    p["out.skp.weight"] = lin(CH, 1, bias=False).weight.detach()
    p = O.clone_params(p)
    rows_full = O.pixelize(O.grid_linspace(H, W)[None])
    un_full = synth_unaries(42).reshape(-1)

    def step(n_rows: int) -> float:
        O.fit_icnn(p, rows_full[:n_rows], un_full[:n_rows], steps=1, optimizer="adam", lr=1e-3)
        return 0.0
    return step, "port"


def cpu_reference_throughput(steps: int, warmup: int, budget_s: float = 240.0):
    """The reference's own CPU implementation of one fit step on ALL host cores (torchrun pins OMP_NUM_THREADS=1: reset).
    Each step fits the FULL 640x480 frame; only when warmup+steps full-frame steps would not end within ``budget_s`` is the
    sample cut to a horizontal band of the frame (and said so in ``sample``)."""
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    step, kind = _reference_fit_step()
    t0 = time.perf_counter()
    step(N_PIX)                                                     # calibration = first warm-up step, full frame
    t_full = time.perf_counter() - t0
    frac = 1.0
    while frac > 1 / 64 and t_full * frac * (steps + warmup) > budget_s:
        frac /= 2
    n = int(H * frac) * W
    for _ in range(max(0, warmup - 1)):
        step(n)
    t0 = time.perf_counter()
    for _ in range(steps):
        step(n)
    dt = time.perf_counter() - t0
    cores = torch.get_num_threads()
    what = "the full 640x480 frame" if frac == 1.0 else f"the top {n} of {N_PIX} pixel rows of the frame ({frac:g} frame)"
    impl = ("reference package (baseline/_ref): awesome.model.convex_net.ConvexNextNet + UnariesWeightedLoss(SE) + "
            "torch.optim.Adam + enforce_convexity" if kind == "reference" else "oracle port of the reference's loop")
    sample = f"{steps} fit steps on {what}, {impl}, torch CPU fp32, {cores} threads (os.cpu_count()={os.cpu_count()})"
    return n * steps / dt, dt / steps * 1e3, cores, sample, kind


def _time_fitter(fitter, steps: int) -> float:
    import torch
    fitter.run(max(5, fitter.K), record=False)        # includes the CUDA-graph capture: keep it out of the timed region
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fitter.run(steps, record=False)
    e1.record()
    torch.cuda.synchronize()
    fitter.raise_if_nonfinite()
    return e0.elapsed_time(e1) / steps


def sustained_leg(fitter, pool, dev, gpu_index: int, G: int, seconds: float = 10.0):
    """The headline loop, unchanged, for >= ``seconds`` of device time: ms per step with the clocks settled, median SM
    clock, power and clock-event reasons sampled over the whole region (nvidia-smi, 20 ms period)."""
    import torch
    fitter.set_target_pool(pool)
    fitter.run(200, record=False)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fitter.run(1000, record=False); e1.record()
    torch.cuda.synchronize(dev)
    n_steps = max(2000, int(seconds * 1e3 / (e0.elapsed_time(e1) / 1000.0)))
    sampler = ClockSampler(gpu_index)
    sampler.query_power = True
    sampler.start()
    time.sleep(0.3)
    t0 = time.time()
    e0.record()
    done = 0
    while done < n_steps:
        k = min(2000, n_steps - done)
        fitter.run(k, record=False)
        done += k
    e1.record()
    torch.cuda.synchronize(dev)
    t1 = time.time()
    clk = sampler.stop(t0, t1)
    ms = e0.elapsed_time(e1)
    fitter.raise_if_nonfinite()
    return {"seconds": ms * 1e-3, "steps": n_steps, "ms_per_step": ms / n_steps,
            "pixel_samples_per_s": G * N_PIX * n_steps / (ms * 1e-3), "sm_mhz_median": clk["sm_mhz"],
            "sm_max_mhz": clk["sm_max_mhz"], "power_w_median": clk.get("power_w"), "reasons": clk["reasons"],
            "clock_samples": clk["samples"]}


def frames_per_s_leg(A, dev, rank: int, world: int, G: int, precision: str, barrier, n_frames: int = 60, n_segments: int = 8):
    """The second half of BASELINE's metric, MEASURED: wall-clock frames/s of fitting the whole synthetic 60-frame 640x480
    sequence (configs[1]) with ``awesome_b200.fit_sequence_sharded`` -- 8 fixed segments over the ranks, inside a segment
    the reference's chain (4000 steps cold for its first frame, 400 warm for every following one; G = 1 frame per launch),
    native step loops, no-foreground skip, IoU check + retry, every frame's unaries copied from pinned host memory, masks /
    states / IoUs gathered on every rank at the end.  Time = barrier to barrier, max over ranks.  ``digest`` hashes every
    fitted state: it is the same for any number of GPUs."""
    import hashlib
    import torch
    import torch.distributed as dist
    from awesome_b200 import synth
    segs = A.plan_segments(n_frames, n_segments)
    mine = [i for si in A.segments_of_rank(len(segs), rank, world) for i in segs[si]]
    host = {i: synth.c2_unaries(H, W, seed=42 + i, t=0.1 * i).pin_memory() for i in mine}     # outside the timed region
    sched = A.FitSchedule(num_epochs=4000, reuse_state_epochs=400, optimizer="adam", plateau=False, lr=1e-3,
                          steps_per_graph=50, proper_prior_fit_retrys=1)
    grid = A.GridSpecHost("linspace", 1, H, W)
    args = dict(n_hidden=HID, in_features=CH, n_hidden_layers=LAYERS, precision=precision)
    # warm-up: library / graph-capture costs of a first call are not part of a sequence fit's steady state
    A.fit_sequence_sharded(A.ConvexNextNet, args, grid, lambda i: host[mine[0]], G, A.FitSchedule(
        num_epochs=100, reuse_state_epochs=50, optimizer="adam", plateau=False, lr=1e-3, steps_per_graph=50), n_segments=1,
        group=G, rank=0, world=1, device=dev, gather=False, keep_states=False)
    barrier()
    t0 = time.perf_counter()
    res = A.fit_sequence_sharded(A.ConvexNextNet, args, grid, lambda i: host[i], n_frames, sched, n_segments=n_segments,
                                 group=G, rank=rank, world=world, device=dev, gather=True)
    barrier()
    wall = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([wall], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall = float(t[0])
    h = hashlib.sha256()
    for i in sorted(res):
        if res[i]["state"] is not None:
            h.update(res[i]["state"].numpy().tobytes())
    fitted = [r for r in res.values() if not r["skipped"]]
    return {"value": n_frames / wall, "unit": "frames/s", "measured": True, "frames": n_frames, "wall_s": wall,
            "segments": n_segments, "frames_per_launch": G, "schedule": "4000 steps cold (first frame of a segment) / 400 warm (every following frame), Adam 1e-3",
            "steps_total_per_rank_max": max(sum(4000 if k == 0 else 400 for k in range((len(sg) + G - 1) // G))
                                            for sg in segs) * len(A.segments_of_rank(len(segs), 0, world)),
            "mean_iou": sum(r["iou"] for r in fitted) / max(1, len(fitted)), "min_iou": min(r["iou"] for r in fitted),
            "proper_fits": sum(1 for r in fitted if r["proper_fit"]), "retries": sum(r["retries"] for r in fitted),
            "skipped": sum(1 for r in res.values() if r["skipped"]), "digest": h.hexdigest()[:16],
            "includes": "H2D of every frame's unaries, skip check, fit, IoU check / retry, mask packing, D2H + gather of results"}


def joint_leg(A, dev, rank: int, world: int, barrier, precision: str, steps: int = 10):
    """BASELINE configs[4] on hardware: the data-parallel joint UNet + (x, y, t) prior step of the spatio-temporal configs
    (``awesome/agent/torch_agent.py:428-551``) -- a stock U-Net of the reference's size (13 395 905 parameters), the
    RealNVP(18 flows, m = 32) o ICNN(L = 2) prior on the tensor path, ``FBMSJointLoss``, Adam 1e-4, 2 frames of 640x480 per
    GPU and step, ONE exchange step: the all-reduce of the 53.8 MB flat gradient bucket between ``backward`` and
    ``optimizer.step`` (``:489-492``).  Timed three ways (CUDA events, max over ranks): bucketed all-reduce overlapped with
    the backward pass (the product), one all-reduce after backward, no exchange; plus the collective alone.  Replicas are
    checked bit-identical after the overlapped run."""
    import torch
    import torch.distributed as dist
    from awesome_b200 import measures as M
    from awesome_b200 import synth
    B, T = 2, 200
    torch.manual_seed(42)
    seg = synth.stock_unet(4).to(dev)
    pri = A.real_nvp_path_connected_net(channels=3, hidden_units=32, flow_n_flows=18, flow_output_fn="tanh", norm="minmax",
                                        convex_net_hidden_units=130, convex_net_hidden_layers=2, precision=precision).to(dev)
    g = torch.Generator().manual_seed(1000 + rank)
    img = torch.randn(B, 4, H, W, generator=g).to(dev)                       # random RGB + edge channel
    grid = A.GridSpecHost("linspace", B, H, W, t0=rank * B / (T - 1), t_step=1.0 / (T - 1)).materialize(3, dev)
    lab = torch.full((B, 1, H, W), 2.0)                                      # sparse weak labels: 0 fg, 1 bg, 2 none
    lab[torch.rand(B, 1, H, W, generator=g) < 0.05] = 0.0
    lab[torch.rand(B, 1, H, W, generator=g) < 0.10] = 1.0
    lab = lab.to(dev)
    with torch.no_grad():
        pri(grid)                                                            # ActNorm data-dependent init
    init = ({k: v.clone() for k, v in seg.state_dict().items()}, {k: v.clone() for k, v in pri.state_dict().items()})
    out = {"workload": "joint UNet + spatio-temporal prior step (BASELINE configs[4])", "frames_per_gpu_per_step": B,
           "frames_per_step": world * B, "unet_params": sum(p.numel() for p in seg.parameters()),
           "prior_params": sum(p.numel() for p in pri.parameters()), "n_gpus": world}

    def run(mode):
        seg.load_state_dict(init[0]); pri.load_state_dict(init[1])
        tr = A.JointTrainer(seg, pri, M.FBMSJointLoss(), optimizer_args=dict(lr=1e-4), n_buckets=4, comm=mode)
        tr.broadcast_parameters(0)
        for _ in range(3):
            tr.step(img, grid, lab)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            loss = tr.step(img, grid, lab)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / steps
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        tr.bucket.remove_hooks()
        return tr, ms, float(loss)

    # default mode of JointTrainer: ONE all-reduce of the flat bucket between backward and optimizer.step (measured faster than
    # the bucketed overlap on NVSwitch: the collective takes ~0.5 % of the step, the hooks and the concurrent NCCL kernels cost more)
    tr, ms_after, loss = run("after")
    out.update(bucket_bytes=tr.bucket.nbytes, ms_per_step=ms_after, frames_per_s=world * B / ms_after * 1e3, final_loss=loss,
               exchange="one NCCL all-reduce (AVG) of the flat fp32 gradient bucket after backward")
    if world > 1:
        flat = torch.cat([p.detach().reshape(-1) for p in list(seg.parameters()) + list(pri.parameters())])
        ref = flat.clone()
        dist.broadcast(ref, src=0)
        same = torch.tensor([float(torch.equal(ref, flat))], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        out["replicas_bit_identical"] = bool(same.item() > 0)
        buf = tr.bucket.flat
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            dist.all_reduce(buf, op=dist.ReduceOp.AVG)
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) / 10], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ar = float(t[0])
        del tr
        tr, ms_overlap, _ = run("overlap")
        nb = tr.bucket.n_buckets
        del tr
        _, ms_off, _ = run("off")
        hidden = (ms_after - ms_overlap) / ar if ar > 0 else 0.0
        out.update(ms_per_step_bucketed_overlap=ms_overlap, n_buckets_overlap=nb, ms_per_step_no_exchange=ms_off,
                   allreduce_ms_alone=ar, allreduce_share_of_step=ar / ms_after,
                   allreduce_busbw_GBps=2 * (world - 1) / world * buf.numel() * 4 / (ar * 1e-3) / 1e9,
                   exposed_comm_ms=ms_after - ms_off, overlap_gain_ms=ms_after - ms_overlap,
                   overlapped_fraction=max(0.0, min(1.0, hidden)))
    del seg, pri
    torch.cuda.empty_cache()
    return out


def secondary_workloads(A, dev, unaries640):
    """Short device-timed runs of the other BASELINE configs (ms per fused fit step, pixel-samples/s):
    configs[0] 256x256 ICNN(L=1) notebook fit, configs[2] RealNVP path-connectedness fit, configs[3] 8 objects per
    frame in one grouped launch.  Same rules as the headline (tensor path, inputs resident, CUDA events)."""
    import torch
    out = {}
    torch.manual_seed(0)
    # configs[0]: how_to/convexity -- ConvexNextNet(L=1), index grid, fg/bg-weighted SE, Adam 2e-3
    m = A.ConvexNextNet(n_hidden_layers=1, precision="f16").to(dev)
    hard = (torch.nn.functional.interpolate(unaries640[None, None], size=(256, 256))[0, 0] > 0.5).float()
    f = m.make_fitter(A.GridSpecHost("index", 1, 256, 256), hard, A.LossConfig("fgbg_se", fg_weight=0.4),
                      A.OptimConfig("adam", lr=2e-3), steps_per_graph=50)
    ms = _time_fitter(f, 200)
    out["c0_convexity_256x256_L1"] = {"ms_per_step": ms, "pixel_samples_per_s": 256 * 256 / ms * 1e3}
    # configs[1] one frame per launch (the headline groups --frames-per-step frames): 2400 tiles over 148 SMs
    grid640 = A.GridSpecHost("linspace", 1, H, W)
    m1 = A.ConvexNextNet(n_hidden=HID, in_features=CH, n_hidden_layers=LAYERS, precision="f16").to(dev)
    f = m1.make_fitter(grid640, unaries640, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    ms = _time_fitter(f, 200)
    out["c1_convexity_single_frame_640x480"] = {"ms_per_step": ms, "pixel_samples_per_s": N_PIX / ms * 1e3}
    del f, m1
    # configs[2]: path-connectedness -- RealNVP(12 flows, m=32, tanh) o ICNN(L=2), Adamax + plateau, flow wd 1e-5
    pc = A.real_nvp_path_connected_net(channels=2, hidden_units=32, flow_n_flows=12, flow_output_fn="tanh", norm="minmax",
                                       convex_net_hidden_units=130, convex_net_hidden_layers=2, precision="f16").to(dev)
    grid = A.GridSpecHost("linspace", 1, H, W)
    opt = A.OptimConfig("adamax", lr=1e-3, weight_decay=[1e-5, 0.0, 0.0, 0.0], plateau=True)
    f = pc.make_fitter(grid, unaries640, A.LossConfig("mse"), opt, steps_per_graph=25)
    ms = _time_fitter(f, 50)
    out["c2_path_connected_640x480"] = {"ms_per_step": ms, "pixel_samples_per_s": N_PIX / ms * 1e3}
    del f, pc
    # configs[3]: 8 objects per frame, one grouped launch per kernel
    multi = A.NumberBasedMultiPriorModule(
        prior_type=A.real_nvp_path_connected_net,
        prior_args=dict(channels=2, hidden_units=32, flow_n_flows=12, flow_output_fn="tanh", norm="minmax",
                        convex_net_hidden_units=130, convex_net_hidden_layers=2, precision="f16"), min_priors=8).to(dev)
    tg = torch.stack([torch.roll(unaries640, shifts=(17 * k, 29 * k), dims=(0, 1)) for k in range(8)])
    f = multi.make_fitter(grid, tg, A.LossConfig("mse"), opt, steps_per_graph=10)
    ms = _time_fitter(f, 20)
    out["c3_multi_object_8x640x480"] = {"ms_per_step": ms, "pixel_samples_per_s": 8 * N_PIX / ms * 1e3}
    del f, multi
    # configs[4], prior side only: the (x, y, t) RealNVP(18 flows) o ICNN prior of the spatio-temporal configs fitted on a batch of
    # 2 frames (the prefit / pretrain step of path_connected_net.py:511-728 with cached unaries; the joint step is `joint_unet_prior`)
    st = A.real_nvp_path_connected_net(channels=3, hidden_units=32, flow_n_flows=18, flow_output_fn="tanh", norm="minmax",
                                       convex_net_hidden_units=130, convex_net_hidden_layers=2, precision="f16").to(dev)
    grid3 = A.GridSpecHost("linspace", 2, H, W, t0=0.0, t_step=1.0 / 199)
    tg3 = torch.stack([unaries640, torch.roll(unaries640, shifts=(5, 9), dims=(0, 1))])
    f = st.make_fitter(grid3, tg3, A.LossConfig("mse"), opt, steps_per_graph=10)
    ms = _time_fitter(f, 30)
    out["c4_spatio_temporal_prior_2x640x480"] = {"ms_per_step": ms, "pixel_samples_per_s": 2 * N_PIX / ms * 1e3}
    del f, st
    torch.cuda.empty_cache()
    out["n4_image_preprocess_640x480"] = image_preprocess_throughput(A, dev)
    return out


def image_preprocess_throughput(A, dev, reps: int = 80):
    """SURVEY 8f N4: the dataset layer's per-frame OpenCV preprocessing on the device (awb_image.cu), HBM bound.
    Frames rotate through a pool larger than L2; achieved GB/s = algorithmic bytes (12 B read + 12 / 4 B written per
    pixel) / CUDA-event time, against the measured copy bandwidth; OpenCV on the host timed beside it when importable."""
    import torch
    pk, pk_src = peaks()
    pool = torch.rand((40, 3, H, W), device=dev)                 # 147 MB > 126 MB L2
    res = {}
    for name, fn, nbytes in (("process_image_blur5", A.image.process_image, 24 * N_PIX),
                             ("create_edge_map", A.image.create_edge_map, 16 * N_PIX)):
        fn(pool)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(reps // 8):
            fn(pool)                                              # one launch over the 40-frame batch
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) / (reps // 8) / pool.shape[0] * 1e3
        res[name] = {"us_per_frame": us, "GBps": nbytes / us / 1e3, "frac_of_hbm_peak": nbytes / us / 1e3 / pk["hbm_gbs"],
                     "peak_source": pk_src}
    try:
        import cv2
        import numpy as np
        img = pool[0].cpu().numpy()

        def cpu_proc():
            im = (img.transpose(1, 2, 0) * 255).astype(np.uint8)
            return cv2.GaussianBlur(im, (5, 5), 0).astype(np.float32).transpose(2, 0, 1) / np.float32(255)

        def cpu_edge():
            im = (img.transpose(1, 2, 0) * 255).astype(np.uint8)
            gray = cv2.cvtColor(cv2.GaussianBlur(im, (3, 3), 0), cv2.COLOR_RGB2GRAY)
            gx, gy = cv2.Sobel(gray, cv2.CV_16S, 1, 0, ksize=3), cv2.Sobel(gray, cv2.CV_16S, 0, 1, ksize=3)
            g = cv2.addWeighted(cv2.convertScaleAbs(gx), 0.5, cv2.convertScaleAbs(gy), 0.5, 0) / 255
            return cv2.GaussianBlur(g, (5, 5), 0).astype(np.float32)
        for name, fn in (("process_image_blur5", cpu_proc), ("create_edge_map", cpu_edge)):
            fn()
            t0 = time.perf_counter()
            for _ in range(20):
                fn()
            res[name]["opencv_host_us_per_frame"] = (time.perf_counter() - t0) / 20 * 1e6
        res["opencv"] = cv2.__version__
    except Exception as e:            # a baseline leg must never take the bench line down
        res["opencv"] = f"unavailable: {e!r}"[:120]
    del pool
    torch.cuda.empty_cache()
    return res


def eager_gpu_throughput(dev, steps: int = 10):
    """The same oracle port (the reference's eager ATen op sequence: per-op kernels, autograd, per-tensor Adam, one
    clamp per tensor, a host sync on the loss every step) on the SAME B200 -- the GPU-vs-GPU comparison SURVEY 8d
    asks for beside the CPU arm.  Reported as a baseline only."""
    import torch
    from oracle import prior_oracle as O
    torch.manual_seed(42)
    lin = torch.nn.Linear
    p = {}
    l = lin(CH, HID); p["input.weight"], p["input.bias"] = l.weight.detach(), l.bias.detach()
    for i in range(LAYERS):
        l = lin(HID, HID); p[f"skip.{i}.ln.weight"], p[f"skip.{i}.ln.bias"] = l.weight.detach(), l.bias.detach()
        p[f"skip.{i}.skp.weight"] = lin(CH, HID, bias=False).weight.detach()
    l = lin(HID, 1); p["out.ln.weight"], p["out.ln.bias"] = l.weight.detach(), l.bias.detach()
    p["out.skp.weight"] = lin(CH, 1, bias=False).weight.detach()
    p = {k: v.to(dev) for k, v in O.clone_params(p).items()}
    rows = O.pixelize(O.grid_linspace(H, W)[None]).to(dev)
    un = synth_unaries(42).reshape(-1).to(dev)
    O.fit_icnn(p, rows, un, steps=3, optimizer="adam", lr=1e-3)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    O.fit_icnn(p, rows, un, steps=steps, optimizer="adam", lr=1e-3)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    return {"value": N_PIX * steps / dt, "unit": "pixel-samples/s", "kind": "port", "device": torch.cuda.get_device_name(dev),
            "ms_per_step": dt / steps * 1e3,
            "sample": f"{steps} fit steps on the full 640x480 frame, eager PyTorch fp32 ops of the reference's loop on cuda"}


def dump_outputs(out_dir: str, fitter, G: int) -> None:
    """What a caller of the timed path receives after its last step: the G fitted priors and that step's loss per frame
    (kept by the optimizer state on the device).  Called right after the timed region, before any other leg fits."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    params = fitter.params.detach().reshape(G, -1).cpu().numpy().astype(np.float32)
    loss = np.array([fitter.scalars(o).last_loss for o in range(G)], dtype=np.float64)
    np.save(os.path.join(out_dir, "params.npy"), params)
    np.save(os.path.join(out_dir, "loss.npy"), loss)


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    thr, ms, cores, sample, kind = cpu_reference_throughput(args.steps, max(1, args.warmup), budget_s=240.0)
    G = max(1, args.frames_per_step)
    line = {
        "impl": "reference", "metric": "prior-fit pixel-samples/sec (fwd+bwd+step)", "value": thr,
        "unit": "pixel-samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": max(1, args.warmup),
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(G, args.precision),
        "cpu_baseline": {"value": thr, "unit": "pixel-samples/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": thr, "unit": "pixel-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "one CPU process on rank 0 (the reference fits one frame at a time); value does not grow with --gpus",
    }
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("AWB_BENCH_PRECISION", "f16"), choices=["fp32", "f16"])
    ap.add_argument("--frames-per-step", type=int, default=4,
                    help="independent frames of the rank's share of the sequence fitted together per fused launch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the short runs of BASELINE configs 0, 2, 3")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 10 s leg behind roofline.sustained")
    ap.add_argument("--no-joint", action="store_true", help="skip the joint UNet + prior step leg (BASELINE configs[4])")
    ap.add_argument("--no-frames", action="store_true", help="skip the measured frames/s leg (60-frame sharded sequence fit)")
    ap.add_argument("--sustained-seconds", type=float, default=10.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the fitted parameters and the per-frame loss of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries exactly ONE line, the JSON: everything any library prints to file descriptor 1 (NCCL's version
    # banner, warnings of child processes) is sent to stderr, and the JSON line is written to the saved descriptor.
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import __graft_entry__ as entry
    entry.build()
    import awesome_b200 as A
    from awesome_b200 import _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left to the caller (stdout carries only the JSON line either way: fd 1 is redirected above)
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    sampler = ClockSampler(local_rank)
    sampler.start()
    warmup = max(3, args.warmup)

    # ---- the fit: frames are independent units (rank r owns its share of the 60-frame sequence); a rank fits
    # G = --frames-per-step of its frames together, one ConvexNextNet prior per frame, one fused launch per kernel.
    # With G frames per launch the next frame's CTAs fill the SMs that the 16-tile CTAs of the previous one leave idle
    # (2400 tiles of one frame over 148 SMs = 16.2 per SM with 17 on the critical path) and the per-launch fixed cost
    # is shared; G = 4 keeps the 4 x 23 MB of weight-gradient partials inside the 126 MB L2.
    G = max(1, args.frames_per_step)
    torch.manual_seed(42 + rank)
    model = A.NumberBasedMultiPriorModule(
        prior_type=A.ConvexNextNet,
        prior_args=dict(n_hidden=HID, in_features=CH, n_hidden_layers=LAYERS, precision=args.precision), min_priors=G).to(dev)
    unaries_host = torch.stack([synth_unaries(42 + rank * G + k, t=0.1 * (rank * G + k)) for k in range(G)]).pin_memory()
    unaries = unaries_host.to(dev, non_blocking=True)                       # [G,H,W]
    grid = A.GridSpecHost("linspace", 1, H, W)
    fitter = model.make_fitter(grid, unaries, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    # The per-step input (G frames of unaries, 1.2 MB each) would sit in the 126 MB L2: rotate through a pool of
    # >= POOL_FRAMES distinct frames (> L2) so that every timed step reads its unaries from HBM.
    n_groups = (POOL_FRAMES + G - 1) // G
    base = unaries.reshape(1, G, -1)
    shifts = torch.arange(n_groups, device=dev).view(-1, 1, 1)
    idx = (torch.arange(N_PIX, device=dev).view(1, 1, -1) + 37 * shifts) % N_PIX     # cheap distinct frames: rolled copies
    pool = torch.gather(base.expand(n_groups, G, N_PIX), 2, idx.expand(n_groups, G, N_PIX)).contiguous()
    pool[0].copy_(base[0])
    fitter.set_target_pool(pool)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-timed K steps, inputs resident in HBM
    fitter.run(warmup, record=False)
    barrier()
    launches0 = lib.awb_launch_count()
    t_load0 = time.time()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    fitter.run(args.steps, record=False)
    ev1.record()
    barrier()
    launches = lib.awb_launch_count() - launches0
    ms_total = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fitter, G)

    # ---- end to end through the public API: the step's unaries arrive from pinned host memory, loss read back
    fitter.set_target_pool(None)
    e2e_warm = 3
    host_pool = [unaries_host.reshape(G, -1)] + [torch.roll(unaries_host, 13 * k, 2).reshape(G, -1).pin_memory() for k in (1, 2, 3)]
    fitter.run_host_frames(host_pool, e2e_warm)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    # one C-ABI call with HOST buffers: every step copies its G frames (4*N_PIX bytes each) host->device (copy stream, double
    # buffered) and stores its loss into pinned host memory; both inside the timed region
    loss_host = fitter.run_host_frames(host_pool, args.steps)
    e1.record()
    barrier()
    t_e2e = e0.elapsed_time(e1)
    clocks = sampler.stop(t_load0, time.time())      # samples under load: the device-timed and the end-to-end region
    if not bool(torch.isfinite(loss_host).all()):
        raise SystemExit("e2e: non-finite loss read back from the host-frame fit")
    fitter.raise_if_nonfinite()

    # ---- frames/s over the sharded 60-frame sequence, measured (every rank takes part)
    frames_leg = None
    if not args.no_frames:
        fitter.set_target_pool(None)
        frames_leg = frames_per_s_leg(A, dev, rank, world, 1, args.precision, barrier)      # the warm-start chain: one frame per launch

    # ---- configs[4]: joint UNet + prior step with its gradient all-reduce (every rank takes part)
    joint = None
    if not args.no_joint:
        try:
            joint = joint_leg(A, dev, rank, world, barrier, args.precision)
        except Exception as e:           # a secondary leg must never take the bench line down
            joint = {"unavailable": repr(e)[:300]}

    # ---- the same loop for >= 10 s: earns (or not) the sustained-clock reading of the roofline (N = 1 only)
    sustained = None
    if rank == 0 and world == 1 and not args.no_sustained:
        sustained = sustained_leg(fitter, pool, dev, local_rank, G, seconds=args.sustained_seconds)
        fitter.set_target_pool(None)

    # ---- the other BASELINE configs, briefly (N = 1 only; device-timed, not part of `value`)
    secondary = None
    if rank == 0 and world == 1 and not args.no_secondary:
        secondary = secondary_workloads(A, dev, unaries[0])

    # ---- per-kernel timing of the step, live with CUDA events on the launch stream (profile mode brackets every launch
    # with events, which removes the programmatic-dependent-launch overlap: used for SHARES, not for the roofline)
    fitter.set_target_pool(pool)
    n_cls = lib.awb_profile_classes()
    lib.awb_profile_enable(1)
    fitter.run(6, record=False)
    tot = (C.c_double * n_cls)()
    cnt = (C.c_int32 * n_cls)()
    _lib.check(lib.awb_profile_read(tot, cnt))
    lib.awb_profile_enable(0)
    names = [lib.awb_profile_class_name(i).decode() for i in range(n_cls)]
    per_class = {names[i]: {"ms_per_launch": tot[i] / cnt[i], "launches_per_step": cnt[i] / 6.0,
                            "ms_per_step": tot[i] / 6.0} for i in range(n_cls) if cnt[i] > 0}
    step_ms_prof = sum(v["ms_per_step"] for v in per_class.values())
    pk, pk_src = peaks()

    if world > 1:
        t = torch.tensor([ms_total, t_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, t_e2e = float(t[0]), float(t[1])
        ln = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(ln, op=dist.ReduceOp.SUM)
        launches = int(ln[0])

    if rank == 0:
        units = world * G * N_PIX * args.steps
        value = units / (ms_total * 1e-3)
        e2e_val = units / (t_e2e * 1e-3)
        ms_step = ms_total / args.steps
        burst, sust = pk["bf16_tflops"], pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
        if args.precision == "f16" and "tc_fused" in per_class:
            dom, dom_flop = "tc_fused", FLOP_PER_PX_STEP * N_PIX * G
            # The fused kernel IS the step (one launch per step; the optimizer kernel overlaps its tail through programmatic
            # dependent launch), and a kernel cannot take longer than the step that contains it: the launch duration used
            # for `achieved` is the device-timed step.  The timed region is short (K steps of ~0.36 ms), so the applicable
            # peak is the BURST figure; `sustained` below repeats the measurement over >= 10 s against the sustained one.
            ms_launch = ms_step
            note = ("fused fit kernel = all layer contractions of one step; achieved = algorithmic FLOP per step / device-timed "
                    "ms_per_step; peak = measured cuBLAS bf16 burst (short timed region)")
        else:
            gemm = [k for k in ("gemm_fwd", "gemm_wgrad", "gemm_dgrad") if k in per_class]
            dom = max(gemm, key=lambda k: per_class[k]["ms_per_step"])
            dom_flop = GEMM_FLOP_PER_PX_LAUNCH * N_PIX * G
            ms_launch = per_class[dom]["ms_per_launch"]
            note = ("fp32 CUDA-core contraction (exact-parity path); reported against the cuBLAS bf16 tensor peak the north "
                    "star names")
        traffic = None
        tp = os.path.join(ROOT, "profiles", "r2_headline_f16_tc_traffic.json")     # from the committed ncu --set full capture
        if dom == "tc_fused" and os.path.exists(tp):
            for name, rec in json.load(open(tp)).get("kernels", {}).items():
                if "k_icnn_fit_tc" in name:
                    traffic = rec.get("dram_bytes_per_launch")
        ach = dom_flop / (ms_launch * 1e-3) / 1e12
        roofline = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": burst, "unit": "TFLOP/s",
                    "frac": ach / burst, "traffic": traffic, "traffic_unit": "bytes/launch (ncu dram read+write)",
                    "peaks": {"bf16_tflops_burst": burst, "bf16_tflops_sustained": sust, "source": pk_src},
                    "frac_of_burst": ach / burst, "frac_of_sustained": ach / sust,
                    "algorithmic_flop_per_launch": dom_flop, "ms_per_launch": ms_launch,
                    "ms_per_launch_event_bracketed": per_class[dom]["ms_per_launch"],
                    "share_of_step_event_bracketed": per_class[dom]["ms_per_step"] / step_ms_prof,
                    "note": note, "per_class_ms_per_step": {k: round(v["ms_per_step"], 4) for k, v in per_class.items()}}
        if sustained is not None:
            roofline["sustained"] = {
                **sustained, "achieved": FLOP_PER_PX_STEP * N_PIX * G / (sustained["ms_per_step"] * 1e-3) / 1e12,
                "peak": sust, "frac": FLOP_PER_PX_STEP * N_PIX * G / (sustained["ms_per_step"] * 1e-3) / 1e12 / sust}
        # HBM-bound kernels of the step (north star item 4): the optimizer pass
        roofline_hbm = None
        if "reduce_opt" in per_class:
            P_prior = int(sum(p.numel() for p in model.priors[0].parameters()))
            n_part = min(148 // G if G <= 148 else 1, (N_PIX + 127) // 128) if args.precision == "f16" else min(148, (N_PIX + 255) // 256)
            G_aug = 4 * HID + LAYERS * HID * 136 + 136
            alg = 28 * P_prior * G + (2 * P_prior * G if args.precision == "f16" else 0)      # p, m, v read + written, g read (+ fp16 image)
            moved = alg + 4 * n_part * G * G_aug                                                  # + the per-CTA gradient partials it reduces
            us = per_class["reduce_opt"]["ms_per_launch"] * 1e3
            roofline_hbm = {"kernel": "k_reduce_opt_aug (cross-CTA gradient reduction + Adam + clamp + fp16 image)",
                            "bound": "hbm", "unit": "GB/s", "peak": pk["hbm_gbs"], "us_per_launch": us,
                            "algorithmic_bytes_per_launch": alg, "achieved": alg / us / 1e3, "frac": alg / us / 1e3 / pk["hbm_gbs"],
                            "bytes_moved_per_launch": moved, "moved_GBps": moved / us / 1e3,
                            "moved_frac_of_peak": moved / us / 1e3 / pk["hbm_gbs"], "partials_per_object": n_part,
                            "share_of_step": per_class["reduce_opt"]["ms_per_step"] / step_ms_prof,
                            "note": "latency bound: 28 B/parameter of optimizer traffic (+ the L2-resident gradient partials); "
                                    "runs in the shadow of the next fit kernel's prologue (PDL), < 5 % of the step"}
        cpu, eager = None, None
        if not args.no_cpu_baseline:
            try:
                eager = eager_gpu_throughput(dev)
            except Exception as e:       # a baseline leg must never take the bench line down
                eager = {"unavailable": repr(e)[:200]}
            thr, ms_cpu, cores, sample, kind = cpu_reference_throughput(steps=8, warmup=1, budget_s=30.0)
            cpu = {"value": thr, "unit": "pixel-samples/s", "cores": cores, "kind": kind, "sample": sample,
                   "ms_per_step_sample": ms_cpu}
        line = {
            "metric": "prior-fit pixel-samples/sec (fwd+bwd+step)", "value": value, "unit": "pixel-samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else "f16 operands / f32 accumulate", "data": "synthetic",
            "config": workload_config(G, args.precision),
            "e2e": {"value": e2e_val, "unit": "pixel-samples/s", "h2d_bytes_per_step": 4 * N_PIX * G,
                    "d2h_bytes_per_step": 4 * G, "ms_per_step": t_e2e / args.steps},
            "gpu_launches": int(launches),
            "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"],
                       "samples": clocks["samples"]},
            "frames_per_s": frames_leg,
            "joint_unet_prior": joint,
            "roofline": roofline,
            "roofline_hbm": roofline_hbm,
            "cpu_baseline": cpu,
            "eager_gpu_baseline": eager,
            "secondary": secondary,
            "final_loss": float(loss_host[-1].mean()),
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
