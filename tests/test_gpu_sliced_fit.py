"""GPU tests of the pixel-sliced fit step (awb_prior_slice_grads / awb_prior_rows_opt_step, SlicedFitter,
fit_sequence(n_slices=...)): rows add up to the fused step, the optimizer is the fused step's, the result does not depend on
the number of ranks, error paths, and a real two-GPU NCCL run when the machine has two GPUs."""
import ctypes as C
import os
import socket

import pytest
import torch

import __graft_entry__ as entry

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


def blob(H, W, cx=0.5, cy=0.5, rx=0.27, ry=0.31, tau=0.08):
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    return torch.sigmoid((torch.sqrt(((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2) - 1) / tau)


def _model(A, kind, C_, precision, seed=0):
    torch.manual_seed(seed)
    if kind == "icnn":
        m = A.ConvexNextNet(in_features=C_, n_hidden_layers=2, precision=precision)
    else:
        m = A.real_nvp_path_connected_net(channels=C_, hidden_units=32, flow_n_flows=6, flow_output_fn="tanh",
                                          convex_net_hidden_layers=2, precision=precision)
    m = m.to(DEV)
    arena = m._ensure_flat()
    return m, m._prior_for(arena.device), arena


def _grid(A, mode, B, H, W, C_):
    if mode == "explicit":
        g = A.GridSpecHost("linspace", B, H, W, t0=0.1, t_step=0.2).materialize(C_, DEV)
        g = (g * 0.9 + 0.03).contiguous()                    # not what the generated modes produce
        return A.GridSpecHost.from_tensor(g)
    return A.GridSpecHost(mode, B, H, W, t0=0.1, t_step=0.2)


def _target(B, H, W):
    return torch.stack([blob(H, W, cx=0.4 + 0.05 * b, rx=0.2, ry=0.25) for b in range(B)]).reshape(1, -1).to(DEV)


def _rows(A, prior, params, grid, target, spec, windows):
    """Gradient rows of the given windows, one workspace reused window after window."""
    ws = prior.new_workspace(max(e - b for b, e in windows), A._lib.AWB_WS_FIT_STEP, DEV)
    rows = torch.empty((len(windows), prior.grad_row_floats), dtype=torch.float32, device=DEV)
    for k, (b, e) in enumerate(windows):
        prior.slice_grads(params, grid, b, e, target, spec, rows[k], ws)
    return rows


CASES = [  # kind, C, precision, grid mode
    ("icnn", 2, "fp32", "linspace"), ("icnn", 3, "fp32", "index"), ("icnn", 2, "f16", "explicit"),
    ("icnn", 3, "f16", "linspace"), ("flow", 2, "f16", "linspace"), ("flow", 2, "fp32", "explicit"),
    ("flow", 3, "fp32", "linspace"), ("flow", 3, "f16", "index"), ("flow", 3, "f16", "explicit"),
]


@pytest.mark.parametrize("kind,C_,precision,mode", CASES)
def test_rows_add_up_to_the_full_batch_step(A, kind, C_, precision, mode):
    """Sum of the gradient rows of a ragged window plan (a one-row window, windows off the 128-row grid, one crossing a
    frame boundary) == the full-batch gradient of awb_prior_backward with dlogits of the same loss; loss == the fused step's."""
    B, H, W = 3, 24, 40                                       # 960 rows per frame
    m, prior, params = _model(A, kind, C_, precision)
    grid = _grid(A, mode, B, H, W, C_)
    N = grid.n_pixels
    target = _target(B, H, W)
    spec = A.LossConfig("mse").to_specs(target)[0]
    windows = [(0, 1), (1, 700), (700, 1280), (1280, 2000), (2000, N)]
    rows = _rows(A, prior, params, grid, target, spec, windows)
    total = rows.double().sum(0).cpu()
    # full-batch reference: forward (exact fp32, or the tensor path's training forward), dlogits in torch, backward
    ws = prior.new_workspace(N, A._lib.AWB_WS_TRAINING, DEV)
    mode = A._lib.AWB_FWD_TC_TRAINING if precision == "f16" else A._lib.AWB_FWD_EXACT_TRAINING
    logits, _ = prior.forward(params, grid, mode, ws)
    y = logits.detach().double()
    s = torch.sigmoid(y)
    t = target.double()
    dlog = (2.0 * (s - t) * s * (1 - s) / N).float().contiguous()
    grads, _ = prior.backward(params, grid, dlog, ws, False)
    g_full = grads[0].double().cpu()
    P = prior.n_params
    err = float((total[:P] - g_full).norm() / g_full.norm())
    tol = 1e-5 if precision == "fp32" else (2e-2 if kind == "flow" else 1e-2)
    assert err < tol, (err, tol)
    # the loss slot against the fused step's loss on the same parameters (same per-pixel arithmetic, other summation order)
    f = A.PriorFitter(prior, params.detach().clone(), grid, target, A.LossConfig("mse"), A.OptimConfig(), use_graph=False)
    fused_loss = float(f.run(1)[0, 0])
    assert float(total[P]) == pytest.approx(fused_loss, rel=1e-6)
    # the slice plan's rows add up alike
    plan_rows = _rows(A, prior, params, grid, target, spec, [w for w in A.slice_plan(N, 8) if w[0] < w[1]])
    assert float(plan_rows.double().sum(0)[P]) == pytest.approx(fused_loss, rel=1e-6)


@pytest.mark.parametrize("kind", ["icnn", "flow"])
def test_sliced_steps_run_the_fused_optimizer(A, kind):
    """30 sliced steps (S = 4) against 30 awb_prior_fit_step steps from the same state (fp32 handle, Adam + per-step plateau):
    loss histories agree to 1e-4, the convexity clamp holds."""
    B, H, W = 2, 32, 48
    m, prior, params = _model(A, kind, 3, "fp32", seed=1)
    grid = A.GridSpecHost("linspace", B, H, W, t0=0.0, t_step=1.0)
    target = _target(B, H, W)
    opt = A.OptimConfig("adamax", lr=2e-3, weight_decay=[1e-5, 0.0, 0.0, 0.0], plateau=True, patience=3)
    p_fused = params.detach().clone()
    fused = A.PriorFitter(prior, p_fused, grid, target, A.LossConfig("mse"), opt, use_graph=False).run(30)[:, 0].cpu()
    sliced = A.SlicedFitter(prior, params, grid, target, A.LossConfig("mse"), opt, n_slices=4)
    hist = sliced.run(30)[:, 0].cpu()
    torch.testing.assert_close(hist, fused, rtol=1e-4, atol=0)
    assert sliced.scalars().step == 30 and not sliced.scalars().nonfinite
    for k, v in m.state_dict().items():
        if k.endswith("ln.weight") and ("skip." in k or "out." in k):
            assert float(v.min()) >= 0.0, k


def _simulated_world(A, prior, params0, grid, target, spec, hyper, S, world, steps):
    """`world` ranks one after another on one GPU: each rank computes its slices with its own parameter copy, the rows are
    merged in slice order like all_gather_into_tensor, every rank runs the optimizer on the merged rows."""
    plan = A.slice_plan(grid.n_pixels, S)
    ps = [params0.detach().clone() for _ in range(world)]
    states = []
    for _ in range(world):
        st = torch.empty(prior.opt_state_bytes(), dtype=torch.uint8, device=DEV)
        lrs = (C.c_double * 4)(*[2e-3] * 4)
        A._lib.check(prior.lib.awb_opt_state_init(prior.handle, st.data_ptr(), lrs, A._lib.stream_ptr()))
        states.append(st)
    ws = prior.new_workspace(max(e - b for b, e in plan), A._lib.AWB_WS_FIT_STEP, DEV)
    losses = [torch.empty(steps, device=DEV) for _ in range(world)]
    for s in range(steps):
        merged = []
        for r in range(world):
            mine = A.rank_slices(S, r, world)
            local = torch.zeros((len(mine), prior.grad_row_floats), device=DEV)
            for j, k in enumerate(mine):
                prior.slice_grads(ps[r], grid, plan[k][0], plan[k][1], target, spec, local[j], ws)
            merged.append(local)
        rows = torch.cat(merged).contiguous()
        for r in range(world):
            prior.rows_opt_step(ps[r], states[r], rows, hyper, losses[r][s:s + 1])
    return ps, losses


def _world_case(A):
    m, prior, params = _model(A, "flow", 3, "f16", seed=5)
    B, H, W = 2, 40, 56                                       # 4480 rows: slices of 1024 / 1152 / 1152 / 1152
    grid = A.GridSpecHost("linspace", B, H, W, t0=0.0, t_step=0.5)
    target = _target(B, H, W)
    opt = A.OptimConfig("adamax", lr=2e-3, weight_decay=[1e-5, 0.0, 0.0, 0.0])
    return m, prior, params, grid, target, opt


def test_parameters_do_not_depend_on_the_number_of_ranks(A):
    """S = 4 at world = 1, 2, 4: parameters and loss histories are torch.equal after 50 steps, on every rank, and equal to
    SlicedFitter's one-rank run."""
    m, prior, params, grid, target, opt = _world_case(A)
    spec = A.LossConfig("mse").to_specs(target)[0]
    hyper = opt.to_c()
    p0 = params.detach().clone()
    results = {w: _simulated_world(A, prior, p0, grid, target, spec, hyper, 4, w, 50) for w in (1, 2, 4)}
    ref_p, ref_l = results[1][0][0], results[1][1][0]
    assert bool(torch.isfinite(ref_l).all()) and float(ref_l[-1]) < float(ref_l[0])
    for w, (ps, ls) in results.items():
        for r in range(w):
            assert torch.equal(ps[r], ref_p), (w, r)
            assert torch.equal(ls[r], ref_l), (w, r)
    f = A.SlicedFitter(prior, params, grid, target, A.LossConfig("mse"), opt, n_slices=4)
    hist = f.run(50)[:, 0]
    assert torch.equal(params, ref_p) and torch.equal(hist, ref_l)


def _iou_per_frame(A, m, un, T, H, W):
    t_step = 1.0 / (T - 1)
    out = []
    with torch.no_grad():
        for i in range(T):
            g = A.GridSpecHost("linspace", 1, H, W, t0=i * t_step).materialize(3, DEV)
            prob = torch.sigmoid(m(g)).reshape(1, -1)
            out.append(A.pretrain.mask_iou(prob, un[i].reshape(1, -1).to(DEV)))
    return out


@pytest.mark.parametrize("shuffle", [False, True])
def test_fit_sequence_sliced_matches_the_fused_loop(A, shuffle):
    """fit_sequence(n_slices=4) against fit_sequence() from the same seed (C = 3 flow prior, both prefits, T = 6 at 48x64):
    the same batches and step count, loss histories within 2e-3 over the first 10 steps (the fp16 tensor path: a step's
    gradient differs only in summation order, which moves later steps by fp16 rounding), the same lr trace of the epoch
    plateau steps over the first 100 epochs, and per-frame IoU > 0.9 for both."""
    T, H, W = 6, 48, 64
    un = torch.stack([blob(H, W, cx=0.4 + 0.04 * i, rx=0.2, ry=0.25) for i in range(T)])
    sched = A.FitSchedule(num_epochs=150, batch_size=2, lr=3e-3, prefit_flow_net_identity=True,
                          prefit_flow_net_identity_num_epochs=10, prefit_convex_net=True, prefit_convex_net_num_epochs=40,
                          dataloader_shuffle=shuffle, plateau_patience=10, plateau_factor=0.9, plateau_threshold=0.3)
    runs = []
    for n_slices in (None, 4):
        torch.manual_seed(11)
        m = A.real_nvp_path_connected_net(channels=3, hidden_units=32, flow_n_flows=6, flow_output_fn="tanh",
                                          convex_net_hidden_layers=2, precision="f16").to(DEV)
        lrs = []
        hist = A.fit_sequence(m, T, H, W, un, sched, lr_trace=lrs, n_slices=n_slices).cpu()
        runs.append((hist, lrs, _iou_per_frame(A, m, un, T, H, W)))
    (h0, lr0, iou0), (h1, lr1, iou1) = runs
    assert h0.shape == h1.shape == (150 * 3,)
    torch.testing.assert_close(h1[:10], h0[:10], rtol=2e-3, atol=0)
    # the plateau fires at the same epochs while the trajectories stay close (late in the fit a decision at the
    # threshold can move by an epoch)
    assert lr0[:100] == lr1[:100] and lr0[99][0] < lr0[0][0]
    assert min(iou0) > 0.9 and min(iou1) > 0.9, (iou0, iou1)


def _status(A, prior, params, grid, b, e, target, spec, row, ws, nbytes=None):
    return prior.lib.awb_prior_slice_grads(prior.handle, params.data_ptr(), C.byref(grid.to_c()), b, e, target.data_ptr(),
                                           C.byref(spec), row.data_ptr(), ws.data_ptr(),
                                           ws.numel() if nbytes is None else nbytes, 0, A._lib.stream_ptr())


def test_error_paths(A):
    L = A._lib
    m, prior, params = _model(A, "icnn", 2, "fp32")
    B, H, W = 1, 16, 24
    grid = A.GridSpecHost("linspace", B, H, W)
    N = grid.n_pixels
    target = _target(B, H, W)
    spec = A.LossConfig("mse").to_specs(target)[0]
    row = torch.zeros(prior.grad_row_floats, device=DEV)
    ws = prior.new_workspace(N, L.AWB_WS_FIT_STEP, DEV)
    assert prior.grad_row_floats == prior.n_params + 1
    assert _status(A, prior, params, grid, 0, N, target, spec, row, ws) == 0
    assert _status(A, prior, params, grid, 0, N + 1, target, spec, row, ws) == -1           # past the batch
    assert _status(A, prior, params, grid, -1, 5, target, spec, row, ws) == -1              # negative begin
    assert _status(A, prior, params, grid, 7, 7, target, spec, row, ws) == -1               # empty
    assert _status(A, prior, params, grid, 9, 3, target, spec, row, ws) == -1               # reversed
    assert _status(A, prior, params, grid, 0, -1, target, spec, row, ws) == -1              # negative end
    assert _status(A, prior, params, grid, -64, -1, target, spec, row, ws) == -1            # entirely before the batch
    small = prior.workspace_bytes(128, L.AWB_WS_FIT_STEP)
    assert _status(A, prior, params, grid, 0, N, target, spec, row, ws, nbytes=small) == -4  # short workspace
    assert _status(A, prior, params, grid, 0, 128, target, spec, row, ws, nbytes=small) == 0  # ... enough for its window
    # several objects, NormalizingFlow1D: unsupported
    multi = A.Prior(L.AWB_KIND_ICNN, 2, 130, 2, n_objects=2)
    pm = torch.zeros(2 * multi.n_params, device=DEV)
    assert _status(A, multi, pm, grid, 0, N, target, spec, torch.zeros(multi.n_params + 1, device=DEV),
                   multi.new_workspace(N, L.AWB_WS_FIT_STEP, DEV)) == -2
    diffeo = A.Prior(L.AWB_KIND_DIFFEO_ICNN, 2, 130, 2, n_flows=2, flow_hidden=16)
    pd = torch.zeros(diffeo.n_params, device=DEV)
    assert _status(A, diffeo, pd, grid, 0, N, target, spec, torch.zeros(diffeo.n_params + 1, device=DEV),
                   diffeo.new_workspace(N, L.AWB_WS_FIT_STEP, DEV)) == -2
    st = torch.empty(diffeo.opt_state_bytes(), dtype=torch.uint8, device=DEV)
    rows = torch.zeros((2, diffeo.n_params + 1), device=DEV)
    assert diffeo.lib.awb_prior_rows_opt_step(diffeo.handle, pd.data_ptr(), st.data_ptr(), rows.data_ptr(), 2,
                                              C.byref(A.OptimConfig().to_c()), None, None, 0, L.stream_ptr()) == -2
    # world must divide S
    with pytest.raises(ValueError, match="multiple"):
        A.rank_slices(8, 0, 3)
    # a NaN in one slice's target: sticky non-finite flag, parameters untouched
    grid2 = A.GridSpecHost("linspace", 2, 32, 40)
    t2 = _target(2, 32, 40)
    t2[0, 1500] = float("nan")
    f = A.SlicedFitter(prior, params, grid2, t2, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-2), n_slices=4)
    before = params.detach().clone()
    f.step()
    sc = f.scalars()
    assert sc.nonfinite == 1 and sc.step == 0
    assert torch.equal(params, before)
    with pytest.raises(ValueError, match="nan or inf"):
        f.raise_if_nonfinite()


def _nccl_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import awesome_b200 as A
        global DEV
        DEV = f"cuda:{rank}"
        m, prior, params, grid, target, opt = _world_case(A)
        f = A.SlicedFitter(prior, params, grid, target, A.LossConfig("mse"), opt, n_slices=4, group=dist.group.WORLD)
        hist = f.run(50)
        torch.cuda.synchronize()
        torch.save({"params": params.cpu(), "hist": hist.cpu()}, os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_real_nccl_two_ranks_match_one_rank(A, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs for a real NCCL world of 2")
    import torch.multiprocessing as mp
    m, prior, params, grid, target, opt = _world_case(A)
    A.SlicedFitter(prior, params, grid, target, A.LossConfig("mse"), opt, n_slices=4).run(50)
    ref = params.detach().cpu()
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, str(tmp_path))) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
        assert p.exitcode == 0
    for r in range(2):
        got = torch.load(os.path.join(tmp_path, f"rank{r}.pt"))
        assert torch.equal(got["params"], ref), r


def _seq_schedule(A, shuffle):
    return A.FitSchedule(num_epochs=12, batch_size=2, lr=3e-3, prefit_flow_net_identity=True,
                         prefit_flow_net_identity_num_epochs=5, prefit_convex_net=True, prefit_convex_net_num_epochs=10,
                         dataloader_shuffle=shuffle, noisy_percentage=0.34 if shuffle else 0.0, plateau_patience=2,
                         plateau_factor=0.9, plateau_threshold=0.3)


def _seq_run(A, shuffle, seed, n_slices, group):
    """fit_sequence of a small C = 3 flow prior from the given seed (torch and numpy global RNGs)."""
    import numpy as np
    T, H, W = 6, 48, 64
    un = torch.stack([blob(H, W, cx=0.4 + 0.04 * i, rx=0.2, ry=0.25) for i in range(T)])
    torch.manual_seed(seed)
    np.random.seed(seed)
    m = A.real_nvp_path_connected_net(channels=3, hidden_units=32, flow_n_flows=6, flow_output_fn="tanh",
                                      convex_net_hidden_layers=2, precision="f16").to(DEV)
    lrs = []
    hist = A.fit_sequence(m, T, H, W, un, _seq_schedule(A, shuffle), lr_trace=lrs, n_slices=n_slices, group=group)
    return m._ensure_flat().detach().cpu(), hist.cpu(), lrs


def _seq_worker(rank, world, port, backend, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dev = rank if backend == "nccl" else 0
    torch.cuda.set_device(dev)
    global DEV
    DEV = f"cuda:{dev}"
    kw = dict(device_id=torch.device("cuda", dev)) if backend == "nccl" else {}
    dist.init_process_group(backend, rank=rank, world_size=world, **kw)
    try:
        import awesome_b200 as A
        out = {}
        for shuffle in (False, True):
            # rank 1 starts from other random states: the broadcasts of fit_sequence must make that irrelevant
            out[shuffle] = _seq_run(A, shuffle, 11 if rank == 0 else 12345, 4, dist.group.WORLD)
        torch.save(out, os.path.join(out_dir, f"seq_rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_fit_sequence_on_two_ranks_matches_one_rank(A, tmp_path):
    """The multi-rank branch of fit_sequence(n_slices=4, group=...) with two processes (NCCL on two GPUs, else gloo with
    both processes on one GPU): rank 1 starts from different RNG states, yet after the broadcasts of the prefit result, the
    noisy unaries and the shuffled batch order both ranks end with the parameters, loss history and lr trace of the
    one-process run, bit for bit, in ordered and shuffled mode."""
    import torch.multiprocessing as mp
    backend = "nccl" if torch.cuda.device_count() >= 2 else "gloo"
    ref = {shuffle: _seq_run(A, shuffle, 11, 4, None) for shuffle in (False, True)}
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_seq_worker, args=(r, 2, port, backend, str(tmp_path))) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(900)
        assert p.exitcode == 0
    for r in range(2):
        got = torch.load(os.path.join(tmp_path, f"seq_rank{r}.pt"))
        for shuffle in (False, True):
            p_ref, h_ref, lr_ref = ref[shuffle]
            p_got, h_got, lr_got = got[shuffle]
            assert torch.equal(p_got, p_ref), (r, shuffle)
            assert torch.equal(h_got, h_ref), (r, shuffle)
            assert lr_got == lr_ref, (r, shuffle)
