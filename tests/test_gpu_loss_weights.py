"""Per-pixel loss weights and the ignore label of the fused fit steps (awb_loss_spec.weight / ignore_enabled) on the GPU:
gradient rows against float64 on both kernel paths, the reference's weak-label loss, and the properties the weighted
epilogue must keep (all-ones map == no map bit for bit, ignored pixels inert, NaN weights flagged, grouped == single,
sliced == unsliced, host frames == device frames, error returns)."""
import ctypes as C

import pytest
import torch

import __graft_entry__ as entry
from oracle import prior_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
IGN = 2.0                    # the FBMS none class

# Bounds of tests/test_gpu_launch_regimes.py (exact path per entry relative to the tensor's largest entry; tensor path
# normwise, DESIGN section 4), restated here.
TOL_GRAD, TOL_LOSS = 5e-4, 1e-6
TC_TOL_LOSS, TC_TOL_GRAD_ICNN, TC_TOL_GRAD_FLOW = 2e-4, 1e-2, 2e-2


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


def entry_err(got, ref):
    d = float((got.double() - ref).abs().max())
    s = float(ref.abs().max())
    return d / s if s > 0 else d


def make_model(A, kind, C_, precision, seed=0, F=None):
    torch.manual_seed(seed)
    if kind == "flow":
        m = A.real_nvp_path_connected_net(channels=C_, hidden_units=32, flow_n_flows=F or (12 if C_ == 2 else 18),
                                          flow_output_fn="tanh", norm="minmax", convex_net_hidden_units=130,
                                          convex_net_hidden_layers=2, precision=precision)
        sd = m.state_dict()
        for k in sd:
            if ".net.2." in k:
                sd[k] = 0.05 * torch.randn_like(sd[k])
            elif k.endswith((".s", ".t")) and ".flows." in k:
                sd[k] = 0.1 * torch.randn_like(sd[k])
            elif k.endswith("data_dep_init_done"):
                sd[k] = torch.ones_like(sd[k])
        m.load_state_dict(sd)
    else:
        m = A.ConvexNextNet(n_hidden=130, in_features=C_, n_hidden_layers=2, precision=precision)
    return m.to(DEV)


def torch_grid(B, H, W, C_, t0=0.1, t_step=0.3):
    y, x = torch.linspace(0, 1, H), torch.linspace(0, 1, W)
    yy, xx = torch.meshgrid(y, x, indexing="ij")
    ch = [xx.expand(B, H, W), yy.expand(B, H, W)]
    if C_ == 3:
        t = torch.full((B,), t0, dtype=torch.float32) + torch.arange(B, dtype=torch.float32) * torch.tensor(t_step)
        ch.append(t.view(B, 1, 1).expand(B, H, W))
    return torch.stack(ch, 1).contiguous().to(DEV)


def weak_target(B, H, W, seed=0, frac_ignored=0.3, hard=False):
    """Soft (or {0, 1}) unaries of a blob with about ``frac_ignored`` of the pixels set to the none class, and a weight map
    uniform in [0, 2]."""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    if H == 1:                                           # one pixel row: through the blob, so that both classes occur
        yy = torch.full_like(yy, 0.5)
    t = torch.sigmoid((torch.sqrt(((xx - 0.45) / 0.25) ** 2 + ((yy - 0.5) / 0.3) ** 2) - 1) / 0.08).expand(B, H, W).reshape(-1)
    if hard:
        t = (t >= 0.5).float()
    t = torch.where(torch.rand(t.shape, generator=g) < frac_ignored, torch.full_like(t, IGN), t)
    w = 2.0 * torch.rand(t.shape, generator=g)
    return t.contiguous().to(DEV), w.contiguous().to(DEV)


def reference(model, kind, rows, target, weight, loss_kind, mode):
    """float64: loss = mean over kept pixels of w * class weight * l, and every parameter gradient (arena order)."""
    by_id = {id(q): k for k, q in model.named_parameters()}
    names = [by_id[id(q)] for q in model._arena_params()]
    p = {k: v.detach().to(DEV, torch.float64).clone() for k, v in model.state_dict().items()}
    for k in names:
        p[k].requires_grad_(True)
    N, C_ = rows.shape
    x = rows.double().t().reshape(1, C_, 1, N)
    if kind == "flow":
        y = O.icnn_forward(p, O.pathconnected_deformation(p, x), "convex_net.").reshape(-1)
    else:
        y = O.icnn_forward(p, O.pixelize(x)).reshape(-1)
    keep = target != IGN
    t, yk, wk = target[keep].double(), y[keep], weight[keep].double()
    cw = O.unaries_weight(t.float(), mode).double()     # class weights from the counts over the kept pixels
    if loss_kind == "mse":
        l = (t - torch.sigmoid(yk)) ** 2
    else:
        l = torch.nn.functional.binary_cross_entropy_with_logits(yk, t, reduction="none")
    loss = (l * cw * wk).sum() / keep.sum()
    grads = torch.autograd.grad(loss, [p[k] for k in names])
    return names, float(loss), grads


def split(flat, grads):
    out, off = [], 0
    for g in grads:
        out.append(flat[off:off + g.numel()].view(g.shape))
        off += g.numel()
    assert off == flat.numel()
    return out


def grad_row(A, model, spec, target, loss):
    prior = model._prior_for(model._ensure_flat().device)
    params = model._ensure_flat().detach().reshape(1, -1).contiguous()
    specs = loss.to_specs(target.reshape(1, -1))
    row = torch.zeros(prior.grad_row_floats, dtype=torch.float32, device=DEV)
    ws = prior.new_workspace(spec.n_pixels, A._lib.AWB_WS_FIT_STEP, DEV)
    prior.slice_grads(params, spec, 0, spec.n_pixels, target, specs[0], row, ws)
    torch.cuda.synchronize()
    return row, prior.n_params


# (kind, C, B, H, W): both sides of the exact path's n_splits branch (148 full ranges / empty trailing ranges; one / two
# ranges) for the ICNN and the RealNVP prior at C = 2 and 3
SIZES = [("icnn", 2, 1, 148, 256), ("icnn", 2, 1, 1, 37889), ("flow", 2, 1, 15, 17), ("flow", 2, 1, 1, 257),
         ("flow", 3, 1, 148, 256), ("flow", 3, 1, 1, 37889)]
LOSSES = [("mse", "none"), ("mse", "sssdms"), ("bce", "none"), ("bce", "sssdms")]


@pytest.mark.parametrize("loss_kind,mode", LOSSES)
@pytest.mark.parametrize("kind,C_,B,H,W", SIZES)
def test_exact_path_weighted_rows_against_float64(A, kind, C_, B, H, W, loss_kind, mode):
    m = make_model(A, kind, C_, "fp32")
    target, weight = weak_target(B, H, W, seed=C_ + W)
    spec = A.GridSpecHost("linspace", B, H, W, t0=0.1, t_step=0.3)
    row, P = grad_row(A, m, spec, target, A.LossConfig(loss_kind, mode=mode, weight=weight, ignore_value=IGN))
    names, loss, grads = reference(m, kind, O.pixelize(torch_grid(B, H, W, C_)), target, weight, loss_kind, mode)
    errs = {k: entry_err(g, g64) for k, g, g64 in zip(names, split(row[:P], grads), grads)}
    l_err = abs(float(row[P]) - loss) / loss
    print(f"[weights exact {kind} C={C_} N={B * H * W} {loss_kind}/{mode}] loss {l_err:.2e} "
          f"gradients {max(errs.values()):.2e} ({max(errs, key=errs.get)})")
    assert l_err <= TOL_LOSS
    bad = {k: v for k, v in errs.items() if not v <= TOL_GRAD}
    assert not bad, bad


@pytest.mark.parametrize("kind,C_,B,H,W,loss_kind,mode", [
    ("icnn", 2, 1, 149, 128, "mse", "sssdms"), ("icnn", 2, 1, 1, 37889, "bce", "sssdms"), ("icnn", 3, 1, 148, 256, "bce", "none"),
    ("flow", 2, 1, 149, 128, "bce", "sssdms"), ("flow", 3, 2, 74, 128, "mse", "none")])
def test_tensor_path_weighted_rows_against_float64(A, kind, C_, B, H, W, loss_kind, mode):
    m = make_model(A, kind, C_, "f16", seed=3)
    target, weight = weak_target(B, H, W, seed=7 + C_)
    spec = A.GridSpecHost("linspace", B, H, W, t0=0.1, t_step=0.3)
    row, P = grad_row(A, m, spec, target, A.LossConfig(loss_kind, mode=mode, weight=weight, ignore_value=IGN))
    names, loss, grads = reference(m, kind, O.pixelize(torch_grid(B, H, W, C_)), target, weight, loss_kind, mode)
    l_err = abs(float(row[P]) - loss) / loss
    errs, flow = {}, []
    for k, g, g64 in zip(names, split(row[:P], grads), grads):
        if k.startswith(("flow_net.", "linear.")):
            flow.append((float((g.double() - g64).norm()), float(g64.norm())))
        elif float(g64.norm()) > 1e-7:
            errs[k] = (float((g.double() - g64).norm() / g64.norm()), TC_TOL_GRAD_ICNN)
    if flow:
        errs["flow_net + linear"] = (sum(d ** 2 for d, _ in flow) ** 0.5 / sum(r ** 2 for _, r in flow) ** 0.5,
                                     TC_TOL_GRAD_FLOW)
    print(f"[weights tensor {kind} C={C_} {loss_kind}/{mode}] loss {l_err:.2e} worst normwise "
          f"{max(v for v, _ in errs.values()):.2e}")
    assert l_err <= TC_TOL_LOSS
    bad = {k: v for k, (v, tol) in errs.items() if not v <= tol}
    assert not bad, bad


def test_diffeo_weighted_fit_step_matches_autograd_adam(A, golden):
    """ConvexDiffeomorphismNet, one fused step with a weight map and ignore label == autograd (the module's native
    backward) of the same weighted loss in float64 on the logits, then torch.optim.Adam and enforce_convexity."""
    g = golden("diffeo.pt")

    def make(prec="fp32"):
        m = A.ConvexDiffeomorphismNet(n_hidden=130, n_hidden_layers=1, nf_layers=4, nf_hidden=70, precision=prec)
        m.load_state_dict(g["pert"])
        return m.to(DEV)

    H, W = 48, 64
    target, weight = weak_target(1, H, W, seed=11)
    grid = A.GridSpecHost("linspace", 1, H, W)
    m_ref = make()
    opt = torch.optim.Adam(m_ref.parameters(), lr=1e-3)
    y = m_ref(grid.materialize(2, DEV)).reshape(-1)
    keep = target != IGN
    yd = y.double()
    l = torch.where(keep, weight.double() * (torch.where(keep, target, 0.0).double() - torch.sigmoid(yd)) ** 2, 0.0)
    loss_ref = l.sum() / keep.sum()
    loss_ref.backward()
    opt.step()
    m_ref.convex_net.enforce_convexity()
    m = make()
    f = m.make_fitter(grid, target, A.LossConfig("mse", weight=weight, ignore_value=IGN), A.OptimConfig("adam", lr=1e-3),
                      use_graph=False)
    loss = float(f.run(1)[0, 0])
    assert abs(loss - loss_ref.item()) <= 1e-5 * abs(loss_ref.item())
    # Adam's first step is lr * g / (|g| + eps): an entry whose gradient is within a few eps of 0 moves by a fraction of lr
    # that the last bits of g decide (the weight map puts more of them there than the unweighted test sees): atol = lr / 10
    for k, v in m_ref.state_dict().items():
        torch.testing.assert_close(m.state_dict()[k], v, rtol=1e-4, atol=1e-4, msg=lambda s: f"{k}: {s}")


def test_weak_label_criterion_matches_reference_weighted_bce(A):
    """``WeightedLoss(BCELoss, "sssdms", noneclass=2)`` on a {0, 1, 2} weak-label target: the loss of the fused step equals
    the oracle's ``loss_weighted_bce_sssdms`` on the same logits."""
    class BCELoss:
        pass

    class WeightedLoss:
        def __init__(self):
            self.criterion, self.mode, self.noneclass = BCELoss(), "sssdms", 2

    cfg = A.LossConfig.from_reference(WeightedLoss())
    assert (cfg.kind, cfg.mode, cfg.ignore_value) == ("bce", "sssdms", 2.0)
    H, W = 60, 80
    target, _ = weak_target(1, H, W, seed=5, frac_ignored=0.7, hard=True)
    m = make_model(A, "icnn", 2, "fp32", seed=1)
    grid = A.GridSpecHost("linspace", 1, H, W)
    with torch.no_grad():
        prob = torch.sigmoid(m(grid.materialize(2, DEV)).reshape(-1).double())
    ref = float(O.loss_weighted_bce_sssdms(prob.cpu(), target.double().cpu(), noneclass=2.0))
    f = m.make_fitter(grid, target, cfg, A.OptimConfig("adam", lr=1e-3), use_graph=False)
    loss = float(f.run(1)[0, 0])
    assert abs(loss - ref) <= 1e-5 * ref, (loss, ref)


# ------------------------------------------------------------------------------------------------------------ properties
def opt_bytes(f):
    """The optimizer state that steps write: moments [2][O][P] and the per-object scalars (not the allocation's padding)."""
    O_, P = f.prior.n_objects, f.prior.n_params
    sc = [f.scalars(o) for o in range(O_)]
    return torch.cat([f.opt_state[:8 * O_ * P].cpu(),
                      torch.tensor([[s.step, s.num_bad, s.nonfinite] + list(s.lr) + [s.best, s.last_loss] for s in sc],
                                   dtype=torch.float64).view(torch.uint8).reshape(-1)])


def _fit(A, m, grid, target, loss, steps=4, graph=False):
    f = m.make_fitter(grid, target, loss, A.OptimConfig("adam", lr=1e-3), use_graph=graph, steps_per_graph=2)
    hist = f.run(steps)
    torch.cuda.synchronize()
    return hist.clone(), m._ensure_flat().detach().clone(), opt_bytes(f), f


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_all_ones_map_is_bit_identical_to_no_map(A, precision):
    H, W = 96, 128
    target, _ = weak_target(1, H, W, seed=2, frac_ignored=0.0)
    grid = A.GridSpecHost("linspace", 1, H, W)
    out = []
    for loss in (A.LossConfig("mse"), A.LossConfig("mse", weight=torch.ones(H * W, device=DEV))):
        out.append(_fit(A, make_model(A, "icnn", 2, precision), grid, target, loss, graph=True))
    for a, b in zip(out[0][:3], out[1][:3]):
        assert torch.equal(a, b)


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_ignored_pixels_change_nothing(A, precision):
    """Another ignore value at the same pixels (so other targets there) and NaN / huge weights there: same bits."""
    H, W = 96, 128
    target, weight = weak_target(1, H, W, seed=4)
    ign = target == IGN
    grid = A.GridSpecHost("linspace", 1, H, W)
    a = _fit(A, make_model(A, "flow", 2, precision), grid, target, A.LossConfig("bce", weight=weight, ignore_value=IGN))
    t2 = torch.where(ign, torch.full_like(target, -7.0), target)
    w2 = torch.where(ign, torch.where(torch.rand_like(weight) < 0.5, float("nan"), 1e30), weight)
    b = _fit(A, make_model(A, "flow", 2, precision), grid, t2, A.LossConfig("bce", weight=w2, ignore_value=-7.0))
    for x, y in zip(a[:3], b[:3]):
        assert torch.equal(x, y)
    assert not b[3].scalars().nonfinite


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_nan_weight_on_a_kept_pixel_flags_and_skips(A, precision):
    H, W = 48, 64
    target, weight = weak_target(1, H, W, seed=6)
    kept = int(torch.nonzero(target != IGN)[0])
    weight[kept] = float("nan")
    m = make_model(A, "icnn", 2, precision)
    before = m._ensure_flat().detach().clone()
    f = m.make_fitter(A.GridSpecHost("linspace", 1, H, W), target, A.LossConfig("mse", weight=weight, ignore_value=IGN),
                      A.OptimConfig("adam", lr=1e-3), use_graph=False)
    f.run(1)
    assert f.scalars().nonfinite
    assert torch.equal(m._ensure_flat().detach(), before)
    with pytest.raises(ValueError):
        f.raise_if_nonfinite()


def test_grouped_objects_with_own_maps_equal_single_fits(A):
    H, W, G = 48, 64, 3
    grid = A.GridSpecHost("linspace", 1, H, W)
    tw = [weak_target(1, H, W, seed=20 + k) for k in range(G)]
    multi = A.NumberBasedMultiPriorModule(prior_type=A.ConvexNextNet, prior_args=dict(n_hidden_layers=2), min_priors=G).to(DEV)
    assert len(multi.priors) == G
    for p in multi.priors:
        p.load_state_dict(make_model(A, "icnn", 2, "fp32").state_dict())
    tg = torch.stack([t for t, _ in tw])
    wg = torch.stack([w for _, w in tw])
    f = multi.make_fitter(grid, tg, A.LossConfig("mse", mode="sssdms", weight=wg, ignore_value=IGN),
                          A.OptimConfig("adam", lr=1e-3), use_graph=False)
    hg = f.run(3)
    big = multi._group_arena().detach().clone()
    for k in range(G):
        h1, p1, _, _ = _fit(A, make_model(A, "icnn", 2, "fp32"), grid, tw[k][0],
                            A.LossConfig("mse", mode="sssdms", weight=tw[k][1], ignore_value=IGN), steps=3)
        assert torch.equal(hg[:, k], h1[:, 0])
        assert torch.equal(big[k], p1.reshape(-1))


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_sliced_weighted_fit_does_not_depend_on_the_world_size(A, precision):
    """Sliced steps with a weight map (windows starting mid-row) give the same bits for world = 1, 2 and 4: the rows of
    every rank's slices are the same rows."""
    from awesome_b200.fit import slice_plan
    H, W, S = 37, 53, 8
    target, weight = weak_target(1, H, W, seed=9)
    grid = A.GridSpecHost("linspace", 1, H, W)
    plan = slice_plan(H * W, S)
    assert any(b % W for b, _ in plan if b)         # windows that start mid-row
    m0 = make_model(A, "flow", 2, precision)
    prior = m0._prior_for(m0._ensure_flat().device)
    params0 = m0._ensure_flat().detach().reshape(1, -1).clone()
    spec = A.LossConfig("bce", mode="sssdms", weight=weight, ignore_value=IGN).to_specs(target.reshape(1, -1))[0]
    R = prior.grad_row_floats
    ws = prior.new_workspace(max(e - b for b, e in plan), A._lib.AWB_WS_FIT_STEP, DEV)
    results = []
    for world in (1, 2, 4):
        rows = torch.zeros((S, R), dtype=torch.float32, device=DEV)
        for rank in range(world):                    # each simulated rank computes its own slices
            for k in range(rank * S // world, (rank + 1) * S // world):
                b, e = plan[k]
                prior.slice_grads(params0, grid, b, e, target, spec, rows[k], ws)
        results.append(rows.clone())
        full = torch.zeros(R, dtype=torch.float32, device=DEV)
        if world == 1:
            ws_full = prior.new_workspace(H * W, A._lib.AWB_WS_FIT_STEP, DEV)
            prior.slice_grads(params0, grid, 0, H * W, target, spec, full, ws_full)
            tol = 5e-4 if precision == "fp32" else 2e-2
            assert float((rows.sum(0) - full).norm() / full.norm()) <= tol
    assert torch.equal(results[0], results[1]) and torch.equal(results[0], results[2])


def test_host_frames_equal_device_frames(A):
    H, W = 48, 64
    target, weight = weak_target(1, H, W, seed=12)
    t2, _ = weak_target(1, H, W, seed=13)
    grid = A.GridSpecHost("linspace", 1, H, W)
    loss = A.LossConfig("mse", weight=weight, ignore_value=IGN)
    m1 = make_model(A, "icnn", 2, "f16")
    f1 = m1.make_fitter(grid, target, loss, A.OptimConfig("adam", lr=1e-3), use_graph=False)
    f1.set_target_pool(torch.stack([target, t2]).reshape(2, 1, -1).contiguous())
    f1.run(4, record=False)
    m2 = make_model(A, "icnn", 2, "f16")
    f2 = m2.make_fitter(grid, target, loss, A.OptimConfig("adam", lr=1e-3), use_graph=False)
    f2.run_host_frames([target.cpu().reshape(1, -1).pin_memory(), t2.cpu().reshape(1, -1).pin_memory()], 4)
    torch.cuda.synchronize()
    assert torch.equal(m1._ensure_flat(), m2._ensure_flat())
    assert torch.equal(opt_bytes(f1), opt_bytes(f2))


def test_set_target_with_a_new_map_recaptures(A):
    H, W = 48, 64
    target, w1 = weak_target(1, H, W, seed=14)
    _, w2 = weak_target(1, H, W, seed=15)
    grid = A.GridSpecHost("linspace", 1, H, W)
    m = make_model(A, "icnn", 2, "fp32")
    f = m.make_fitter(grid, target, A.LossConfig("mse", weight=w1), A.OptimConfig("adam", lr=1e-3), steps_per_graph=2)
    f.run(2)
    f.set_target(target, A.LossConfig("mse", weight=w2))        # same shape: copied into the fitter's map
    assert f._graph is not None and torch.equal(f._weight.reshape(-1), w2)
    f.set_target(target, A.LossConfig("mse", weight=w2, ignore_value=IGN))
    assert f._graph is None
    f.set_target(target, A.LossConfig("mse"))
    assert f._weight is None
    h = f.run(2)
    assert torch.isfinite(h).all()


def test_c_abi_errors(A):
    L = A._lib
    lib = L.load()
    m = make_model(A, "icnn", 2, "fp32")
    H, W = 16, 16
    target, weight = weak_target(1, H, W)
    grid = A.GridSpecHost("linspace", 1, H, W)
    f = m.make_fitter(grid, target, A.LossConfig("mse"), A.OptimConfig("adam", lr=1e-3), use_graph=False)
    bad = L.LossSpec(L.AWB_LOSS_SE_SIGMOID, L.AWB_CLS_UNARY_LT_HALF, 1.0, 1.0, None, 1, float("nan"))
    gs = grid.to_c()
    rc = lib.awb_prior_fit_step(f.prior.handle, f.params.data_ptr(), f.opt_state.data_ptr(), C.byref(gs),
                                target.data_ptr(), C.byref(bad), C.byref(f._hyper), None, f.ws.data_ptr(), f.ws.numel(), 0,
                                L.stream_ptr())
    assert rc == -1                                  # AWB_ERR_INVALID: a NaN ignore label
    counts = torch.zeros((1, 2), dtype=torch.int64, device=DEV)
    assert lib.awb_target_counts_ignore(target.data_ptr(), H * W, 1, 0, 1, float("inf"), counts.data_ptr(),
                                        L.stream_ptr()) == -1
    assert lib.awb_target_counts_ignore(target.data_ptr(), H * W, 1, 0, 1, IGN, counts.data_ptr(), L.stream_ptr()) == 0
    kept = target[target != IGN]
    assert counts.cpu().tolist() == [[int((kept < 0.5).sum()), int((kept >= 0.5).sum())]]
    # the star fit step takes no weight map or ignore label
    star = A.Prior(L.AWB_KIND_STAR, 2, 32, 0)
    sp = torch.zeros((1, star.n_params), device=DEV)
    st = torch.zeros(star.opt_state_bytes(), dtype=torch.uint8, device=DEV)
    x = torch.rand((64, 2), device=DEV)
    t = torch.rand(64, device=DEV)
    sws = torch.zeros(int(lib.awb_star_workspace_bytes(star.handle, 64)), dtype=torch.uint8, device=DEV)
    for spec in (L.LossSpec(0, 0, 1.0, 1.0, weight.data_ptr(), 0, 0.0), L.LossSpec(0, 0, 1.0, 1.0, None, 1, 2.0)):
        rc = lib.awb_star_fit_step(star.handle, sp.data_ptr(), st.data_ptr(), x.data_ptr(), t.data_ptr(), 64, C.byref(spec),
                                   C.byref(f._hyper), None, sws.data_ptr(), sws.numel(), L.stream_ptr())
        assert rc == -2


def test_weak_label_fit_iou_against_the_fully_labelled_fit(A):
    """640x480 synthetic frame: fit to weak labels (10 % of the pixels labelled, the rest none class) and to the full
    labels; report the IoU of the two fitted masks.  Nothing is asserted beyond a sane fit: no target has been set."""
    H, W = 480, 640
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    full = (torch.sqrt(((xx - 0.45) / 0.25) ** 2 + ((yy - 0.5) / 0.3) ** 2) >= 1).float().reshape(-1).to(DEV)
    g = torch.Generator().manual_seed(0)
    weak = torch.where(torch.rand(H * W, generator=g).to(DEV) < 0.1, full, torch.full_like(full, IGN))
    grid = A.GridSpecHost("linspace", 1, H, W)
    masks = []
    for t, loss in ((full, A.LossConfig("bce", mode="sssdms")), (weak, A.LossConfig("bce", mode="sssdms", ignore_value=IGN))):
        m = make_model(A, "icnn", 2, "f16", seed=0)
        f = m.make_fitter(grid, t, loss, A.OptimConfig("adam", lr=1e-3), steps_per_graph=50)
        f.run(1000)
        f.raise_if_nonfinite()
        with torch.no_grad():
            masks.append(m(grid.materialize(2, DEV)).reshape(-1) <= 0)
    inter = float((masks[0] & masks[1]).sum())
    iou = inter / float((masks[0] | masks[1]).sum())
    gt = full <= 0.5
    iou_gt = float((masks[1] & gt).sum()) / float((masks[1] | gt).sum())
    print(f"[weak labels] 640x480, 10 % labelled, 1000 steps: IoU(weak fit, full fit) = {iou:.4f}, "
          f"IoU(weak fit, ground truth) = {iou_gt:.4f}")
    assert iou > 0.5
