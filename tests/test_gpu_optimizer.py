"""The fused optimizer kernels (``k_reduce_opt``, ``k_reduce_opt_aug``, ``k_plateau_step`` in awb_simt.cu) against a
float64 reference, formula by formula.

Every output is recomputed in float64 from the kernel's own fp32 inputs to that formula: ``m`` from (m_old, g), ``v`` from
(v_old, g), ``p`` from (p_old, the kernel's m_new and v_new, step size and bias correction), with the fp32
hyper-parameters ``awb_opt_hyper`` carries.  The bounds are a few fp32 roundings of the terms involved, so a parameter in
the wrong group, a wrong lr, weight decay or bias-correction step, a clamp on the wrong entries or a dropped block fails by
orders of magnitude.  Groups, clamp entries and per-group step counts come from the state_dict keys and from the test's
own bookkeeping (torch keeps a step count per parameter and skips a parameter whose grad is None; the host test
``test_optimizer_oracle_host.py`` pins that bookkeeping against torch), never from the handle's arrays."""
import ctypes as C
import math

import pytest
import torch

import __graft_entry__ as entry
from oracle import prior_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24                 # unit roundoff of fp32
SCAL_BYTES = 80                # sizeof(OptScal): lr[4] and best (f64), step, num_bad, nonfinite, pad, last_loss, pad2, group_start[4]
LRS = [2e-3, 1e-3, 3e-3, 4e-3]
WDS = [1e-3, 1e-2, 0.0, 5e-2]


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


# ---------------------------------------------------------------------------------------------------- models and layout
def _model(A, kind, C_=2, L_=1, h=130, precision="fp32", F=6, m=32, seed=0):
    torch.manual_seed(seed)
    if kind == "icnn":
        return A.ConvexNextNet(n_hidden=h, in_features=C_, n_hidden_layers=L_, precision=precision)
    if kind == "flow":
        net = A.real_nvp_path_connected_net(channels=C_, hidden_units=m, flow_n_flows=F, flow_output_fn="tanh",
                                            convex_net_hidden_units=h, convex_net_hidden_layers=L_, precision=precision)
        sd = net.state_dict()
        for k in sd:
            if ".net.2." in k:                                 # zero-initialised couplings would make the flow trivial
                sd[k] = 0.05 * torch.randn_like(sd[k])
            elif k.endswith("data_dep_init_done"):
                sd[k] = torch.ones_like(sd[k])
        net.load_state_dict(sd)
        return net
    if kind == "diffeo":
        return A.ConvexDiffeomorphismNet(n_hidden=h, n_hidden_layers=L_, precision=precision)
    return A.StarShapedNet(h)


def _layout(model):
    """Optimizer group and clamp flag of every arena entry, from the parameter names: ICNN 1; RealNVP / NormalizingFlow1D
    prior: convex_net 1, flow 0 (weight-norm gains 3), linear 2; star: offset 2, the rest 1, clamp on W2_r.weight."""
    sd = dict(model.state_dict())
    star = type(model).__name__ == "StarShapedNet"
    if star:
        clamp_keys = {"W2_r.weight"}
    elif type(model).__name__ == "ConvexNextNet":
        clamp_keys = set(O.icnn_clamp_keys(sd))
    else:
        clamp_keys = set(O.icnn_clamp_keys(sd, "convex_net."))
    assert clamp_keys and clamp_keys <= set(sd)

    def grp(n):
        if star:
            return 2 if n == "offset" else 1
        if n.startswith("diffeo_net.") or n.startswith("flow_net."):
            return 3 if n.endswith("weight_g") else 0
        return 2 if n.startswith("linear.") else 1

    group, clamp, names = [], [], []
    for n, p in model.named_parameters():
        group += [grp(n)] * p.numel()
        clamp += [n in clamp_keys] * p.numel()
        names.append((n, p.numel()))
    return torch.tensor(group, device=DEV), torch.tensor(clamp, device=DEV), names


def _handle(A, model, O_):
    """Native handle of ``O_`` objects with the model's layout (flow constants pushed)."""
    d = model.to(DEV)._prior_for(torch.device(DEV)).desc
    prior = A.Prior(d.kind, d.C, d.h, d.L, d.F, d.m, bool(d.flow_tanh), O_, d.precision)
    if d.kind == A._lib.AWB_KIND_FLOW_ICNN:
        model._push_consts(prior)
    return prior


def _icnn_P(h, C_, L_):
    return h * (C_ + 1) + L_ * (h * h + h + h * C_) + h + 1 + C_


def _h_with_tail(C_, L_, tail):
    """ICNN width whose parameter count leaves ``tail`` parameters in the last 32-parameter block (0: a full block)."""
    return next(h for h in range(8, 200) if _icnn_P(h, C_, L_) % 32 == tail % 32)


# ---------------------------------------------------------------------------------------------------- optimizer state
def _round_up(a, b):
    return (a + b - 1) // b * b


def _new_state(A, prior, lrs=LRS):
    L = A._lib
    st = torch.empty(prior.opt_state_bytes(), dtype=torch.uint8, device=DEV)
    L.check(prior.lib.awb_opt_state_init(prior.handle, st.data_ptr(), (C.c_double * 4)(*lrs), L.stream_ptr()))
    return st


def _mv(prior, st):
    """m [O][P] and v [O][P] as views of the blob; the scalars follow at round_up(8 O P, 256)."""
    O_, P = prior.n_objects, prior.n_params
    assert st.numel() == prior.opt_state_bytes() == _round_up(8 * O_ * P, 256) + _round_up(SCAL_BYTES * O_, 256)
    f = st[:8 * O_ * P].view(torch.float32).view(2, O_, P)
    return f[0], f[1]


def _scal(A, prior, st, o=0):
    L = A._lib
    out = L.OptScalars()
    L.check(prior.lib.awb_opt_read_scalars(prior.handle, st.data_ptr(), o, C.byref(out), L.stream_ptr()))
    return out


def _lrs(A, prior, st):
    return torch.tensor([list(_scal(A, prior, st, o).lr) for o in range(prior.n_objects)], dtype=torch.float64,
                        device=DEV)


def _hyper(A, kind, wds=WDS, active=0, plateau=0, patience=0, factor=0.5, threshold=1e-4, min_lr=0.0, plateau_eps=1e-8):
    L = A._lib
    k = L.AWB_OPT_ADAM if kind == "adam" else L.AWB_OPT_ADAMAX
    return L.OptHyper(k, 0.9, 0.999, 1e-8, (C.c_float * 4)(*wds), plateau, patience, factor, threshold, min_lr,
                      plateau_eps, active)


def _snap(params, prior, st):
    m, v = _mv(prior, st)
    return params.detach().clone(), m.clone(), v.clone()


# ---------------------------------------------------------------------------------------------------- the reference
def _within(got, ref, tol, mask, what):
    err = (got.double() - ref).abs()
    bad = (err > tol) & mask
    if bool(bad.any()):
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} entries outside the bound, first {idx}: got {float(got[idx])!r}, "
                             f"ref {float(ref[idx])!r}, tol {float(tol[idx]):.3e}")
    return float((err / tol).masked_fill(~mask, 0).max()) if bool(mask.any()) else 0.0


def check_step(hy, lr, own, before, after, group, clamp, g=None, gtol=None, what=""):
    """One optimizer step, per formula.  ``lr`` [O][4] float64 (in force during the step), ``own`` [4] 1-based step
    count of each group at this step, ``before`` / ``after`` (p, m, v) [O][P] fp32.  ``g`` (float64 [O][P]): the
    gradient (weight decay not yet added) with an absolute error bound ``gtol``; None: recovered from the first moment,
    ``g + wd p = m_old + (m_new - m_old) / (1 - beta1)`` (the m formula then only bounds that recovery)."""
    p0, m0, v0 = (t.double() for t in before)
    p1, m1, v1 = after
    m1d, v1d = m1.double(), v1.double()
    b1, b2, eps = hy.beta1, hy.beta2, hy.eps                 # the fp32 values, widened
    grp = group.long()
    on = torch.ones_like(grp, dtype=torch.bool) if hy.active_groups == 0 else ((hy.active_groups >> grp) & 1).bool()
    on = on.expand_as(p0)
    for x0, x1, n in zip(before, after, "pmv"):
        assert torch.equal(x0[~on], x1[~on]), f"{what}: an inactive entry of {n} changed"
    wd = torch.tensor(list(hy.weight_decay), dtype=torch.float64, device=DEV)[grp]
    if g is None:
        ge = m0 + (m1d - m0) / (1.0 - b1)
        getol = 4 * U * (m0.abs() + m1d.abs()) / (1.0 - b1)
    else:
        ge = g + wd * p0
        getol = (gtol if gtol is not None else 0.0) + 2 * U * ge.abs()
        m_ref = m0 + (ge - m0) * (1.0 - b1)
        _within(m1, m_ref, 4 * U * (m0.abs() + ge.abs()) + (1.0 - b1) * getol + 1e-38, on, f"{what} m")
    own_t = torch.tensor(own, dtype=torch.float64, device=DEV)
    ss = (lr / (1.0 - b1 ** own_t))[:, grp]
    bc2s = torch.sqrt(1.0 - b2 ** own_t)[grp]
    if hy.kind == 0:
        v_ref = v0 * b2 + (1.0 - b2) * ge * ge
        _within(v1, v_ref, 6 * U * v_ref + 2 * (1.0 - b2) * ge.abs() * getol + 1e-38, on, f"{what} v")
        delta = ss * m1d / (v1d.sqrt() / bc2s + eps)
    else:
        v_ref = torch.maximum(v0 * b2, ge.abs() + eps)
        _within(v1, v_ref, 4 * U * v_ref + getol, on, f"{what} v")
        delta = ss * m1d / v1d
    p_free = p0 - delta
    cl = clamp.expand_as(p0)
    p_ref = torch.where(cl, p_free.clamp_min(0.0), p_free)
    r = _within(p1, p_ref, 12 * U * delta.abs() + 2 * U * p_ref.abs() + 1e-38, on, f"{what} p")
    return dict(ratio=r, clamped=int((cl & on & (p_free < -1e-3)).sum()))


# ---------------------------------------------------------------------------------------------------- awb_optim_step
OPTIM_CASES = [  # id, kind, C, L, h, O
    ("icnn-L1-tail1", "icnn", 2, 1, _h_with_tail(2, 1, 1), 1),
    ("icnn-L1-full", "icnn", 3, 1, _h_with_tail(3, 1, 0), 1),
    ("icnn-L2", "icnn", 2, 2, 130, 1),
    ("icnn-O3", "icnn", 2, 2, 130, 3),
    ("icnn-O16-tail1", "icnn", 2, 1, _h_with_tail(2, 1, 1), 16),
    ("flow-C2", "flow", 2, 2, 130, 1),
    ("flow-C3", "flow", 3, 2, 130, 1),
    ("flow-C2-O3", "flow", 2, 1, 130, 3),
    ("flow-C3-O16", "flow", 3, 1, 130, 16),
    ("diffeo", "diffeo", 2, 1, 130, 1),
    ("star", "star", 2, 0, 150, 1),
]


@pytest.mark.parametrize("opt", ["adam", "adamax"])
@pytest.mark.parametrize("case", OPTIM_CASES, ids=[c[0] for c in OPTIM_CASES])
def test_optim_step_per_formula(A, case, opt):
    """Caller gradients, different per object; four steps: all groups, one group masked out, all groups again (it rejoins
    with its own step count), then only that group."""
    _, kind, C_, L_, h, O_ = case
    model = _model(A, kind, C_, L_, h)
    group, clamp, _ = _layout(model)
    prior = _handle(A, model, O_)
    P = prior.n_params
    assert group.numel() == P
    if kind == "icnn" and h != 130:
        assert P == _icnn_P(h, C_, L_) and P % 32 in (0, 1)
    gen = torch.Generator(device=DEV).manual_seed(7)
    params = (0.5 * torch.randn(O_, P, device=DEV, generator=gen)).contiguous()
    st = _new_state(A, prior)
    present = sorted(set(group.tolist()))
    off = present[-1]
    masks = [0, 0b1111 & ~(1 << off), 0, 1 << off]
    own = [0, 0, 0, 0]
    clamped = 0
    for k, active in enumerate(masks):
        hy = _hyper(A, opt, active=active)
        for g in range(4):
            if active == 0 or (active >> g) & 1:
                own[g] += 1
        grads = (torch.randn(O_, P, device=DEV, generator=gen) * (1 + torch.arange(O_, device=DEV)[:, None])).contiguous()
        lr = _lrs(A, prior, st)
        before = _snap(params, prior, st)
        A._lib.check(prior.lib.awb_optim_step(prior.handle, params.data_ptr(), grads.data_ptr(), st.data_ptr(),
                                              C.byref(hy), A._lib.stream_ptr()))
        torch.cuda.synchronize()
        res = check_step(hy, lr, own, before, _snap(params, prior, st), group, clamp, g=grads.double(),
                         what=f"step {k}")
        clamped += res["clamped"]
        assert all(_scal(A, prior, st, o).step == k + 1 for o in range(O_))
    assert clamped > 0                                                    # the clamp was exercised


@pytest.mark.parametrize("opt", ["adam", "adamax"])
def test_optim_step_2000_step_trajectory(A, opt):
    """2,000 steps of a flow prior's groups (lr and weight decay per group, the flow group masked out on every 7th step)
    against the float64 oracle: the fp32 state may drift only by rounding, |p - p64| <= 1e-4 (|p64| + |p64 - p_init|)."""
    model = _model(A, "flow", 2, 1, 130)
    group, clamp, _ = _layout(model)
    prior = _handle(A, model, 2)
    P = prior.n_params
    gen = torch.Generator(device=DEV).manual_seed(11)
    params = (0.5 * torch.randn(2, P, device=DEV, generator=gen)).contiguous()
    init = params.double().clone()
    st = _new_state(A, prior)
    p64, m64, v64 = init.clone(), torch.zeros_like(init), torch.zeros_like(init)
    hy_all, hy_mask = _hyper(A, opt), _hyper(A, opt, active=0b1110)
    wd = torch.tensor([float(hy_all.weight_decay[g]) for g in range(4)], dtype=torch.float64, device=DEV)[group]
    lr = torch.tensor(LRS, dtype=torch.float64, device=DEV)[group]
    b1, b2, eps = hy_all.beta1, hy_all.beta2, hy_all.eps
    own = torch.zeros(4, dtype=torch.float64, device=DEV)
    mu = 0.3 * torch.randn(2, P, device=DEV, generator=gen)               # a drift per entry: the parameters travel
    for k in range(2000):
        hy = hy_mask if k % 7 == 6 else hy_all
        on = torch.ones(4, dtype=torch.bool, device=DEV) if hy.active_groups == 0 else \
            torch.tensor([(hy.active_groups >> g) & 1 == 1 for g in range(4)], device=DEV)
        own += on.double()
        grads = (mu + torch.randn(2, P, device=DEV, generator=gen)).contiguous()
        A._lib.check(prior.lib.awb_optim_step(prior.handle, params.data_ptr(), grads.data_ptr(), st.data_ptr(),
                                              C.byref(hy), A._lib.stream_ptr()))
        e = on[group]
        ge = grads.double() + wd * p64                                         # the oracle's arithmetic, vectorised over groups
        m_new = m64 + (ge - m64) * (1 - b1)
        if opt == "adam":
            v_new = v64 * b2 + (1 - b2) * ge * ge
            upd = lr / (1 - b1 ** own[group]) * m_new / (v_new.sqrt() / torch.sqrt(1 - b2 ** own[group]) + eps)
        else:
            v_new = torch.maximum(v64 * b2, ge.abs() + eps)
            upd = lr / (1 - b1 ** own[group]) * m_new / v_new
        p_new = p64 - upd
        p_new = torch.where(clamp & e, p_new.clamp_min(0.0), p_new)
        p64, m64, v64 = (torch.where(e, a, b) for a, b in ((p_new, p64), (m_new, m64), (v_new, v64)))
    torch.cuda.synchronize()
    err = (params.double() - p64).abs()
    bound = 1e-4 * (p64.abs() + (p64 - init).abs()) + 1e-9
    worst = float((err / bound).max())
    print(f"[trajectory {opt}] max |p - p64| = {float(err.max()):.3e}, worst share of the bound {worst:.3f}")
    assert worst <= 1.0
    assert float((p64 - init).abs().max()) > 0.5                           # the parameters really moved


# ---------------------------------------------------------------------------------------------------- awb_prior_rows_opt_step
# dyadic learning rates and losses: every comparison of the scheduler is exact in float64 on both sides
MIN_LR, P_EPS, THR = 2.0 ** -10, 2.0 ** -27, 0.25
ROW_LRS = [2.0 ** -8, 2.0 ** -10 + 2.0 ** -29, 2.0 ** -7, 2.0 ** -9]   # group 1: its reductions are eps-suppressed
SCRIPT = [1.0, 0.75, 0.5, 0.5, 0.5, 0.5, 0.625, 0.5, 0.5, 0.25, 0.25, 0.25, 0.25, float("nan"), 0.25, 0.25]


def _row_losses(total, n):
    """``n`` loss slots that add up to ``total`` exactly in any order (integer multiples of 2^-12)."""
    if math.isnan(total):
        out = [0.0] * n
        out[n // 2] = float("nan")
        return out
    K = int(total * 4096)
    q, r = divmod(K, n)
    return [(q + (i < r)) / 4096.0 for i in range(n)]


@pytest.mark.parametrize("n_rows", [1, 2, 7, 8, 9, 33])
def test_rows_opt_step_per_formula_and_plateau(A, n_rows):
    model = _model(A, "flow", 2, 1, 130)
    group, clamp, _ = _layout(model)
    prior = _handle(A, model, 1)
    P = prior.n_params
    gen = torch.Generator(device=DEV).manual_seed(5)
    params = (0.5 * torch.randn(1, P, device=DEV, generator=gen)).contiguous()
    st = _new_state(A, prior, ROW_LRS)
    hy = _hyper(A, "adam", plateau=1, patience=2, factor=0.5, threshold=THR, min_lr=MIN_LR, plateau_eps=P_EPS)
    ref = O.Plateau(ROW_LRS, patience=2, factor=hy.factor, threshold=hy.threshold, min_lr=hy.min_lr, eps=hy.plateau_eps)
    loss_out = torch.zeros(1, device=DEV)
    steps, seen_nan = 0, False
    for k, total in enumerate(SCRIPT):
        rows = torch.randn(n_rows, P + 1, device=DEV, generator=gen)
        rows[:, P] = torch.tensor(_row_losses(total, n_rows), device=DEV)
        rows = rows.contiguous()
        lr = _lrs(A, prior, st)
        before = _snap(params, prior, st)
        prior.rows_opt_step(params, st, rows, hy, loss_out)
        torch.cuda.synchronize()
        after = _snap(params, prior, st)
        s = _scal(A, prior, st)
        if math.isnan(total):
            seen_nan = True
            for x0, x1 in zip(before, after):
                assert torch.equal(x0, x1)
            assert s.step == steps and s.nonfinite == 1 and math.isnan(s.last_loss) and math.isnan(float(loss_out))
        else:
            steps += 1
            g64 = rows[:, :P].double().sum(0, keepdim=True)
            gtol = 2 * n_rows * U * rows[:, :P].double().abs().sum(0, keepdim=True)
            check_step(hy, lr, [steps] * 4, before, after, group, clamp, g=g64, gtol=gtol, what=f"step {k}")
            ref.step(total)
            assert s.step == steps and s.last_loss == total and float(loss_out) == total
            assert s.nonfinite == int(seen_nan)                          # sticky
        assert list(s.lr) == ref.lrs and s.best == ref.best and s.num_bad == ref.num_bad, (k, list(s.lr), ref.lrs)
    # the script reached what it is there for: three reductions down to min_lr, and the eps-suppressed group
    assert ref.lrs == [MIN_LR, ROW_LRS[1], MIN_LR, MIN_LR]


# ---------------------------------------------------------------------------------------------------- fit step (k_reduce_opt_aug)
def _blob(H, W, o=0):
    yy, xx = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    return torch.sigmoid((torch.sqrt(((xx - 0.45 - 0.01 * o) / 0.25) ** 2 + ((yy - 0.5) / 0.3) ** 2) - 1) / 0.08)


def _fit_setup(A, kind, C_, L_, h, precision, O_, m=32, seed=0):
    models = [_model(A, kind, C_, L_, h, precision, m=m, seed=seed + o).to(DEV) for o in range(O_)]
    group, clamp, names = _layout(models[0])
    prior = _handle(A, models[0], O_)
    params = torch.stack([mm._ensure_flat().detach() for mm in models]).contiguous().clone()
    assert params.shape[1] == prior.n_params == group.numel()
    return models, prior, params, group, clamp, names


def _fit_step(A, prior, params, st, spec, target, hy, ws, flags=0, loss_out=None):
    L = A._lib
    O_ = prior.n_objects
    specs = (L.LossSpec * O_)(*[L.LossSpec(L.AWB_LOSS_SE_SIGMOID, L.AWB_CLS_UNARY_LT_HALF, 1.0 / spec.n_pixels,
                                           1.0 / spec.n_pixels)] * O_)
    gs = spec.to_c()
    L.check(prior.lib.awb_prior_fit_step(prior.handle, params.data_ptr(), st.data_ptr(), C.byref(gs), target.data_ptr(),
                                         specs, C.byref(hy), loss_out.data_ptr() if loss_out is not None else None,
                                         ws.data_ptr(), ws.numel(), flags, L.stream_ptr()))


def _aug_blocks(h, C_, L_):
    ld = _round_up(h + C_ + 1, 8)
    return 4 * h + L_ * h * ld + ld


FIT_CASES = [  # id, kind, C, L, h, precision, O, flow hidden m
    ("icnn-fp32-Gfull", "icnn", 2, 1, next(h for h in range(8, 200) if _aug_blocks(h, 2, 1) % 128 == 0), "fp32", 1, 32),
    ("icnn-fp32-O16", "icnn", 2, 2, 130, "fp32", 16, 32),
    ("icnn-f16-L1", "icnn", 2, 1, 130, "f16", 1, 32),
    ("icnn-f16-L2-O16", "icnn", 3, 2, 130, "f16", 16, 32),
    ("flow-fp32-PFfull", "flow", 2, 1, 130, "fp32", 1, 29),
    ("flow-fp32-O16", "flow", 3, 1, 130, "fp32", 16, 32),
    ("flow-f16", "flow", 2, 2, 130, "f16", 1, 32),
    ("flow-f16-O16-PFfull", "flow", 2, 1, 130, "f16", 16, 29),
    ("diffeo", "diffeo", 2, 1, 130, "fp32", 1, 32),
]


@pytest.mark.parametrize("opt", ["adam", "adamax"])
@pytest.mark.parametrize("case", FIT_CASES, ids=[c[0] for c in FIT_CASES])
def test_fit_step_per_formula(A, case, opt):
    """Two fused fit steps.  The gradient is formed inside the kernel: it is taken back from the first moment, v and p
    are checked per formula with it, and (single-object exact fp32 handles) compared per tensor with ``awb_prior_backward``."""
    _, kind, C_, L_, h, precision, O_, m = case
    models, prior, params, group, clamp, names = _fit_setup(A, kind, C_, L_, h, precision, O_, m)
    P = prior.n_params
    if kind == "icnn" and precision == "fp32" and O_ == 1:
        assert _aug_blocks(h, C_, L_) % 128 == 0
    if kind == "flow" and m == 29:
        assert (P - _icnn_P(h, C_, L_)) % 128 == 0                       # flow + linear parameters: whole 128-blocks
    H, W = 37, 45
    spec = A.GridSpecHost("linspace", 1, H, W, t0=0.1, t_step=0.2)
    target = torch.stack([_blob(H, W, o).reshape(-1) for o in range(O_)]).to(DEV).contiguous()
    st = _new_state(A, prior)
    ws = prior.new_workspace(spec.n_pixels, A._lib.AWB_WS_FIT_STEP, DEV)
    hy = _hyper(A, opt)
    for k in range(2):
        lr = _lrs(A, prior, st)
        before = _snap(params, prior, st)
        _fit_step(A, prior, params, st, spec, target, hy, ws, flags=A._lib.AWB_FIT_REUSE_PACKED if k else 0)
        torch.cuda.synchronize()
        after = _snap(params, prior, st)
        check_step(hy, lr, [k + 1] * 4, before, after, group, clamp, what=f"step {k}")
        if k == 0 and O_ == 1 and precision == "fp32":
            # the gradient the kernel used, per tensor, against awb_prior_backward at the same parameters
            p0, m0 = before[0].double(), before[1].double()
            wd = torch.tensor(list(hy.weight_decay), dtype=torch.float64, device=DEV)[group.long()]
            g_k = (m0 + (after[1].double() - m0) / (1 - hy.beta1)) - wd * p0
            wsb = prior.new_workspace(spec.n_pixels, A._lib.AWB_WS_TRAINING, DEV)
            logits, _ = prior.forward(before[0], spec, A._lib.AWB_FWD_EXACT_TRAINING, wsb)
            s = torch.sigmoid(logits.double())
            dlog = (2.0 * (s - target.double()) * s * (1 - s) / spec.n_pixels).float().contiguous()
            g_b, _ = prior.backward(before[0], spec, dlog, wsb, False)
            # summation order only (a misrouted column is off by O(1)); a tensor whose gradient is a sum of cancelling
            # terms (the weight-norm gains) is measured against a tenth of its group's largest entry
            tol = 1e-3
            grp0 = group.clone().masked_fill(group == 3, 0)
            off = 0
            for n, cnt in names:
                a, b = g_k[0, off:off + cnt], g_b[0, off:off + cnt].double()
                block = g_b[0][grp0 == grp0[off]].double()
                scale = max(float(b.abs().max()), 0.1 * float(block.abs().max()), 1e-12)
                assert float((a - b).abs().max()) <= tol * scale, f"{n}: {float((a - b).abs().max()) / scale:.3e}"
                off += cnt
    assert _scal(A, prior, st).step == 2


# ---------------------------------------------------------------------------------------------------- defect 1 and 2
@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_flow_identity_then_fit_bias_corrects_each_group_from_its_own_step(A, precision):
    """k steps of ``awb_flow_identity_step`` (flow group only), then the main fit on the same state: the ICNN and linear
    groups take their first step with bias correction 1, the flow group its (k+1)-th -- in ``awb_prior_fit_step``
    (k_reduce_opt_aug) exactly as in ``awb_prior_rows_opt_step`` (k_reduce_opt) on a copy of the same state."""
    k = 5
    models, prior, params, group, clamp, names = _fit_setup(A, "flow", 2, 1, 130, precision, 1)
    H, W = 30, 41
    spec = A.GridSpecHost("linspace", 1, H, W)
    target = _blob(H, W).reshape(1, -1).to(DEV).contiguous()
    st = _new_state(A, prior)
    wsi = prior.new_workspace(spec.n_pixels, A._lib.AWB_WS_TRAINING, DEV)
    hy = _hyper(A, "adamax")
    gs = spec.to_c()
    for _ in range(k):
        A._lib.check(prior.lib.awb_flow_identity_step(prior.handle, params.data_ptr(), st.data_ptr(), C.byref(gs),
                                                      C.byref(hy), None, wsi.data_ptr(), wsi.numel(),
                                                      A._lib.stream_ptr()))
    torch.cuda.synchronize()
    assert _scal(A, prior, st).step == k
    own = [k + 1, 1, 1, 1]
    lr = _lrs(A, prior, st)
    # rows path on a copy: the gradient row of the whole batch
    p_rows, st_rows = params.clone(), st.clone()
    row = torch.empty(1, prior.grad_row_floats, device=DEV)
    prior.slice_grads(p_rows, spec, 0, spec.n_pixels, target.reshape(-1),
                      A._lib.LossSpec(A._lib.AWB_LOSS_SE_SIGMOID, A._lib.AWB_CLS_UNARY_LT_HALF, 1.0 / spec.n_pixels,
                                      1.0 / spec.n_pixels), row[0],
                      prior.new_workspace(spec.n_pixels, A._lib.AWB_WS_FIT_STEP, DEV))
    before = _snap(p_rows, prior, st_rows)
    prior.rows_opt_step(p_rows, st_rows, row, hy)
    torch.cuda.synchronize()
    check_step(hy, lr, own, before, _snap(p_rows, prior, st_rows), group, clamp, g=row[:, :-1].double(), what="rows")
    # fused fit step (k_reduce_opt_aug) on the original
    before = _snap(params, prior, st)
    _fit_step(A, prior, params, st, spec, target, hy, prior.new_workspace(spec.n_pixels, A._lib.AWB_WS_FIT_STEP, DEV))
    torch.cuda.synchronize()
    check_step(hy, lr, own, before, _snap(params, prior, st), group, clamp, what="fit_step")


def test_star_offset_toggled_off_and_on_keeps_its_step_count(A):
    """``StarFitter.train_offset`` on, off, on (active_groups 0b110 -> 0b010 -> 0b110): the offset group rejoins with its
    own step count 2, not a restarted 1 (torch does not advance the step of a parameter whose grad is None)."""
    torch.manual_seed(2)
    model = A.StarShapedNet(150).to(DEV)
    group, clamp, _ = _layout(model)
    f = model.make_fitter(optim=A.OptimConfig("adam", lr=[0.0, 1e-2, 3e-2, 0.0], weight_decay=[0.0, 1e-3, 1e-2, 0.0]))
    prior, params, st = f.prior, f.arena.view(1, -1), f.opt_state
    x = torch.rand(400, 2, device=DEV) - 0.5
    t = (x.norm(dim=1) < 0.3).float()
    own = [0, 0, 0, 0]
    for k, on in enumerate([True, False, True, True]):
        f.train_offset = on
        own[1] += 1
        own[2] += int(on)
        hy = f.optim.to_c()
        hy.active_groups = 0b110 if on else 0b010
        lr = _lrs(A, prior, st)
        before = _snap(params, prior, st)
        f.step(x, t)
        torch.cuda.synchronize()
        check_step(hy, lr, list(own), before, _snap(params, prior, st), group, clamp, what=f"step {k}")


# ---------------------------------------------------------------------------------------------------- awb_opt_plateau_step
@pytest.mark.parametrize("stride", [1, 0])
def test_plateau_step_per_object(A, stride):
    model = _model(A, "icnn", 2, 1, 130)
    prior = _handle(A, model, 16)
    st = _new_state(A, prior, ROW_LRS)
    hy = _hyper(A, "adam", plateau=1, patience=1, factor=0.5, threshold=THR, min_lr=MIN_LR, plateau_eps=P_EPS)
    refs = [O.Plateau(ROW_LRS, patience=1, factor=hy.factor, threshold=hy.threshold, min_lr=hy.min_lr,
                      eps=hy.plateau_eps) for _ in range(16)]
    m0, v0 = (t.clone() for t in _mv(prior, st))
    for k in range(8):
        if stride:
            losses = [1.0 / (1 + (k if o % 3 else k // 3)) * (1 + o / 16) for o in range(16)]
            if k == 5:
                losses[4] = float("inf")
        else:
            losses = [1.0 if k == 0 else 0.5 if k == 1 else 0.45] * 16
        dl = torch.tensor(losses, device=DEV, dtype=torch.float32)
        A._lib.check(prior.lib.awb_opt_plateau_step(prior.handle, st.data_ptr(), dl.data_ptr(), stride, C.byref(hy),
                                                    A._lib.stream_ptr()))
        for o in range(16):
            lo = float(dl[o if stride else 0])
            if math.isfinite(lo):
                refs[o].step(lo)
            s = _scal(A, prior, st, o)
            assert list(s.lr) == refs[o].lrs and s.best == refs[o].best and s.num_bad == refs[o].num_bad, (k, o)
            assert s.step == 0 and s.nonfinite == int(stride == 1 and o == 4 and k >= 5)
    assert len({tuple(r.lrs) for r in refs}) > 1 if stride else len({tuple(r.lrs) for r in refs}) == 1
    assert any(r.lrs != ROW_LRS for r in refs)
    m1, v1 = _mv(prior, st)
    assert torch.equal(m0, m1) and torch.equal(v0, v1)


# ---------------------------------------------------------------------------------------------------- tensor-path weight image
@pytest.mark.parametrize("kind,L_,O_", [("icnn", 1, 1), ("icnn", 2, 16), ("icnn", 2, 1), ("flow", 1, 16), ("flow", 2, 1)])
def test_reused_weight_image_matches_a_fresh_pack(A, kind, L_, O_):
    """f16 handles, plateau on: ``awb_prior_fit_steps(8)`` (the optimizer's in-place update of the fp16 weight image is
    reused from step to step) against 8 ``awb_prior_fit_step(flags = 0)`` calls (repacked every step).  Parameters, the
    whole optimizer blob and every step's loss must be bit-identical."""
    L = A._lib
    models, prior, params, group, clamp, names = _fit_setup(A, kind, 2, L_, 130, "f16", O_)
    H, W = 40, 52
    spec = A.GridSpecHost("linspace", 1, H, W)
    targets = [torch.stack([_blob(H, W, o + 3 * s).reshape(-1) for o in range(O_)]).to(DEV).contiguous() for s in range(3)]
    hy = _hyper(A, "adamax", plateau=1, patience=1, threshold=0.5)
    specs = (L.LossSpec * O_)(*[L.LossSpec(L.AWB_LOSS_SE_SIGMOID, L.AWB_CLS_UNARY_LT_HALF, 1.0 / spec.n_pixels,
                                           1.0 / spec.n_pixels)] * O_)
    gs = spec.to_c()
    p_a, st_a = params.clone(), _new_state(A, prior)
    p_b, st_b = params.clone(), st_a.clone()
    ws_a, ws_b = (prior.new_workspace(spec.n_pixels, L.AWB_WS_FIT_STEP, DEV) for _ in range(2))
    loss_a = torch.zeros(8, O_, device=DEV)
    loss_b = torch.zeros(8, O_, device=DEV)
    ptrs = (C.c_void_p * 3)(*[t.data_ptr() for t in targets])
    L.check(prior.lib.awb_prior_fit_steps(prior.handle, p_a.data_ptr(), st_a.data_ptr(), C.byref(gs), ptrs, 3, 0, 8, specs,
                                          C.byref(hy), loss_a.data_ptr(), ws_a.data_ptr(), ws_a.numel(), 0, L.stream_ptr()))
    for s in range(8):
        _fit_step(A, prior, p_b, st_b, spec, targets[s % 3], hy, ws_b, flags=0, loss_out=loss_b[s])
    torch.cuda.synchronize()
    assert torch.equal(loss_a, loss_b)
    assert torch.equal(p_a, p_b)
    assert torch.equal(st_a, st_b)
    assert not torch.equal(p_a, params)
    s = _scal(A, prior, st_a)
    assert s.step == 8 and s.lr[1] < LRS[1]                           # the plateau reduced the lr along the way
