"""Gradient penalties through the ICNN priors (``second_order=True``) against a float64 reference.

A penalty on ``g = d prior / d grid`` (built with ``create_graph=True``) is trained through
``awb_prior_grid_grad_backward``: the gradient ``u`` on ``g`` becomes ``ydot = J u`` on the upstream gradient ``w`` of the
first backward and ``sum_n w_n d(J_n u_n) / d params`` on the parameters; the grid receives only the first-order part.
The reference is ``oracle/prior_oracle.py`` run in float64 on the GPU with torch autograd (``create_graph=True``, then
``.backward()``), as in ``test_gpu_coord_grad.py``, whose kink exclusion is reused: ``w`` and ``u`` are 0 at the pixels
whose ReLU input is within KINK of zero (the masks of the second-order terms are those of the forward, and a pixel on a
kink can take the other side in fp32).  The sizes sit on both sides of the ``n_splits`` branch restated in
``test_gpu_launch_regimes.py``: a few hundred rows, 37 889 rows (one more than 148 ranges of 256) and the 640x480 frame."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as Fn

import __graft_entry__ as entry
from oracle import prior_oracle as O
from test_gpu_coord_grad import CHUNK, KINK_MAX_FRACTION, _KinkProbe, make_flow
from test_gpu_launch_regimes import entry_err, n_splits, torch_grid

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Parameter gradients of the penalised loss, ydot and x.grad on the exact path, per entry relative to the tensor's largest
# float64 entry: the TOL_GRAD of test_gpu_launch_regimes.py.  Calibrated on the 640x480 frame (case ``calib``).
TOL_MEASURED = 1.6e-6      # calib, worst tensor (skip.1.ln.bias), one B200 at a 1000 W power limit
TOL = 5e-4
TC_TOL = 2e-2                 # f16 modules, normwise per tensor (with a floor): the flow bound of DESIGN section 4
LAM = 0.1


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


def make(A, kind, C_, h, L, precision="fp32", second_order=True, seed=0):
    torch.manual_seed(seed)
    if kind == "convexnet":
        m = A.ConvexNet(n_hidden=h, in_channels=C_, precision=precision, second_order=second_order)
    else:
        m = A.ConvexNextNet(n_hidden=h, in_features=C_, n_hidden_layers=L, precision=precision, second_order=second_order)
    return m.to(DEV)


def forward64(kind):
    return O.convexnet_forward if kind == "convexnet" else O.icnn_forward


def p64(m):
    return {k: v.detach().to(DEV, torch.float64).clone().requires_grad_(True) for k, v in m.state_dict().items()}


def rows_of(x4):
    return x4.permute(0, 2, 3, 1).reshape(-1, x4.shape[1])


def kink_mask(kind, m, rows):
    """Float ``[N]``: 0 at the pixel rows within KINK of a ReLU kink of the float64 forward, 1 elsewhere."""
    p = {k: v.detach() for k, v in p64(m).items()}
    near = torch.zeros(rows.shape[0], dtype=torch.bool, device=DEV)
    saved = O.F
    try:
        for a in range(0, rows.shape[0], CHUNK):
            O.F = probe = _KinkProbe(min(CHUNK, rows.shape[0] - a))
            with torch.no_grad():
                forward64(kind)(p, rows[a:a + CHUNK].double())
            near[a:a + CHUNK] = probe.near
    finally:
        O.F = saved
    frac = float(near.float().mean())
    assert frac <= KINK_MAX_FRACTION, frac
    return (~near).float(), frac


def penalised(y, x, pen, mask, wt, v, t):
    """First-order term + LAM * penalty on g = d inner / d x.  Channel dim 1 in both layouts ([B,C,H,W] and [N,C])."""
    if pen == "bce":
        inner = (mask * Fn.binary_cross_entropy_with_logits(y, t, reduction="none")).sum()
    else:
        inner = (wt * y).sum()
    g = torch.autograd.grad(inner, x, create_graph=True)[0]
    if pen == "eikonal":
        p = (mask * ((g.pow(2).sum(1, keepdim=True) + 1e-12).sqrt() - 1).pow(2)).sum()
    else:
        p = (mask * g).pow(2).sum()
    return (mask * v * y).sum() + LAM * p


def inputs(case, N, mask):
    g = torch.Generator(device=DEV).manual_seed(11)
    wt = torch.randn(N, device=DEV, generator=g) * mask
    v = torch.randn(N, device=DEV, generator=g)
    t = torch.rand(N, device=DEV, generator=g)
    return wt, v, t


def reference(case, m, rows, mask, wt, v, t):
    """float64 gradients of the penalised loss w.r.t. the parameters, the rows and wt, chunk by chunk."""
    p = p64(m)
    fwd = forward64(case["kind"])
    dx = torch.empty(rows.shape, dtype=torch.float64, device=DEV)
    dw = torch.empty(rows.shape[0], dtype=torch.float64, device=DEV)
    for a in range(0, rows.shape[0], CHUNK):
        s = slice(a, a + CHUNK)
        r = rows[s].double().requires_grad_(True)
        w = wt[s].double().reshape(-1, 1).requires_grad_(True)
        y = fwd(p, r)
        loss = penalised(y, r, case["pen"], mask[s].double().reshape(-1, 1), w, v[s].double().reshape(-1, 1),
                         t[s].double().reshape(-1, 1))
        loss.backward()
        dx[s] = r.grad
        if w.grad is not None:          # not for bce, whose w is a function of the logits
            dw[s] = w.grad.reshape(-1)
    return {k: q.grad for k, q in p.items()}, dx, dw


def module_run(m, x4, rows_input, case, mask, wt, v, t):
    """The penalised step through the module: parameter gradients, x.grad and wt.grad (= ydot for sq / eikonal)."""
    x0 = rows_of(x4) if rows_input else x4
    x = x0.clone().requires_grad_(True)
    m.zero_grad()
    y = m(x)
    shp = y.shape
    w = wt.reshape(shp).clone().requires_grad_(True)
    penalised(y, x, case["pen"], mask.reshape(shp), w, v.reshape(shp), t.reshape(shp)).backward()
    grads = {k: q.grad.clone() for k, q in m.named_parameters()}
    dx = x.grad if rows_input else rows_of(x.grad)
    return grads, dx, (w.grad.reshape(-1) if w.grad is not None else None)


def _c(id_, kind, C_, h, L, B, H, W, pen, rows=False):
    return dict(id=id_, kind=kind, C=C_, h=h, L=L, B=B, H=H, W=W, pen=pen, rows=rows)


EXACT = [
    _c("calib", "icnn", 2, 130, 2, 1, 480, 640, "sq"),
    _c("calib-bce", "icnn", 2, 130, 2, 1, 480, 640, "bce"),
    _c("L1-c2-n300-rows", "icnn", 2, 130, 1, 1, 1, 300, "sq", rows=True),
    _c("L1-c3-n37889-eik", "icnn", 3, 130, 1, 1, 1, 37889, "eikonal", rows=True),
    _c("L2-c3-b2-bce", "icnn", 3, 130, 2, 2, 96, 160, "bce"),
    _c("L3-c2-n37889-bce-rows", "icnn", 2, 130, 3, 1, 1, 37889, "bce", rows=True),
    _c("L3-c3-n257-eik", "icnn", 3, 130, 3, 1, 1, 257, "eikonal"),
    _c("h37-L2-c2-b2-eik", "icnn", 2, 37, 2, 2, 120, 160, "eikonal"),
    _c("h37-L3-c3-calib-bce", "icnn", 3, 37, 3, 1, 480, 640, "bce"),
    _c("convexnet-bce", "convexnet", 2, 130, 1, 1, 240, 320, "bce"),
    _c("convexnet-rows-sq", "convexnet", 2, 130, 1, 1, 1, 37888, "sq", rows=True),
]


@pytest.mark.parametrize("case", EXACT, ids=[c["id"] for c in EXACT])
def test_penalty_exact_path_against_float64(A, case):
    m = make(A, case["kind"], case["C"], case["h"], case["L"], seed=1)
    x4 = torch_grid("linspace", case["B"], case["H"], case["W"], case["C"])
    rows = rows_of(x4)
    N = rows.shape[0]
    mask, frac = kink_mask(case["kind"], m, rows)
    wt, v, t = inputs(case, N, mask)
    grads, dx, dw = module_run(m, x4, case["rows"], case, mask, wt, v, t)
    ref, dx64, dw64 = reference(case, m, rows, mask, wt, v, t)
    errs = {k: entry_err(grads[k], ref[k]) for k in grads if float(ref[k].abs().max()) > 0}
    worst = max(errs, key=errs.get)
    err_x = entry_err(dx, dx64)
    line = (f"[second-order {case['id']}] N={N} S={n_splits(N)}: parameters {errs[worst]:.2e} ({worst})  x.grad "
            f"{err_x:.2e}")
    if case["pen"] != "bce":
        err_y = entry_err(dw, dw64)
        line += f"  ydot {err_y:.2e}"
        assert err_y <= TOL, err_y
    print(line + f"  kink pixels {frac:.2%}")
    assert errs[worst] <= TOL, errs
    assert err_x <= TOL, err_x


@pytest.mark.parametrize("pen", ["sq", "bce"])
def test_penalty_f16_module_against_float64(A, pen):
    """f16 modules: first order on the tensor path, the second-order pass on the exact kernels."""
    case = _c("f16", "icnn", 2, 130, 2, 1, 480, 640, pen)
    m = make(A, "icnn", 2, 130, 2, precision="f16", seed=2)
    x4 = torch_grid("linspace", 1, 480, 640, 2)
    rows = rows_of(x4)
    mask, frac = kink_mask("icnn", m, rows)
    wt, v, t = inputs(case, rows.shape[0], mask)
    grads, dx, _ = module_run(m, x4, False, case, mask, wt, v, t)
    ref, dx64, _ = reference(case, m, rows, mask, wt, v, t)
    # each tensor against the larger of its own norm and a tenth of the block's, as the flow gradients of
    # test_gpu_launch_regimes.py: a bias whose pixel sum cancels carries the tensor path's first-order error on a small norm
    block = float(torch.cat([r.reshape(-1) for r in ref.values()]).norm())
    errs = {k: float((grads[k].double() - ref[k]).norm()) / max(float(ref[k].norm()), 0.1 * block) for k in grads}
    worst = max(errs, key=errs.get)
    err_x = float((dx.double() - dx64).norm() / dx64.norm())
    print(f"[second-order f16 {pen}] parameters normwise {errs[worst]:.2e} ({worst})  x.grad {err_x:.2e}  "
          f"kink pixels {frac:.2%}")
    assert errs[worst] <= TC_TOL, errs
    assert err_x <= TC_TOL, err_x


# -------------------------------------------------------------------------------------------------------- properties
def _pen_only(m, x4, w):
    x = x4.clone().requires_grad_(True)
    g = torch.autograd.grad((w * m(x)).sum(), x, create_graph=True)[0]
    return g.pow(2).sum()


def test_exact_properties(A):
    """Penalty-only loss: every bias gradient exactly 0; two runs and a second backward on a retained graph give the same
    bits."""
    m = make(A, "icnn", 2, 130, 2, seed=3)
    x4 = torch_grid("linspace", 1, 240, 320, 2)
    w = torch.randn(1, 1, 240, 320, device=DEV, generator=torch.Generator(device=DEV).manual_seed(4))

    def grads():
        return torch.cat([q.grad.reshape(-1) for q in m.parameters()]).clone()

    m.zero_grad()
    pen = _pen_only(m, x4, w)
    pen.backward(retain_graph=True)
    g1 = grads()
    for k, q in m.named_parameters():
        if k.endswith("bias"):
            assert int(torch.count_nonzero(q.grad)) == 0, k
        else:
            assert float(q.grad.abs().max()) > 0, k
    m.zero_grad()
    pen.backward()
    assert torch.equal(grads(), g1)
    m.zero_grad()
    _pen_only(m, x4, w).backward()
    assert torch.equal(grads(), g1)


@pytest.mark.parametrize("precision", ["fp32", "f16"])
def test_first_order_bits_do_not_depend_on_the_flag(A, precision):
    """Logits, first-order parameter gradients and dgrid are the same bits with and without second_order, also when the
    first backward builds a graph."""
    ms = [make(A, "icnn", 2, 130, 2, precision=precision, second_order=s, seed=5) for s in (False, True)]
    x4 = torch_grid("linspace", 2, 96, 160, 2)
    w = torch.randn(2, 1, 96, 160, device=DEV, generator=torch.Generator(device=DEV).manual_seed(6))
    out = []
    for m in ms:
        with torch.no_grad():
            y0 = m(x4)
        x = x4.clone().requires_grad_(True)
        y = m(x)
        first = torch.autograd.grad((w * y).sum(), [x] + list(m.parameters()))
        x = x4.clone().requires_grad_(True)
        graph = torch.autograd.grad((w * m(x)).sum(), [x] + list(m.parameters()), create_graph=True)
        out.append([y0, y.detach()] + [g.detach() for g in first] + [g.detach() for g in graph])
    for a, b in zip(*out):
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------------------ errors
def test_penalty_on_parameter_gradients_raises(A):
    m = make(A, "icnn", 2, 130, 2, seed=7)
    x = torch_grid("linspace", 1, 32, 48, 2).requires_grad_(True)
    gs = torch.autograd.grad(m(x).sum(), list(m.parameters()) + [x], create_graph=True)
    with pytest.raises(RuntimeError, match="parameter gradients"):
        gs[0].pow(2).sum().backward()


def test_c_abi_errors(A):
    L = A._lib
    lib = L.load()
    spec = A.GridSpecHost("linspace", 1, 24, 32)
    N = spec.n_pixels
    gs = spec.to_c()
    d_dgrid = torch.randn(1, 2, 24, 32, device=DEV)
    dl = torch.zeros(2, N, device=DEV)
    ydot = torch.empty(2, N, device=DEV)

    def rc(prior, params, ws):
        grads = torch.empty(params.numel(), device=DEV)
        return lib.awb_prior_grid_grad_backward(prior.handle, params.data_ptr(), C.byref(gs), dl.data_ptr(),
                                                d_dgrid.data_ptr(), ydot.data_ptr(), grads.data_ptr(), ws.data_ptr(),
                                                ws.numel(), L.stream_ptr())

    big = torch.empty(1 << 26, dtype=torch.uint8, device=DEV)
    flow = make_flow(A, 2, 4, "fp32", 1, seed=50)
    assert rc(flow._prior_for(torch.device(DEV)), flow._ensure_flat(), big) == -2
    assert b"ICNN" in lib.awb_last_error()
    grouped = A.Prior(L.AWB_KIND_ICNN, 2, 130, 2, n_objects=2)
    assert rc(grouped, torch.zeros(2, grouped.n_params, device=DEV), big) == -2
    star = A.Prior(L.AWB_KIND_STAR, 2, 32, 0)
    assert rc(star, torch.zeros(star.n_params, device=DEV), big) == -2
    for precision in ("fp32", "f16"):
        prior = A.Prior(L.AWB_KIND_ICNN, 2, 130, 2, precision=L.AWB_PREC_FP32 if precision == "fp32" else L.AWB_PREC_F16)
        params = make(A, "icnn", 2, 130, 2, seed=8)._ensure_flat()
        need = prior.workspace_bytes(N, L.AWB_WS_SECOND_ORDER)
        assert need > prior.workspace_bytes(N, L.AWB_WS_TRAINING)
        ws = torch.empty(need, dtype=torch.uint8, device=DEV)
        prior.forward(params, spec, L.AWB_FWD_EXACT_TRAINING, ws)
        assert rc(prior, params, torch.empty(need - 1, dtype=torch.uint8, device=DEV)) == -4
        assert rc(prior, params, ws) == 0
    torch.cuda.synchronize()
