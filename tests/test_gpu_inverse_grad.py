"""Gradients of ``PathConnectedNet.inverse`` against a float64 reference.

``inverse(x)`` maps points back through the flow (MinMax, the flows inverted in reverse order, inverse MinMax, inverse
1x1 conv).  With grad mode on it runs ``awb_prior_inverse(training)`` and ``awb_prior_inverse_backward`` (``k_flow_inv_rec``,
``k_flow_inv_bwd``): gradients w.r.t. the flow and 1x1-conv parameters and the input points.

The reference is the oracle's inverse chain (as in ``test_gpu_flow.py::test_inverse_undoes_get_deformation``) in float64
with torch autograd; with MeanStd buffers or an output scale the same chain restated with ``(x - mean) / std`` and
``s, t = scale * tanh(MLP)``.  The upstream gradient is 0 on the pixels within KINK of a ReLU kink of the coupling MLPs as
the inverse evaluates them (``test_gpu_coord_grad.py``), and TOL_GRAD / TOL_DGRID are that file's.  Which backward variant
every case hits is named through ``flow_bwd_geometry``: the inverse backward shares the unit-loop kernel's geometry."""
import ctypes as C

import pytest
import torch

import __graft_entry__ as entry
from oracle import prior_oracle as O
from test_gpu_coord_grad import CHUNK, TOL_DGRID, TOL_GRAD, _KinkProbe, p64, randomize_linear, rows_of
from test_gpu_launch_regimes import entry_err, flow_bwd_geometry, torch_grid

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KINK_MAX_FRACTION = 0.05


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


def make_flow(A, C_, F, hidden=32, output_fn="tanh", scale=None, norm="minmax", precision="fp32", seed=0,
              spatial=(1000, 1000)):
    """RealNVP prior with non-trivial couplings, initialised ActNorms and a random 1x1 conv."""
    torch.manual_seed(seed)
    m = A.real_nvp_path_connected_net(channels=C_, hidden_units=hidden, flow_n_flows=F, flow_output_fn=output_fn,
                                      flow_output_scale=scale, norm=norm, spatial_shape=spatial,
                                      convex_net_hidden_units=130, convex_net_hidden_layers=2, precision=precision)
    sd = m.state_dict()
    for k in sd:
        if ".net.2." in k:
            sd[k] = 0.05 * torch.randn_like(sd[k])
        elif k.endswith((".s", ".t")) and ".flows." in k:
            sd[k] = 0.1 * torch.randn_like(sd[k])
        elif k.endswith("data_dep_init_done"):
            sd[k] = torch.ones_like(sd[k])
    m.load_state_dict(sd)
    randomize_linear(m, seed + 1)
    return m.to(DEV)


def inverse64(p, x4, output_fn="tanh", scale=None):
    """float64 ``PathConnectedNet.inverse`` of ``x4`` ``[B, C, H, W]``: pixel rows ``[N, C]``."""
    B, C_, H, W = x4.shape
    if "flow_net.norm.mean" in p:
        mean, std = p["flow_net.norm.mean"], p["flow_net.norm.std"]
        z = O.pixelize((x4 - mean) / std)
    else:
        mn, mx, nmn, nmx = (p["flow_net.norm." + k] for k in ("min", "max", "new_min", "new_max"))
        z = O.pixelize(O.minmax(x4, mn, mx, nmn, nmx))
    sc = 1.0 if scale is None else scale
    pre = O.FLOW_PREFIX
    for f in range(O.flow_num(p, pre) - 1, -1, -1):
        a, n = f"{pre}flows.{2 * f}.", f"{pre}flows.{2 * f + 1}."
        z = (z - p[n + "t"]) * torch.exp(-p[n + "s"])
        b = p[a + "b"].to(z.dtype)
        zm = b * z
        s = sc * O._mlp(p, a + "s.", zm, output_fn)
        t = sc * O._mlp(p, a + "t.", zm, output_fn)
        z = zm + (1 - b) * (z - t) * torch.exp(-s)
    z = O.unpixelize(z, B, H, W)
    if "flow_net.norm.mean" in p:
        z = z * std + mean
    else:
        z = O.minmax(z, nmn, nmx, mn, mx)
    z = (z - p["linear.bias"].view(1, C_, 1, 1)) / p["linear.weight"].view(1, C_, 1, 1)
    return O.pixelize(z)


def rows4(rows):
    """Pixel rows ``[n, C]`` as the ``[1, C, 1, n]`` grid the reference takes (every pixel's result depends on its row)."""
    return rows.t().reshape(1, rows.shape[1], 1, rows.shape[0])


def away_from_kinks(m, rows, w4, output_fn, scale):
    """``w4`` with the upstream gradient of the pixels near a coupling-MLP kink of the inverse set to 0, and their fraction."""
    p = p64(m)
    near = torch.zeros(rows.shape[0], dtype=torch.bool, device=DEV)
    saved = O.F
    try:
        for a in range(0, rows.shape[0], CHUNK):
            O.F = probe = _KinkProbe(min(CHUNK, rows.shape[0] - a))
            with torch.no_grad():
                inverse64(p, rows4(rows[a:a + CHUNK].double()), output_fn, scale)
            near[a:a + CHUNK] = probe.near
    finally:
        O.F = saved
    frac = float(near.float().mean())
    assert frac <= KINK_MAX_FRACTION, frac
    B, C_, H, W = w4.shape
    w = rows_of(w4).clone()
    w[near] = 0
    return w.reshape(B, H, W, C_).permute(0, 3, 1, 2).contiguous(), frac


def ref_inverse_grads(m, rows, w_rows, output_fn, scale):
    """float64 gradients of sum(w * inverse(rows)) w.r.t. the flow / linear parameters and the rows."""
    keys = [k for k, _ in m.named_parameters() if not k.startswith("convex_net.")]
    p = p64(m, keys)
    grads = {k: torch.zeros_like(p[k]) for k in keys}
    dx = torch.empty(rows.shape, dtype=torch.float64, device=DEV)
    for a in range(0, rows.shape[0], CHUNK):
        r = rows[a:a + CHUNK].double().requires_grad_(True)
        loss = (w_rows[a:a + CHUNK].double() * inverse64(p, rows4(r), output_fn, scale)).sum()
        gs = torch.autograd.grad(loss, [p[k] for k in keys] + [r])
        for k, g in zip(keys, gs[:-1]):
            grads[k] += g
        dx[a:a + CHUNK] = gs[-1]
    return grads, dx


# ------------------------------------------------------------------------------------------------------------ cases
def _c(id_, C_, F, B, H, W, kernel_extra, hidden=32, output_fn="tanh", scale=None, norm="minmax", precision="fp32"):
    return dict(id=id_, C=C_, F=F, B=B, H=H, W=W, extra=kernel_extra, hidden=hidden, output_fn=output_fn, scale=scale,
                norm=norm, precision=precision)


CASES = [
    _c("c2-n1", 2, 4, 1, 1, 1, {"S": 1, "T": 32, "R": 0}, hidden=8),
    _c("c2-n37-none", 2, 4, 1, 1, 37, {"S": 1, "T": 64, "R": 0}, hidden=8, output_fn=None),
    _c("c2-b3", 2, 12, 3, 24, 32, {"S": 9, "T": 256, "R": 0, "rounds1": 1}),
    _c("c2-meanstd-scale", 2, 12, 1, 96, 128, {"dz_smem": True}, norm="meanstd", scale=0.5),
    _c("c2-frame", 2, 12, 1, 480, 640, {"dz_smem": True, "R": 2, "rounds1": 1}),
    _c("c2-frame-f16", 2, 12, 1, 480, 640, {"dz_smem": True, "R": 2}, precision="f16"),
    _c("c2-global", 2, 12, 1, 1, 2610721, {"dz_smem": False}),
    _c("c3-n37", 3, 6, 1, 1, 37, {"S": 1, "T": 64}, hidden=8),
    _c("c3-none-b2", 3, 6, 2, 48, 64, {"dz_smem": True, "R": 0}, output_fn=None),
    _c("c3-f16-scale-b3", 3, 18, 3, 32, 48, {"dz_smem": True}, hidden=8, scale=0.5, precision="f16"),
    _c("c3-smem-edge", 3, 18, 1, 736, 777, {"dz_smem": True, "R": 3}),
    _c("c3-two-frames", 3, 18, 2, 480, 640, {"dz_smem": False, "R": 4}),
]


def check_variant(case):
    n = case["B"] * case["H"] * case["W"]
    got = flow_bwd_geometry(case["C"], case["F"], n, False)
    for k, v in case["extra"].items():
        assert got[k] == v, (case["id"], k, got[k], v)
    return n


def build(A, case, seed=0):
    return make_flow(A, case["C"], case["F"], case["hidden"], case["output_fn"], case["scale"], case["norm"],
                     case["precision"], seed, spatial=(case["H"], case["W"]))


def deformed_points(m, case):
    """Points to map back: the deformation of the case's coordinate grid, moved by a small seeded offset (another frame's
    points, say).  Without it the only point of a 1x1 grid, (0, 0), maps back to about 0, where the gradient of the conv
    weight (-d_out out / w) is at rounding level."""
    g = torch.Generator(device=DEV).manual_seed(case["B"] * case["H"] * case["W"])
    with torch.no_grad():
        xd = m.get_deformation(torch_grid("linspace", case["B"], case["H"], case["W"], case["C"]))
        return (xd + 0.05 * torch.randn(xd.shape, device=DEV, generator=g)).contiguous()


@pytest.mark.parametrize("case", CASES, ids=[c["id"] for c in CASES])
def test_inverse_gradients_against_float64(A, case):
    """Flow and 1x1-conv gradients and d / d x of inverse against float64; ICNN gradients exactly 0; the output equals the
    no-grad output bit for bit."""
    n = check_variant(case)
    m = build(A, case, seed=21)
    B, C_, H, W = case["B"], case["C"], case["H"], case["W"]
    xd = deformed_points(m, case)
    torch.manual_seed(22)
    w, frac = away_from_kinks(m, rows_of(xd), torch.randn(B, C_, H, W, device=DEV), case["output_fn"], case["scale"])
    with torch.no_grad():
        back_ng = m.inverse(xd)
    m.zero_grad()
    x = xd.clone().requires_grad_(True)
    back = m.inverse(x)
    assert back.requires_grad and torch.equal(back.detach(), back_ng)
    (w * back).sum().backward()
    grads, dx64 = ref_inverse_grads(m, rows_of(xd), rows_of(w), case["output_fn"], case["scale"])
    errs = {}
    for k, prm in m.named_parameters():
        if k.startswith("convex_net."):
            assert prm.grad is not None and int(torch.count_nonzero(prm.grad)) == 0, k
        else:
            errs[k] = entry_err(prm.grad, grads[k])
    err_d = entry_err(rows_of(x.grad), dx64)
    worst = max(errs, key=errs.get)
    print(f"[inverse-grad {case['id']}] N={n}: parameters {errs[worst]:.2e} ({worst})  dx {err_d:.2e}  "
          f"kink pixels {frac:.2%}")
    assert errs[worst] <= TOL_GRAD, errs
    assert err_d <= TOL_DGRID, err_d


# ----------------------------------------------------------------------------------------------------- properties
@pytest.mark.parametrize("C_,F,B,H,W", [(2, 12, 1, 96, 128), (3, 18, 2, 480, 640)], ids=["c2", "c3-global"])
def test_bits_reproducible_and_dgrid_independent(A, C_, F, B, H, W):
    """The training inverse's out equals awb_prior_flow_inverse and the module's no-grad inverse bit for bit; grads are
    bit-identical with and without dgrid and across repeated calls."""
    case = _c("p", C_, F, B, H, W, {})
    m = build(A, case, seed=31)
    xd = deformed_points(m, case)
    arena = m._ensure_flat()
    prior = m._prior_for(arena.device)
    spec = A.GridSpecHost.from_tensor(xd)
    ws = prior.new_workspace(spec.n_pixels, A._lib.AWB_WS_DEFORMATION, DEV)
    out = prior.inverse(arena, spec, True, ws)
    ref = torch.empty_like(out)
    gs = spec.to_c()
    A._lib.check(prior.lib.awb_prior_flow_inverse(prior.handle, arena.data_ptr(), C.byref(gs), ref.data_ptr(),
                                                  A._lib.stream_ptr()))
    assert torch.equal(out, ref)
    assert torch.equal(out, prior.inverse(arena, spec, False, ws))
    with torch.no_grad():
        assert torch.equal(rows_of(m.inverse(xd)), out)
    d_out = torch.randn_like(out)
    g0, none = prior.inverse_backward(arena, spec, d_out, ws, False)
    g1, dg1 = prior.inverse_backward(arena, spec, d_out, ws, True)
    g2, dg2 = prior.inverse_backward(arena, spec, d_out, ws, True)
    assert none is None and dg1 is not None
    assert torch.equal(g0, g1) and torch.equal(g1, g2) and torch.equal(dg1, dg2)
    assert bool(torch.isfinite(g1).all()) and float(g1.abs().max()) > 0


def test_round_trip_cancels(A):
    """sum(w * inverse(get_deformation(x))): d / d x = w, and the flow and 1x1-conv gradients of the two halves cancel."""
    case = _c("rt", 2, 12, 1, 96, 128, {})
    m = build(A, case, seed=41)
    x4 = torch_grid("linspace", 1, 96, 128, 2)
    torch.manual_seed(42)
    w = torch.randn(1, 2, 96, 128, device=DEV)
    m.zero_grad()
    x = x4.clone().requires_grad_(True)
    (w * m.inverse(m.get_deformation(x))).sum().backward()
    g_rt = {k: p.grad.clone() for k, p in m.named_parameters() if not k.startswith("convex_net.")}
    err_x = float((x.grad - w).abs().max() / w.abs().max())
    m.zero_grad()
    (w * m.inverse(m.get_deformation(x4).detach())).sum().backward()       # the inverse half alone
    g_inv = {k: p.grad.clone() for k, p in m.named_parameters() if not k.startswith("convex_net.")}
    scale = max(float(g.abs().max()) for g in g_inv.values())
    resid = max(float(g.abs().max()) for g in g_rt.values()) / scale
    print(f"[inverse-grad round trip] dx - w: {err_x:.2e}  parameter residual {resid:.2e} of the inverse half's")
    assert err_x <= 1e-3, err_x
    assert resid <= 1e-3, resid


def test_adam_steps_match_float64_loop(A):
    """A few Adam steps on a loss through inverse (points mapped back onto fixed targets) against the same loop on the
    float64 oracle chain."""
    case = _c("adam", 2, 12, 1, 48, 64, {})
    m = build(A, case, seed=51)
    xd = deformed_points(m, case)
    torch.manual_seed(52)
    target = torch_grid("linspace", 1, 48, 64, 2) + 0.05 * torch.randn(1, 2, 48, 64, device=DEV)
    keys = [k for k, _ in m.named_parameters() if not k.startswith("convex_net.")]
    p = p64(m, keys)
    for k, prm in m.named_parameters():
        prm.requires_grad_(not k.startswith("convex_net."))
    named = dict(m.named_parameters())
    lr, steps = 1e-3, 4
    opt = torch.optim.Adam([named[k] for k in keys], lr=lr)
    opt64 = torch.optim.Adam([p[k] for k in keys], lr=lr)
    hist, hist64 = [], []
    for _ in range(steps):
        opt.zero_grad()
        loss = ((m.inverse(xd) - target) ** 2).mean()
        loss.backward()
        opt.step()
        hist.append(float(loss))
        opt64.zero_grad()
        loss64 = ((O.unpixelize(inverse64(p, xd.double()), 1, 48, 64) - target.double()) ** 2).mean()
        loss64.backward()
        opt64.step()
        hist64.append(float(loss64))
    print(f"[inverse-grad adam] losses {hist} float64 {hist64}")
    torch.testing.assert_close(torch.tensor(hist), torch.tensor(hist64), rtol=1e-4, atol=1e-9)
    for k in keys:
        # Adam's first steps move every entry by about lr; an entry whose float64 gradient is at rounding level may move
        # either way in both loops, so the comparison is of the moved distance
        torch.testing.assert_close(named[k].detach().double(), p[k].detach(), rtol=0, atol=0.1 * lr * steps,
                                   msg=lambda s: f"{k}: {s}")


def test_graph_only_when_needed_and_first_order_only(A):
    m = make_flow(A, 2, 4, seed=61)
    xd = deformed_points(m, _c("g", 2, 4, 1, 16, 24, {}))
    with torch.no_grad():
        y = m.inverse(xd.clone().requires_grad_(True))
    assert y.grad_fn is None and not y.requires_grad
    for prm in m.parameters():
        prm.requires_grad_(False)
    assert m.inverse(xd).grad_fn is None
    for prm in m.parameters():
        prm.requires_grad_(True)
    x = xd.clone().requires_grad_(True)
    y = m.inverse(x)
    g = torch.autograd.grad(y.sum(), x, create_graph=True)[0]
    with pytest.raises(RuntimeError, match="differentiate twice"):
        g.pow(2).sum().backward()
    y = m.inverse(x[0])                   # [C, H, W] in, [C, H, W] out
    assert y.shape == x[0].shape
    y.sum().backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="once per forward"):
        y.sum().backward()


def test_c_abi_errors(A):
    L = A._lib
    lib = L.load()
    m = make_flow(A, 2, 4, seed=71)
    xd = deformed_points(m, _c("e", 2, 4, 1, 24, 32, {}))
    spec = A.GridSpecHost.from_tensor(xd)
    N = spec.n_pixels
    gs = spec.to_c()
    out = torch.empty(N, 2, device=DEV)
    dgrid = torch.empty(1, 2, 24, 32, device=DEV)

    def rcs(prior, params, ws, grid=gs, nbytes=None, params_ptr=None):
        grads = torch.empty(params.shape[-1], device=DEV)
        nb = ws.numel() if nbytes is None else nbytes
        pp = params.data_ptr() if params_ptr is None else params_ptr
        return (lib.awb_prior_inverse(prior.handle, pp, C.byref(grid), out.data_ptr(), 1, ws.data_ptr(), nb,
                                      L.stream_ptr()),
                lib.awb_prior_inverse_backward(prior.handle, pp, C.byref(grid), out.data_ptr(), grads.data_ptr(),
                                               dgrid.data_ptr(), ws.data_ptr(), nb, L.stream_ptr()))

    big = torch.empty(1 << 26, dtype=torch.uint8, device=DEV)
    # ICNN and NormalizingFlow1D handles: invalid
    icnn = A.Prior(L.AWB_KIND_ICNN, 2, 130, 2)
    assert rcs(icnn, torch.zeros(icnn.n_params, device=DEV), big) == (-1, -1)
    diffeo = A.ConvexDiffeomorphismNet(n_hidden=130, n_hidden_layers=1, nf_layers=2, nf_hidden=70).to(DEV)
    dp = diffeo._prior_for(torch.device(DEV))
    assert rcs(dp, diffeo._ensure_flat(), big) == (-1, -1)
    # grouped flow handle: unsupported
    grouped = A.Prior(L.AWB_KIND_FLOW_ICNN, 2, 130, 2, n_flows=4, flow_hidden=32, flow_tanh=True, n_objects=2)
    m._push_consts(grouped)
    params2 = torch.stack([m._ensure_flat().detach()] * 2).contiguous()
    assert rcs(grouped, params2, big) == (-2, -2)
    single = m._prior_for(torch.device(DEV))
    arena = m._ensure_flat()
    # a generated grid: invalid
    lin = A.GridSpecHost("linspace", 1, 24, 32).to_c()
    assert rcs(single, arena, big, grid=lin) == (-1, -1)
    # a workspace one byte short of the deformation layout
    need = single.workspace_bytes(N, L.AWB_WS_DEFORMATION)
    assert rcs(single, arena, big, nbytes=need - 1) == (-4, -4)
    # null params
    assert rcs(single, arena, big, params_ptr=0) == (-1, -1)
    # the full workspace works
    assert rcs(single, arena, big, nbytes=need) == (0, 0)
