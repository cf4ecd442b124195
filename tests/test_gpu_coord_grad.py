"""Coordinate gradients of the flow priors against a float64 reference.

``PathConnectedNet`` (RealNVP o ICNN, C = 2 and 3) and ``ConvexDiffeomorphismNet`` (NormalizingFlow1D o ICNN) are
differentiable w.r.t. the coordinate grid: the flow backward forms ``dgrid = linear^T (gradient at the 1x1-conv / linear
output)`` in its last pass over each pixel range.  ``get_deformation`` is differentiable w.r.t. the parameters and the
grid through ``awb_prior_deformation`` / ``awb_prior_deformation_backward``.  Second derivatives raise.

dgrid is the gradient of a piecewise-linear function of the coordinates (ReLU units in the ICNN and the coupling MLPs):
it jumps where a pixel crosses a unit's kink.  A pixel whose pre-activation lies within fp32 rounding of zero can sit on
one side of the kink in fp32 and on the other in float64, and its gradient then differs by a whole weight.  The float64
reference therefore records the pixels with a ReLU input within KINK of zero (relative to the largest input of that
layer) and the upstream gradient is 0 there, in the kernels' run and in the reference alike; every other pixel is compared
per entry.  The excluded fraction is printed and bounded by KINK_MAX_FRACTION.

The reference is ``oracle/prior_oracle.py`` run in float64 on the GPU with torch autograd, as in
``test_gpu_launch_regimes.py``, whose restatement of the host dispatch (``flow_bwd_geometry``, ``n_splits``, ...) names the
backward variant every case is meant to hit.  The upstream gradient is random (``(w * y).sum()``), and the 1x1 conv /
2x2 linear has random weight and bias, so that the ``linear^T`` factor is tested."""
import pytest
import torch

import __graft_entry__ as entry
from oracle import prior_oracle as O
from test_gpu_launch_regimes import entry_err, flow_bwd_geometry, n_splits, split_chunk, torch_grid

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# d logits / d grid on the exact fp32 path, per entry relative to max |dgrid64|.  One tolerance for every case, calibrated
# on the 640x480 C = 2 frame (case ``calib``); see TOL_DGRID_MEASURED for the error measured there on a B200.
TOL_DGRID_MEASURED = None
TOL_DGRID = 5e-4
TOL_GRAD = 5e-4              # parameter gradients of get_deformation, as TOL_GRAD of test_gpu_launch_regimes.py
TC_TOL_DGRID = 2e-2          # tensor path, normwise: the flow bound of DESIGN section 4
CHUNK = 1 << 18              # float64 reference: pixel rows per autograd chunk
KINK = 1e-5                  # |ReLU input| < KINK * max |input of the layer|: the pixel is excluded (module docstring)
KINK_MAX_FRACTION = 0.05


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


# ------------------------------------------------------------------------------------------------------------- models
def randomize_linear(m, seed):
    g = torch.Generator().manual_seed(seed)
    sd = m.state_dict()
    sd["linear.weight"] = 1.0 + 0.3 * torch.randn(sd["linear.weight"].shape, generator=g)
    sd["linear.bias"] = 0.1 * torch.randn(sd["linear.bias"].shape, generator=g)
    m.load_state_dict(sd)


def make_flow(A, C_, F, precision="fp32", flow_eval=0, seed=0, norm="minmax", scale=None, spatial=(1000, 1000), L=2):
    """RealNVP prior with non-trivial couplings, initialised ActNorms and a random 1x1 conv."""
    torch.manual_seed(seed)
    m = A.real_nvp_path_connected_net(channels=C_, hidden_units=32, flow_n_flows=F, flow_output_fn="tanh",
                                      flow_output_scale=scale, norm=norm, spatial_shape=spatial,
                                      convex_net_hidden_units=130, convex_net_hidden_layers=L, precision=precision)
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
    m.flow_eval = flow_eval
    return m.to(DEV)


def make_diffeo(A, nc, precision="fp32", seed=0):
    torch.manual_seed(seed)
    m = A.ConvexDiffeomorphismNet(n_hidden=130, n_hidden_layers=1, nf_layers=nc, nf_hidden=70, precision=precision)
    randomize_linear(m, seed + 1)
    return m.to(DEV)


def p64(m, grad_keys=()):
    p = {k: v.detach().to(DEV, torch.float64).clone() for k, v in m.state_dict().items()}
    for k in grad_keys:
        p[k].requires_grad_(True)
    return p


# ----------------------------------------------------------------------------------------------- float64 reference
def flow_deform64(p, x4, scale=None):
    """``pathconnected_deformation`` of the oracle; with MeanStd buffers or an output scale, the same map restated with
    ``(x - mean) / std`` and ``s, t = scale * tanh(MLP)``."""
    if scale is None and "flow_net.norm.mean" not in p:
        return O.pathconnected_deformation(p, x4)
    B, C_, H, W = x4.shape
    x = x4 * p["linear.weight"].reshape(1, C_, 1, 1) + p["linear.bias"].reshape(1, C_, 1, 1)
    mean, std = p["flow_net.norm.mean"], p["flow_net.norm.std"]
    z = O.pixelize((x - mean) / std)
    sc = 1.0 if scale is None else scale
    pre = O.FLOW_PREFIX
    for f in range(O.flow_num(p, pre)):
        a, n = f"{pre}flows.{2 * f}.", f"{pre}flows.{2 * f + 1}."
        b = p[a + "b"].to(z.dtype)
        zm = b * z
        s = sc * O._mlp(p, a + "s.", zm, "tanh")
        t = sc * O._mlp(p, a + "t.", zm, "tanh")
        z = zm + (1 - b) * (z * torch.exp(s) + t)
        z = z * torch.exp(p[n + "s"]) + p[n + "t"]
    return O.pixelize(O.unpixelize(z, B, H, W) * std + mean)


def deform64(kind, p, rows, scale=None):
    """Deformed pixel rows ``[n, C]`` of pixel rows ``rows`` (a ``[1, C, 1, n]`` grid for the RealNVP prior)."""
    if kind == "diffeo":
        return O.flow1d_forward(p, rows @ p["linear.weight"].T + p["linear.bias"], "diffeo_net.")
    return flow_deform64(p, rows.t().reshape(1, rows.shape[1], 1, rows.shape[0]), scale)


def logits64(kind, p, rows, scale=None):
    if kind == "icnn":
        return O.icnn_forward(p, rows).reshape(-1)
    if kind == "convexnet":
        return O.convexnet_forward(p, rows).reshape(-1)
    return O.icnn_forward(p, deform64(kind, p, rows, scale), "convex_net.").reshape(-1)


class _KinkProbe:
    """Stands in for ``torch.nn.functional`` inside the oracle while it evaluates: marks the pixel rows with a ReLU input
    (a ``[n, units]`` pre-activation) within KINK of zero."""

    def __init__(self, n):
        self.near = torch.zeros(n, dtype=torch.bool, device=DEV)

    def _note(self, a):
        a = a.detach().abs()
        self.near |= (a < KINK * a.max()).any(dim=1)

    def relu(self, a, *args, **kw):
        self._note(a)
        return torch.nn.functional.relu(a, *args, **kw)

    def leaky_relu(self, a, *args, **kw):
        self._note(a)
        return torch.nn.functional.leaky_relu(a, *args, **kw)

    def __getattr__(self, name):
        return getattr(torch.nn.functional, name)


def kink_rows(kind, m, rows, scale=None, deformation_only=False):
    """Boolean ``[N]``: pixel rows within KINK of a ReLU kink of the float64 forward (of the deformation alone when
    ``deformation_only``)."""
    p = p64(m)
    out = torch.zeros(rows.shape[0], dtype=torch.bool, device=DEV)
    saved = O.F
    try:
        for a in range(0, rows.shape[0], CHUNK):
            r = rows[a:a + CHUNK].double()
            O.F = probe = _KinkProbe(r.shape[0])
            with torch.no_grad():
                deform64(kind, p, r, scale) if deformation_only else logits64(kind, p, r, scale)
            out[a:a + CHUNK] = probe.near
    finally:
        O.F = saved
    return out


def away_from_kinks(kind, m, rows, w, scale=None, deformation_only=False, max_fraction=KINK_MAX_FRACTION):
    """``w`` with the upstream gradient of the kink pixels set to 0, and the excluded fraction."""
    near = kink_rows(kind, m, rows, scale, deformation_only)
    frac = float(near.float().mean())
    assert frac <= max_fraction, frac
    B, C_, H, W = w.shape
    w = w.permute(0, 2, 3, 1).reshape(-1, C_).clone()
    w[near] = 0
    return w.reshape(B, H, W, C_).permute(0, 3, 1, 2).contiguous(), frac


def ref_dgrid(kind, m, rows, w_rows, scale=None):
    """float64 ``d sum(w * logits) / d rows`` (``[N, C]``), chunk by chunk (every pixel's logit depends on its row only)."""
    p = p64(m)
    out = torch.empty(rows.shape, dtype=torch.float64, device=DEV)
    for a in range(0, rows.shape[0], CHUNK):
        r = rows[a:a + CHUNK].double().requires_grad_(True)
        y = logits64(kind, p, r, scale)
        out[a:a + CHUNK] = torch.autograd.grad((w_rows[a:a + CHUNK].double() * y).sum(), r)[0]
    return out


def last_range(n):
    """Rows of the flow backward's last non-empty pixel range (ranges of ``split_chunk(n)`` rows, ``n_splits(n)`` of them)."""
    chunk = split_chunk(n)
    nonempty = (n + chunk - 1) // chunk
    assert nonempty <= n_splits(n)
    return (nonempty - 1) * chunk, n


def rows_of(x4):
    return x4.permute(0, 2, 3, 1).reshape(-1, x4.shape[1])


def module_dgrid(m, x4, w):
    x = x4.clone().requires_grad_(True)
    y = m(x)
    return torch.autograd.grad((w * y).sum(), x)[0]


# --------------------------------------------------------------------------------------- exact fp32 path: the cases
def _c(id_, kind, C_, F, B, H, W, kernel, flow_eval=1, extra=None, **kw):
    return dict(id=id_, kind=kind, C=C_, F=F, B=B, H=H, W=W, kernel=kernel, flow_eval=flow_eval, extra=extra or {}, **kw)


EXACT = [
    _c("calib", "flow", 2, 12, 1, 480, 640, "k_flow_bwd<2>", extra={"dz_smem": True}),
    _c("bwd2-global", "flow", 2, 12, 1, 1, 2610721, "k_flow_bwd<2>", extra={"dz_smem": False}),
    _c("bwd3-smem-edge", "flow", 3, 18, 1, 736, 777, "k_flow_bwd<3>", extra={"dz_smem": True}),
    _c("bwd3-global-edge", "flow", 3, 18, 1, 1, 571873, "k_flow_bwd<3>", extra={"dz_smem": False}),
    _c("seg-smem-edge", "flow", 2, 12, 1, 592, 1094, "k_flow_bwd_seg<true>", flow_eval=2),
    _c("seg-global-edge", "flow", 2, 12, 1, 747, 867, "k_flow_bwd_seg<false>", flow_eval=2),
    _c("c2-seg-n37", "flow", 2, 12, 1, 1, 37, "k_flow_bwd_seg<true>", flow_eval=2, extra={"S": 1}),
    # MeanStd norm and output_scale != 1: the segment tables are specialised for scale 1, flow_eval = 2 falls back
    _c("meanstd-scale", "flow", 2, 12, 1, 96, 128, "k_flow_bwd<2>", flow_eval=2, norm="meanstd", scale=0.5),
]
for C_, F in ((2, 12), (3, 18)):
    EXACT += [
        _c(f"c{C_}-n1", "flow", C_, F, 1, 1, 1, f"k_flow_bwd<{C_}>", extra={"S": 1, "T": 32}),
        _c(f"c{C_}-n37", "flow", C_, F, 1, 1, 37, f"k_flow_bwd<{C_}>", extra={"S": 1, "T": 64}),
        _c(f"c{C_}-n257", "flow", C_, F, 1, 1, 257, f"k_flow_bwd<{C_}>", extra={"S": 2, "T": 160}),
        _c(f"c{C_}-n37889", "flow", C_, F, 1, 1, 37889, f"k_flow_bwd<{C_}>", extra={"empty": 4}),
    ]
EXACT += [_c(f"diffeo-nc{nc}", "diffeo", 2, nc, 1, 240, 320, f"k_diffeo_bwd<{nc}>") for nc in (2, 4, 8)]


def check_variant(case):
    n = case["B"] * case["H"] * case["W"]
    if case["kind"] == "diffeo":
        got = dict(kernel=f"k_diffeo_bwd<{case['F']}>", S=n_splits(n))
    else:
        seg = case["flow_eval"] == 2 and case["C"] == 2 and case.get("scale") is None
        got = flow_bwd_geometry(case["C"], case["F"], n, seg)
    assert got["kernel"] == case["kernel"], (case["id"], got)
    for k, v in case["extra"].items():
        assert got[k] == v, (case["id"], k, got[k], v)
    return n


def build(A, case, precision="fp32", seed=0):
    if case["kind"] == "diffeo":
        return make_diffeo(A, case["F"], precision, seed)
    spatial = (case["H"], case["W"])
    return make_flow(A, case["C"], case["F"], precision, case["flow_eval"], seed, case.get("norm", "minmax"),
                     case.get("scale"), spatial)


@pytest.mark.parametrize("case", EXACT, ids=[c["id"] for c in EXACT])
def test_dgrid_exact_path_against_float64(A, case):
    """d sum(w * logits) / d grid per entry against float64, and the float64 self-check that zeroing the rows of the last
    non-empty pixel range moves some entry by more than the tolerance."""
    n = check_variant(case)
    m = build(A, case)
    x4 = torch_grid("linspace", case["B"], case["H"], case["W"], case["C"])
    torch.manual_seed(5)
    w, frac = away_from_kinks(case["kind"], m, rows_of(x4), torch.randn(case["B"], 1, case["H"], case["W"], device=DEV),
                              case.get("scale"))
    dgrid = module_dgrid(m, x4, w)
    ref = ref_dgrid(case["kind"], m, rows_of(x4), w.reshape(-1), case.get("scale"))
    err = entry_err(rows_of(dgrid), ref)
    r0, r1 = last_range(n)
    dropped = ref.clone()
    dropped[r0:r1] = 0
    sens = entry_err(dropped, ref)
    print(f"[coord-grad {case['id']}] N={n} {case['kernel']}: dgrid {err:.2e}  last range [{r0}, {r1}) zeroed {sens:.2e}  "
          f"kink pixels {frac:.2%}")
    assert err <= TOL_DGRID, (case["id"], err)
    assert sens > TOL_DGRID, (case["id"], sens)


# ------------------------------------------------------------------------------------------------------- tensor path
TC = [
    _c("tc-c2-tables", "flow", 2, 12, 1, 480, 640, "k_flow_bwd_seg<true>", flow_eval=0),
    _c("tc-c3", "flow", 3, 18, 1, 240, 320, "k_flow_bwd<3>", flow_eval=0),
    _c("tc-diffeo-nc4", "diffeo", 2, 4, 1, 240, 320, "k_diffeo_bwd<4>"),
]


@pytest.mark.parametrize("case", TC, ids=[c["id"] for c in TC])
def test_dgrid_tensor_path_against_float64(A, case):
    c = dict(case)
    c["flow_eval"] = 2 if case["kind"] == "flow" and case["C"] == 2 else 1     # f16 handles use the tables by default
    check_variant(c)
    m = build(A, case, precision="f16", seed=3)
    x4 = torch_grid("linspace", case["B"], case["H"], case["W"], case["C"])
    torch.manual_seed(6)
    w = torch.randn(case["B"], 1, case["H"], case["W"], device=DEV)
    dgrid = rows_of(module_dgrid(m, x4, w)).double()
    ref = ref_dgrid(case["kind"], m, rows_of(x4), w.reshape(-1))
    err = float((dgrid - ref).norm() / ref.norm())
    print(f"[coord-grad {case['id']}] tensor path: dgrid normwise {err:.2e}")
    assert err <= TC_TOL_DGRID, (case["id"], err)


# -------------------------------------------------------------------------------------------------------- properties
PROPS = [
    ("fp32-c2-tables", lambda A: make_flow(A, 2, 12, "fp32", 2, seed=7), 2),
    ("fp32-c3", lambda A: make_flow(A, 3, 18, "fp32", 1, seed=8), 3),
    ("f16-c2", lambda A: make_flow(A, 2, 12, "f16", 0, seed=9), 2),
    ("f16-c3", lambda A: make_flow(A, 3, 18, "f16", 0, seed=10), 3),
    ("fp32-diffeo", lambda A: make_diffeo(A, 4, "fp32", seed=11), 2),
    ("f16-diffeo", lambda A: make_diffeo(A, 4, "f16", seed=12), 2),
]


@pytest.mark.parametrize("make,C_", [(mk, c) for _, mk, c in PROPS], ids=[i for i, _, _ in PROPS])
def test_dgrid_properties(A, make, C_):
    """Parameter gradients do not depend on whether dgrid is requested (bit for bit); dgrid is the same bits from run to
    run; pixel rows [N, C] give the [B, C, H, W] result permuted, bit for bit."""
    m = make(A)
    B, H, W = 2, 96, 160
    x4 = torch_grid("linspace", B, H, W, C_)
    torch.manual_seed(4)
    w = torch.randn(B, 1, H, W, device=DEV)

    def run(want_dgrid):
        m.zero_grad()
        x = x4.clone().requires_grad_(want_dgrid)
        (w * m(x)).sum().backward()
        return torch.cat([p.grad.reshape(-1) for p in m.parameters()]).clone(), (x.grad.clone() if want_dgrid else None)

    g0, _ = run(False)
    g1, d1 = run(True)
    g2, d2 = run(True)
    assert torch.equal(g0, g1)
    assert torch.equal(d1, d2)
    assert float(d1.abs().max()) > 0
    rows = rows_of(x4).clone().requires_grad_(True)
    (w.reshape(-1, 1) * m(rows)).sum().backward()
    assert torch.equal(rows.grad, rows_of(d1))


def test_multi_object_container_sums_single_priors(A):
    """A MultipleObjectsAwarePathConnectedNet of three flow priors: d / d grid of sum_k (w_k * y_k) is the sum of the three
    single-prior dgrids (the container needs no code of its own)."""
    cont = A.MultipleObjectsAwarePathConnectedNet(prior=make_flow(A, 2, 12, "fp32", 1, seed=20), min_priors=3).to(DEV)
    for k in range(3):
        src = make_flow(A, 2, 12, "fp32", 1, seed=21 + 3 * k)
        cont.priors[k].load_state_dict(src.state_dict())
    B, H, W = 1, 120, 160
    x4 = torch_grid("linspace", B, H, W, 2)
    torch.manual_seed(2)
    w = torch.randn(B, 3, 1, H, W, device=DEV)
    x = x4.clone().requires_grad_(True)
    y = cont(x)
    assert y.shape == (B, 3, 1, H, W)
    d_all = torch.autograd.grad((w * y).sum(), x)[0]
    d_sum = sum(module_dgrid(cont.priors[k], x4, w[:, k]) for k in range(3))
    rel = float((d_all - d_sum).abs().max() / d_sum.abs().max())
    assert rel <= 1e-6, rel


# --------------------------------------------------------------------------------------------------- get_deformation
DEFORM = [
    _c("c2-640x480", "flow", 2, 12, 1, 480, 640, "k_flow_bwd<2>"),
    _c("c2-tables", "flow", 2, 12, 1, 240, 320, "k_flow_bwd_seg<true>", flow_eval=2),
    _c("c3-configs4", "flow", 3, 18, 2, 480, 640, "k_flow_bwd<3>", extra={"dz_smem": False}),
    _c("diffeo-nc4", "diffeo", 2, 4, 1, 240, 320, "k_diffeo_bwd<4>"),
]


def ref_deformation(kind, m, rows, w_rows):
    """float64 gradients of sum(w * get_deformation(rows)) w.r.t. the flow / linear parameters and the rows."""
    keys = [k for k, _ in m.named_parameters() if not k.startswith("convex_net.")]
    p = p64(m, keys)
    grads = {k: torch.zeros_like(p[k]) for k in keys}
    dgrid = torch.empty(rows.shape, dtype=torch.float64, device=DEV)
    for a in range(0, rows.shape[0], CHUNK):
        r = rows[a:a + CHUNK].double().requires_grad_(True)
        l = (w_rows[a:a + CHUNK].double() * deform64(kind, p, r)).sum()
        gs = torch.autograd.grad(l, [p[k] for k in keys] + [r])
        for k, g in zip(keys, gs[:-1]):
            grads[k] += g
        dgrid[a:a + CHUNK] = gs[-1]
    return grads, dgrid


@pytest.mark.parametrize("case", DEFORM, ids=[c["id"] for c in DEFORM])
def test_get_deformation_gradients_against_float64(A, case):
    """Flow and linear gradients and dgrid of get_deformation against float64; ICNN gradients exactly 0; the output equals
    the no_grad output bit for bit, which is what the inference forward returns."""
    n = check_variant(case)
    m = build(A, case, seed=13)
    B, C_, H, W = case["B"], case["C"], case["H"], case["W"]
    x4 = torch_grid("linspace", B, H, W, C_)
    torch.manual_seed(14)
    w, frac = away_from_kinks(case["kind"], m, rows_of(x4), torch.randn(B, C_, H, W, device=DEV), deformation_only=True)
    with torch.no_grad():
        d_ng = m.get_deformation(x4)
        arena = m._ensure_flat()
        prior = m._prior_for(arena.device)
        spec = A.GridSpecHost.from_tensor(x4)
        ws = prior.new_workspace(n, A._lib.AWB_WS_INFERENCE, DEV)
        _, d_fwd = prior.forward(arena, spec, A._lib.AWB_FWD_EXACT, ws, want_deformed=True)
    assert torch.equal(rows_of(d_ng), d_fwd[0])
    m.zero_grad()
    x = x4.clone().requires_grad_(True)
    d = m.get_deformation(x)
    assert d.requires_grad and torch.equal(d.detach(), d_ng)
    (w * d).sum().backward()
    grads, dgrid64 = ref_deformation(case["kind"], m, rows_of(x4), rows_of(w))
    errs = {}
    biggest = max(float(g.abs().max()) for g in grads.values())
    for k, prm in m.named_parameters():
        if k.startswith("convex_net."):
            assert prm.grad is not None and int(torch.count_nonzero(prm.grad)) == 0, k
        elif k.endswith("scale.weight_v"):
            # WNScale's weight is 1x1: g * v / |v| = g * sign(v), whose derivative in v is identically 0.  The kernel returns
            # exactly 0; float64 autograd returns the rounding of (1/|v| - v^2/|v|^3), which is no error to measure against.
            assert int(torch.count_nonzero(prm.grad)) == 0, k
            assert float(grads[k].abs().max()) <= 1e-12 * biggest, (k, float(grads[k].abs().max()), biggest)
        else:
            errs[k] = entry_err(prm.grad, grads[k])
    err_d = entry_err(rows_of(x.grad), dgrid64)
    worst = max(errs, key=errs.get)
    print(f"[coord-grad deformation {case['id']}] N={n}: parameters {errs[worst]:.2e} ({worst})  dgrid {err_d:.2e}  "
          f"kink pixels {frac:.2%}")
    assert errs[worst] <= TOL_GRAD, errs
    assert err_d <= TOL_DGRID, err_d


def test_get_deformation_parameter_gradients_without_grid_grad(A):
    """A parameter-only loss on get_deformation (x without requires_grad) gives the same parameter gradients, bit for bit."""
    m = make_flow(A, 2, 12, "fp32", 1, seed=30)
    x4 = torch_grid("linspace", 1, 96, 128, 2)
    w = torch.randn(1, 2, 96, 128, device=DEV)
    out = []
    for want in (False, True):
        m.zero_grad()
        (w * m.get_deformation(x4.clone().requires_grad_(want))).sum().backward()
        out.append(torch.cat([p.grad.reshape(-1) for p in m.parameters()]))
    assert torch.equal(out[0], out[1])


# ------------------------------------------------------------------------------------------------------------ errors
@pytest.mark.parametrize("kind", ["icnn", "flow", "flow-deformation"])
def test_second_derivatives_raise(A, kind):
    """A gradient penalty through a prior would silently lose its second-order term: it raises instead."""
    if kind == "icnn":
        m = A.ConvexNextNet(in_features=2, n_hidden_layers=2).to(DEV)
    else:
        m = make_flow(A, 2, 12, "fp32", 1, seed=40)
    x = torch_grid("linspace", 1, 32, 48, 2).requires_grad_(True)
    y = m.get_deformation(x) if kind == "flow-deformation" else m(x)
    g = torch.autograd.grad(y.sum(), x, create_graph=True)[0]
    with pytest.raises(RuntimeError, match="differentiate twice"):
        g.pow(2).sum().backward()
    y = m.get_deformation(x) if kind == "flow-deformation" else m(x)
    g = torch.autograd.grad(y.sum(), x, create_graph=True)[0]
    with pytest.raises(RuntimeError, match="differentiate twice"):
        (y.sum() + g.pow(2).sum()).backward()


def test_c_abi_errors(A):
    import ctypes as C
    L = A._lib
    lib = L.load()
    spec = A.GridSpecHost("linspace", 1, 24, 32)
    N = spec.n_pixels
    gs = spec.to_c()
    dd = torch.zeros(N, 2, device=DEV)
    dgrid = torch.empty(1, 2, 24, 32, device=DEV)

    def deform_rcs(prior, params, ws):
        grads = torch.empty(params.shape[-1], device=DEV)
        return (lib.awb_prior_deformation(prior.handle, params.data_ptr(), C.byref(gs), dd.data_ptr(), 1, ws.data_ptr(),
                                          ws.numel(), L.stream_ptr()),
                lib.awb_prior_deformation_backward(prior.handle, params.data_ptr(), C.byref(gs), dd.data_ptr(),
                                                   grads.data_ptr(), dgrid.data_ptr(), ws.data_ptr(), ws.numel(),
                                                   L.stream_ptr()))

    # dgrid on a grouped (2-object) flow handle: unsupported
    m = make_flow(A, 2, 4, "fp32", 1, seed=50)
    grouped = A.Prior(L.AWB_KIND_FLOW_ICNN, 2, 130, 2, n_flows=4, flow_hidden=32, flow_tanh=True, n_objects=2)
    m._push_consts(grouped)
    params2 = torch.stack([m._ensure_flat().detach()] * 2).contiguous()
    ws = grouped.new_workspace(N, L.AWB_WS_TRAINING, DEV)
    rc = lib.awb_prior_backward(grouped.handle, params2.data_ptr(), C.byref(gs), torch.zeros(2, N, device=DEV).data_ptr(),
                                torch.empty_like(params2).data_ptr(), dgrid.data_ptr(), ws.data_ptr(), ws.numel(),
                                L.stream_ptr())
    assert rc == -2
    assert b"grouped" in lib.awb_last_error()
    assert deform_rcs(grouped, params2, grouped.new_workspace(N, L.AWB_WS_DEFORMATION, DEV)) == (-2, -2)
    # an ICNN handle has no deformation
    icnn = A.Prior(L.AWB_KIND_ICNN, 2, 130, 2)
    p_icnn = torch.zeros(icnn.n_params, device=DEV)
    assert deform_rcs(icnn, p_icnn, icnn.new_workspace(N, L.AWB_WS_DEFORMATION, DEV)) == (-1, -1)
    assert b"no deformation" in lib.awb_last_error()
    # the star prior: unsupported
    star = A.Prior(L.AWB_KIND_STAR, 2, 32, 0)
    p_star = torch.zeros(star.n_params, device=DEV)
    assert deform_rcs(star, p_star, torch.empty(1 << 20, dtype=torch.uint8, device=DEV)) == (-2, -2)
    # a workspace one byte short of the deformation layout
    single = m._prior_for(torch.device(DEV))
    arena = m._ensure_flat()
    need = single.workspace_bytes(N, L.AWB_WS_DEFORMATION)
    assert 0 < need < single.workspace_bytes(N, L.AWB_WS_FIT_STEP)   # the deformation layout carries no ICNN activations
    assert deform_rcs(single, arena, torch.empty(need - 1, dtype=torch.uint8, device=DEV)) == (-4, -4)
    assert deform_rcs(single, arena, torch.empty(need, dtype=torch.uint8, device=DEV)) == (0, 0)
    torch.cuda.synchronize()
