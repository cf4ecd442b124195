"""Autograd through the star-shape prior: ``awb_star_backward`` (``k_star_bwd``) against a float64 reference.

``StarShapedNet.forward`` is differentiable w.r.t. its parameters and the sample points.  The reference is
``oracle/prior_oracle.py``'s ``star_forward`` run in float64 on the GPU with torch autograd, for a random upstream gradient
``w`` (``(w * net(x)).sum()``).  Parameter gradients and ``dx`` are compared per tensor, relative to the tensor's largest
reference entry.

The network is piecewise linear in its ReLU inputs: a point whose float64 pre-activation (of ``a`` or of ``b``) lies
within fp32 rounding of zero can sit on the other side of the kink in fp32, and its gradient then differs by a whole
weight.  As in ``test_gpu_coord_grad.py``, such points (pre-activation within KINK of zero, relative to the largest
pre-activation of that layer) get ``w = 0`` in the kernel's run and in the reference alike; the excluded fraction is
printed and bounded.

``geometry()`` restates the host dispatch of ``k_star_bwd`` (``star_bwd_ctas`` in ``awb_star.cu``); every size names the
branch it is meant to hit and the test asserts the restatement agrees, as ``test_gpu_launch_regimes.py`` does.  A
float64-only self-check shows that dropping the last CTA's points moves some gradient entry by more than the bound."""
import pytest
import torch

import __graft_entry__ as entry
from oracle import prior_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Per-tensor error relative to the tensor's largest float64 entry.  Measured on one B200 over every case below (each
# case prints its values): parameter gradients at most 2.2e-6 (W2_r.weight, n = 1000), dx at most 7.7e-7; the bounds
# leave a margin of about 10x.  Dropping the last CTA's points moves some float64 gradient entry by more than 10x the bound
# in every case (the self-check at the end of the comparison).
TOL_GRAD = 2e-5
TOL_DX = 1e-5
KINK = 1e-5                  # |ReLU input| < KINK * max |input of the layer|: the point is excluded (module docstring)
KINK_MAX_FRACTION = 0.05
OFFSET = (0.05, -0.03)

# ----------------------------------------------------------------------------------------------- host dispatch, restated
K_STAR_T = 64                # awb_star.cu kStarT: points per tile
K_MAX_SPLITS = 148           # awb_internal.cuh kMaxSplits


def cdiv(a, b):
    return (a + b - 1) // b


def geometry(n):
    """awb_star.cu ``star_bwd_ctas``: tiles per CTA, CTA count, points per CTA; and the two size-dependent branches."""
    tiles = cdiv(n, K_STAR_T)
    per = cdiv(tiles, K_MAX_SPLITS)
    S = cdiv(tiles, per)
    return dict(S=S, chunk=per * K_STAR_T, multi_tile=per > 1, remainder=n % K_STAR_T != 0)


# (h, n, expected branches).  h = 150 is the notebook's width (5 lane groups of 32 units, the last partly padding);
# h = 37 has an odd width that pads both the lane groups and the products' K loop.
CASES = [
    (150, 1, dict(multi_tile=False, remainder=True)),
    (150, 5, dict(multi_tile=False, remainder=True)),
    (150, 1000, dict(multi_tile=False, remainder=True)),
    (150, 64 * 48, dict(multi_tile=False, remainder=False)),
    (150, 148 * 64, dict(multi_tile=False, remainder=False, S=148)),   # the last size with one tile per CTA
    (150, 148 * 64 + 1, dict(multi_tile=True, remainder=True)),
    (150, 149 * 64, dict(multi_tile=True, remainder=False)),
    (150, 640 * 480, dict(multi_tile=True, remainder=False)),           # a full likelihood image
    (37, 1000, dict(multi_tile=False, remainder=True)),
    (37, 64 * 48, dict(multi_tile=False, remainder=False)),
    (37, 148 * 64 + 1, dict(multi_tile=True, remainder=True)),
    (37, 149 * 64, dict(multi_tile=True, remainder=False)),
]


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


@pytest.fixture(scope="module")
def A():
    import awesome_b200
    return awesome_b200


def make_star(A, h, seed=0):
    torch.manual_seed(seed)
    m = A.StarShapedNet(h)
    sd = m.state_dict()
    sd["offset"] = torch.tensor([OFFSET])
    m.load_state_dict(sd)
    m = m.to(DEV)
    m.offset.requires_grad_(True)
    return m


def points(n, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(n, 2, generator=g) - 0.5).to(DEV)


def p64(m):
    return {k: v.detach().to(DEV, torch.float64).clone().requires_grad_(True) for k, v in m.state_dict().items()}


def near_kinks(p, x):
    """Boolean ``[n]``: float64 ReLU inputs of the point within KINK of zero (the star forward, restated)."""
    with torch.no_grad():
        z = x.double() + p["offset"]
        r = torch.sqrt(torch.sum(z ** 2, dim=1, keepdim=True))
        apre = (z / (0.01 + r)) @ p["W0.weight"].T + p["W0.bias"]
        a = torch.relu(apre)
        bpre = a @ p["W1.weight"].T + p["W1.bias"] + r @ p["W1_r.weight"].T + p["W1_r.bias"]
        near = torch.zeros(x.shape[0], dtype=torch.bool, device=DEV)
        for v in (apre, bpre):
            near |= (v.abs() < KINK * v.abs().max()).any(dim=1)
    return near


def ref_grads(p, x, w):
    """float64 ``d sum(w * y) / d (params, x)``."""
    xr = x.double().clone().requires_grad_(True)
    y = O.star_forward(p, xr).reshape(-1)
    keys = list(p)
    gs = torch.autograd.grad((w.double() * y).sum(), [p[k] for k in keys] + [xr])
    return dict(zip(keys, gs[:-1])), gs[-1]


def native_grads(m, x, w):
    xr = x.clone().requires_grad_(True)
    y = m(xr).reshape(-1)
    names = [k for k, _ in m.named_parameters()]
    gs = torch.autograd.grad((w * y).sum(), [dict(m.named_parameters())[k] for k in names] + [xr])
    return dict(zip(names, gs[:-1])), gs[-1]


def rel_err(a, ref):
    return float((a.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize("h,n,branches", CASES, ids=[f"h{h}-n{n}" for h, n, _ in CASES])
def test_star_backward_vs_float64(A, h, n, branches):
    geo = geometry(n)
    for k, v in branches.items():
        assert geo[k] == v, (k, geo)
    m = make_star(A, h, seed=h)
    x = points(n, seed=n)
    w = torch.randn(n, generator=torch.Generator().manual_seed(n + 1)).to(DEV)
    p = p64(m)
    near = near_kinks(p, x)
    frac = float(near.float().mean())
    assert frac <= KINK_MAX_FRACTION, frac
    w[near] = 0
    g, dx = native_grads(m, x, w)
    g64, dx64 = ref_grads(p, x, w)
    errs = {k: rel_err(g[k], g64[k]) for k in g64}
    err_dx = rel_err(dx, dx64)
    # the bound sees one dropped CTA: the float64 gradients without the last CTA's points move past it
    w_drop = w.clone()
    w_drop[(geo["S"] - 1) * geo["chunk"]:] = 0
    gd, _ = ref_grads(p, x, w_drop)
    moved = max(rel_err(gd[k], g64[k]) for k in g64)
    print(f"h={h} n={n} S={geo['S']} chunk={geo['chunk']} kink fraction {frac:.2e}: max param err "
          f"{max(errs.values()):.2e} ({max(errs, key=errs.get)}), dx err {err_dx:.2e}; last CTA dropped: {moved:.2e}")
    for k, e in errs.items():
        assert e <= TOL_GRAD, (k, e)
    assert err_dx <= TOL_DX, err_dx
    assert moved > 10 * TOL_GRAD, moved
    # both biases of a pair receive the same gradient (the forward adds them)
    assert torch.equal(g["W1.bias"], g["W1_r.bias"]) and torch.equal(g["W2.bias"], g["W2_r.bias"])


def test_star_autograd_vs_notebook_fixture(A, golden):
    """The notebook's loss through the drop-in reproduces the notebook class's loss and gradients."""
    g = golden("star.pt")
    m = A.StarShapedNet(150)
    m.load_state_dict(g["init"])
    m = m.to(DEV)
    m.offset.requires_grad = True
    loss = torch.nn.functional.mse_loss(torch.sigmoid(m(g["x"].to(DEV))).squeeze(), g["t"].to(DEV))
    loss.backward()
    torch.testing.assert_close(loss.detach().cpu(), g["loss"], rtol=1e-5, atol=1e-8)
    for k, p in m.named_parameters():
        torch.testing.assert_close(p.grad.cpu(), g["grads"][k], rtol=2e-3, atol=2e-7, msg=lambda s: f"{k}: {s}")


def test_star_notebook_loop_vs_oracle_and_fitter(A, golden):
    """Cell 3 run literally for 5 steps: Adam on the drop-in's parameters, ``loss.backward()``, the W2_r clamp, and the
    offset unfrozen at step 2 with its own optimizer.  Matches the CPU oracle loop (tolerances of
    test_star_fit_steps_vs_oracle_adam_with_late_offset) and the fused StarFitter."""
    g = golden("star.pt")
    x, t = g["x"].to(DEV), g["t"].to(DEV)
    m = A.StarShapedNet(150)
    m.load_state_dict(g["init"])
    m = m.to(DEV)
    opt = torch.optim.Adam([p for k, p in m.named_parameters() if k != "offset"], lr=1e-2)
    opt_off = torch.optim.Adam([m.offset], lr=1e-2)
    mf = A.StarShapedNet(150)
    mf.load_state_dict(g["init"])
    mf = mf.to(DEV)
    f = mf.make_fitter(optim=A.OptimConfig("adam", lr=1e-2))
    p = O.clone_params(g["init"], requires_grad=True)
    keys = list(g["grads"])
    ref_opt = torch.optim.Adam([p[k] for k in keys if k != "offset"], lr=1e-2)
    ref_opt_off = torch.optim.Adam([p["offset"]], lr=1e-2)
    ours, fused, ref = [], [], []
    for step in range(5):
        if step == 2:
            m.offset.requires_grad = True
        opt.zero_grad(); opt_off.zero_grad()
        loss = torch.nn.functional.mse_loss(torch.sigmoid(m(x)).squeeze(), t)
        loss.backward()
        if step < 2:
            assert m.offset.grad is None
        opt.step()
        if step >= 2:
            opt_off.step()
        with torch.no_grad():
            m.W2_r.weight.clamp_(min=0)
        ours.append(float(loss.detach()))
        f.train_offset = step >= 2
        fused.append(float(f.step(g["x"], g["t"])))
        ref_opt.zero_grad(); ref_opt_off.zero_grad()
        rl = torch.nn.functional.mse_loss(torch.sigmoid(O.star_forward(p, g["x"])).squeeze(), g["t"])
        rl.backward()
        ref_opt.step()
        if step >= 2:
            ref_opt_off.step()
        with torch.no_grad():
            p["W2_r.weight"].clamp_(min=0)
        ref.append(float(rl.detach()))
    torch.testing.assert_close(torch.tensor(ours), torch.tensor(ref), rtol=2e-4, atol=1e-7)
    torch.testing.assert_close(torch.tensor(ours), torch.tensor(fused), rtol=2e-4, atol=1e-7)
    sd, sdf = m.state_dict(), mf.state_dict()
    for k in keys:
        torch.testing.assert_close(sd[k].cpu(), p[k].detach(), rtol=2e-3, atol=2e-5, msg=lambda s: f"{k}: {s}")
        torch.testing.assert_close(sd[k], sdf[k], rtol=2e-3, atol=2e-5, msg=lambda s: f"{k} vs StarFitter: {s}")
    assert float(sd["W2_r.weight"].min()) >= 0.0


def test_star_autograd_properties(A):
    m = make_star(A, 150, seed=3)
    n = 3000
    x = points(n, seed=7)
    x[17] = -m.offset.detach()[0]                    # exactly at -offset: r = 0
    w = torch.randn(n, generator=torch.Generator().manual_seed(8)).to(DEV)
    params = list(m.parameters())
    prior = m._prior_for(torch.device(DEV))
    # logits: no_grad, grad enabled with nothing requiring grad, and a graph-building forward give the bits of a plain
    # awb_star_forward call
    plain = torch.empty(n, device=DEV)
    A._lib.check(prior.lib.awb_star_forward(prior.handle, m._ensure_flat().data_ptr(), x.data_ptr(), n, plain.data_ptr(),
                                            A._lib.stream_ptr()))
    with torch.no_grad():
        y0 = m(x)
    assert y0.grad_fn is None and torch.equal(y0.reshape(-1), plain)
    xr = x.clone().requires_grad_(True)
    y = m(xr)
    assert y.grad_fn is not None and torch.equal(y.detach().reshape(-1), plain)
    # two backward calls: the same bits
    g1 = torch.autograd.grad((w * y.reshape(-1)).sum(), params + [xr], retain_graph=True)
    g2 = torch.autograd.grad((w * y.reshape(-1)).sum(), params + [xr], retain_graph=True)
    assert all(torch.equal(a, b) for a, b in zip(g1, g2))
    # the point at -offset: finite gradients, dx = 0 (every term carries a factor r = 0)
    assert all(bool(torch.isfinite(a).all()) for a in g1)
    assert torch.equal(g1[-1][17], torch.zeros(2, device=DEV))
    # dx not wanted: the parameter gradients keep their bits
    yp = m(x)
    gp = torch.autograd.grad((w * yp.reshape(-1)).sum(), params)
    assert all(torch.equal(a, b) for a, b in zip(gp, g1[:-1]))
    # the offset frozen (the default): no gradient for it
    m2 = make_star(A, 150, seed=3)
    m2.offset.requires_grad_(False)
    (w * m2(x).reshape(-1)).sum().backward()
    assert m2.offset.grad is None and m2.W1.weight.grad is not None
    # first order only
    xr = x.clone().requires_grad_(True)
    gx = torch.autograd.grad(m(xr).sum(), xr, create_graph=True)[0]
    with pytest.raises(RuntimeError, match="differentiate twice"):
        gx.sum().backward()


def test_star_backward_c_abi_errors(A):
    from awesome_b200 import _lib as L
    star = A.Prior(L.AWB_KIND_STAR, 2, 32, 0)
    lib = star.lib
    n = 100
    params = torch.zeros(star.n_params, device=DEV)
    x, dy = torch.zeros(n, 2, device=DEV), torch.ones(n, device=DEV)
    grads, dx = torch.empty(star.n_params, device=DEV), torch.empty(n, 2, device=DEV)
    need = int(lib.awb_star_backward_workspace_bytes(star.handle, n))
    assert need > 0
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)

    def call(h=star.handle, params=params.data_ptr(), x=x.data_ptr(), n=n, dy=dy.data_ptr(), grads=grads.data_ptr(),
             dx=dx.data_ptr(), ws=ws.data_ptr(), ws_bytes=need):
        return lib.awb_star_backward(h, params, x, n, dy, grads, dx, ws, ws_bytes, L.stream_ptr())

    icnn = A.Prior(L.AWB_KIND_ICNN, 2, 130, 2)
    assert call(h=icnn.handle) == -1 and b"not a star prior" in lib.awb_last_error()
    assert lib.awb_star_backward_workspace_bytes(icnn.handle, n) == -1
    assert lib.awb_star_backward_workspace_bytes(star.handle, 0) == -1
    assert call(n=0) == -1
    for name in ("params", "x", "dy", "grads", "ws"):
        assert call(**{name: None}) == -1, name
    assert call(h=None) == -1
    assert call(ws_bytes=need - 1) == -4
    assert call(dx=None) == 0
    assert call() == 0
    torch.cuda.synchronize()
