"""``second_order=True`` on the ICNN priors, without a GPU.

The flag travels through the constructors (and so through the reference's ``prior_model_args``), leaves the state_dict
alone, and is refused by the priors that have no second-order backward.  The autograd wiring of the second-order path
(``_PriorFunction`` -> ``_GridGradFunction``: which output goes where, pixel rows vs grids, the ``ydot`` -> dlogits path,
retained graphs) is checked against plain float64 autograd of the oracle, with a float64 stand-in for the native prior
that implements the same three calls the module makes (``backward``, ``grid_grad_backward`` and the forwards)."""
import pytest
import torch

import awesome_b200 as A
from awesome_b200.model.base import _PriorFunction
from oracle import prior_oracle as O


@pytest.mark.parametrize("cls,kw", [(A.ConvexNextNet, dict(n_hidden=16, n_hidden_layers=2)),
                                    (A.ConvexNet, dict(n_hidden=16))])
def test_flag_leaves_state_dict_unchanged(cls, kw):
    sds = []
    for args in (dict(kw), dict(kw, second_order=True), dict(kw, **{"second_order": False})):
        torch.manual_seed(3)
        m = cls(**args)                       # prior_model_type(**prior_model_args)
        assert m.second_order == args.get("second_order", False)
        sds.append(m.state_dict())
    for sd in sds[1:]:
        assert list(sd) == list(sds[0])
        for k in sd:
            assert torch.equal(sd[k], sds[0][k]), k


def test_other_priors_reject_the_flag():
    with pytest.raises(ValueError, match="second_order"):
        A.ConvexDiffeomorphismNet(n_hidden=16, nf_hidden=8, second_order=True)
    with pytest.raises(ValueError, match="second_order"):
        A.StarShapedNet(n_hidden=16, second_order=True)
    with pytest.raises(ValueError, match="second_order"):
        A.real_nvp_path_connected_net(channels=2, hidden_units=8, flow_n_flows=2, convex_net_hidden_units=16,
                                      second_order=True)
    m = A.real_nvp_path_connected_net(channels=2, hidden_units=8, flow_n_flows=2, convex_net_hidden_units=16)
    with pytest.raises(ValueError, match="second_order"):
        A.PathConnectedNet(convex_net=A.ConvexNextNet(n_hidden=16, second_order=True), flow_net=m.flow_net)
    A.StarShapedNet(n_hidden=16, second_order=False)


# --------------------------------------------------------------------------------- wiring, float64 stand-in prior
class _Float64Prior:
    """The native prior's calls, restated with float64 autograd on the oracle (pixel rows depend on their own row only)."""

    def __init__(self, module):
        self.names = [k for k, _ in module.named_parameters()]
        self.shapes = [p.shape for _, p in module.named_parameters()]

    def _params(self, arena):
        p, off = {}, 0
        for k, s in zip(self.names, self.shapes):
            n = s.numel()
            p[k] = arena[off:off + n].detach().double().reshape(s).requires_grad_(True)
            off += n
        return p

    @staticmethod
    def _rows(spec):
        g = spec.grid.double()
        return g.permute(0, 2, 3, 1).reshape(-1, g.shape[1]).clone().requires_grad_(True)

    def new_workspace(self, n_pixels, layout, device):
        return {"layout": layout}

    def forward(self, arena, spec, mode, ws, want_deformed=False):
        with torch.no_grad():
            y = O.icnn_forward(self._params(arena), self._rows(spec)).reshape(1, -1)
        return y.float(), None

    @torch.enable_grad()
    def backward(self, arena, spec, dlogits, ws, want_dgrid):
        p, x = self._params(arena), self._rows(spec)
        gs = torch.autograd.grad((dlogits.double().reshape(-1, 1) * O.icnn_forward(p, x)).sum(), list(p.values()) + [x])
        grads = torch.cat([g.reshape(-1) for g in gs[:-1]]).float().reshape(1, -1)
        dgrid = gs[-1].reshape(spec.B, spec.H, spec.W, -1).permute(0, 3, 1, 2).float() if want_dgrid else None
        return grads, dgrid

    @torch.enable_grad()
    def grid_grad_backward(self, arena, spec, w, u, ws):
        assert ws["layout"] == A._lib.AWB_WS_SECOND_ORDER
        assert u.is_contiguous() and u.shape == (spec.B, len(spec.grid[0]), spec.H, spec.W)
        p, x = self._params(arena), self._rows(spec)
        y = O.icnn_forward(p, x)
        J = torch.autograd.grad(y.sum(), x, create_graph=True)[0]
        ur = u.double().permute(0, 2, 3, 1).reshape(x.shape)
        ydot = (J * ur).sum(1)
        gs = torch.autograd.grad((w.double().reshape(-1) * ydot).sum(), list(p.values()), allow_unused=True)
        gs = [torch.zeros_like(q) if g is None else g for g, q in zip(gs, p.values())]
        return ydot.detach().float().reshape(1, -1), torch.cat([g.reshape(-1) for g in gs]).float().reshape(1, -1)


def _model(second_order=True):
    torch.manual_seed(0)
    m = A.ConvexNextNet(n_hidden=12, n_hidden_layers=2, second_order=second_order)
    fake = _Float64Prior(m)
    m._prior_for = lambda device: fake
    return m


def _apply(m, x):
    """``ArenaPriorModule._forward_any`` without the CUDA device guard."""
    params = m._arena_params()
    if x.dim() == 2:
        spec = A.GridSpecHost.from_tensor(x.t().reshape(1, x.shape[1], 1, x.shape[0]))
        return _PriorFunction.apply(m, spec, True, x, *params).reshape(-1, 1)
    spec = A.GridSpecHost.from_tensor(x)
    return _PriorFunction.apply(m, spec, True, x, *params).reshape(x.shape[0], 1, x.shape[2], x.shape[3])


def _penalised(model_out, x, which):
    y = model_out
    if which == "bce":
        g = torch.autograd.grad(torch.nn.functional.binary_cross_entropy_with_logits(y, torch.full_like(y, 0.3)), x,
                                create_graph=True)[0]
    else:
        g = torch.autograd.grad(y.sum(), x, create_graph=True)[0]
    if which == "eikonal":
        pen = (g.norm(dim=1 if x.dim() == 4 else -1) - 1).pow(2).mean()
    else:
        pen = g.pow(2).sum()
    return (torch.sigmoid(y) - 0.5).pow(2).mean() + 0.1 * pen


@pytest.mark.parametrize("which", ["sq", "eikonal", "bce"])
@pytest.mark.parametrize("rows", [False, True])
def test_wiring_against_float64_autograd(which, rows):
    m = _model()
    torch.manual_seed(1)
    x4 = torch.rand(2, 2, 5, 7)
    x0 = x4.permute(0, 2, 3, 1).reshape(-1, 2) if rows else x4
    x = x0.clone().requires_grad_(True)
    _penalised(_apply(m, x), x, which).backward()
    got = {k: p.grad for k, p in m.named_parameters()}

    ref = {k: v.detach().double().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    xr = x0.double().clone().requires_grad_(True)
    xrows = xr if rows else xr.permute(0, 2, 3, 1).reshape(-1, 2)
    y = O.icnn_forward(ref, xrows)
    y = y if rows else y.reshape(2, 5, 7, 1).permute(0, 3, 1, 2)
    _penalised(y, xr, which).backward()
    for k, p in ref.items():
        torch.testing.assert_close(got[k].double(), p.grad, rtol=1e-4, atol=1e-6, msg=k)
    # the grid receives the first-order part only (the ICNN is piecewise linear in it: float64 autograd agrees)
    torch.testing.assert_close(x.grad.double(), xr.grad, rtol=1e-4, atol=1e-6)


def test_retained_graph_and_parameter_gradient_penalty():
    m = _model()
    x = torch.rand(1, 2, 4, 6).requires_grad_(True)
    g = torch.autograd.grad(_apply(m, x).sum(), x, create_graph=True)[0]
    pen = g.pow(2).sum()
    pen.backward(retain_graph=True)
    first = [p.grad.clone() for p in m.parameters()]
    m.zero_grad()
    pen.backward()
    for a, p in zip(first, m.parameters()):
        assert torch.equal(a, p.grad)
    y = _apply(m, x)
    gp = torch.autograd.grad(y.sum(), list(m.parameters()) + [x], create_graph=True)
    with pytest.raises(RuntimeError, match="parameter gradients"):
        gp[0].pow(2).sum().backward()


def test_default_double_backward_still_raises():
    m = _model(second_order=False)
    x = torch.rand(1, 2, 4, 6).requires_grad_(True)
    g = torch.autograd.grad(_apply(m, x).sum(), x, create_graph=True)[0]
    with pytest.raises(RuntimeError, match="differentiate twice"):
        g.pow(2).sum().backward()
