"""Autograd wiring of ``PathConnectedNet.inverse`` (``_InverseFunction``), without a GPU.

A float64 stand-in for the native prior implements the two calls the function makes (``inverse`` and
``inverse_backward``) with torch autograd of the oracle's inverse chain; the function's gradients must then equal plain
float64 autograd of the same chain: which gradient goes to which parameter, ``dgrid`` only when the points require grad,
one backward per forward, and no double backward."""
import pytest
import torch

import awesome_b200 as A
from awesome_b200 import _lib as L
from awesome_b200.model.base import _InverseFunction
from oracle import prior_oracle as O


def inverse_rows(p, x4):
    B, C_, H, W = x4.shape
    mn, mx, nmn, nmx = (p["flow_net.norm." + k] for k in ("min", "max", "new_min", "new_max"))
    z = O.flow_inverse(p, O.pixelize(O.minmax(x4, mn, mx, nmn, nmx)), O.FLOW_PREFIX)
    z = O.minmax(O.unpixelize(z, B, H, W), nmn, nmx, mn, mx)
    return O.pixelize((z - p["linear.bias"].view(1, C_, 1, 1)) / p["linear.weight"].view(1, C_, 1, 1))


class _Float64Prior:
    def __init__(self, module):
        self.module = module
        self.names = [k for k, _ in module.named_parameters()]
        self.shapes = [p.shape for _, p in module.named_parameters()]

    def _params(self, arena):
        p, off = {k: v.detach().double() for k, v in self.module.state_dict().items()}, 0
        for k, s in zip(self.names, self.shapes):
            n = s.numel()
            p[k] = arena[off:off + n].detach().double().reshape(s).requires_grad_(True)
            off += n
        return p

    def new_workspace(self, n_pixels, layout, device):
        return {"layout": layout, "records": False}

    def inverse(self, arena, spec, training, ws):
        assert ws["layout"] == L.AWB_WS_DEFORMATION and training
        ws["records"] = True
        with torch.no_grad():
            return inverse_rows(self._params(arena), spec.grid.double()).float()

    @torch.enable_grad()
    def inverse_backward(self, arena, spec, d_out, ws, want_dgrid):
        assert ws["records"] and d_out.is_contiguous() and d_out.dtype == torch.float32
        p, x = self._params(arena), spec.grid.double().clone().requires_grad_(True)
        leaves = [p[k] for k in self.names]
        gs = torch.autograd.grad((d_out.double() * inverse_rows(p, x)).sum(), leaves + [x], allow_unused=True)
        grads = torch.cat([(torch.zeros_like(q) if g is None else g).reshape(-1) for g, q in zip(gs[:-1], leaves)]).float()
        return grads, (gs[-1].float() if want_dgrid else None)


def _model():
    torch.manual_seed(0)
    m = A.real_nvp_path_connected_net(channels=2, hidden_units=8, flow_n_flows=4, flow_output_fn="tanh",
                                      convex_net_hidden_units=16)
    sd = m.state_dict()
    for k in sd:
        if ".net.2." in k:
            sd[k] = 0.05 * torch.randn_like(sd[k])
        elif k.endswith((".s", ".t")) and ".flows." in k:
            sd[k] = 0.1 * torch.randn_like(sd[k])
    sd["linear.weight"] = 1.0 + 0.3 * torch.randn_like(sd["linear.weight"])
    m.load_state_dict(sd)
    fake = _Float64Prior(m)
    m._prior_for = lambda device: fake
    return m


def _inverse(m, x):
    """``PathConnectedNet.inverse`` with grad, without the CUDA device guard."""
    m._ensure_flat()
    spec = A.GridSpecHost.from_tensor(x)
    rows = _InverseFunction.apply(m, spec, x if x.requires_grad else None, *m._arena_params())
    B, C_, H, W = x.shape
    return rows.reshape(B, H, W, C_).permute(0, 3, 1, 2)


@pytest.mark.parametrize("x_grad", [True, False])
def test_wiring_against_float64_autograd(x_grad):
    m = _model()
    torch.manual_seed(1)
    x0 = torch.rand(2, 2, 5, 7)
    w = torch.randn(2, 2, 5, 7)
    x = x0.clone().requires_grad_(x_grad)
    (w * _inverse(m, x)).sum().backward()
    ref = {k: v.detach().double().clone().requires_grad_(k in dict(m.named_parameters()))
           for k, v in m.state_dict().items()}
    xr = x0.double().clone().requires_grad_(True)
    y = inverse_rows(ref, xr).reshape(2, 5, 7, 2).permute(0, 3, 1, 2)
    (w.double() * y).sum().backward()
    for k, p in m.named_parameters():
        if k.startswith("convex_net."):
            assert int(torch.count_nonzero(p.grad)) == 0, k
        else:
            torch.testing.assert_close(p.grad.double(), ref[k].grad, rtol=1e-4, atol=1e-6, msg=k)
    if x_grad:
        torch.testing.assert_close(x.grad.double(), xr.grad, rtol=1e-4, atol=1e-6)
    else:
        assert x.grad is None


def test_once_per_forward_and_first_order_only():
    m = _model()
    x = torch.rand(1, 2, 3, 4, requires_grad=True)
    y = _inverse(m, x)
    y.sum().backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="once per forward"):
        y.sum().backward()
    y = _inverse(m, x)
    g = torch.autograd.grad(y.sum(), x, create_graph=True)[0]
    with pytest.raises(RuntimeError, match="differentiate twice"):
        g.pow(2).sum().backward()
