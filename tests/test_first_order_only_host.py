"""The first-order-only backward of the prior autograd Functions (``awesome_b200/model/base.py``), on a CPU stand-in:
first derivatives are unchanged, and a double backward raises even when the upstream gradient is a constant (the case
torch's ``once_differentiable`` alone lets through as a silently constant gradient)."""
import pytest
import torch

from awesome_b200.model.base import _first_order_only


class _Cube(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return x ** 3

    @staticmethod
    @_first_order_only
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return g * 3 * x ** 2


def test_first_derivative_unchanged():
    x = torch.linspace(-1, 1, 7, dtype=torch.float64, requires_grad=True)
    w = torch.randn(7, dtype=torch.float64)
    (g,) = torch.autograd.grad((w * _Cube.apply(x)).sum(), x)
    assert torch.equal(g, w * 3 * x.detach() ** 2)
    assert not g.requires_grad


@pytest.mark.parametrize("upstream", ["constant", "weighted"])
def test_double_backward_raises(upstream):
    x = torch.linspace(-1, 1, 7, dtype=torch.float64, requires_grad=True)
    y = _Cube.apply(x)
    out = y.sum() if upstream == "constant" else (torch.randn(7, dtype=torch.float64, requires_grad=True) * y).sum()
    (g,) = torch.autograd.grad(out, x, create_graph=True)
    assert torch.equal(g.detach(), (3 * x ** 2).detach() if upstream == "constant" else g.detach())
    with pytest.raises(RuntimeError, match="differentiate twice"):
        (out + g.pow(2).sum()).backward()
