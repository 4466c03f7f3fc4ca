"""CPU checks of the batched reverse-mode glue that need no GPU."""
import pytest
import torch

from pdivgnn_b200 import _lib


class _Toy(torch.autograd.Function):
    """y = 2 x whose backward hands its cotangent to the library's pointer path, as _EPDFunction.backward does."""

    @staticmethod
    def forward(ctx, x):
        return 2 * x

    @staticmethod
    def backward(ctx, g):
        _lib.raw(g)
        return 2 * g


def test_legacy_batched_cotangent_is_refused():
    """torch.autograd.grad(..., is_grads_batched=True) runs the backward under torch's legacy vmap, whose tensors have no
    storage: the library refuses them and points to the torch.func entry points."""
    x = torch.ones(3, requires_grad=True)
    with pytest.raises(NotImplementedError, match="torch.func.jacrev"):
        torch.autograd.grad(_Toy.apply(x), x, torch.eye(3), is_grads_batched=True)
    (g,) = torch.autograd.grad(_Toy.apply(x), x, torch.ones(3))  # a plain cotangent passes
    assert torch.equal(g, torch.full((3,), 2.0))


def test_is_vmapped():
    t = torch.zeros(2, 3)
    assert not _lib.is_vmapped(t)
    seen = []
    torch.func.vmap(lambda r: seen.append(_lib.is_vmapped(r)) or r)(t)
    assert seen == [True]
    assert _lib.raw(t) is t
