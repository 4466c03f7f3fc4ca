"""The yardstick of the forward-mode tests (test_gpu_jvp.py): the oracle's fp64 JVP (torch.func.jvp through O.forward)
agrees with central finite differences on the 3x3 grid, along each input direction alone and all three together.
h = 1e-6: larger steps cross ReLU kinks (the combined direction is off by 2e-3 at h = 1e-5)."""
from types import SimpleNamespace

import pytest
import torch
import torch.autograd.forward_ad as fwAD

import pdg_helpers as H
from oracle import pdg_oracle as O
from test_input_grads_cpu import _grid_batch

KEYS = ("mean_stress", "pos", "edge_attr")


def _setup():
    b = _grid_batch()
    t = torch.tensor
    stats = dict(mean_pos=t(0.5), std_pos=t(0.35), mean_mean_stress=t(0.), std_mean_stress=t(30.), mean_local_stress=t(0.),
                 std_local_stress=t(45.), mean_edge_weight=t(0.4), std_edge_weight=t(0.2))
    sd = {k: v.double() for k, v in O.init_state_dict(seed=69).items()}

    def f(*xs):
        bb = SimpleNamespace(**{**vars(b), **dict(zip(KEYS, xs))})
        return O.forward(sd, bb, stats, 3, scale_output=True, scale_input=True, dtype=torch.float64)
    return b, f, tuple(getattr(b, k) for k in KEYS)


def _direction(x0, which, seed=3):
    g = torch.Generator().manual_seed(seed)
    return tuple(torch.randn(x.shape, generator=g, dtype=torch.float64) if which in ("all", k) else torch.zeros_like(x)
                 for k, x in zip(KEYS, x0))


@pytest.mark.parametrize("which", ["mean_stress", "pos", "edge_attr", "all"])
def test_oracle_fp64_jvp_matches_central_differences(which):
    _, f, x0 = _setup()
    v = _direction(x0, which)
    _, jv = torch.func.jvp(f, x0, v)
    h = 1e-6
    fd = (f(*[x + h * d for x, d in zip(x0, v)]) - f(*[x - h * d for x, d in zip(x0, v)])) / (2 * h)
    linf, l2 = H.rel_err(jv, fd)
    assert jv.abs().max() > 0
    assert linf < 1e-5 and l2 < 1e-5, (which, linf, l2)


def test_oracle_forward_ad_equals_func_jvp():
    """The two forward-mode front ends torch offers give the same fp64 bits on the oracle."""
    _, f, x0 = _setup()
    v = _direction(x0, "all")
    _, jv = torch.func.jvp(f, x0, v)
    with fwAD.dual_level():
        t = fwAD.unpack_dual(f(*[fwAD.make_dual(x, d) for x, d in zip(x0, v)])).tangent
    assert torch.equal(t, jv)
