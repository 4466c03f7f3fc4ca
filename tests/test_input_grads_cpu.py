"""The yardstick of the input-gradient tests (test_gpu_input_grads.py): the oracle's fp64 gradients with respect to
mean_stress, pos and edge_attr agree with central finite differences on the 3x3 grid (SURVEY 2.4)."""
from types import SimpleNamespace

import numpy as np
import torch

import pdg_helpers as H
from oracle import pdg_oracle as O


def _grid_batch():
    g = H.load_golden("grid3x3")
    pos = torch.from_numpy(np.asarray(g["pos"], dtype=np.float64))[:, :2]
    ei = torch.from_numpy(np.asarray(g["edge_index"], dtype=np.int64))
    ea = torch.from_numpy(np.asarray(g["edge_attr"], dtype=np.float64))
    n = pos.shape[0]
    gen = torch.Generator().manual_seed(4)
    ms = (torch.rand(1, 3, generator=gen, dtype=torch.float64) * 2 - 1).expand(n, 3) * 40.0
    ms = ms + 0.5 * torch.randn(n, 3, generator=gen, dtype=torch.float64)  # per-node values: every entry is exercised
    types = torch.tensor([1, 1, 1, 1, 0, 1, 1, 1, 1], dtype=torch.int64)[:, None]
    return SimpleNamespace(pos=pos, edge_index=ei, edge_attr=ea, mean_stress=ms, nodes_types=types, batch_size=1,
                           ptr=torch.tensor([0, n]), batch=torch.zeros(n, dtype=torch.int64), num_nodes=n)


def test_oracle_fp64_input_gradients_match_central_differences():
    b = _grid_batch()
    t = torch.tensor
    stats = dict(mean_pos=t(0.5), std_pos=t(0.35), mean_mean_stress=t(0.), std_mean_stress=t(30.), mean_local_stress=t(0.),
                 std_local_stress=t(45.), mean_edge_weight=t(0.4), std_edge_weight=t(0.2))
    sd = {k: v.double() for k, v in O.init_state_dict(seed=69).items()}
    w = torch.randn(b.num_nodes, 3, generator=torch.Generator().manual_seed(5), dtype=torch.float64)

    def loss(**inputs):
        bb = SimpleNamespace(**{**vars(b), **inputs})
        return (O.forward(sd, bb, stats, 3, scale_output=False, scale_input=True, dtype=torch.float64) * w).sum()

    keys = ("mean_stress", "pos", "edge_attr")
    leaves = {k: getattr(b, k).clone().requires_grad_(True) for k in keys}
    grads = dict(zip(keys, torch.autograd.grad(loss(**leaves), list(leaves.values()))))
    for k in keys:
        x0 = getattr(b, k)
        fd = torch.empty_like(x0).reshape(-1)
        h = 1e-6 * max(1.0, x0.abs().max().item())
        for i in range(x0.numel()):
            xp, xm = x0.clone().reshape(-1), x0.clone().reshape(-1)
            xp[i] += h
            xm[i] -= h
            with torch.no_grad():
                fd[i] = (loss(**{k: xp.view_as(x0)}) - loss(**{k: xm.view_as(x0)})) / (2 * h)
        linf, l2 = H.rel_err(grads[k], fd.view_as(x0))
        assert grads[k].abs().max() > 0, k
        assert linf < 1e-5 and l2 < 1e-5, (k, linf, l2)
