"""The yardstick of the loss-kernel tests (test_gpu_loss.py): ``O.loss_fp64``, the vectorised fp64 restatement of the
training loss and its gradient, agrees to 1e-12 with the oracle's per-graph loop of ``train_loss``
(``normalized_mse_loss_single``, ``compute_divergence`` on the densified, column-sliced row block, autograd for the
gradient), run in fp64 from the same fp32 inputs.  Batches: the goldens, the synthetic batch, and random ragged batches
with empty rows, columns past 2 N_i, duplicates, a graph whose every entry is dropped and labels outside {-1, 0, 1}.

The random batch builder below is shared with test_gpu_loss.py."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import pdg_helpers as H
from oracle import pdg_oracle as O


# ---- batch builder ----------------------------------------------------------------------------------------------
def p1_operator(n, rng):
    """(row, col, val) of the nodal-average P1 divergence (synth._p1_divergence_operator) on a Delaunay triangulation of
    n random points of the unit square: about 14 entries a row, columns in [0, 2n)."""
    from scipy.spatial import Delaunay
    from pdivgnn_b200 import synth
    pts = rng.random((n, 2))
    tri = Delaunay(pts).simplices.copy()
    x, y = pts[:, 0], pts[:, 1]
    i, j, k = tri.T
    cw = (x[j] - x[i]) * (y[k] - y[i]) - (x[k] - x[i]) * (y[j] - y[i]) < 0
    tri[cw, 1], tri[cw, 2] = tri[cw, 2], tri[cw, 1].copy()
    return synth._p1_divergence_operator(pts, tri)


def random_operator(n, rng, per_row=4, empty=0.2):
    """Random sparse rows: Poisson(per_row) entries each (a share `empty` forced empty), columns in [0, 2n)."""
    k = rng.poisson(per_row, n)
    k[rng.random(n) < empty] = 0
    row = np.repeat(np.arange(n), k)
    col = rng.integers(0, 2 * n, row.size)
    return row, col, rng.standard_normal(row.size)


def make_batch(sizes, seed=0, op="mix", labels="mixed", values="normal", width=None, wide=0, dups=0.0, dropped=(),
               hub_row=None, hub_col=None, exact=(), illcond=(), empty_op=False, mean_ls=2.5, std_ls=40.0):
    """A collated batch on the CPU: raw ground truth, standardised prediction, row-stacked fp32 operator with
    graph-local columns (width = max 2 N_i unless given, uncoalesced when `dups`), labels [N, 1].

    op: "p1" (mesh operators with their values, random rows below 4 nodes), "rand", or "mix" (alternating).  values: "normal" or "wide"
    (magnitudes 1e-6 .. 1e6).  wide: entries per graph with columns in [2 N_i, width).  dups: share of entries
    repeated with a second value.  dropped: graphs whose every column lies past 2 N_i.  hub_row / hub_col: graph
    index with one row of 2 500 entries / one stacked-stress column read by 2 500 rows.  exact: graphs with
    pred == gt.  illcond: graphs whose ground truth has mean 1e4 x its spread.  labels: "zero", "pm1", "mixed"
    ({-1, 0, 1}) or "two" (also 2, -2, 3)."""
    rng = np.random.default_rng(seed)
    sizes = [int(s) for s in sizes]
    ptr = np.concatenate([[0], np.cumsum(sizes)])
    n = int(ptr[-1])
    if width is None:
        width = 2 * max(sizes)
    if dropped or wide:
        width = max(width, 2 * max(sizes) + 16)
    rows, cols, vals = [], [], []

    def add(r, c, v=None):
        rows.append(r + ptr[gi])
        cols.append(c)
        vals.append(rng.standard_normal(r.size) * 10.0 ** rng.uniform(-1, 1, r.size) if v is None else v)

    for gi, ni in enumerate(sizes):
        if empty_op:
            break
        kind = op if op != "mix" else ("p1" if gi % 2 == 0 else "rand")
        r, c, v = p1_operator(ni, rng) if kind == "p1" and ni >= 4 else random_operator(ni, rng)
        if gi in dropped:
            c = rng.integers(2 * ni, width, c.size)
        add(r, c, v)
        if hub_row == gi:
            c = rng.choice(2 * ni, min(2500, 2 * ni), replace=False)
            add(np.full(c.size, ni // 2), c)
        if hub_col == gi:
            r = rng.choice(ni, min(2500, ni), replace=False)
            add(r, np.full(r.size, ni + ni // 3))
        if wide:
            add(rng.integers(0, ni, wide), rng.integers(2 * ni, width, wide))
    cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)  # noqa: E731
    row, col, val = cat(rows, np.int64), cat(cols, np.int64), cat(vals, np.float64)
    _, first = np.unique(row * width + col, return_index=True)  # one value per position, duplicates added below
    row, col, val = row[first], col[first], val[first]
    if values == "wide":
        val = rng.choice([-1.0, 1.0], row.size) * 10.0 ** rng.uniform(-6, 6, row.size)
    if dups:
        pick = np.nonzero(rng.random(row.size) < dups)[0]
        row, col = np.concatenate([row, row[pick]]), np.concatenate([col, col[pick]])
        val = np.concatenate([val, rng.standard_normal(pick.size)])
        perm = rng.permutation(row.size)
        row, col, val = row[perm], col[perm], val[perm]
    opm = torch.sparse_coo_tensor(torch.from_numpy(np.stack([row, col]).astype(np.int64)),
                                  torch.from_numpy(val.astype(np.float32)), (n, width))
    if not dups:
        opm = opm.coalesce()
    lab = {"zero": lambda: np.zeros(n), "pm1": lambda: rng.choice([-1, 1], n), "mixed": lambda: rng.integers(-1, 2, n),
           "two": lambda: rng.choice([-2, -1, 0, 1, 2, 3], n)}[labels]()
    mean_ls, std_ls = float(np.float32(mean_ls)), float(np.float32(std_ls))
    ls = mean_ls + std_ls * rng.standard_normal((n, 3))
    for gi in illcond:
        ls[ptr[gi]:ptr[gi + 1]] = mean_ls + std_ls * (1e4 + rng.standard_normal((sizes[gi], 3)))
    ls = torch.from_numpy(ls.astype(np.float32))
    gt = O.loss_fp64(torch.zeros(n, 3), ls, mean_ls, std_ls, torch.from_numpy(ptr), divergence=False).gt
    pred = gt + torch.from_numpy(rng.standard_normal((n, 3)).astype(np.float32))
    for gi in exact:
        pred[ptr[gi]:ptr[gi + 1]] = gt[ptr[gi]:ptr[gi + 1]]
    return SimpleNamespace(pred=pred, local_stress=ls, mean_ls=mean_ls, std_ls=std_ls, ptr=torch.from_numpy(ptr),
                           op_div_matrix=opm, surfaces_nodes_for_div=torch.from_numpy(lab.astype(np.int64))[:, None],
                           batch_size=len(sizes))


# ---- the oracle's loop ------------------------------------------------------------------------------------------
def loop_fp64(b, divergence, penalty, upstream):
    """train_loss's per-graph loop (gnn_train.py:162-202) on fp64 copies of the fp32 prediction and standardised
    ground truth; per-node divergence from the same densified, column-sliced block compute_divergence multiplies."""
    t = torch.tensor
    gt = ((b.local_stress - t(b.mean_ls, dtype=torch.float32)) / t(b.std_ls, dtype=torch.float32)).double()
    p = b.pred.double().requires_grad_(True)
    op = b.op_div_matrix.coalesce().double()
    ptr = b.ptr.tolist()
    nmse_g, div_g, div_node = [], [], []
    for i in range(b.batch_size):
        s, e = ptr[i], ptr[i + 1]
        nmse_g.append(O.normalized_mse_loss_single(gt[s:e], p[s:e]))
        if divergence:
            blk = O.op_div_row_block(op, s, e)
            lab = b.surfaces_nodes_for_div[s:e]
            div_g.append(O.compute_divergence(p[s:e], blk, lab))
            d = blk.to_dense()[:, : (e - s) * 2] @ O._stack_stress(p[s:e])
            d[lab.squeeze(1) == 1] = 0
            d[lab.squeeze(1) == -1] = 0
            div_node.append(d)
    nmse = sum(nmse_g) / b.batch_size
    div = sum(g * penalty for g in div_g) / b.batch_size if divergence else torch.zeros((), dtype=torch.float64)
    outs = [o for o, w in zip((nmse, div), upstream) if o.requires_grad]
    ws = [torch.tensor(w, dtype=torch.float64) for o, w in zip((nmse, div), upstream) if o.requires_grad]
    grad, = torch.autograd.grad(outs, p, ws)
    return SimpleNamespace(gt=gt, nmse_graph=torch.stack(nmse_g).detach(), nmse=nmse.detach(), div=div.detach(),
                           div_graph=torch.stack(div_g).detach() if divergence else None,
                           div_node=torch.cat(div_node).detach() if divergence else None, grad=grad)


def _close(a, b, what):
    """|a - b| <= 1e-12 max|b| element by element; inf / NaN (graphs of one node have a zero norm) in the same places."""
    a, b = torch.as_tensor(a, dtype=torch.float64), torch.as_tensor(b, dtype=torch.float64)
    fin = torch.isfinite(b)
    assert torch.equal(torch.isfinite(a), fin) and torch.equal(a[~fin].nan_to_num(), b[~fin].nan_to_num()), what
    scale = b[fin].abs().max().item() if fin.any() else 0.0
    err = (a[fin] - b[fin]).abs().max().item() if fin.any() else 0.0
    assert err <= 1e-12 * scale, (what, err, scale)


def _pin(b, divergence=True, penalty=10.0, upstream=(1.0, 1.0)):
    r = O.loss_fp64(b.pred, b.local_stress, b.mean_ls, b.std_ls, b.ptr, b.op_div_matrix, b.surfaces_nodes_for_div,
                    divergence, penalty, upstream)
    o = loop_fp64(b, divergence, penalty, upstream)
    assert torch.equal(r.gt.double(), o.gt)  # the same fp32 standardisation
    _close(r.nmse_graph, o.nmse_graph, "nmse_graph")
    _close(r.nmse, o.nmse, "nmse")
    _close(r.div, o.div, "div")
    _close(r.total, o.nmse + o.div, "total")
    _close(r.grad, o.grad, "grad")
    if divergence:
        _close(r.div_graph, o.div_graph, "div_graph")
        _close(r.div_node, o.div_node, "div_node")
        lab = b.surfaces_nodes_for_div.squeeze(1)
        assert r.div_node.abs().max() > 0 or ((lab == 1) | (lab == -1)).all() or b.op_div_matrix._nnz() == 0
    return r


GOLDEN = ["train2_div", "train2_nodiv", "train3_noperiodic", "train2_quad"]


@pytest.mark.parametrize("name", GOLDEN)
def test_restatement_matches_oracle_loop_on_goldens(name):
    g = H.load_golden(name)
    _, batch, stats = H.oracle_batch_from_samples(H.golden_samples(g), bool(g["periodic"]))
    b = SimpleNamespace(pred=torch.from_numpy(g["pred_std"]), local_stress=batch.local_stress,
                        mean_ls=stats["mean_local_stress"].item(), std_ls=stats["std_local_stress"].item(), ptr=batch.ptr,
                        op_div_matrix=batch.op_div_matrix, surfaces_nodes_for_div=batch.surfaces_nodes_for_div,
                        batch_size=batch.batch_size)
    r = _pin(b, bool(g["divergence"]), float(g["penalty"]))
    # and the fp32 reference's own loss, as written by the golden, to fp32 accuracy
    assert abs(r.total.item() - float(g["loss"])) <= 1e-5 * abs(float(g["loss"]))


def test_restatement_matches_oracle_loop_on_synthetic_batch():
    _, _, batch, stats = H.synthetic_batch(3, 600, seed0=69)
    b = SimpleNamespace(pred=torch.randn(batch.num_nodes, 3, generator=torch.Generator().manual_seed(5)),
                        local_stress=batch.local_stress, mean_ls=stats["mean_local_stress"].item(),
                        std_ls=stats["std_local_stress"].item(), ptr=batch.ptr, op_div_matrix=batch.op_div_matrix,
                        surfaces_nodes_for_div=batch.surfaces_nodes_for_div, batch_size=batch.batch_size)
    _pin(b, True, 10.0, (0.3, -2.5))


RAGGED = {
    "mixed_ops": dict(sizes=[1, 2, 5, 40, 257], op="mix"),
    "wide_columns_dups": dict(sizes=[3, 17, 60, 9], op="rand", wide=5, dups=0.3, labels="pm1"),
    "dropped_graph_label_two": dict(sizes=[30, 12, 45], op="mix", dropped=(1,), labels="two", values="wide"),
    "hubs_exact_illcond": dict(sizes=[1300, 20, 8], op="rand", hub_row=0, hub_col=0, exact=(1,), illcond=(2,)),
    "empty_operator": dict(sizes=[4, 9], empty_op=True),
}


@pytest.mark.parametrize("case", list(RAGGED))
@pytest.mark.parametrize("upstream", [(1.0, 1.0), (0.3, -2.5), (1.0, 0.0), (0.0, 1.0)])
def test_restatement_matches_oracle_loop_on_ragged_batches(case, upstream):
    b = make_batch(seed=len(case), **RAGGED[case])
    _pin(b, True, 10.0, upstream)
    _pin(b, False, 10.0, upstream)


def test_restatement_mask_and_empty_operator():
    """Labels other than 1 and -1 keep their row; an operator without entries gives a divergence of exactly 0."""
    b = make_batch([6, 7], seed=3, op="rand", labels="two")
    r = O.loss_fp64(b.pred, b.local_stress, b.mean_ls, b.std_ls, b.ptr, b.op_div_matrix, b.surfaces_nodes_for_div)
    lab = b.surfaces_nodes_for_div.squeeze(1)
    assert (r.div_node[(lab == 1) | (lab == -1)] == 0).all()
    assert (r.div_node[(lab == 2) | (lab == 3)] != 0).any()
    e = make_batch([6, 7], seed=3, empty_op=True)
    r = O.loss_fp64(e.pred, e.local_stress, e.mean_ls, e.std_ls, e.ptr, e.op_div_matrix, e.surfaces_nodes_for_div)
    r0 = O.loss_fp64(e.pred, e.local_stress, e.mean_ls, e.std_ls, e.ptr, divergence=False)
    assert r.div.item() == 0.0 and (r.div_node == 0).all() and torch.equal(r.grad, r0.grad)
