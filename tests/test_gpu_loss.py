"""The fused loss kernels (pdg_loss.cu: k_loss_graph, k_loss_finish, k_loss_backward and the operator plan) against
the fp64 restatement ``O.loss_fp64`` (pinned to the oracle's loop by test_loss_cpu.py), element by element.

Every value is judged against its own a-priori rounding bound and the test fails when error / bound > 1 anywhere.
The bounds are first-order bounds, u = 2^-24, gamma_m = m u / (1 - m u), times SAFETY = 2 for the second-order terms
and for using exact rather than computed magnitudes inside them.  fp64 sums of k terms add (k + 16) 2^-53 of the sum
of magnitudes.  The kernel's arithmetic, step by step:

* divergence of node n over its m kept entries: the fmaf chain d = sum_k v_k s_k gives
  |dd| <= gamma_m sum_k |v_k s_k|.  Rows labelled 1 or -1 are exactly 0.
* per-graph divergence D = sum_c sum_n d_nc^2 / N: each fl(d^2) is off by |dd| (2|d| + |dd|) + u (|d| + |dd|)^2; the
  fp64 sum is rounded to fp32 (u), N to fp32 (u), the quotient (u), the two columns added and rounded (u):
  sum_c E_c / N + 4 u D.
* NMSE of a graph, q_c = mse_c / norm_c, nmse = mean_c q_c:
  - mse: fl(gt - p) and fl(d * d) are fp32 roundings, the fp64 sum is rounded to fp32: gamma_3 d^2 per node, u mse.
  - norm: the mean is an fp64 sum rounded to fp32, |dm| <= u |m| (+ the fp64 sum's error); e = fl(gt - m~) is then off
    by de = |dm| + u (|e| + |dm|), and fl(e~^2) by de (2|e| + de) + u (|e| + de)^2, i.e. u |e| (2|m| + 3|e|) at first
    order: the bound scales with |mean_gt| |e|, not with norm, so a mean 1e4 x the spread is judged fairly.  The sum
    is rounded to fp32 (u norm).
  - q~ = fl(mse~ / norm~): |dq| <= E_mse / norm + q E_norm / norm + u q; the fp64 mean of three is rounded (u).
* d loss / d pred, NMSE part G = g_nmse 2 (p - gt) / (3 B norm_c): fl(p - gt), 1 / fl(norm~), the product, the
  upstream product, fl(3B) and the quotient: |dG| <= |G| (E_norm / norm + 6 u).
* divergence part: coefficient C = g_div penalty 2 / (N B) (four fp32 roundings) times a CSC gather
  X = sum_k v_k d_row(k) over the m' entries that read this stacked-stress value (fmaf chain):
  |dX| <= gamma_m' sum |v d| + sum |v| |dd_row|; sxy adds two such sums (u); the product with C (u):
  |C| (|dX| + 5 u |X|).  The two parts are added (u |G_total|).
* totals: k_loss_finish adds the B per-graph terms in order in fp32 (gamma_B sum |term|, and for the divergence one
  product with the penalty each) and divides by B (u), on top of the per-term bounds.

Graphs of one node have a zero norm (and so an infinite NMSE); where the restatement is not finite the kernel must
give the same inf or NaN.

The cases mix triangle-mesh P1 operators (about 14 entries a row) with random sparse rows, and cover: graph sizes
around the 256-thread block stride, one graph, 4096 graphs of 1-5 nodes, total N at 2^16 - 1, 2^16 and 2^16 + 1 (the
CSC radix sort's bit count changes at 2^16), empty rows, a 2 500-entry row and a 2 500-entry column, columns in
[2 N_i, width), uncoalesced duplicates, a graph with every entry dropped, values 1e-6 .. 1e6, an empty operator,
labels all 0 / all +-1 / mixed / outside {-1, 0, 1}, pred == gt, an ill-conditioned norm, penalties 0 .. 1e4, the
upstream weights of nmse + div, (0.3, -2.5), nmse alone, div alone, divergence off, and one graph of 2^24 + 1 nodes
(N_i does not survive a round trip through fp32 there).

The per-graph terms and per-node divergences are read from the workspace of the C ABI (``pdg_loss``'s layout: B
rows of 8 floats {nmse_i, div_i, ...}, then the [N, 2] divergence at the next 256-byte boundary); the same call
through ``nmse_div_loss`` must give the same bits."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import pdg_helpers as H
from oracle import pdg_oracle as O
from test_loss_cpu import make_batch

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
E64 = 2.0 ** -53
SAFETY = 2.0
F32 = torch.float32


def gamma(m):
    m = torch.as_tensor(m, dtype=torch.float64)
    return m * U / (1 - m * U)


def _f32(x):
    return float(np.float32(x))


_MODELS = {}


def _model(mean_ls, std_ls):
    key = (mean_ls, std_ls)
    if key not in _MODELS:
        t = torch.tensor
        stats = dict(mean_pos=t(0.), std_pos=t(1.), mean_mean_stress=t(0.), std_mean_stress=t(1.),
                     mean_local_stress=t(mean_ls), std_local_stress=t(std_ls), mean_edge_weight=t(0.),
                     std_edge_weight=t(1.))
        _MODELS[key] = H.make_model(stats, steps=1)
    return _MODELS[key]


def _device(b):
    return SimpleNamespace(**{k: (v.cuda() if torch.is_tensor(v) else v) for k, v in vars(b).items()})


# ---- the kernels, through loss.py and through the C ABI ----------------------------------------------------------
def run_loss(db, divergence, penalty, upstream):
    """nmse_div_loss + torch.autograd.grad.  upstream: (g_nmse, g_div), "nmse" (nmse.backward() alone) or "div"."""
    from pdivgnn_b200 import nmse_div_loss
    pred = db.pred.clone().requires_grad_(True)
    nmse, div = nmse_div_loss(pred, db, _model(db.mean_ls, db.std_ls), divergence, penalty)
    if upstream == "nmse":
        grad, = torch.autograd.grad(nmse, pred)
    elif upstream == "div":
        grad, = torch.autograd.grad(div, pred)
    else:
        w = [torch.tensor(_f32(x), device="cuda") for x in upstream]
        grad, = torch.autograd.grad((nmse, div), pred, w)
    return torch.stack([nmse.detach(), div.detach()]), grad


def upstream_pair(upstream):
    return {"nmse": (1.0, 0.0), "div": (0.0, 1.0)}.get(upstream, upstream) if isinstance(upstream, str) else \
        tuple(_f32(x) for x in upstream)


def run_abi(db, divergence, penalty, upstream, poison=None):
    """pdg_opdiv_plan_build + pdg_loss + pdg_loss_backward on buffers filled with `poison` first (None: not filled).
    Returns (out2, per-graph [B, 2] {nmse_i, div_i}, divergence [N, 2], grad)."""
    from pdivgnn_b200 import _lib
    L = _lib.lib()
    op = db.op_div_matrix.coalesce()
    idx, val = op.indices().contiguous(), op.values().contiguous()
    n, b, nnz = db.pred.shape[0], db.ptr.numel() - 1, idx.shape[1]
    plan = torch.empty(L.pdg_opdiv_plan_bytes(n, nnz), dtype=torch.uint8, device="cuda")
    tb = L.pdg_opdiv_tmp_bytes(n, nnz)
    tmp = torch.empty(tb, dtype=torch.uint8, device="cuda")
    wsb = L.pdg_loss_ws_bytes(n, b)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    if poison is not None:
        for t in (plan, tmp, ws):
            t.fill_(poison)
    st = _lib.stream_ptr()
    norm = _lib.PdgNorm(mean_local_stress=db.mean_ls, std_local_stress=db.std_ls)
    P = _lib.ptr
    lab = db.surfaces_nodes_for_div.reshape(-1).contiguous()
    _lib.check(L.pdg_opdiv_plan_build(P(idx[0]), P(idx[1]), nnz, P(db.ptr), b, n, P(plan), P(tmp), tb, st), "plan")
    out2 = torch.empty(2, dtype=F32, device="cuda")
    _lib.check(L.pdg_loss(P(db.pred), P(db.local_stress), C.byref(norm), P(db.ptr), b, n, P(lab), P(plan), P(val), nnz,
                          int(divergence), float(penalty), P(ws), P(out2), st), "pdg_loss")
    up = torch.tensor(upstream_pair(upstream), dtype=F32, device="cuda")
    grad = torch.empty_like(db.pred)
    _lib.check(L.pdg_loss_backward(P(db.pred), P(db.local_stress), C.byref(norm), P(db.ptr), b, n, P(plan), P(val), nnz,
                                   int(divergence), float(penalty), P(ws), P(up), P(grad), st), "pdg_loss_backward")
    off = -(-(b * 8 * 4) // 256) * 256
    per_graph = ws[: b * 32].view(F32).view(b, 8)[:, :2].clone()
    gdiv = ws[off: off + n * 8].view(F32).view(n, 2).clone()
    return out2, per_graph, gdiv, grad


# ---- bounds ---------------------------------------------------------------------------------------------------------
def bounds(db, divergence, penalty, upstream):
    """The restatement's values and the bound of each kernel output (module docstring)."""
    g_nmse, g_div = upstream_pair(upstream)
    r = O.loss_fp64(db.pred, db.local_stress, db.mean_ls, db.std_ls, db.ptr, db.op_div_matrix,
                    db.surfaces_nodes_for_div, divergence, penalty, (g_nmse, g_div))
    f64, dev = torch.float64, db.pred.device
    ptr = db.ptr
    b, n = ptr.numel() - 1, db.pred.shape[0]
    cnt = ptr[1:] - ptr[:-1]
    ni = cnt.to(f64)
    gid = torch.repeat_interleave(torch.arange(b, device=dev), cnt)
    seg = lambda x: torch.zeros(b, *x.shape[1:], dtype=f64, device=dev).index_add_(0, gid, x)  # noqa: E731
    s64 = ((ni + 16) * E64)[:, None]
    p, t = db.pred.to(f64), r.gt.to(f64)
    # NMSE
    mean = seg(t) / ni[:, None]
    dm = U * mean.abs() + s64 * seg(t.abs()) / ni[:, None]
    e = t - mean[gid]
    de = dm[gid] + U * (e.abs() + dm[gid])
    norm = seg(e.square())
    e_norm = seg(de * (2 * e.abs() + de) + U * (e.abs() + de).square()) + (U + s64) * norm
    d = p - t
    mse = seg(d.square())
    e_mse = (gamma(3) + U + s64) * mse
    q = mse / norm
    nmse_b = (e_mse / norm + q * e_norm / norm + U * q).sum(1) / 3 + U * r.nmse_graph
    grad_b = (r.grad.abs() if not divergence else (g_nmse * 2 * d / norm[gid] / (3 * b)).abs()) * \
        (e_norm / norm + 6 * U)[gid]
    out = SimpleNamespace(r=r, nmse_graph=nmse_b, div_graph=None, div_node=None)
    if divergence:
        row, node, first, val = O.opdiv_entries(db.op_div_matrix, ptr)
        v = val.to(f64).abs()[:, None]
        s = torch.where(first[:, None], p[node][:, [0, 2]], p[node][:, [2, 1]]).abs()
        m = torch.zeros(n, dtype=f64, device=dev).index_add_(0, row, torch.ones_like(val, dtype=f64))
        a = torch.zeros(n, 2, dtype=f64, device=dev).index_add_(0, row, v * s)
        lab = db.surfaces_nodes_for_div.reshape(-1)
        kept = ((lab != 1) & (lab != -1)).to(f64)[:, None]
        dd = gamma(m)[:, None] * a * kept
        dn = r.div_node.abs()
        e_sq = dd * (2 * dn + dd) + U * (dn + dd).square()
        div_b = (seg(e_sq) + s64 * seg(dn.square())).sum(1) / ni + 4 * U * r.div_graph
        out.div_node, out.div_graph = dd, div_b
        # CSC gathers: [node, first?, column of d] sums of |v d| and |v| dd, and entry counts per stacked-stress value
        k = node * 2 + first.long()
        zs = lambda w: torch.zeros(2 * n, *w.shape[1:], dtype=f64, device=dev).index_add_(0, k, w).view(n, 2, *w.shape[1:])  # noqa: E731
        mc = zs(torch.ones_like(val, dtype=f64))
        xa, xd = zs(v * dn[row]), zs(v * dd[row])
        xs = zs(val.to(f64)[:, None] * r.div_node[row])
        ex = gamma(mc)[..., None] * xa + xd  # [n, first?, c]
        coef = (g_div * penalty * 2.0 / (ni * b))[gid].abs()
        # sxx = a0 (first, c0); syy = b1 (second, c1); sxy = b0 + a1 (second c0 + first c1)
        e0 = ex[:, 1, 0] + 5 * U * xs[:, 1, 0].abs()
        e1 = ex[:, 0, 1] + 5 * U * xs[:, 0, 1].abs()
        x2 = xs[:, 0, 0] + xs[:, 1, 1]
        e2 = ex[:, 0, 0] + ex[:, 1, 1] + U * x2.abs() + 5 * U * x2.abs()
        gdiv_b = coef[:, None] * torch.stack([e0, e1, e2], 1)
        g_nm = (g_nmse * 2 * d / norm[gid] / (3 * b)).abs() * (e_norm / norm + 6 * U)[gid]
        grad_b = g_nm + gdiv_b
    out.grad = grad_b + U * r.grad.abs()
    # totals
    out.nmse = (nmse_b.sum() + gamma(b) * r.nmse_graph.abs().sum()) / b + U * r.nmse.abs()
    out.div = penalty * ((out.div_graph.sum() if divergence else 0.0) + gamma(b + 1) * r.div_graph.abs().sum()) / b + \
        U * r.div.abs()
    return out


def ratio(got, want, bound, what):
    """Worst |got - want| / bound; inf / NaN of the restatement must be matched exactly; bound 0 means exactly equal."""
    got, want, bound = got.to(torch.float64), want.to(torch.float64), torch.as_tensor(bound, dtype=torch.float64)
    fin = torch.isfinite(want)
    assert torch.equal(torch.isfinite(got), fin), (what, "non-finite in other places")
    assert torch.equal(got[~fin].nan_to_num(), want[~fin].nan_to_num()), (what, "other inf / NaN")
    err = (got - want).abs()[fin]
    bnd = (SAFETY * bound.expand_as(want))[fin]
    zero = bnd == 0
    assert (err[zero] == 0).all(), (what, "not exact where the bound is 0")
    return (err[~zero] / bnd[~zero]).max().item() if (~zero).any() else 0.0


def judge(name, db, divergence=True, penalty=10.0, upstream=(1.0, 1.0)):
    """Kernels vs restatement, element by element; bitwise: loss.py == C ABI, and the ABI on 0x00- and 0xFF-filled
    plan / tmp / workspace buffers.  Returns the restatement and the kernel outputs."""
    out2, grad = run_loss(db, divergence, penalty, upstream)
    a = run_abi(db, divergence, penalty, upstream, poison=0x00)
    z = run_abi(db, divergence, penalty, upstream, poison=0xFF)
    for i, (x, y) in enumerate(zip(a, z)):
        if i != 2 or divergence:  # without divergence the per-node divergence is not written
            assert torch.equal(x.view(torch.int32), y.view(torch.int32)), (name, "poisoned buffers change bits")
    assert torch.equal(out2.view(torch.int32), a[0].view(torch.int32)), (name, "loss.py and ABI differ")
    assert torch.equal(grad.view(torch.int32), a[3].view(torch.int32)), (name, "loss.py and ABI differ")
    _, per_graph, gdiv, _ = a
    bd = bounds(db, divergence, penalty, upstream)
    r = bd.r
    w = {"nmse_graph": ratio(per_graph[:, 0], r.nmse_graph, bd.nmse_graph, (name, "nmse_graph")),
         "nmse": ratio(out2[0], r.nmse, bd.nmse, (name, "nmse")),
         "div": ratio(out2[1], r.div, bd.div, (name, "div")),
         "grad": ratio(grad, r.grad, bd.grad, (name, "grad"))}
    if divergence:
        w["div_node"] = ratio(gdiv, r.div_node, bd.div_node, (name, "div_node"))
        w["div_graph"] = ratio(per_graph[:, 1], r.div_graph, bd.div_graph, (name, "div_graph"))
    else:
        assert out2[1].item() == 0.0
    print(f"\n{name}: worst error / bound " + " ".join(f"{k} {v:.3g}" for k, v in w.items()))
    for k, v in w.items():
        assert v <= 1.0, (name, k, v)
    return r, SimpleNamespace(out2=out2, per_graph=per_graph, gdiv=gdiv, grad=grad)


def _tiny_sizes(seed=11):
    return np.random.default_rng(seed).integers(1, 6, 4096)


CASES = {
    # name: (make_batch arguments, divergence, penalty, upstream)
    "tile_sizes_ragged": (dict(sizes=[1, 2, 255, 256, 257, 511, 512, 513, 4097], op="mix"), True, 10.0, (1.0, 1.0)),
    "one_graph_p1": (dict(sizes=[3000], op="p1", labels="zero"), True, 1.0, (0.3, -2.5)),
    "4096_tiny_graphs": (dict(sizes=_tiny_sizes(), op="rand"), True, 10.0, (1.0, 1.0)),
    "n_65535": (dict(sizes=[40000, 25535], op="mix"), True, 1.0, (1.0, 1.0)),
    "n_65536": (dict(sizes=[40000, 25536], op="mix", dropped=(1,), width=80016), True, 1.0, (1.0, 1.0)),
    "n_65537": (dict(sizes=[40000, 25537], op="mix", wide=50), True, 1.0, (0.3, -2.5)),
    "hub_row_and_column": (dict(sizes=[4097, 300], op="p1", hub_row=0, hub_col=0), True, 10.0, (1.0, 1.0)),
    "wide_columns_dups_dropped": (dict(sizes=[50, 700, 20, 90], op="rand", wide=30, dups=0.3, dropped=(2,)), True, 10.0,
                                  (1.0, 1.0)),
    "values_1e-6_1e6": (dict(sizes=[600, 900], op="rand", values="wide"), True, 10.0, (1.0, 1.0)),
    "empty_operator": (dict(sizes=[100, 37], empty_op=True), True, 10.0, (1.0, 1.0)),
    "labels_all_pm1": (dict(sizes=[300, 200], op="p1", labels="pm1"), True, 10.0, (1.0, 1.0)),
    "labels_outside_pm1": (dict(sizes=[300, 200], op="mix", labels="two"), True, 10.0, (1.0, 1.0)),
    "pred_equals_gt_div_off": (dict(sizes=[300, 200, 50], op="p1", exact=(1,)), False, 10.0, (1.0, 1.0)),
    "pred_equals_gt": (dict(sizes=[300, 200, 50], op="p1", exact=(1,)), True, 10.0, (1.0, 1.0)),
    "illconditioned_norm": (dict(sizes=[500, 300], op="p1", illcond=(0,)), True, 10.0, (1.0, 1.0)),
    "penalty_0": (dict(sizes=[400, 123], op="mix"), True, 0.0, (1.0, 1.0)),
    "penalty_1e4_div_alone": (dict(sizes=[400, 123], op="mix"), True, 1e4, "div"),
    "nmse_alone": (dict(sizes=[400, 123], op="mix"), True, 10.0, "nmse"),
    "divergence_off": (dict(sizes=[400, 123], op="mix"), False, 10.0, (0.3, -2.5)),
}


@pytest.mark.parametrize("name", list(CASES))
def test_loss_kernels_within_rounding_bounds(name):
    kw, divergence, penalty, upstream = CASES[name]
    b = make_batch(seed=len(name), **kw)
    db = _device(b)
    r, k = judge(name, db, divergence, penalty, upstream)
    lab = b.surfaces_nodes_for_div.reshape(-1).cuda()
    if divergence:
        masked = (lab == 1) | (lab == -1)
        assert torch.equal(k.gdiv[masked], torch.zeros_like(k.gdiv[masked]))
        assert (k.gdiv[~masked] != 0).any() or not (~masked).any() or "empty" in name or "dropped" in name
    if "outside_pm1" in name:  # rows labelled 2, -2, 3 carry a divergence like the reference
        other = (lab != 0) & (lab != 1) & (lab != -1)
        assert other.any() and (k.gdiv[other] != 0).any() and (r.div_node[other] != 0).any()
    for gi in kw.get("exact", ()):
        s, e = int(b.ptr[gi]), int(b.ptr[gi + 1])
        assert k.per_graph[gi, 0].item() == 0.0
        if not divergence:
            assert (k.grad[s:e] == 0).all()
    if kw.get("empty_op"):
        assert k.out2[1].item() == 0.0 and (k.gdiv == 0).all()
        _, g0 = run_loss(db, False, penalty, upstream)
        assert torch.equal(k.grad, g0)


def test_loss_kernels_graph_of_2p24_plus_1_nodes():
    """N_i = 2^24 + 1 (fp32 rounds it to 2^24), two entries a row, columns over all of [0, 2 N_i), mixed labels."""
    n = 2 ** 24 + 1
    g = torch.Generator(device="cuda").manual_seed(7)
    mean_ls, std_ls = _f32(2.5), _f32(40.0)
    ls = mean_ls + std_ls * torch.randn(n, 3, generator=g, device="cuda")
    row = torch.arange(n, device="cuda").repeat_interleave(2)
    col = torch.randint(0, 2 * n, (2 * n,), generator=g, device="cuda")
    val = torch.randn(2 * n, generator=g, device="cuda")
    op = torch.sparse_coo_tensor(torch.stack([row, col]), val, (n, 2 * n)).coalesce()
    db = SimpleNamespace(local_stress=ls, mean_ls=mean_ls, std_ls=std_ls, ptr=torch.tensor([0, n], device="cuda"),
                         op_div_matrix=op, surfaces_nodes_for_div=torch.randint(-1, 2, (n, 1), generator=g, device="cuda"),
                         batch_size=1)
    db.pred = O.loss_fp64(ls, ls, mean_ls, std_ls, db.ptr, divergence=False).gt + \
        torch.randn(n, 3, generator=g, device="cuda")
    judge("graph_2p24_plus_1", db, True, 10.0, (1.0, 1.0))


def _base(seed=3):
    return _device(make_batch([300, 257, 40], seed=seed, op="mix"))


def test_two_runs_identical_bits():
    db = _base()
    a, b = run_loss(db, True, 10.0, (0.3, -2.5)), run_loss(db, True, 10.0, (0.3, -2.5))
    for x, y in zip(a, b):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))


@pytest.mark.parametrize("k", [8, -8, 40, -40])
def test_upstream_scaling_by_power_of_two_is_exact(k):
    db = _base()
    _, g = run_loss(db, True, 10.0, (0.3, -2.5))
    _, gk = run_loss(db, True, 10.0, (0.3 * 2.0 ** k, -2.5 * 2.0 ** k))
    assert torch.equal(gk, g * 2.0 ** k)


def test_unbatched_input_is_one_graph():
    """A Data without `ptr` (benchmark_gnn_fem.py:97) is one graph."""
    db = _device(make_batch([700], seed=5, op="p1"))
    a = run_loss(db, True, 10.0, (1.0, 1.0))
    del db.ptr
    b = run_loss(db, True, 10.0, (1.0, 1.0))
    for x, y in zip(a, b):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))


def test_plan_cache_same_and_different_operator():
    """The same operator and ptr twice reuse one plan and give the same bits; another operator with the same ptr gets
    its own plan and its own, correct, result."""
    from pdivgnn_b200 import loss
    db = _base()
    p1 = loss.build_opdiv_plan(db.op_div_matrix, db.ptr)
    a = run_loss(db, True, 10.0, (1.0, 1.0))
    assert loss.build_opdiv_plan(db.op_div_matrix, db.ptr) is p1
    b = run_loss(db, True, 10.0, (1.0, 1.0))
    for x, y in zip(a, b):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))
    other = _device(make_batch([300, 257, 40], seed=4, op="rand"))
    db.op_div_matrix = other.op_div_matrix
    assert loss.build_opdiv_plan(db.op_div_matrix, db.ptr) is not p1
    _, k = judge("plan_cache_other_operator", db)
    assert not torch.equal(k.grad, a[1])
