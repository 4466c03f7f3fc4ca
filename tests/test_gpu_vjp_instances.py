"""GPU checks of reverse-mode derivatives through the batched forward: torch.func.grad, vjp and jacrev of a function that
vmaps the model over loads or shapes, and autograd through that vmap, reach pdg_forward_batched_saved (one saved forward
per instance) and pdg_vjp_instances (one adjoint pass for up to 64 (instance, cotangent) pairs).

Row k of the saved forward, and every saved tensor of instance k, must have the bits of pdg_forward with PDG_FLAG_SAVE on
instance k's inputs.  Row (i, m) of the adjoint must have the bits of pdg_vjp_batched with K = 1 on a separate saved
forward of instance i, i.e. the input gradients of pdg_backward_inputs: so every per-instance gradient through torch
equals a separate torch.autograd.grad call."""
import ctypes as C
from types import SimpleNamespace

import pytest
import torch

import pdg_helpers as H
import test_gpu_fwd_batched as FB
from oracle import pdg_oracle as O

pytestmark = pytest.mark.gpu
INPUTS = FB.INPUTS
GRAPHS = ["train2_div", "train2_quad", "synthetic", "mesh1024", "seg_spans_rows_127_128"]
KS = [1, 2, 3, 8, 64]
TOL, GUARD = 1e-5, 1.25


def _save_flags(**kw):
    from pdivgnn_b200 import _lib
    return FB._flags(**kw) | _lib.FLAG_SAVE


# ---- C ABI helpers ---------------------------------------------------------------------------------------------------
def _saved_single(s, xs, flags, steps=None):
    """pdg_forward with PDG_FLAG_SAVE on one instance: (out, zero-filled workspace after the call)"""
    from pdivgnn_b200 import _lib
    steps = s.steps if steps is None else steps
    nbytes = s.L.pdg_forward_ws_bytes(s.n, s.e, steps, flags)
    ws = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    out = torch.full((s.n, 3), float("nan"), device="cuda")
    _lib.check(s.L.pdg_forward(C.byref(s.ps), C.byref(s.norm), s.p(xs["mean_stress"]), s.p(xs["pos"]), s.p(s.types),
                               s.p(xs["edge_attr"]), s.p(s.plan.buf), s.n, s.e, steps, flags, 0, s.p(ws), nbytes,
                               s.p(out), _lib.stream_ptr()), "pdg_forward")
    return out, ws


def _saved_batched(s, k, xs, strides, flags, ws_bytes=None, precision=0, n=None):
    """pdg_forward_batched_saved: (rc, out, workspace, bytes of one instance)"""
    from pdivgnn_b200 import _lib
    one = s.L.pdg_forward_batched_saved_ws_bytes(s.n, s.e, s.steps, flags, 1)
    ws = torch.zeros(max(k, 1) * max(one, 1), dtype=torch.uint8, device="cuda")
    out = torch.full((max(k, 1), s.n, 3), float("nan"), device="cuda")
    rc = s.L.pdg_forward_batched_saved(C.byref(s.ps), C.byref(s.norm), s.p(xs["mean_stress"]), strides["mean_stress"],
                                       s.p(xs["pos"]), strides["pos"], s.p(s.types), s.p(xs["edge_attr"]),
                                       strides["edge_attr"], s.p(s.plan.buf), s.n if n is None else n, s.e, s.steps, flags,
                                       precision, s.p(ws), k * one if ws_bytes is None else ws_bytes, k, s.p(out),
                                       _lib.stream_ptr())
    return rc, out, ws, one


def _saved_views(s, flags, steps=None):
    """(label, byte offset, bytes) of every tensor a PDG_FLAG_SAVE forward keeps (pdg_ws_offset what = 0..11, every t)"""
    steps = s.steps if steps is None else steps
    ts = {0: steps + 1, 1: steps, 2: steps - 1, 3: steps, 4: steps, 5: steps, 6: steps, 7: steps, 8: 1, 9: 1, 10: 1,
          11: 2 + 3 * steps}
    views = []
    for what, nt in ts.items():
        for t in range(nt):
            off, elems = C.c_size_t(), C.c_size_t()
            rc = s.L.pdg_ws_offset(s.n, s.e, steps, flags, what, t, C.byref(off), C.byref(elems))
            assert rc == 0, (what, t, s.L.pdg_last_error())
            views.append((f"what {what} t {t}", off.value, elems.value * (8 if what == 11 else 4)))
    return views


def _vjp_instances(s, I, M, xs, strides, fwd_ws, U, flags, outs=(True, True, True), vws=None, ws_bytes=None, steps=None,
                   precision=0, n=None):
    """pdg_vjp_instances; U [I, M, N, 3].  Returns (rc, [grad_mean_stress, grad_pos, grad_edge_attr] each [I, M, ...])"""
    from pdivgnn_b200 import _lib
    steps = s.steps if steps is None else steps
    nbytes = s.L.pdg_vjp_batched_ws_bytes(s.n, s.e, steps, max(1, min(I * M, 64)))
    if vws is None:
        vws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device="cuda")
    shapes = ((s.n, 3), (s.n, 2), (s.e,))
    o = [torch.full((max(I, 1), max(M, 1)) + sh, float("nan"), device="cuda") if w else None for w, sh in zip(outs, shapes)]
    rc = s.L.pdg_vjp_instances(C.byref(s.ps), C.byref(s.norm), s.p(xs["mean_stress"]), strides["mean_stress"],
                               s.p(xs["pos"]), strides["pos"], s.p(s.types), s.p(xs["edge_attr"]), strides["edge_attr"],
                               s.p(s.plan.buf), s.n if n is None else n, s.e, steps, flags, precision, s.p(fwd_ws), I,
                               s.p(vws), nbytes if ws_bytes is None else ws_bytes, M, s.p(U), *(s.p(t) for t in o),
                               _lib.stream_ptr())
    return rc, o


def _vjp_single(s, xs, u, flags, steps=None):
    """pdg_vjp_batched with K = 1 on a separate saved forward of one instance"""
    from pdivgnn_b200 import _lib
    steps = s.steps if steps is None else steps
    _, ws = _saved_single(s, xs, flags, steps)
    nbytes = s.L.pdg_vjp_batched_ws_bytes(s.n, s.e, steps, 1)
    vws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    o = [torch.empty(s.n, 3, device="cuda"), torch.empty(s.n, 2, device="cuda"), torch.empty(s.e, device="cuda")]
    _lib.check(s.L.pdg_vjp_batched(C.byref(s.ps), C.byref(s.norm), s.p(xs["mean_stress"]), s.p(xs["pos"]), s.p(s.types),
                                   s.p(xs["edge_attr"]), s.p(s.plan.buf), s.n, s.e, steps, flags, 0, s.p(ws), s.p(vws),
                                   nbytes, 1, s.p(u), *(s.p(t) for t in o), _lib.stream_ptr()), "pdg_vjp_batched")
    return o


def _cot(s, I, M, seed=5):
    return torch.randn((I, M, s.n, 3), generator=torch.Generator().manual_seed(seed)).cuda()


# ---- ABI: the saved batched forward ----------------------------------------------------------------------------------
@pytest.mark.parametrize("shared", [None, "mean_stress", "pos", "edge_attr"])
@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("name", GRAPHS)
def test_saved_forward_rows_and_state_equal_single(name, k, shared):
    s = FB._setup(name)
    flags = _save_flags()
    xs, strides = FB._instances(s, k, tuple(n for n in INPUTS if n != shared), seed=k)
    rc, out, ws, one = _saved_batched(s, k, xs, strides, flags)
    assert rc == 0, s.L.pdg_last_error()
    assert 0 < one <= s.L.pdg_forward_ws_bytes(s.n, s.e, s.steps, flags) and one % 256 == 0
    assert s.L.pdg_forward_batched_saved_ws_bytes(s.n, s.e, s.steps, flags, k) == k * one
    views = _saved_views(s, flags)
    for i in range(k):
        ref, ref_ws = _saved_single(s, FB._row(xs, strides, i), flags)
        assert torch.equal(out[i], ref), i
        inst = ws[i * one:(i + 1) * one]
        for label, off, nb in views:
            assert torch.equal(inst[off:off + nb], ref_ws[off:off + nb]), (i, label)


def test_saved_forward_refusals():
    from pdivgnn_b200 import _lib
    s = FB._setup("train2_div")
    xs, strides = FB._instances(s, 2, seed=23)
    big = 1 << 30

    def refused(what, k=2, flags=None, **kw):
        kw.setdefault("ws_bytes", big)
        rc, *_ = _saved_batched(s, k, xs, kw.pop("strides", strides), _save_flags() if flags is None else flags, **kw)
        assert rc == -1 and what in s.L.pdg_last_error(), (what, s.L.pdg_last_error())
    refused(b"PDG_FLAG_SAVE", flags=FB._flags())
    refused(b"n_instances", k=0)
    refused(b"n_instances", k=65)
    refused(b"fp32", precision=_lib.PREC_BF16)
    refused(b"stride", strides=dict(strides, edge_attr=-1))
    refused(b"empty graph", n=0)
    refused(b"workspace", ws_bytes=s.L.pdg_forward_batched_saved_ws_bytes(s.n, s.e, s.steps, _save_flags(), 2) - 1)
    assert s.L.pdg_forward_batched_saved_ws_bytes(s.n, s.e, s.steps, FB._flags(), 2) == 0
    for k in (0, 65):
        assert s.L.pdg_forward_batched_saved_ws_bytes(s.n, s.e, s.steps, _save_flags(), k) == 0


# ---- ABI: the instance adjoint ---------------------------------------------------------------------------------------
IMS = [(1, 1), (3, 1), (8, 1), (2, 3), (4, 16), (64, 1), (1, 64)]


def _check_adjoint(s, I, M, xs, strides, flags, U, got, steps=None):
    for i in range(I):
        row = FB._row(xs, strides, i)
        for m in range(M):
            ref = _vjp_single(s, row, U[i, m].contiguous(), flags, steps)
            for j in range(3):
                assert torch.equal(got[j][i, m], ref[j]), (i, m, INPUTS[j])


@pytest.mark.parametrize("shared", [None, "pos"])
@pytest.mark.parametrize("I,M", IMS)
@pytest.mark.parametrize("name", ["train2_div", "mesh1024"])
def test_adjoint_rows_equal_single(name, I, M, shared):
    s = FB._setup(name)
    flags = _save_flags()
    xs, strides = FB._instances(s, I, tuple(n for n in INPUTS if n != shared), seed=I + M)
    rc, _, ws, _ = _saved_batched(s, I, xs, strides, flags)
    assert rc == 0, s.L.pdg_last_error()
    U = _cot(s, I, M, seed=I * M)
    rc, got = _vjp_instances(s, I, M, xs, strides, ws, U, flags)
    assert rc == 0, s.L.pdg_last_error()
    assert all(torch.isfinite(t).all() and t.abs().max() > 0 for t in got)
    _check_adjoint(s, I, M, xs, strides, flags, U, got)


@pytest.mark.parametrize("steps", [1, 3])
def test_adjoint_steps(steps):
    s = FB._setup("train2_div", steps)
    flags = _save_flags()
    xs, strides = FB._instances(s, 3, seed=steps)
    rc, _, ws, _ = _saved_batched(s, 3, xs, strides, flags)
    assert rc == 0, s.L.pdg_last_error()
    U = _cot(s, 3, 2, seed=steps)
    rc, got = _vjp_instances(s, 3, 2, xs, strides, ws, U, flags)
    assert rc == 0, s.L.pdg_last_error()
    _check_adjoint(s, 3, 2, xs, strides, flags, U, got)


@pytest.mark.parametrize("scale_input,scale_output", [(False, True), (True, False), (False, False)])
def test_adjoint_scale_flags(scale_input, scale_output):
    s = FB._setup("train2_div")
    flags = _save_flags(scale_input=scale_input, scale_output=scale_output)
    xs, strides = FB._instances(s, 2, seed=9)
    rc, _, ws, _ = _saved_batched(s, 2, xs, strides, flags)
    assert rc == 0, s.L.pdg_last_error()
    U = _cot(s, 2, 3, seed=9)
    rc, got = _vjp_instances(s, 2, 3, xs, strides, ws, U, flags)
    assert rc == 0, s.L.pdg_last_error()
    _check_adjoint(s, 2, 3, xs, strides, flags, U, got)


def test_adjoint_properties():
    """zero-load instance, NULL outputs, read-only forward workspace, poisoned vjp workspace, repeats, launch count"""
    s = FB._setup("train2_div")
    flags = _save_flags()
    I, M = 4, 3
    xs, strides = FB._instances(s, I, seed=13)
    xs["mean_stress"][2].zero_()
    rc, out, ws, _ = _saved_batched(s, I, xs, strides, flags)
    assert rc == 0, s.L.pdg_last_error()
    assert (out[2] == 0).all()
    ws0 = ws.clone()
    U = _cot(s, I, M, seed=29)
    nbytes = s.L.pdg_vjp_batched_ws_bytes(s.n, s.e, s.steps, I * M)
    runs = []
    for fill in (0x00, 0xFF, 0x7F, 0x00):
        rc, got = _vjp_instances(s, I, M, xs, strides, ws, U, flags,
                                 vws=torch.full((nbytes,), fill, dtype=torch.uint8, device="cuda"))
        assert rc == 0, s.L.pdg_last_error()
        runs.append(got)
    for got in runs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(runs[0], got))
    assert torch.equal(ws, ws0)
    for j in range(3):  # the all-zero load: exact zeros, +0.0
        assert (runs[0][j][2] == 0).all() and not (runs[0][j][2].view(torch.int32) != 0).any(), j
        assert all(runs[0][j][i].abs().max() > 0 for i in (0, 1, 3)), j
    _check_adjoint(s, I, M, xs, strides, flags, U, runs[0])
    for want in ((False, True, False), (True, False, False), (False, False, True), (True, True, False)):
        rc, got = _vjp_instances(s, I, M, xs, strides, ws, U, flags, outs=want)
        assert rc == 0, s.L.pdg_last_error()
        for j in range(3):
            assert (got[j] is None) == (not want[j])
            if want[j]:
                assert torch.equal(got[j], runs[0][j]), (want, j)


def test_adjoint_launch_count():
    s = FB._setup("train2_div")
    flags = _save_flags()
    counts = []
    for I, M in ((1, 1), (64, 1), (1, 1)):
        xs, strides = FB._instances(s, I, seed=31)
        rc, _, ws, _ = _saved_batched(s, I, xs, strides, flags)
        assert rc == 0, s.L.pdg_last_error()
        U = _cot(s, I, M)
        _vjp_instances(s, I, M, xs, strides, ws, U, flags)  # function attributes set
        s.L.pdg_launch_count(1)
        rc, _ = _vjp_instances(s, I, M, xs, strides, ws, U, flags)
        assert rc == 0, s.L.pdg_last_error()
        counts.append(s.L.pdg_launch_count(1))
    assert counts == [5 * s.steps + 4] * 3, counts


def test_adjoint_refusals():
    from pdivgnn_b200 import _lib
    s = FB._setup("train2_div")
    flags = _save_flags()
    xs, strides = FB._instances(s, 2, seed=37)
    rc, _, ws, _ = _saved_batched(s, 2, xs, strides, flags)
    assert rc == 0, s.L.pdg_last_error()
    U = _cot(s, 2, 64)
    big = 1 << 30

    def refused(what, I=2, M=2, **kw):
        kw.setdefault("ws_bytes", big)
        f = kw.pop("flags", flags)
        rc, _ = _vjp_instances(s, I, M, xs, kw.pop("strides", strides), ws, U, f, **kw)
        assert rc == -1 and what in s.L.pdg_last_error(), (what, s.L.pdg_last_error())
    refused(b"n_instances", I=0)
    refused(b"n_instances", I=65)
    refused(b"n_cotangents", M=0)
    refused(b"n_cotangents", M=65)
    refused(b"> 64", I=2, M=33)
    refused(b"stride", strides=dict(strides, mean_stress=-3))
    refused(b"fp32", precision=_lib.PREC_BF16)
    refused(b"SAVE", flags=FB._flags())
    refused(b"steps", steps=0)
    refused(b"steps", steps=63)
    refused(b"no output", outs=(False, False, False))
    refused(b"empty graph", n=0)
    refused(b"workspace", ws_bytes=s.L.pdg_vjp_batched_ws_bytes(s.n, s.e, s.steps, 4) - 1)


# ---- torch: derivatives taken outside the vmap -----------------------------------------------------------------------
def _weights(c, k, seed=3):
    return torch.randn((k, c.batch.num_nodes, 3), generator=torch.Generator().manual_seed(seed)).cuda()


def _obj(f, w):
    """a scalar objective of one instance: <w, local_stress>"""
    return lambda *x: (f(*x) * w).sum()


def _separate(f, W, xs, argnums=0):
    """one torch.autograd.grad per instance: d <W[k], f(xs[k])> / d xs[k][argnums]"""
    rows = []
    for k in range(W.shape[0]):
        leaves = [x[k].detach().clone().requires_grad_(i == argnums) for i, x in enumerate(xs)]
        rows.append(torch.autograd.grad((f(*leaves) * W[k]).sum(), leaves[argnums])[0])
    return torch.stack(rows)


def _vm_obj(f, W):
    """the sum over instances of <W[k], f(x_k)>, with the model vmapped over the instances"""
    return lambda *xs: (torch.func.vmap(f)(*xs) * W).sum()


@pytest.mark.parametrize("name", ["train2_div", "mesh1024"])
@pytest.mark.parametrize("case", ["mean_stress", "load_expanded", "pos", "edge_attr"])
def test_grad_of_vmap_equals_separate_grads(name, case):
    """torch.func.grad outside the vmap: each row has the bits of a separate torch.autograd.grad (at the parent commit
    this returned zeros).  A load S [3] expanded to the N nodes: torch reduces the per-node rows over N, as a [K, N, 3]
    sum under vmap and as an [N, 3] sum per call, and those two reductions may round differently; the per-node rows
    have the bits of separate calls, so the expanded load must equal their sum over N formed the batched way, and the
    separate gradients within 1e-6."""
    c = FB._graph(name)
    s = FB._setup(name)
    k = 5
    W = _weights(c, k)
    xs, _ = FB._instances(s, k, seed=29)
    if case == "load_expanded":
        f0, _ = FB._model_fn(c, FB._frozen(c), ("mean_stress",))
        x = xs["mean_stress"][:, 0].contiguous()
        ours = torch.func.grad(_vm_obj(lambda S: f0(S.expand(s.n, 3)), W))(x)
        rows = _separate(f0, W, (x.unsqueeze(1).expand(k, s.n, 3).contiguous(),))  # [K, N, 3], per node
        assert torch.equal(ours, rows.sum(1))
        sep = _separate(lambda S: f0(S.expand(s.n, 3)), W, (x,))
        assert H.rel_err(ours, sep)[0] < 1e-6, H.rel_err(ours, sep)
        return
    f, _ = FB._model_fn(c, FB._frozen(c), (case,))
    x = xs[case]
    ours = torch.func.grad(_vm_obj(f, W))(x)
    ref = _separate(f, W, (x,))
    assert ours.shape == x.shape
    assert ours.abs().max() > 0
    assert torch.equal(ours, ref)


def test_autograd_through_vmap():
    c = FB._graph("train2_div")
    s = FB._setup("train2_div")
    f, _ = FB._model_fn(c, FB._frozen(c), ("mean_stress",))
    xs, _ = FB._instances(s, 4, seed=41)
    W = _weights(c, 4, seed=41)
    loads = xs["mean_stress"].clone().requires_grad_(True)
    out = torch.func.vmap(f)(loads)
    assert out.requires_grad
    out.backward(W)
    assert torch.equal(loads.grad, _separate(f, W, (xs["mean_stress"],)))


def test_vjp_of_vmap_with_shared_pos():
    """K loads on one shape: d / d pos of the sum of the K objectives.  Through the model's pos input alone it equals
    the sum of K separate gradients bit for bit (both are sum(0) of the same rows); with the edge lengths computed from pos
    in torch, torch reduces the K edge-weight rows before the edge-length backward instead of after it, which reassociates
    fp32 sums: held to 1e-6 relative."""
    c = FB._graph("mesh1024")
    s = FB._setup("mesh1024")
    model = FB._frozen(c)
    k = 4
    xs, _ = FB._instances(s, k, ("mean_stress",), seed=43)
    W = _weights(c, k, seed=43)
    for ea_from_pos in (False, True):
        f, _ = FB._model_fn(c, model, ("mean_stress", "pos"), ea_from_pos=ea_from_pos)
        ours = torch.func.grad(lambda p: (torch.func.vmap(lambda L: f(L, p))(xs["mean_stress"]) * W).sum())(s.x["pos"])
        sep = []
        for i in range(k):
            p = s.x["pos"].detach().clone().requires_grad_(True)
            sep.append(torch.autograd.grad((f(xs["mean_stress"][i], p) * W[i]).sum(), p)[0])
        ref = torch.stack(sep).sum(0)
        assert ours.abs().max() > 0
        if not ea_from_pos:
            assert torch.equal(ours, ref)
        else:
            assert H.rel_err(ours, ref)[0] < 1e-6, H.rel_err(ours, ref)


def _objectives(pred):
    """four objectives of one instance: the mean of each stress component and the mean von Mises measure"""
    sxx, syy, sxy = pred[:, 0], pred[:, 1], pred[:, 2]
    return torch.stack([sxx.mean(), syy.mean(), sxy.mean(), (sxx * sxx + syy * syy - sxx * syy + 3.0 * sxy * sxy).mean()])


def test_jacrev_of_vmap_equals_separate_grads():
    c = FB._graph("train2_div")
    s = FB._setup("train2_div")
    f, _ = FB._model_fn(c, FB._frozen(c), ("mean_stress",))
    k = 3
    xs, _ = FB._instances(s, k, ("mean_stress",), seed=47)
    L = xs["mean_stress"]
    jac = torch.func.jacrev(lambda x: torch.func.vmap(lambda l: _objectives(f(l)))(x))(L)
    assert jac.shape == (k, 4, k, s.n, 3)
    for i in range(k):
        for j in range(4):  # one forward per objective: a single backward releases the forward state
            leaf = L[i].detach().clone().requires_grad_(True)
            g = torch.autograd.grad(_objectives(f(leaf))[j], leaf)[0]
            assert torch.equal(jac[i, j, i], g), (i, j)
            for o in range(k):
                if o != i:
                    assert (jac[i, j, o] == 0).all(), (i, j, o)


def test_nested_in_dims_and_chunks():
    c = FB._graph("train2_div")
    s = FB._setup("train2_div")
    f, _ = FB._model_fn(c, FB._frozen(c), INPUTS)
    xs, _ = FB._instances(s, 6, seed=53)
    W = _weights(c, 6, seed=53)
    ref = [_separate(f, W, (xs["mean_stress"], xs["pos"], xs["edge_attr"]), argnums=j) for j in range(3)]
    args = tuple(xs[n] for n in INPUTS)
    flat = torch.func.grad(lambda *x: (torch.func.vmap(f)(*x) * W).sum(), argnums=(0, 1, 2))(*args)
    for j in range(3):
        assert torch.equal(flat[j], ref[j]), INPUTS[j]
    nest = torch.func.grad(lambda *x: (torch.func.vmap(torch.func.vmap(f))(*x) * W.reshape(2, 3, *W.shape[1:])).sum(),
                           argnums=(0, 1, 2))(*(x.reshape(2, 3, *x.shape[1:]) for x in args))
    for j in range(3):
        assert torch.equal(nest[j].reshape(ref[j].shape), ref[j]), ("nested", INPUTS[j])
    # a non-zero in_dims
    ms_t = xs["mean_stress"].movedim(0, 1).contiguous()
    g = torch.func.grad(lambda m: (torch.func.vmap(f, in_dims=(1, 0, 0))(m, xs["pos"], xs["edge_attr"]) * W).sum())(ms_t)
    assert torch.equal(g.movedim(1, 0), ref[0])
    chunked = torch.func.grad(lambda *x: (torch.func.vmap(f, chunk_size=4)(*x) * W).sum(), argnums=(0, 1, 2))(*args)
    for j in range(3):
        assert torch.equal(chunked[j], ref[j]), ("chunk_size", INPUTS[j])


@pytest.mark.parametrize("k", [65, 130])
def test_more_than_64_instances(k):
    c = FB._graph("train2_div")
    s = FB._setup("train2_div")
    f, _ = FB._model_fn(c, FB._frozen(c), ("mean_stress",))
    xs, _ = FB._instances(s, k, ("mean_stress",), seed=59)
    W = _weights(c, k, seed=59)
    assert torch.equal(torch.func.grad(_vm_obj(f, W))(xs["mean_stress"]), _separate(f, W, (xs["mean_stress"],)))


def test_refusals():
    c = FB._graph("train2_div")
    s = FB._setup("train2_div")
    xs, _ = FB._instances(s, 2, ("mean_stress",), seed=61)
    W = _weights(c, 2)
    f, db = FB._model_fn(c, H.make_model(c.stats, params=c.sd), ("mean_stress",))
    with pytest.raises(NotImplementedError, match="forward only"):
        torch.func.grad(_vm_obj(f, W))(xs["mean_stress"])  # a trainable model
    h, _ = FB._model_fn(c, FB._frozen(c, precision="bf16"), ("mean_stress",), db)
    with pytest.raises(NotImplementedError, match="fp32"):
        torch.func.grad(_vm_obj(h, W))(xs["mean_stress"])
    frozen = FB._frozen(c)
    with torch.no_grad():
        frozen(db, scale_output=True)  # the model's own parameter list is cached before functional_call swaps it
    params = {k: v.detach().clone() for k, v in frozen.named_parameters()}

    def fp(ms):
        b = SimpleNamespace(**vars(db))
        b.mean_stress = ms
        return torch.func.functional_call(frozen, params, (b,), {"scale_output": True, "scale_input": True}).local_stress
    with pytest.raises(NotImplementedError, match="functional_call"):
        torch.func.grad(_vm_obj(fp, W))(xs["mean_stress"])


# ---- against the oracle ----------------------------------------------------------------------------------------------
# per-load gradients measured on a B200 (1 000 W) to miss the input-gradient bar, with their (L-inf, L2) errors: none
# (all 12 rows met it)
MEASURED_MISSES = {}


def test_per_load_gradients_match_oracle():
    """one 1 089-node mesh under three uniform loads S_k (mean_stress = S_k on every node): d obj_k / d S_k of the four
    objectives of each load, by jacrev over the vmapped model, against the fp64 oracle on that load alone, with the bar
    of tests/test_gpu_input_grads.py: 4x L-inf / 3x L2 of the oracle's own fp32 error, floor 1e-5."""
    c = FB._graph("mesh1024")
    s = FB._setup("mesh1024")
    f, _ = FB._model_fn(c, FB._frozen(c), ("mean_stress",))
    S0 = c.batch.mean_stress[0].float()
    loads = torch.stack([S0, -0.5 * S0.flip(0), torch.tensor([S0.abs().max(), 0.0, -S0.abs().max()])]).cuda()
    k, n = loads.shape[0], s.n
    jac = torch.func.jacrev(lambda L: torch.func.vmap(lambda l: _objectives(f(l.expand(n, 3))))(L))(loads)  # [k,4,k,3]
    fails, misses = [], []
    for i in range(k):
        def oracle(dtype):
            S = loads[i].cpu().to(dtype).clone().requires_grad_(True)
            b = SimpleNamespace(**vars(c.batch))
            b.mean_stress = S.expand(n, 3).clone()
            obj = _objectives(O.forward(c.sd, b, c.stats, 10, scale_output=True, scale_input=True, dtype=dtype))
            return torch.stack([torch.autograd.grad(obj[j], S, retain_graph=True)[0] for j in range(4)]).double()
        t64, t32 = oracle(torch.float64), oracle(torch.float32)
        for j in range(4):
            label = f"load {i} objective {('sxx', 'syy', 'sxy', 'von Mises')[j]}"
            e, r = H.rel_err(jac[i, j, i].double().cpu(), t64[j]), H.rel_err(t32[j], t64[j])
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


# ---- adjoint passes that start inside a forward pass -----------------------------------------------------------------
def test_adjoint_from_a_later_instance():
    """pdg_vjp_instances given the workspace from instance 13 on of a 20-instance saved forward (every instance keeps the
    packed weights): the rows of instances 13..17 equal separate calls"""
    s = FB._setup("train2_div")
    flags = _save_flags()
    xs, strides = FB._instances(s, 20, ("mean_stress", "edge_attr"), seed=67)
    rc, _, ws, one = _saved_batched(s, 20, xs, strides, flags)
    assert rc == 0, s.L.pdg_last_error()
    sub = {n: xs[n][13:18] if strides[n] else xs[n] for n in INPUTS}
    U = _cot(s, 5, 2, seed=67)
    rc, got = _vjp_instances(s, 5, 2, sub, strides, ws[13 * one:], U, flags)
    assert rc == 0, s.L.pdg_last_error()
    _check_adjoint(s, 5, 2, sub, strides, flags, U, got)


def _vjp_loop(f, L, U):
    """separate torch.autograd.grad calls: row [m, k] = d <U[m, k], f(L[k])> / d L[k]"""
    rows = torch.empty_like(U)
    for m in range(U.shape[0]):
        for k in range(U.shape[1]):
            leaf = L[k].detach().clone().requires_grad_(True)
            rows[m, k] = torch.autograd.grad(f(leaf), leaf, U[m, k])[0]
    return rows


@pytest.mark.parametrize("k,m", [(20, 4), (2, 65)])
def test_vmap_over_vjp_of_vmap_in_several_passes(k, m):
    """M cotangents for each of K instances: passes of 64 // M instances that start inside a forward pass (K = 20,
    M = 4: the second pass starts at instance 16), and M > 64 (cotangents in passes of 64, one instance each)"""
    c = FB._graph("train2_div")
    s = FB._setup("train2_div")
    f, _ = FB._model_fn(c, FB._frozen(c), ("mean_stress",))
    xs, _ = FB._instances(s, k, ("mean_stress",), seed=71)
    L = xs["mean_stress"]
    U = torch.randn((m, k, s.n, 3), generator=torch.Generator().manual_seed(71)).cuda()
    _, vjp_fn = torch.func.vjp(lambda x: torch.func.vmap(f)(x), L)
    ours = torch.func.vmap(vjp_fn)(U)[0]
    assert ours.shape == U.shape
    assert torch.equal(ours, _vjp_loop(f, L, U))


@pytest.mark.parametrize("k", [20, 70])
def test_jacrev_of_vmap_in_several_passes(k):
    """jacrev of four objectives per load at K = 20 and 70 loads: 4K cotangents for each instance, in passes of 64
    cotangents of one instance, over two forward passes at K = 70"""
    c = FB._graph("train2_div")
    s = FB._setup("train2_div")
    f, _ = FB._model_fn(c, FB._frozen(c), ("mean_stress",))
    xs, _ = FB._instances(s, k, ("mean_stress",), seed=73)
    L = xs["mean_stress"]
    jac = torch.func.jacrev(lambda x: torch.func.vmap(lambda l: _objectives(f(l)))(x))(L)
    assert jac.shape == (k, 4, k, s.n, 3)
    norms = jac.abs().sum((3, 4))  # [k, 4, k]
    off = ~torch.eye(k, dtype=torch.bool, device=norms.device)
    assert (norms.permute(1, 0, 2)[:, off] == 0).all()
    for i in range(k):
        for j in range(4):
            leaf = L[i].detach().clone().requires_grad_(True)
            g = torch.autograd.grad(_objectives(f(leaf))[j], leaf)[0]
            assert torch.equal(jac[i, j, i], g), (i, j)


# ---- derivatives inside the vmap stay refused when the inputs also require grad outside it ---------------------------
def test_grad_inside_vmap_refused_with_inputs_requiring_grad():
    c = FB._graph("train2_div")
    s = FB._setup("train2_div")
    g, _ = FB._model_fn(c, FB._frozen(c), ("mean_stress", "pos"))
    xs, _ = FB._instances(s, 2, ("mean_stress",), seed=79)
    loads = xs["mean_stress"][:, 0].contiguous().requires_grad_(True)  # optimised in an outer loop
    with pytest.raises(NotImplementedError, match="forward only"):
        torch.func.vmap(torch.func.grad(lambda S: g(S.expand(s.n, 3), s.x["pos"]).sum()))(loads)
    pos = s.x["pos"].clone().requires_grad_(True)
    with pytest.raises(NotImplementedError, match="forward only"):
        torch.func.vmap(lambda S: torch.func.grad(lambda p: g(S.expand(s.n, 3), p).sum())(pos))(loads.detach())


# ---- the saved forwards are released after a plain backward ----------------------------------------------------------
def test_saved_forwards_released_after_backward():
    c = FB._graph("mesh1024")
    s = FB._setup("mesh1024")
    f, _ = FB._model_fn(c, FB._frozen(c), ("mean_stress",))
    k = 8
    xs, _ = FB._instances(s, k, ("mean_stress",), seed=83)
    W = _weights(c, k, seed=83)
    loads = xs["mean_stress"].clone().requires_grad_(True)
    torch.cuda.synchronize()
    m0 = torch.cuda.memory_allocated()
    out = torch.func.vmap(f)(loads)
    held = torch.cuda.memory_allocated() - m0
    saved = k * s.L.pdg_forward_batched_saved_ws_bytes(s.n, s.e, s.steps, _save_flags(), 1)
    assert held >= saved
    out.backward(W, retain_graph=True)  # the graph stays; the saved forwards do not
    # what stays: the output, the inputs' copies and the gradient (allocator blocks: a 1 MB margin against K saved forwards)
    assert torch.cuda.memory_allocated() - m0 <= held - saved + loads.numel() * 4 + (1 << 20)
    assert torch.equal(loads.grad, _separate(f, W, (xs["mean_stress"],)))
    with pytest.raises(RuntimeError, match="second backward"):
        out.backward(W)
