"""GPU checks of the batched forward: K instances of one graph (their own mean_stress, pos and edge_attr) in one
pdg_forward_batched pass, and torch.func.vmap over the model's inputs, which reaches it.

Row k must have the bits of pdg_forward on instance k's inputs: instance k = blockIdx.y runs the x-grid of one
pdg_forward, in a workspace of its own with the same LayerNorm partial slots, so every sum is formed in the same order.
A batch of K copies of the mesh is not the same model: its graph-LayerNorm statistics mix the copies."""
import ctypes as C
import functools
from types import SimpleNamespace

import pytest
import torch

import pdg_helpers as H
import test_gpu_jvp as JV
import test_gpu_shapes as S
from oracle import pdg_oracle as O

pytestmark = pytest.mark.gpu
INPUTS = ("mean_stress", "pos", "edge_attr")
# golden cases, the synthetic 3 x 600 batch as one instance, one 1 024-node mesh, a receiver segment cut by a tile
# boundary, and G + 1 node tiles (G = SM count, read at run time: the y-grid runs many waves)
GRAPHS = ["train2_div", "infer1", "train2_quad", "synthetic", "mesh1024", "seg_spans_rows_127_128", "ntG+1"]
KS = [1, 2, 3, 8, 64]


def _flags(scale_input=True, scale_output=True, zero_check=True):
    from pdivgnn_b200 import _lib
    return (_lib.FLAG_SCALE_INPUT if scale_input else 0) | (_lib.FLAG_SCALE_OUTPUT if scale_output else 0) \
        | (_lib.FLAG_ZERO_CHECK if zero_check else 0)


@functools.lru_cache(maxsize=None)
def _graph(name):
    """SimpleNamespace(batch, stats, sd)"""
    if name in ("train2_div", "infer1", "train2_quad", "synthetic"):
        return JV._case(name)
    if name == "mesh1024":
        from pdivgnn_b200 import synth
        _, batch, stats = H.oracle_batch_from_samples([synth.make_rve_mesh(69, 1024)], True)
        return SimpleNamespace(batch=batch, stats=stats, sd=O.init_state_dict(seed=69))
    if name == "ntG+1":
        c = S._case("sweep", "etG_r0_ntG+1_r127")
    else:
        c = S._case("layout", name)
    return SimpleNamespace(batch=c.batch, stats=c.stats, sd=c.sd)


@functools.lru_cache(maxsize=None)
def _setup(name, steps=10):
    from pdivgnn_b200 import _lib, autograd as A
    c = _graph(name)
    b = c.batch
    model = H.make_model(c.stats, steps=steps, params=c.sd)
    n = b.num_nodes
    plan = A.build_plan(b.edge_index.cuda(), n)
    params = [p.detach() for p in A.param_list(model)]
    return SimpleNamespace(
        L=_lib.lib(), p=_lib.ptr, model=model, plan=plan, n=n, e=plan.n_edges, steps=steps, params=params,
        ps=A._params_struct(params), norm=model._norm_struct(),
        types=b.nodes_types.reshape(-1).cuda().contiguous(),
        x={"mean_stress": b.mean_stress.float().cuda().contiguous(), "pos": b.pos.float().cuda().contiguous(),
           "edge_attr": b.edge_attr.reshape(-1).float().cuda().contiguous()})


def _single(s, xs, flags, precision=0):
    """pdg_forward on one instance; xs: {input: tensor}"""
    from pdivgnn_b200 import _lib
    nbytes = s.L.pdg_forward_ws_bytes(s.n, s.e, s.steps, flags)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    out = torch.full((s.n, 3), float("nan"), device="cuda")
    _lib.check(s.L.pdg_forward(C.byref(s.ps), C.byref(s.norm), s.p(xs["mean_stress"]), s.p(xs["pos"]), s.p(s.types),
                               s.p(xs["edge_attr"]), s.p(s.plan.buf), s.n, s.e, s.steps, flags, precision, s.p(ws),
                               nbytes, s.p(out), _lib.stream_ptr()), "pdg_forward")
    return out


def _batched(s, k, xs, strides, flags, ws=None, ws_bytes=None, precision=0, steps=None, n=None):
    """pdg_forward_batched; xs: {input: [K, ...] or one instance}, strides: {input: elements}.  Returns (rc, out)."""
    from pdivgnn_b200 import _lib
    steps = s.steps if steps is None else steps
    nbytes = s.L.pdg_forward_batched_ws_bytes(s.n, s.e, steps, flags, k)
    if ws is None:
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device="cuda")
    out = torch.full((max(k, 1), s.n, 3), float("nan"), device="cuda")
    rc = s.L.pdg_forward_batched(C.byref(s.ps), C.byref(s.norm), s.p(xs["mean_stress"]), strides["mean_stress"],
                                 s.p(xs["pos"]), strides["pos"], s.p(s.types), s.p(xs["edge_attr"]), strides["edge_attr"],
                                 s.p(s.plan.buf), s.n if n is None else n, s.e, steps, flags, precision, s.p(ws),
                                 nbytes if ws_bytes is None else ws_bytes, k, s.p(out), _lib.stream_ptr())
    return rc, out


def _instances(s, k, batched=INPUTS, seed=3):
    """Inputs of K instances: loads scaled and turned, node positions jittered, edge weights scaled.  An input outside
    `batched` is the graph's own, passed once with stride 0."""
    g = torch.Generator().manual_seed(seed)
    xs, strides = {}, {}
    for name in INPUTS:
        x = s.x[name].cpu()
        if name not in batched:
            xs[name], strides[name] = s.x[name], 0
            continue
        if name == "mean_stress":
            v = x.unsqueeze(0) * (0.5 + torch.rand(k, 1, 3, generator=g)) + 2.0 * torch.randn(k, 1, 3, generator=g)
        elif name == "pos":
            v = x.unsqueeze(0) + 0.3 * torch.randn((k,) + tuple(x.shape), generator=g)
        else:
            v = x.unsqueeze(0) * (0.8 + 0.4 * torch.rand((k,) + tuple(x.shape), generator=g))
        xs[name], strides[name] = v.cuda().contiguous(), x.numel()
    return xs, strides


def _row(xs, strides, i):
    return {n: xs[n][i] if strides[n] else xs[n] for n in INPUTS}


def _check_rows(s, k, xs, strides, flags, out):
    for i in range(k):
        one = _single(s, _row(xs, strides, i), flags)
        assert torch.equal(out[i], one), i


# ---- bit identity at the C ABI ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("name", GRAPHS)
def test_rows_equal_single_forwards(name, k):
    s = _setup(name)
    xs, strides = _instances(s, k)
    rc, out = _batched(s, k, xs, strides, _flags())
    assert rc == 0, s.L.pdg_last_error()
    assert torch.isfinite(out).all() and out.abs().max() > 0
    _check_rows(s, k, xs, strides, _flags(), out)
    if k > 1:
        assert not torch.equal(out[0], out[1])


@pytest.mark.parametrize("batched", [("mean_stress",), ("pos",), ("edge_attr",), INPUTS, ()])
@pytest.mark.parametrize("name", ["train2_div", "mesh1024"])
def test_input_subsets(name, batched):
    """each input batched alone, all three, and all strides 0 (K identical rows)"""
    s = _setup(name)
    k = 3
    xs, strides = _instances(s, k, batched, seed=7)
    rc, out = _batched(s, k, xs, strides, _flags())
    assert rc == 0, s.L.pdg_last_error()
    _check_rows(s, k, xs, strides, _flags(), out)
    if not batched:
        assert all(torch.equal(out[i], out[0]) for i in range(k))


@pytest.mark.parametrize("scale_input,scale_output", [(False, True), (True, False), (False, False)])
def test_scale_flags(scale_input, scale_output):
    s = _setup("train2_div")
    xs, strides = _instances(s, 3, seed=9)
    flags = _flags(scale_input, scale_output)
    rc, out = _batched(s, 3, xs, strides, flags)
    assert rc == 0, s.L.pdg_last_error()
    _check_rows(s, 3, xs, strides, flags, out)


@pytest.mark.parametrize("steps", [1, 3, 10, 62])
def test_steps(steps):
    s = _setup("train2_div", steps)
    xs, strides = _instances(s, 3, seed=steps)
    rc, out = _batched(s, 3, xs, strides, _flags())
    assert rc == 0, s.L.pdg_last_error()
    _check_rows(s, 3, xs, strides, _flags(), out)


@pytest.mark.parametrize("name", ["train2_div", "mesh1024"])
def test_zero_load_instance(name):
    """PDG_FLAG_ZERO_CHECK is per instance: an all-zero load gives exact zeros, the others keep their single-call bits"""
    s = _setup(name)
    k = 4
    xs, strides = _instances(s, k, seed=13)
    xs["mean_stress"][2].zero_()
    rc, out = _batched(s, k, xs, strides, _flags())
    assert rc == 0, s.L.pdg_last_error()
    assert (out[2] == 0).all() and not (out[2].view(torch.int32) != 0).any()  # +0.0, not -0.0
    assert all(out[i].abs().max() > 0 for i in (0, 1, 3))
    _check_rows(s, k, xs, strides, _flags(), out)


# ---- semantics -------------------------------------------------------------------------------------------------------
def test_loads_against_oracle_and_not_a_batch_of_copies():
    """one mesh under three loads: each row meets the fp32 bar against the fp64 oracle run on that load alone; one
    forward over a batch of three copies (the copies share their LayerNorm statistics) gives other values"""
    from pdivgnn_b200 import autograd as A
    c = _graph("mesh1024")
    s = _setup("mesh1024")
    b = c.batch
    S0 = b.mean_stress[0].float()
    loads = torch.stack([S0, -0.5 * S0.flip(0), torch.tensor([S0.abs().max(), 0.0, -S0.abs().max()])])
    k, n = loads.shape[0], s.n
    xs = {"mean_stress": loads.unsqueeze(1).expand(k, n, 3).contiguous().cuda(), "pos": s.x["pos"],
          "edge_attr": s.x["edge_attr"]}
    strides = {"mean_stress": n * 3, "pos": 0, "edge_attr": 0}
    rc, out = _batched(s, k, xs, strides, _flags())
    assert rc == 0, s.L.pdg_last_error()
    for i in range(k):
        bi = SimpleNamespace(**vars(b))
        bi.mean_stress = loads[i].expand(n, 3).double().clone()
        ref = O.forward(c.sd, bi, c.stats, 10, scale_output=True, scale_input=True, dtype=torch.float64)
        linf, l2 = H.rel_err(out[i].cpu(), ref)
        assert linf < JV.TOL and l2 < JV.TOL, (i, linf, l2)
    # the batch of copies, through pdg_forward on one graph of 3N nodes
    ei = torch.cat([b.edge_index + i * n for i in range(k)], 1).cuda()
    plan = A.build_plan(ei, k * n)
    cp = SimpleNamespace(**vars(s))
    cp.plan, cp.n, cp.e = plan, k * n, plan.n_edges
    cp.types = s.types.repeat(k)
    copies = _single(cp, {"mean_stress": xs["mean_stress"].reshape(-1, 3), "pos": s.x["pos"].repeat(k, 1),
                          "edge_attr": s.x["edge_attr"].repeat(k)}, _flags()).reshape(k, n, 3)
    for i in range(k):
        assert H.rel_err(copies[i].cpu(), out[i].cpu())[0] > 1e-3, i


# ---- properties ------------------------------------------------------------------------------------------------------
def test_workspace_contents_and_repeats_do_not_matter():
    s = _setup("train2_div")
    k = 5
    xs, strides = _instances(s, k, seed=17)
    nbytes = s.L.pdg_forward_batched_ws_bytes(s.n, s.e, s.steps, _flags(), k)
    outs = []
    for fill in (0x00, 0xFF, 0x7F, 0x7F):
        rc, out = _batched(s, k, xs, strides, _flags(), ws=torch.full((nbytes,), fill, dtype=torch.uint8, device="cuda"))
        assert rc == 0, s.L.pdg_last_error()
        outs.append(out)
    assert all(torch.equal(outs[0], o) for o in outs[1:])


def test_launch_count_independent_of_k():
    s = _setup("train2_div")
    L = s.L
    xs, strides = _instances(s, 64, seed=19)
    _batched(s, 64, xs, strides, _flags())
    _single(s, _row(xs, strides, 0), _flags())
    counts = []
    for run in (lambda: _single(s, _row(xs, strides, 0), _flags()),
                lambda: _batched(s, 1, {n: x[:1] if strides[n] else x for n, x in xs.items()}, strides, _flags()),
                lambda: _batched(s, 64, xs, strides, _flags())):
        L.pdg_launch_count(1)
        run()
        counts.append(L.pdg_launch_count(1))
    assert counts[0] == counts[1] == counts[2] == 4 + 3 * s.steps, counts


def test_ws_bytes():
    from pdivgnn_b200 import _lib
    s = _setup("train2_div")
    L = s.L
    for k in (0, 65):
        assert L.pdg_forward_batched_ws_bytes(s.n, s.e, s.steps, 0, k) == 0
    for steps in (0, 63):
        assert L.pdg_forward_batched_ws_bytes(s.n, s.e, steps, 0, 2) == 0
    one = L.pdg_forward_batched_ws_bytes(s.n, s.e, s.steps, 0, 1)
    assert one > 0 and one % 256 == 0 and one <= L.pdg_forward_ws_bytes(s.n, s.e, s.steps, 0)
    assert L.pdg_forward_batched_ws_bytes(s.n, s.e, s.steps, _lib.FLAG_ZERO_CHECK, 64) == 64 * one


def test_refusals():
    from pdivgnn_b200 import _lib
    s = _setup("train2_div")
    xs, strides = _instances(s, 2, seed=23)
    big = 1 << 30

    def refused(what, **kw):
        kw.setdefault("ws_bytes", big)
        rc, _ = _batched(s, kw.pop("k", 2), xs, kw.pop("strides", strides), kw.pop("flags", _flags()), **kw)
        assert rc == -1 and what in s.L.pdg_last_error(), (what, s.L.pdg_last_error())
    ws = torch.empty(big, dtype=torch.uint8, device="cuda")
    refused(b"n_instances", k=0, ws=ws)
    refused(b"n_instances", k=65, ws=ws)
    refused(b"fp32", precision=_lib.PREC_BF16, ws=ws)
    refused(b"SAVE", flags=_flags() | _lib.FLAG_SAVE, ws=ws)
    refused(b"steps", steps=0, ws=ws)
    refused(b"steps", steps=63, ws=ws)
    refused(b"stride", strides=dict(strides, pos=-1), ws=ws)
    refused(b"empty graph", n=0, ws=ws)
    refused(b"workspace", ws_bytes=s.L.pdg_forward_batched_ws_bytes(s.n, s.e, s.steps, _flags(), 2) - 1)


# ---- torch.func.vmap over the model's inputs -------------------------------------------------------------------------
def _model_fn(c, model, keys, db=None, ea_from_pos=False):
    db = db or H.DeviceBatch(c.batch)

    def f(*xs):
        b = SimpleNamespace(**vars(db))
        for k, x in zip(keys, xs):
            setattr(b, k, x)
        if ea_from_pos:  # edge lengths computed in torch from the node positions (elementwise: the same bits batched)
            d = b.pos[db.edge_index[0]] - b.pos[db.edge_index[1]]
            b.edge_attr = torch.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1])
        return model(b, scale_output=True, scale_input=True).local_stress
    return f, db


def _frozen(c, **kw):
    m = H.make_model(c.stats, params=c.sd)
    m.requires_grad_(False)
    for k, v in kw.items():
        setattr(m, k, v)
    return m


def _loop(f, *xs):
    return torch.stack([f(*x) for x in zip(*xs)])


@pytest.mark.parametrize("name", ["train2_div", "mesh1024"])
@pytest.mark.parametrize("case", ["mean_stress", "load_expanded", "pos_edge_lengths", "edge_attr"])
def test_vmap_equals_separate_calls(name, case):
    c = _graph(name)
    s = _setup(name)
    model = _frozen(c)
    k = 5
    xs, _ = _instances(s, k, seed=29)
    if case == "load_expanded":
        f, _ = _model_fn(c, model, ("mean_stress",))
        loads = xs["mean_stress"][:, 0].contiguous()
        ours = torch.func.vmap(lambda S: f(S.expand(s.n, 3)))(loads)
        ref = _loop(lambda S: f(S.expand(s.n, 3).contiguous()), loads)
    elif case == "pos_edge_lengths":
        f, _ = _model_fn(c, model, ("pos",), ea_from_pos=True)
        ours, ref = torch.func.vmap(f)(xs["pos"]), _loop(f, xs["pos"])
    else:
        f, _ = _model_fn(c, model, (case,))
        ours, ref = torch.func.vmap(f)(xs[case]), _loop(f, xs[case])
    assert ours.shape == (k, s.n, 3)
    assert torch.equal(ours, ref)
    assert not torch.equal(ours[0], ours[1])


def test_vmap_in_dims_nested_and_chunks():
    c = _graph("train2_div")
    s = _setup("train2_div")
    model = _frozen(c)
    f, _ = _model_fn(c, model, INPUTS)
    xs, _ = _instances(s, 6, seed=31)
    ref = _loop(f, xs["mean_stress"], xs["pos"], xs["edge_attr"])
    # a non-zero in_dims, an unbatched input
    ours = torch.func.vmap(f, in_dims=(1, 0, None))(xs["mean_stress"].movedim(0, 1), xs["pos"], s.x["edge_attr"])
    assert torch.equal(ours, _loop(lambda ms, p: f(ms, p, s.x["edge_attr"]), xs["mean_stress"], xs["pos"]))
    # nested vmap: [2, 3, ...] flattens into one pass of 6
    nest = torch.func.vmap(torch.func.vmap(f))(*(xs[n].reshape(2, 3, *xs[n].shape[1:]) for n in INPUTS))
    assert torch.equal(nest.reshape(ref.shape), ref)
    # nested, the inner level over mean_stress only
    inner = torch.func.vmap(lambda ms, p: torch.func.vmap(lambda m: f(m, p, s.x["edge_attr"]))(ms))(
        xs["mean_stress"].reshape(2, 3, s.n, 3), xs["pos"][:2])
    for i in range(2):
        for j in range(3):
            assert torch.equal(inner[i, j], f(xs["mean_stress"][3 * i + j], xs["pos"][i], s.x["edge_attr"])), (i, j)
    chunked = torch.func.vmap(f, chunk_size=4)(xs["mean_stress"], xs["pos"], xs["edge_attr"])
    assert torch.equal(chunked, ref)


@pytest.mark.parametrize("k", [65, 130])
def test_vmap_more_than_64_instances(k):
    c = _graph("train2_div")
    s = _setup("train2_div")
    f, _ = _model_fn(c, _frozen(c), ("mean_stress",))
    xs, _ = _instances(s, k, ("mean_stress",), seed=37)
    assert torch.equal(torch.func.vmap(f)(xs["mean_stress"]), _loop(f, xs["mean_stress"]))


def test_vmap_no_grad_and_cuda_graphs():
    c = _graph("train2_div")
    s = _setup("train2_div")
    xs, _ = _instances(s, 3, ("pos",), seed=41)
    trainable = H.make_model(c.stats, params=c.sd)
    f, _ = _model_fn(c, trainable, ("pos",))
    with torch.no_grad():
        ours, ref = torch.func.vmap(f)(xs["pos"]), _loop(f, xs["pos"])
    assert torch.equal(ours, ref)
    g, _ = _model_fn(c, _frozen(c, cuda_graphs=True), ("pos",))
    assert torch.equal(torch.func.vmap(g)(xs["pos"]), ref)
    assert torch.equal(_loop(g, xs["pos"]), ref)


def test_vmap_refusals():
    c = _graph("train2_div")
    s = _setup("train2_div")
    xs, _ = _instances(s, 2, seed=43)
    trainable = H.make_model(c.stats, params=c.sd)
    f, db = _model_fn(c, trainable, ("mean_stress",))
    with pytest.raises(NotImplementedError, match="forward only"):
        torch.func.vmap(f)(xs["mean_stress"])  # grad mode with trainable parameters
    frozen = _frozen(c)
    g, _ = _model_fn(c, frozen, ("mean_stress",), db)
    loads = xs["mean_stress"][:, 0].contiguous()
    with pytest.raises(NotImplementedError, match="forward only"):
        torch.func.vmap(torch.func.grad(lambda S: g(S.expand(s.n, 3)).sum()))(loads)
    with pytest.raises(NotImplementedError, match="forward only"):
        torch.func.vmap(torch.func.jacfwd(lambda S: g(S.expand(s.n, 3))))(loads)
    h, _ = _model_fn(c, _frozen(c, precision="bf16"), ("mean_stress",), db)
    with pytest.raises(NotImplementedError, match="fp32"):
        torch.func.vmap(h)(xs["mean_stress"])
    params = {k: v.detach() for k, v in frozen.named_parameters()}
    w = "node_decoder.2.bias" if "node_decoder.2.bias" in params else list(params)[-1]

    def fp(bias):
        p = dict(params)
        p[w] = bias
        return torch.func.functional_call(frozen, p, (db,), {"scale_output": True}).local_stress
    with pytest.raises(NotImplementedError, match="functional_call"):
        torch.func.vmap(fp)(params[w].unsqueeze(0).repeat(2, 1))
    t, _ = _model_fn(c, frozen, ("nodes_types",), db)
    with pytest.raises(NotImplementedError, match="nodes_types"):
        torch.func.vmap(t)(db.nodes_types.unsqueeze(0).repeat(2, 1, 1))
