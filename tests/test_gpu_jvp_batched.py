"""GPU checks of batched tangents: torch.func.jacfwd and torch.func.vmap over torch.func.jvp reach one pdg_jvp_batched
pass for up to 64 tangents (more in passes of 64).

Every column of a batched pass must have the bits of a single torch.func.jvp call on the same tangent: tangent k runs
the same operations in the same order as a one-tangent pass.  The localisation field and a shape sensitivity, both
from jacfwd, are held to the bar of tests/test_gpu_jvp.py against per-column fp64 oracle JVPs."""
import ctypes as C
import functools
from types import SimpleNamespace

import pytest
import torch

import pdg_helpers as H
import test_gpu_jvp as JV
from oracle import pdg_oracle as O

pytestmark = pytest.mark.gpu
INPUTS = ("mean_stress", "pos", "edge_attr")
# train2_div: golden batch; synthetic: 3 x 600; mesh1024: one 1 024-node mesh (more tangent groups than one in the edge
# kernel: its x-grid leaves most SMs idle); configs1: 32 x 1 024 (one group of all K tangents)
GRAPHS = ["train2_div", "synthetic", "mesh1024", "configs1"]
KS = [1, 2, 3, 8, 65]
# Jacobian columns measured on a B200 (1 000 W) to miss the bar of tests/test_gpu_jvp.py, with their (L-inf, L2) errors
# against fp64.  Every column of a batched pass has the bits of a single pdg_jvp call (tests above), so a miss here is
# one of the single-tangent JVP (tests/test_gpu_jvp.py: ReLU masks that two fp32 evaluations round differently).
MEASURED_MISSES = {
    "mesh1024 localisation column 1": (3.42e-03, 2.86e-04),
}


@functools.lru_cache(maxsize=None)
def _graph(name):
    """SimpleNamespace(batch, stats, sd, model, db)"""
    if name in ("train2_div", "synthetic"):
        c = JV._case(name)
        batch, stats, sd = c.batch, c.stats, c.sd
    elif name == "mesh1024":
        from pdivgnn_b200 import synth
        _, batch, stats = H.oracle_batch_from_samples([synth.make_rve_mesh(69, 1024)], True)
        sd = O.init_state_dict(seed=69)
    else:
        _, _, batch, stats = H.synthetic_batch(32, 1024)
        sd = O.init_state_dict(seed=69)
    c = SimpleNamespace(batch=batch, stats=stats, sd=sd)
    c.model = JV._model(c)
    c.db = H.DeviceBatch(batch)
    return c


def _tangents(c, k, seed=5):
    """[K, *shape] device tangents of the three inputs"""
    g = torch.Generator().manual_seed(seed)
    return {n: torch.randn((k,) + tuple(getattr(c.db, n).shape), generator=g).cuda() for n in INPUTS}


def _f(c, keys):
    def f(*xs):
        b = SimpleNamespace(**vars(c.db))
        for k, x in zip(keys, xs):
            setattr(b, k, x)
        return c.model(b, scale_output=True, scale_input=True).local_stress
    return f, tuple(getattr(c.db, k) for k in keys)


def _loop(c, tan, k):
    """K single-tangent torch.func.jvp calls; tan: {input: [K, ...] or unbatched tensor}"""
    keys = list(tan)
    f, x0 = _f(c, keys)
    return torch.stack([torch.func.jvp(f, x0, tuple(tan[n][i] if tan[n].dim() > x.dim() else tan[n]
                                                     for n, x in zip(keys, x0)))[1] for i in range(k)])


def _vmapped(c, tan, in_dims):
    keys = list(tan)
    f, x0 = _f(c, keys)
    return torch.func.vmap(lambda *v: torch.func.jvp(f, x0, v)[1], in_dims=in_dims)(*(tan[n] for n in keys))


# ---- bit identity with the loop --------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("name", GRAPHS)
def test_vmap_over_jvp_equals_loop(name, k):
    c = _graph(name)
    tan = _tangents(c, k)
    ours = _vmapped(c, tan, (0, 0, 0))
    assert ours.shape == (k, c.batch.num_nodes, 3)
    ref = _loop(c, tan, k)
    assert torch.equal(ours, ref)
    assert ours.abs().max() > 0


@pytest.mark.parametrize("name", GRAPHS)
def test_jacfwd_columns_equal_loop(name):
    """jacfwd over theta in R^3 of f(x0 + sum_k theta_k V_k): column k is the tangent V_k, exactly"""
    c = _graph(name)
    k = 3
    tan = _tangents(c, k, seed=8)
    f, x0 = _f(c, INPUTS)

    def g(theta):
        return f(*(x + torch.tensordot(theta, tan[n], 1) for n, x in zip(INPUTS, x0)))
    jac = torch.func.jacfwd(g)(torch.zeros(k, device="cuda"))
    assert jac.shape == (c.batch.num_nodes, 3, k)
    ref = _loop(c, tan, k)
    for i in range(k):
        assert torch.equal(jac[..., i], ref[i]), i


@pytest.mark.parametrize("name", ["train2_div", "mesh1024"])
@pytest.mark.parametrize("case", ["mean_stress", "pos", "edge_attr", "ms_unbatched", "no_ea_tangent"])
def test_tangent_subsets_equal_loop(name, case):
    """each input alone; mean_stress unbatched (stride 0, the same tangent for every k) while pos and edge_attr are
    batched; edge_attr with no tangent at all"""
    c = _graph(name)
    k = 3
    tan = _tangents(c, k, seed=11)
    if case in INPUTS:
        tan, dims = {case: tan[case]}, (0,)
    elif case == "ms_unbatched":
        tan["mean_stress"] = tan["mean_stress"][1]
        dims = (None, 0, 0)
    else:
        del tan["edge_attr"]
        dims = (0, 0)
    ours = _vmapped(c, tan, dims)
    assert torch.equal(ours, _loop(c, tan, k))
    assert ours.abs().max() > 0


@pytest.mark.parametrize("name", ["train2_div", "mesh1024"])
def test_nested_vmap_equals_flat(name):
    c = _graph(name)
    tan = _tangents(c, 6, seed=13)
    flat = _vmapped(c, tan, (0, 0, 0))
    f, x0 = _f(c, INPUTS)
    inner = torch.func.vmap(lambda *v: torch.func.jvp(f, x0, v)[1])
    nested = torch.func.vmap(inner)(*(tan[n].reshape(2, 3, *tan[n].shape[1:]) for n in INPUTS))
    assert nested.shape == (2, 3, c.batch.num_nodes, 3)
    assert torch.equal(nested.reshape(flat.shape), flat)


@pytest.mark.parametrize("name", ["synthetic", "configs1"])
def test_permuted_tangents_permute_output(name):
    c = _graph(name)
    tan = _tangents(c, 8, seed=17)
    perm = torch.randperm(8, generator=torch.Generator().manual_seed(3)).cuda()
    a = _vmapped(c, tan, (0, 0, 0))
    b = _vmapped(c, {n: t[perm] for n, t in tan.items()}, (0, 0, 0))
    assert torch.equal(b, a[perm])


# ---- against the oracle ----------------------------------------------------------------------------------------------
def _oracle_jacfwd(c, build, theta0, dtype):
    """jacfwd of the oracle's local_stress through build(theta, batch, dtype) -> batch"""
    def g(theta):
        return O.forward(c.sd, build(theta, c.batch, dtype), c.stats, 10, scale_output=True, scale_input=True,
                         dtype=dtype)
    return torch.func.jacfwd(g)(theta0.to(dtype)).double()


def _localisation(theta, b, dtype=None):
    nb = SimpleNamespace(**vars(b))
    nb.mean_stress = theta.expand(b.mean_stress.shape[0], 3)
    return nb


@functools.lru_cache(maxsize=None)
def _shape_dirs_cpu(n):
    return torch.randn(3, n, 2, generator=torch.Generator().manual_seed(23), dtype=torch.float64) * 0.01


def _shape_dirs(b, dtype):
    """three design directions D_k of the node positions (drawn outside jacfwd: vmap refuses random operations)"""
    return _shape_dirs_cpu(b.pos.shape[0]).to(device=b.pos.device, dtype=dtype)


def _shape(theta, b, dtype):
    """pos(theta) = pos + sum_k theta_k D_k and edge_attr = |pos[row] - pos[col]| in torch (periodic edges stay 0)"""
    nb = SimpleNamespace(**vars(b))
    pos = b.pos.to(dtype) + torch.tensordot(theta, _shape_dirs(b, dtype), 1)
    d = pos[b.edge_index[0]] - pos[b.edge_index[1]]
    nb.pos = pos
    nb.edge_attr = torch.where(b.edge_attr == 0, torch.zeros_like(d[:, 0]), d.norm(dim=1))
    return nb


@pytest.mark.parametrize("what", ["localisation", "shape"])
def test_jacfwd_matches_oracle_and_adjoint(what):
    """The [N, 3, 3] Jacobian of one mesh against per-column fp64 oracle JVPs (bar of tests/test_gpu_jvp.py), and the
    adjoint identity <u, J e_k> = <J^T u, e_k> per column against pdg_backward_inputs.  A column in MEASURED_MISSES is
    held to 1.25x its measured error, and the test is then reported as an expected failure once every check has run."""
    c = _graph("mesh1024")
    _shape_dirs_cpu(c.batch.num_nodes)
    build = _localisation if what == "localisation" else _shape
    theta0 = c.batch.mean_stress[0].clone() if what == "localisation" else torch.zeros(3, dtype=torch.float32)

    def ours_f(theta):
        return c.model(build(theta, c.db, torch.float32), scale_output=True, scale_input=True).local_stress
    ours = torch.func.jacfwd(ours_f)(theta0.cuda()).double().cpu()
    t64 = _oracle_jacfwd(c, build, theta0, torch.float64)
    t32 = _oracle_jacfwd(c, build, theta0, torch.float32)
    assert ours.shape == t64.shape == (c.batch.num_nodes, 3, 3)
    misses = []
    for k in range(3):
        label = f"mesh1024 {what} column {k}"
        e, r = H.rel_err(ours[..., k], t64[..., k]), H.rel_err(t32[..., k], t64[..., k])
        print(f"{label}: Linf {e[0]:.2e} L2 {e[1]:.2e} (oracle fp32 {r[0]:.2e} / {r[1]:.2e})")
        if e[0] <= max(JV.TOL, 4 * r[0]) and e[1] <= max(JV.TOL, 3 * r[1]):
            continue
        m = MEASURED_MISSES.get(label)
        assert m is not None and e[0] <= JV.GUARD * m[0] and e[1] <= JV.GUARD * m[1], (label, e, r, m)
        misses.append(f"{label}: {e[0]:.2e} / {e[1]:.2e}")
    u = torch.randn(c.batch.num_nodes, 3, generator=torch.Generator().manual_seed(29), dtype=torch.float64)
    theta = theta0.cuda().clone().requires_grad_(True)
    (gt,) = torch.autograd.grad((ours_f(theta) * u.float().cuda()).sum(), theta)
    th32 = theta0.clone().requires_grad_(True)
    (gt32,) = torch.autograd.grad((O.forward(c.sd, build(th32, c.batch, torch.float32), c.stats, 10, scale_output=True,
                                             scale_input=True, dtype=torch.float32) * u.float()).sum(), th32)
    for k in range(3):
        def gap(jv, g):
            a, b = float((u * jv).sum()), float(g[k])
            return abs(a - b) / max(abs(a), abs(b))
        mine, ref = gap(ours[..., k], gt.double().cpu()), gap(t32[..., k], gt32.double())
        print(f"adjoint mesh1024 {what} column {k}: ours {mine:.2e}, oracle fp32 {ref:.2e}")
        assert mine <= max(JV.TOL, 4 * ref), (k, mine, ref)
    if misses:
        pytest.xfail("measured miss of the bar, within its regression guard: " + "; ".join(misses))


# ---- launches --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 8, 64, 65])
def test_one_pass_per_64_tangents(k):
    from pdivgnn_b200 import _lib
    c = _graph("train2_div")
    L = _lib.lib()
    T = c.model.message_passing_steps
    tan = _tangents(c, k)
    _vmapped(c, tan, (0, 0, 0))  # plan cached, functions attributes set
    L.pdg_launch_count(1)
    _vmapped(c, tan, (0, 0, 0))
    passes = -(-k // 64)
    assert L.pdg_launch_count(1) == (4 + 3 * T) + passes * (3 + 3 * T)


# ---- C ABI -----------------------------------------------------------------------------------------------------------
def _abi_batched(s, k, tans, strides, jws=None, ws_bytes=None):
    from pdivgnn_b200 import _lib
    nbytes = s.L.pdg_jvp_batched_ws_bytes(s.n, s.e, s.steps, k)
    if jws is None:
        jws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device="cuda")
    out = torch.full((max(k, 1), s.n, 3), float("nan"), device="cuda")
    args = []
    for t, st in zip(tans, strides):
        args += [s.p(t), st]
    rc = s.L.pdg_jvp_batched(C.byref(s.ps), C.byref(s.norm), *s.ins, s.p(s.ws), s.p(jws),
                             nbytes if ws_bytes is None else ws_bytes, k, *args, s.p(out), _lib.stream_ptr())
    return rc, out


def _abi_tangents(s, k):
    g = torch.Generator().manual_seed(41)
    shapes = ((s.n, 3), (s.n, 2), (s.e,))
    return [torch.randn((k,) + sh, generator=g).cuda().contiguous() for sh in shapes], \
        [sh[0] * (sh[1] if len(sh) > 1 else 1) for sh in shapes]


def test_c_abi_batched_properties():
    s = JV._abi_setup()
    k = 5
    tans, strides = _abi_tangents(s, k)
    outs = []
    for fill in (0x00, 0xFF, 0x7F):
        nbytes = s.L.pdg_jvp_batched_ws_bytes(s.n, s.e, s.steps, k)
        rc, out = _abi_batched(s, k, tans, strides, torch.full((nbytes,), fill, dtype=torch.uint8, device="cuda"))
        assert rc == 0, s.L.pdg_last_error()
        outs.append(out)
    assert torch.isfinite(outs[0]).all() and outs[0].abs().max() > 0
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    # each column: the bits of pdg_jvp on that tangent
    for i in range(k):
        s.tan = dict(zip(INPUTS, (t[i] for t in tans)))
        rc, one = JV._abi_jvp(s)
        assert rc == 0 and torch.equal(one, outs[0][i]), i
    # pdg_jvp_batched at K = 1 gives the bits of pdg_jvp
    rc, b1 = _abi_batched(s, 1, [t[:1] for t in tans], strides)
    s.tan = dict(zip(INPUTS, (t[0] for t in tans)))
    rc1, one = JV._abi_jvp(s)
    assert rc == 0 and rc1 == 0 and torch.equal(b1[0], one)
    # NULL tangents: exact zeros
    rc, zero = _abi_batched(s, k, [None] * 3, [0] * 3)
    assert rc == 0 and (zero == 0).all()
    # stride 0: the same bits as a materialised copy
    rc, a = _abi_batched(s, k, [t[2:3] for t in tans], [0] * 3)
    rc2, b = _abi_batched(s, k, [t[2:3].expand(k, *t.shape[1:]).contiguous() for t in tans], strides)
    assert rc == 0 and rc2 == 0 and torch.equal(a, b)
    assert all(torch.equal(a[i], outs[0][2]) for i in range(k))


def test_c_abi_batched_refusals():
    from pdivgnn_b200 import _lib
    s = JV._abi_setup()
    tans, strides = _abi_tangents(s, 2)
    for k in (0, 65):
        rc, _ = _abi_batched(s, k, tans, strides, ws_bytes=1 << 30)
        assert rc == -1 and b"n_tangents" in s.L.pdg_last_error(), k
        assert s.L.pdg_jvp_batched_ws_bytes(s.n, s.e, s.steps, k) == 0
    rc, _ = _abi_batched(s, 2, tans, strides, ws_bytes=s.L.pdg_jvp_batched_ws_bytes(s.n, s.e, s.steps, 2) - 1)
    assert rc == -1 and b"workspace" in s.L.pdg_last_error()
    assert s.L.pdg_jvp_batched_ws_bytes(s.n, s.e, s.steps, 2) == 2 * s.L.pdg_jvp_ws_bytes(s.n, s.e, s.steps)
    for steps in (0, 63):
        bad = SimpleNamespace(**vars(s))
        bad.ins = s.ins[:7] + (steps,) + s.ins[8:]
        rc, _ = _abi_batched(bad, 2, tans, strides, ws_bytes=1 << 30)
        assert rc == -1 and b"steps" in s.L.pdg_last_error(), steps
    s = JV._abi_setup(flags=_lib.FLAG_SCALE_INPUT | _lib.FLAG_ZERO_CHECK)  # forward without PDG_FLAG_SAVE
    rc, _ = _abi_batched(s, 2, tans, strides)
    assert rc == -1 and b"SAVE" in s.L.pdg_last_error()
    s = JV._abi_setup(precision="bf16")
    rc, _ = _abi_batched(s, 2, tans, strides)
    assert rc == -1 and b"fp32" in s.L.pdg_last_error()


# ---- Python errors ---------------------------------------------------------------------------------------------------
def test_unsupported_uses_raise():
    from pdivgnn_b200 import _lib
    c = _graph("train2_div")
    f, x0 = _f(c, ("mean_stress",))
    with pytest.raises(NotImplementedError, match="batched tangents"):
        torch.func.vmap(f)(x0[0].unsqueeze(0).repeat(2, 1, 1))
    m16 = JV._model(c, precision="bf16")

    def f16(ms):
        b = SimpleNamespace(**vars(c.db))
        b.mean_stress = ms
        return m16(b).local_stress
    with pytest.raises(NotImplementedError, match="fp32"):
        torch.func.jacfwd(lambda S: f16(S.expand(c.batch.num_nodes, 3)))(x0[0][0].clone())
    params = {k: v.detach() for k, v in c.model.named_parameters()}
    w = "node_decoder.2.bias" if "node_decoder.2.bias" in params else list(params)[-1]

    def fp(bias):
        p = dict(params)
        p[w] = bias
        return torch.func.functional_call(c.model, p, (c.db,), {"scale_output": True}).local_stress
    with pytest.raises(NotImplementedError, match="parameters"):
        torch.func.jacfwd(fp)(params[w])
    with pytest.raises(RuntimeError, match="BatchedTensor"):
        torch.func.vmap(lambda t: (_lib.ptr(t), t)[1])(torch.zeros(2, 3, device="cuda"))
