"""torch.autograd glue: tensors -> raw pointers -> C ABI (include/pdg.h).

Nothing here computes; it validates inputs, builds / caches the device graph plan,
allocates the workspace from torch's caching allocator (so stream semantics hold) and
calls ``pdg_forward`` / ``pdg_forward_batched`` / ``pdg_backward_inputs`` / ``pdg_jvp_batched`` / ``pdg_vjp_batched``
on the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import os
from collections import OrderedDict

import torch
import torch.autograd.forward_ad as fwAD

from . import _lib

_PARAM_KEYS = None


def param_list(model):
    """The 28 parameters in state_dict order (include/pdg.h, PDG_NUM_PARAMS).  The list is cached on the model (walking
    the module tree costs ~30 us per call, twice per training step); `nn.Module._apply` (.to / .cuda / .float) keeps
    Parameter identities, `load_state_dict` copies in place, and replacing a Parameter object invalidates the cache
    through the id check."""
    cache = model.__dict__.get("_pdg_params")
    if cache is not None:
        ps = cache
        ok = True
        for (_, q), p in zip(model.named_parameters(), ps) if getattr(model, "_pdg_params_strict", False) else ():
            ok = ok and q is p
        if ok:
            return ps
    ps = [p for _, p in model.named_parameters()]
    if len(ps) != _lib.PDG_NUM_PARAMS or sum(p.numel() for p in ps) != _lib.PDG_PARAM_ELEMS:
        raise RuntimeError("unexpected parameter layout")
    model.__dict__["_pdg_params"] = ps
    return ps


# ---- graph plan cache -----------------------------------------------------------------
# Keyed by the identity of the edge_index storage; the cached entry keeps the tensor alive
# so its address cannot be recycled while the entry exists; in-place edits bump _version.
_PLAN_CACHE: "OrderedDict[tuple, tuple]" = OrderedDict()
_PLAN_CACHE_SIZE = 8


class GraphPlan:
    __slots__ = ("buf", "n_nodes", "n_edges", "edge_index")

    def __init__(self, buf, n_nodes, n_edges, edge_index):
        self.buf, self.n_nodes, self.n_edges, self.edge_index = buf, n_nodes, n_edges, edge_index

    def views(self):
        """int32 device views (perm, recv, send, rowptr, send_ptr, send_list) for tests."""
        L = _lib.lib()
        ptrs = [C.c_void_p() for _ in range(6)]
        _lib.check(L.pdg_plan_views(_lib.ptr(self.buf), self.n_nodes, self.n_edges, *[C.byref(p) for p in ptrs]),
                   "pdg_plan_views")
        base = _lib.raw(self.buf).data_ptr()
        e_pad = (self.n_edges + 127) // 128 * 128
        sizes = [e_pad, e_pad, e_pad, self.n_nodes + 1, self.n_nodes + 1, self.n_edges]
        i32 = self.buf.view(torch.int32)
        out = []
        for p, n in zip(ptrs, sizes):
            off = (p.value - base) // 4
            out.append(i32[off:off + n])
        return out


# PDG_VALIDATE=1 (or set_validation(True)): every newly built plan is checked for node ids outside [0, N) -- one
# device->host read per distinct edge_index.  Off by default: the kernels are memory-safe either way (ids are clamped),
# and a graph built by this package's own batcher is valid by construction.
_VALIDATE = os.environ.get("PDG_VALIDATE", "0") not in ("", "0")


def set_validation(on: bool) -> None:
    global _VALIDATE
    _VALIDATE = bool(on)


def build_plan(edge_index: torch.Tensor, n_nodes: int, validate=None) -> GraphPlan:
    L = _lib.lib()
    edge_index = _lib.require_cuda(edge_index, "edge_index", torch.int64)
    if edge_index.dim() != 2 or edge_index.shape[0] != 2:
        raise ValueError("edge_index must be [2, E]")
    n_edges = edge_index.shape[1]
    key = (edge_index.data_ptr(), edge_index._version, n_nodes, n_edges, edge_index.device.index)
    hit = _PLAN_CACHE.get(key)
    if hit is not None:
        _PLAN_CACHE.move_to_end(key)
        return hit
    dev = edge_index.device
    with torch.cuda.device(dev):
        buf = torch.empty(L.pdg_plan_bytes(n_nodes, n_edges), dtype=torch.uint8, device=dev)
        tmp_bytes = L.pdg_plan_tmp_bytes(n_nodes, n_edges)
        tmp = torch.empty(tmp_bytes, dtype=torch.uint8, device=dev)
        _lib.check(L.pdg_plan_build(_lib.ptr(edge_index), n_nodes, n_edges, _lib.ptr(buf), _lib.ptr(tmp), tmp_bytes,
                                    _lib.stream_ptr(dev)), "pdg_plan_build")
        if _VALIDATE if validate is None else validate:
            st = C.c_int32(0)
            if L.pdg_plan_status(_lib.ptr(buf), n_nodes, n_edges, C.byref(st), _lib.stream_ptr(dev)) != 0:
                raise IndexError(f"edge_index contains node ids outside [0, {n_nodes}) "
                                 f"({L.pdg_last_error().decode()})")
    plan = GraphPlan(buf, n_nodes, n_edges, edge_index)
    _PLAN_CACHE[key] = plan
    while len(_PLAN_CACHE) > _PLAN_CACHE_SIZE:
        _PLAN_CACHE.popitem(last=False)
    return plan


def _bucket(nbytes: int) -> int:
    """Round a workspace size up to 1/16 of its power of two (<= 6.25 % slack): batches of slightly different
    sizes then reuse the same cached allocator block instead of triggering cudaMalloc / cudaFree (a device sync)."""
    if nbytes < (1 << 20):
        return nbytes
    g = 1 << (nbytes.bit_length() - 5)
    return (nbytes + g - 1) // g * g


def _params_struct(params):
    s = _lib.PdgParams()
    for i, p in enumerate(params):
        s.p[i] = _lib.raw(p).data_ptr()
    return s


class _EPDFunction(torch.autograd.Function):
    """pdg_forward, pdg_backward_inputs (reverse mode), pdg_vjp_batched (vmapped reverse mode) and pdg_jvp (forward
    mode).  Written in setup_context style so that torch.func.jvp accepts it; the forward workspace reaches ctx as a
    second, non-differentiable output.  `swapped`: parameters other than the cached param_list were in the module
    (torch.func.functional_call), so a gradient for them would never reach this Function."""

    @staticmethod
    def forward(model, plan, mean_stress, pos, types, edge_attr, flags, steps, prec, need_grad, need_tan, swapped,
                *params):
        L = _lib.lib()
        dev = mean_stress.device
        n, e = plan.n_nodes, plan.n_edges
        if need_grad or need_tan:
            flags |= _lib.FLAG_SAVE
        params = [_lib.require_cuda(p.detach(), "parameter", torch.float32) for p in params]
        norm = model._norm_struct()
        with torch.cuda.device(dev):
            ws_bytes = L.pdg_forward_ws_bytes(n, e, steps, flags)
            ws = torch.empty(_bucket(ws_bytes), dtype=torch.uint8, device=dev)
            out = torch.empty((n, 3), dtype=torch.float32, device=dev)
            ps = _params_struct(params)
            _lib.check(L.pdg_forward(C.byref(ps), C.byref(norm), _lib.ptr(mean_stress), _lib.ptr(pos), _lib.ptr(types),
                                     _lib.ptr(edge_attr), _lib.ptr(plan.buf), n, e, steps, flags, prec, _lib.ptr(ws),
                                     ws_bytes, _lib.ptr(out), _lib.stream_ptr(dev)), "pdg_forward")
        return out, ws

    @staticmethod
    def setup_context(ctx, inputs, output):
        model, plan, mean_stress, pos, types, edge_attr, flags, steps, prec, need_grad, need_tan, swapped, *params = inputs
        _, ws = output
        ctx.mark_non_differentiable(ws)
        # no zero gradient is materialised for the workspace output (a memset of the whole saved state per backward);
        # tangents that do not exist arrive as None (pdg_jvp reads NULL as a zero tangent)
        ctx.set_materialize_grads(False)
        ctx.pdg = None
        if need_grad or need_tan:
            params = [_lib.require_cuda(p.detach(), "parameter", torch.float32) for p in params]
            ctx.pdg = (model, plan, mean_stress, pos, types, edge_attr, flags | _lib.FLAG_SAVE, steps, prec, params, ws,
                       model._norm_struct())
        ctx.pdg_need_grad = need_grad
        ctx.pdg_swapped = swapped

    @staticmethod
    def jvp(ctx, _model, _plan, t_ms, t_pos, _types, t_ea, *_rest):
        """Tangent of local_stress from the tangents of mean_stress, pos and edge_attr (fp32 mode).  Under vmap the
        tangents are batched and _EPDTangent's vmap rule makes one tangent pass for the whole batch.  Tangents of the
        parameters were refused in epd_forward; whatever arrives for them here is ignored."""
        t_out = _EPDTangent.apply(ctx.pdg, t_ms, t_pos, t_ea)
        if not ctx.pdg_need_grad:
            ctx.pdg = None  # no backward follows: release the forward workspace now
        return t_out, None

    @staticmethod
    def vmap(info, in_dims, model, plan, mean_stress, pos, types, edge_attr, flags, steps, prec, need_grad, need_tan,
             swapped, *params):
        """torch reaches this rule only when a model input or parameter is batched at this vmap level: with unbatched
        primals it skips the level, and batched tangents go to _EPDTangent.vmap.  Batched mean_stress, pos and
        edge_attr (one graph under many loads or shapes) run as instances of pdg_forward_batched: the vmapped dimension
        moves to the front, unbatched inputs are shared (stride 0).  Inference only, fp32 only."""
        if need_grad or need_tan:
            raise NotImplementedError(
                "pdivgnn_b200: vmap over mean_stress, pos or edge_attr runs the forward only (under torch.no_grad(), or "
                "with a model whose parameters and inputs do not require grad); derivatives through it are not "
                "implemented.  Derivatives at one input point are: batched tangents (torch.func.jacfwd, vmap over "
                "torch.func.jvp) and batched cotangents (torch.func.jacrev, vmap over torch.func.vjp)")
        if prec != _lib.PREC_FP32:
            raise NotImplementedError("pdivgnn_b200: vmap over the model's inputs needs precision='fp32'; in the 16-bit "
                                      "mode call the model once per input")
        if any(d is not None for d in in_dims[12:]):
            raise NotImplementedError(_BATCHED_PARAMS)
        if in_dims[4] is not None:
            raise NotImplementedError("pdivgnn_b200: vmap over nodes_types is not implemented; the instances of one "
                                      "vmapped forward share the graph and its node types, and differ in mean_stress, "
                                      "pos and edge_attr")
        xs = [x if d is None else x.movedim(d, 0) for x, d in zip((mean_stress, pos, edge_attr), (in_dims[2], in_dims[3], in_dims[5]))]
        out, ws = _EPDInstances.apply((model, plan, types, flags, steps, params), *xs)
        return (out, ws), (0, None)

    @staticmethod
    def backward(ctx, grad_out, _grad_ws):
        if grad_out is not None and _lib.is_vmapped(grad_out):
            return _EPDFunction._backward_batched(ctx, grad_out)
        L = _lib.lib()
        if not hasattr(L, "pdg_backward_inputs") or getattr(L.pdg_backward_inputs, "argtypes", None) is None:
            raise RuntimeError("libpdivgnn.so was built without pdg_backward_inputs")
        model, plan, mean_stress, pos, types, edge_attr, flags, steps, prec, params, ws, norm = ctx.pdg
        n, e = plan.n_nodes, plan.n_edges
        dev = mean_stress.device
        if grad_out is None:  # local_stress received no gradient: as autograd's materialised zeros
            grad_out = torch.zeros((n, 3), dtype=torch.float32, device=dev)
        grad_out = _lib.require_cuda(grad_out, "grad_local_stress", torch.float32)
        need = ctx.needs_input_grad  # slots 2, 3, 5: mean_stress, pos, edge_attr
        with torch.cuda.device(dev):
            flat = torch.empty(_lib.PDG_PARAM_ELEMS, dtype=torch.float32, device=dev)
            g_ms = torch.empty((n, 3), dtype=torch.float32, device=dev) if need[2] else None
            g_pos = torch.empty((n, 2), dtype=torch.float32, device=dev) if need[3] else None
            g_ea = torch.empty(e, dtype=torch.float32, device=dev) if need[5] else None
            bws_bytes = L.pdg_backward_ws_bytes(n, e, steps)
            bws = torch.empty(_bucket(bws_bytes), dtype=torch.uint8, device=dev)
            ps = _params_struct(params)
            _lib.check(L.pdg_backward_inputs(C.byref(ps), C.byref(norm), _lib.ptr(mean_stress), _lib.ptr(pos),
                                             _lib.ptr(types), _lib.ptr(edge_attr), _lib.ptr(plan.buf), n, e, steps, flags,
                                             prec, _lib.ptr(ws), _lib.ptr(bws), bws_bytes, _lib.ptr(grad_out),
                                             _lib.ptr(flat), _lib.ptr(g_ms), _lib.ptr(g_pos), _lib.ptr(g_ea),
                                             _lib.stream_ptr(dev)), "pdg_backward_inputs")
        dp = getattr(model, "_pdg_dp", None)
        # data parallel: one all-reduce of the flat buffer (dist.py); input gradients stay rank-local, as in torch DDP
        if dp is not None and dp[0]:
            from .dist import allreduce_flat_
            allreduce_flat_(flat, dp[1], getattr(model, "_pdg_peer", None))
        grads, off = [], 0
        for i, p in enumerate(params):
            grads.append(flat[off:off + p.numel()].view(p.shape) if need[12 + i] else None)
            off += p.numel()
        ctx.pdg = None
        return (None, None, g_ms, g_pos, None, g_ea) + (None,) * 6 + tuple(grads)

    @staticmethod
    def _backward_batched(ctx, grad_out):
        """The cotangent carries a vmap level (torch.func.jacrev, torch.func.vmap over torch.func.vjp or torch.func.grad):
        _EPDAdjoint's vmap rule runs every cotangent of the level in one pdg_vjp_batched pass.  Input gradients only;
        under data parallelism they stay rank-local.  The forward state is kept: jacrev may call again (chunk_size)."""
        need = ctx.needs_input_grad
        prec = ctx.pdg[8]
        if prec != _lib.PREC_FP32:
            raise NotImplementedError("pdivgnn_b200: batched reverse-mode derivatives (torch.func.jacrev, vmap over vjp) "
                                      "need precision='fp32'; the 16-bit mode's input gradients miss its 2e-2 tolerance")
        if ctx.pdg_swapped or any(need[12:]):
            raise NotImplementedError("pdivgnn_b200: batched reverse-mode derivatives with respect to the parameters are "
                                      "not implemented (torch.func.jacrev or vmap over vjp of the parameters); those "
                                      "with respect to mean_stress, pos and edge_attr are")
        want = (need[2], need[3], need[5])
        outs = iter(_EPDAdjoint.apply(ctx.pdg, want, grad_out) if any(want) else ())
        g_ms, g_pos, g_ea = (next(outs) if w else None for w in want)
        return (None, None, g_ms, g_pos, None, g_ea) + (None,) * (6 + len(ctx.pdg[9]))


class _EPDAdjoint(torch.autograd.Function):
    """Input gradients for K cotangents of local_stress in one pdg_vjp_batched pass.  `state` is the forward's ctx tuple,
    `want` the (mean_stress, pos, edge_attr) flags of the gradients to form, `g` the cotangent [N, 3] or [K, N, 3].
    Returns the wanted gradients in that order, each [K, *input shape] (or the input's shape when g is [N, 3]).  The
    vmap rule folds the vmapped dimension into K.  There is no backward: second-order derivatives are not implemented."""

    @staticmethod
    def forward(state, want, g):
        L = _lib.lib()
        model, plan, mean_stress, pos, types, edge_attr, flags, steps, prec, params, ws, norm = state
        dev = mean_stress.device
        n, e = plan.n_nodes, plan.n_edges
        k = g.shape[0] if g.dim() == 3 else None
        g = _lib.require_cuda(g.to(torch.float32), "grad_local_stress", torch.float32).reshape(k or 1, n, 3)
        with torch.cuda.device(dev):
            outs = [torch.empty((k or 1,) + s, dtype=torch.float32, device=dev) if w else None
                    for w, s in zip(want, _tangent_shapes(state))]
            vws_bytes = L.pdg_vjp_batched_ws_bytes(n, e, steps, k or 1)
            vws = torch.empty(_bucket(vws_bytes), dtype=torch.uint8, device=dev)
            ps = _params_struct(params)
            _lib.check(L.pdg_vjp_batched(C.byref(ps), C.byref(norm), _lib.ptr(mean_stress), _lib.ptr(pos),
                                         _lib.ptr(types), _lib.ptr(edge_attr), _lib.ptr(plan.buf), n, e, steps, flags,
                                         prec, _lib.ptr(ws), _lib.ptr(vws), vws_bytes, k or 1, _lib.ptr(g),
                                         *(_lib.ptr(o) for o in outs), _lib.stream_ptr(dev)), "pdg_vjp_batched")
        return tuple(o if k is not None else o[0] for o in outs if o is not None)

    @staticmethod
    def setup_context(ctx, inputs, output):
        pass

    @staticmethod
    def vmap(info, in_dims, state, want, g):
        """Moves the vmapped dimension B of the cotangent to the front and merges it with a K that an inner vmap level
        already folded in ([B, K, N, 3] -> [B*K, N, 3]: nested vmap flattens).  One pass per at most VJP_MAX_COTANGENTS
        cotangents."""
        b = info.batch_size
        g = g.unsqueeze(0).expand(b, *g.shape) if in_dims[2] is None else g.movedim(in_dims[2], 0)
        k = g.shape[1] if g.dim() == 4 else None
        g = g.reshape(b * (k or 1), *g.shape[-2:])
        cap = _lib.VJP_MAX_COTANGENTS
        parts = [_EPDAdjoint.apply(state, want, g[i:i + cap]) for i in range(0, g.shape[0], cap)]
        outs = tuple(p[0] if len(parts) == 1 else torch.cat(p) for p in zip(*parts))
        outs = tuple(o.reshape(b, k, *o.shape[1:]) if k is not None else o for o in outs)
        return outs, (0,) * len(outs)


def _tangent_shapes(state):
    plan = state[1]
    return ((plan.n_nodes, 3), (plan.n_nodes, 2), (plan.n_edges,))


_BATCHED_PARAMS = ("pdivgnn_b200: vmap over the model's parameters (model ensembles through torch.func.functional_call) "
                   "is not implemented; vmap over mean_stress, pos and edge_attr is")


class _EPDInstances(torch.autograd.Function):
    """local_stress of K instances of one graph: pdg_forward_batched, one pass per at most FWD_MAX_INSTANCES instances.
    `state` is (model, plan, nodes_types, flags, steps, params).  An input is of its per-graph shape (the same for every
    instance) or [K, *shape], at least one of them the latter; returns local_stress [K, N, 3] and the workspace.  The
    vmap rule folds the vmapped dimension into K.  Inference only: there is no backward."""

    @staticmethod
    def forward(state, mean_stress, pos, edge_attr):
        L = _lib.lib()
        model, plan, types, flags, steps, params = state
        dev = types.device
        n, e = plan.n_nodes, plan.n_edges
        xs, shapes = (mean_stress, pos, edge_attr), _tangent_shapes(state)
        k = next(x.shape[0] for x, s in zip(xs, shapes) if x.dim() == len(s) + 1)
        args = []
        for x, s, name in zip(xs, shapes, ("mean_stress", "pos", "edge_attr")):
            stride = 0
            if x.dim() == len(s) + 1 and x.stride(0) != 0:
                x, stride = x.contiguous(), x[0].numel()
            elif x.dim() == len(s) + 1:
                x = x[0]  # one input expanded over K: passed once, with stride 0
            args.append((_lib.require_cuda(x, name, torch.float32), stride))
        cap = _lib.FWD_MAX_INSTANCES
        with torch.cuda.device(dev):
            ws_bytes = L.pdg_forward_batched_ws_bytes(n, e, steps, flags, min(k, cap))
            ws = torch.empty(_bucket(ws_bytes), dtype=torch.uint8, device=dev)  # reused by every pass (stream order)
            out = torch.empty((k, n, 3), dtype=torch.float32, device=dev)
            ps, norm = _params_struct(params), model._norm_struct()
            for i in range(0, k, cap):
                kk = min(cap, k - i)
                xp = [_lib.ptr(x[i:i + kk] if st else x) for x, st in args]
                _lib.check(L.pdg_forward_batched(C.byref(ps), C.byref(norm), xp[0], args[0][1], xp[1], args[1][1],
                                                 _lib.ptr(types), xp[2], args[2][1], _lib.ptr(plan.buf), n, e, steps,
                                                 flags, _lib.PREC_FP32, _lib.ptr(ws), ws_bytes, kk, _lib.ptr(out[i:i + kk]),
                                                 _lib.stream_ptr(dev)), "pdg_forward_batched")
        return out, ws

    @staticmethod
    def setup_context(ctx, inputs, output):
        ctx.mark_non_differentiable(*output)

    @staticmethod
    def vmap(info, in_dims, state, *xs):
        """Moves the vmapped dimension B of every batched input to the front and merges it with the K that an inner
        vmap level folded in ([B, K, ...] -> [B*K, ...]: nested vmap flattens).  Unbatched inputs stay shared."""
        shapes = _tangent_shapes(state)
        b = info.batch_size
        xs = [x if d is None else x.movedim(d, 0) for x, d in zip(xs, in_dims[1:])]
        k = next(x.shape[1 if d is not None else 0] for x, d, s in zip(xs, in_dims[1:], shapes)
                 if x.dim() == len(s) + 1 + (d is not None))
        flat = []
        for x, d, s in zip(xs, in_dims[1:], shapes):
            if d is not None or x.dim() == len(s) + 1:
                if d is None:
                    x = x.unsqueeze(0)
                elif x.dim() == len(s) + 1:
                    x = x.unsqueeze(1)
                x = x.expand(b, k, *s).reshape(b * k, *s)
            flat.append(x)
        out, ws = _EPDInstances.apply(state, *flat)
        return (out.reshape(b, k, *out.shape[1:]), ws), (0, None)


class _EPDTangent(torch.autograd.Function):
    """Tangents of local_stress for K tangents of (mean_stress, pos, edge_attr) in one pdg_jvp_batched pass.  `state` is
    the forward's ctx tuple.  A tangent is None (zero), of the input's shape (the same for every k) or [K, *shape]; the
    result is [K, N, 3], or [N, 3] when no tangent has the K dimension.  The vmap rule folds the vmapped dimension into
    K.  There is no backward: second-order derivatives are not implemented."""

    @staticmethod
    def forward(state, t_ms, t_pos, t_ea):
        L = _lib.lib()
        model, plan, mean_stress, pos, types, edge_attr, flags, steps, prec, params, ws, norm = state
        dev = mean_stress.device
        n, e = plan.n_nodes, plan.n_edges
        ts, shapes = (t_ms, t_pos, t_ea), _tangent_shapes(state)
        ks = {t.shape[0] for t, s in zip(ts, shapes) if t is not None and t.dim() == len(s) + 1}
        if len(ks) > 1:
            raise ValueError(f"pdivgnn_b200: batched tangents disagree on their count: {sorted(ks)}")
        k = ks.pop() if ks else None
        args = []
        for t, s, name in zip(ts, shapes, ("mean_stress", "pos", "edge_attr")):
            stride = 0
            if t is not None:
                # tangents may arrive non-contiguous (an expanded load direction) or in another dtype; one tangent
                # expanded over K (leading stride 0) is passed once, with stride 0
                t = t.to(torch.float32)
                if t.dim() == len(s) + 1 and t.stride(0) != 0:
                    t, stride = t.reshape(k, *s), t[0].numel()
                elif t.dim() == len(s) + 1:
                    t = t[0]
                t = _lib.require_cuda(t, f"{name} tangent", torch.float32).reshape(-1, *s)
            args += [t, stride]
        with torch.cuda.device(dev):
            jws_bytes = L.pdg_jvp_batched_ws_bytes(n, e, steps, k or 1)
            jws = torch.empty(_bucket(jws_bytes), dtype=torch.uint8, device=dev)
            t_out = torch.empty((k or 1, n, 3), dtype=torch.float32, device=dev)
            ps = _params_struct(params)
            _lib.check(L.pdg_jvp_batched(C.byref(ps), C.byref(norm), _lib.ptr(mean_stress), _lib.ptr(pos),
                                         _lib.ptr(types), _lib.ptr(edge_attr), _lib.ptr(plan.buf), n, e, steps, flags,
                                         prec, _lib.ptr(ws), _lib.ptr(jws), jws_bytes, k or 1,
                                         _lib.ptr(args[0]), args[1], _lib.ptr(args[2]), args[3], _lib.ptr(args[4]),
                                         args[5], _lib.ptr(t_out), _lib.stream_ptr(dev)), "pdg_jvp_batched")
        return t_out if k is not None else t_out[0]

    @staticmethod
    def setup_context(ctx, inputs, output):
        pass

    @staticmethod
    def vmap(info, in_dims, state, *ts):
        """Moves the vmapped dimension B of every batched tangent to the front and merges it with a K that an inner
        vmap level already folded in ([B, K, ...] -> [B*K, ...]: nested vmap flattens).  Unbatched tangents keep the
        input's shape (stride 0 in the kernels).  One pass per at most JVP_MAX_TANGENTS tangents."""
        shapes = _tangent_shapes(state)
        b = info.batch_size
        ts = [t if d is None else t.movedim(d, 0) for t, d in zip(ts, in_dims[1:])]
        ks = {t.shape[1 if d is not None else 0] for t, d, s in zip(ts, in_dims[1:], shapes)
              if t is not None and t.dim() == len(s) + 1 + (d is not None)}
        if len(ks) > 1:
            raise ValueError(f"pdivgnn_b200: batched tangents disagree on their count: {sorted(ks)}")
        k = ks.pop() if ks else None
        flat = []
        for t, d, s in zip(ts, in_dims[1:], shapes):
            if t is not None and k is not None and (d is not None or t.dim() == len(s) + 1):
                if d is None:
                    t = t.unsqueeze(0)
                elif t.dim() == len(s) + 1:
                    t = t.unsqueeze(1)
                t = t.expand(b, k, *s).reshape(b * k, *s)
            flat.append(t)
        total, cap = b * (k or 1), _lib.JVP_MAX_TANGENTS
        outs = []
        for i in range(0, total, cap):
            part = [t[i:i + cap] if t is not None and t.dim() == len(s) + 1 else t for t, s in zip(flat, shapes)]
            outs.append(_EPDTangent.apply(state, *part))
        out = outs[0] if len(outs) == 1 else torch.cat(outs)
        return (out if k is None else out.reshape(b, k, *out.shape[1:])), 0


# ---- CUDA-graph replay of the inference forward (small-N latency) ------------------------------------------------------
# One forward is ~45 dependent kernel launches.  For one ~1 000-node mesh (the reference's own benchmark shape,
# scripts/benchmark_gnn_fem.py:81-100: one graph per call) the kernels themselves take ~0.1 ms while launching them one
# by one costs ~0.4 ms.  With `model.cuda_graphs = True` (or PDG_CUDA_GRAPHS=1) a no-grad forward on the SAME input
# tensors is captured once (pdg_forward on a capture stream: the library only enqueues on the stream it is given, its
# memsets and programmatic-dependent launches are capturable) and replayed afterwards with a single launch.
# The cache key is the identity of every buffer the captured kernels read (inputs, plan, parameters) plus the scalars
# baked into the launch arguments (flags, steps, precision, the 8 statistics); the entry keeps those tensors alive,
# so an address cannot be recycled under it.  In-place edits of inputs or parameters are seen by the replay (same
# addresses).  The result is copied out of the graph's static output buffer.
_GRAPH_CACHE: "OrderedDict[tuple, tuple]" = OrderedDict()
_GRAPH_CACHE_SIZE = 8
_GRAPHS_ENV = os.environ.get("PDG_CUDA_GRAPHS", "0") not in ("", "0")


def _forward_graphed(model, plan, mean_stress, pos, types, edge_attr, flags, steps, prec, params):
    L = _lib.lib()
    dev = mean_stress.device
    norm = model._norm_struct()
    key = (plan.buf.data_ptr(), mean_stress.data_ptr(), pos.data_ptr(), types.data_ptr(), edge_attr.data_ptr(), flags,
           steps, prec, tuple(p.data_ptr() for p in params), tuple(getattr(norm, f[0]) for f in norm._fields_), dev.index)
    hit = _GRAPH_CACHE.get(key)
    if hit is None:
        n, e = plan.n_nodes, plan.n_edges
        dparams = [_lib.require_cuda(p.detach(), "parameter", torch.float32) for p in params]
        ps = _params_struct(dparams)
        ws_bytes = L.pdg_forward_ws_bytes(n, e, steps, flags)

        def enqueue(ws, out):
            _lib.check(L.pdg_forward(C.byref(ps), C.byref(norm), _lib.ptr(mean_stress), _lib.ptr(pos), _lib.ptr(types),
                                     _lib.ptr(edge_attr), _lib.ptr(plan.buf), n, e, steps, flags, prec, _lib.ptr(ws),
                                     ws_bytes, _lib.ptr(out), _lib.stream_ptr(dev)), "pdg_forward")

        with torch.cuda.device(dev):
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):  # one eager run first: module load, function attributes
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
                out = torch.empty((n, 3), dtype=torch.float32, device=dev)
                enqueue(ws, out)
            torch.cuda.current_stream(dev).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                enqueue(ws, out)
        hit = (graph, out, (ws, plan, mean_stress, pos, types, edge_attr, dparams, norm))
        _GRAPH_CACHE[key] = hit
        while len(_GRAPH_CACHE) > _GRAPH_CACHE_SIZE:
            _GRAPH_CACHE.popitem(last=False)
    else:
        _GRAPH_CACHE.move_to_end(key)
    hit[0].replay()
    return hit[1].clone()


def epd_forward(model, mesh_graph, scale_output: bool, scale_input: bool, zero_check: bool = True) -> torch.Tensor:
    """EncodeProcessDecode.forward body past the early exit (models.py:301-321)."""
    mean_stress = _lib.require_cuda(mesh_graph.mean_stress, "mean_stress", torch.float32)
    pos = _lib.require_cuda(mesh_graph.pos, "pos", torch.float32)
    types = _lib.require_cuda(mesh_graph.nodes_types, "nodes_types", torch.int64).reshape(-1)
    edge_attr = _lib.require_cuda(mesh_graph.edge_attr, "edge_attr", torch.float32).reshape(-1)
    n = mean_stress.shape[0]
    if mean_stress.shape != (n, 3) or pos.shape != (n, 2) or types.numel() != n:
        raise ValueError("expected mean_stress [N,3], pos [N,2], nodes_types [N,1]")
    plan = build_plan(mesh_graph.edge_index, n)
    if edge_attr.numel() != plan.n_edges:
        raise ValueError("edge_attr must have one weight per edge")
    flags = (_lib.FLAG_SCALE_INPUT if scale_input else 0) | (_lib.FLAG_SCALE_OUTPUT if scale_output else 0) \
        | (_lib.FLAG_ZERO_CHECK if zero_check else 0)
    prec = _lib.PREC_BF16 if getattr(model, "precision", "fp32") in ("bf16", "fp16", "tc16") else _lib.PREC_FP32
    params = param_list(model)
    # grad mode is off inside Function.forward, so decide here whether the backward state must be kept: a frozen model
    # (no parameter requires grad) differentiated with respect to its inputs keeps it too
    need_grad = torch.is_grad_enabled() and (mean_stress.requires_grad or pos.requires_grad or edge_attr.requires_grad
                                             or any(p.requires_grad for p in params))
    # forward-mode AD (torch.autograd.forward_ad dual tensors, torch.func.jvp): tangents of the inputs keep the forward
    # state for pdg_jvp.  Parameters are looked at only while a dual level is open (no cost on the training path), and
    # through a fresh walk of the module: torch.func.functional_call swaps them under the cached list of param_list.
    need_tan = False
    if fwAD._current_level >= 0:
        need_tan = any(fwAD.unpack_dual(t).tangent is not None for t in (mean_stress, pos, edge_attr))
        if any(fwAD.unpack_dual(p).tangent is not None for _, p in model.named_parameters()):
            raise NotImplementedError("pdivgnn_b200: forward-mode derivatives with respect to the parameters are not "
                                      "implemented; tangents of mean_stress, pos and edge_attr are")
        if need_tan and prec != _lib.PREC_FP32:
            raise NotImplementedError("pdivgnn_b200: forward-mode derivatives need precision='fp32'; in the 16-bit mode "
                                      "per-row derivatives amplify the fp16 rounding beyond its 2e-2 tolerance "
                                      "(DESIGN.md section 5)")
    # inside torch.func transforms, parameters that torch.func.functional_call swapped in are not the cached list above,
    # so their gradient would never reach the library (jacrev over them would return zeros): a reverse-mode derivative
    # with respect to them is refused here, and a batched backward refuses any swapped parameter (a fresh walk only
    # under a transform)
    swapped = False
    transformed = torch._C._functorch.maybe_current_level() is not None
    if transformed:
        fresh = [q for _, q in model.named_parameters()]
        swapped = any(q is not p for q, p in zip(fresh, params))
        if swapped and any(_lib.is_vmapped(q) for q in fresh):
            raise NotImplementedError(_BATCHED_PARAMS)
        if swapped and torch.is_grad_enabled() and any(q is not p and q.requires_grad for q, p in zip(fresh, params)):
            raise NotImplementedError("pdivgnn_b200: reverse-mode derivatives with respect to parameters swapped in by "
                                      "torch.func.functional_call are not implemented (torch.func.jacrev, vjp or grad "
                                      "of the parameters); those with respect to mean_stress, pos and edge_attr are")
    # the CUDA-graph replay reads raw pointers: not under a torch.func transform (a vmapped input has no storage of its
    # own; its forward runs as pdg_forward_batched instances)
    if not (need_grad or need_tan) and (getattr(model, "cuda_graphs", False) or _GRAPHS_ENV) and not transformed \
            and not torch.cuda.is_current_stream_capturing():
        return _forward_graphed(model, plan, mean_stress, pos, types, edge_attr, flags, model.message_passing_steps, prec,
                                params)
    return _EPDFunction.apply(model, plan, mean_stress, pos, types, edge_attr, flags, model.message_passing_steps, prec,
                              need_grad, need_tan, swapped, *params)[0]
