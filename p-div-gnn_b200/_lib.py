"""ctypes binding of the C-ABI library ``lib/libpdivgnn.so`` (include/pdg.h).

There is no fallback: if the library is missing or a call fails, the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libpdivgnn.so")

PDG_NUM_PARAMS = 28
PDG_PARAM_ELEMS = 167299
FLAG_SCALE_INPUT, FLAG_SCALE_OUTPUT, FLAG_SAVE, FLAG_ZERO_CHECK = 1, 2, 4, 8
PREC_FP32, PREC_BF16 = 0, 1
JVP_MAX_TANGENTS = 64  # PDG_JVP_MAX_TANGENTS: tangents of one pdg_jvp_batched call
VJP_MAX_COTANGENTS = 64  # PDG_VJP_MAX_COTANGENTS: cotangents of one pdg_vjp_batched call
FWD_MAX_INSTANCES = 64  # PDG_FWD_MAX_INSTANCES: instances of one pdg_forward_batched call


class PdgParams(C.Structure):
    _fields_ = [("p", C.c_void_p * PDG_NUM_PARAMS)]


class PdgNorm(C.Structure):
    _fields_ = [(k, C.c_float) for k in (
        "mean_pos", "std_pos", "mean_mean_stress", "std_mean_stress",
        "mean_local_stress", "std_local_stress", "mean_edge_weight", "std_edge_weight")]


class PdgAdam(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("lr", "beta1", "beta2", "eps", "weight_decay", "inv_scale")] + [("step", C.c_int)]


_lib = None

_vp, _i64, _i32, _sz, _f = C.c_void_p, C.c_int64, C.c_int, C.c_size_t, C.c_float
_SIGS = {
    "pdg_last_error": (C.c_char_p, []),
    "pdg_version": (_i32, []),
    "pdg_persistent_grid": (_i32, [_i32, _i32]),
    "pdg_num_sms": (_i32, []),
    "pdg_launch_count": (C.c_longlong, [_i32]),
    "pdg_timing_enable": (_i32, [_i32]),
    "pdg_timing_classes": (_i32, []),
    "pdg_timing_class_name": (C.c_char_p, [_i32]),
    "pdg_timing_collect": (_i32, [C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "pdg_tc_selftest": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp]),
    "pdg_plan_bytes": (_sz, [_i64, _i64]),
    "pdg_plan_tmp_bytes": (_sz, [_i64, _i64]),
    "pdg_plan_build": (_i32, [_vp, _i64, _i64, _vp, _vp, _sz, _vp]),
    "pdg_plan_views": (_i32, [_vp, _i64, _i64] + [C.POINTER(_vp)] * 6),
    "pdg_plan_status": (_i32, [_vp, _i64, _i64, C.POINTER(C.c_int32), _vp]),
    "pdg_forward_ws_bytes": (_sz, [_i64, _i64, _i32, _i32]),
    "pdg_forward": (_i32, [C.POINTER(PdgParams), C.POINTER(PdgNorm), _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _i32,
                           _i32, _vp, _sz, _vp, _vp]),
    "pdg_forward_batched_ws_bytes": (_sz, [_i64, _i64, _i32, _i32, _i32]),
    "pdg_forward_batched": (_i32, [C.POINTER(PdgParams), C.POINTER(PdgNorm), _vp, _i64, _vp, _i64, _vp, _vp, _i64, _vp,
                                   _i64, _i64, _i32, _i32, _i32, _vp, _sz, _i32, _vp, _vp]),
    "pdg_forward_batched_saved_ws_bytes": (_sz, [_i64, _i64, _i32, _i32, _i32]),
    "pdg_forward_batched_saved": (_i32, [C.POINTER(PdgParams), C.POINTER(PdgNorm), _vp, _i64, _vp, _i64, _vp, _vp, _i64,
                                         _vp, _i64, _i64, _i32, _i32, _i32, _vp, _sz, _i32, _vp, _vp]),
    "pdg_ws_offset": (_i32, [_i64, _i64, _i32, _i32, _i32, _i32, C.POINTER(_sz), C.POINTER(_sz)]),
    "pdg_backward_ws_bytes": (_sz, [_i64, _i64, _i32]),
    "pdg_backward": (_i32, [C.POINTER(PdgParams), C.POINTER(PdgNorm), _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _i32,
                            _i32, _vp, _vp, _sz, _vp, _vp, _vp]),
    "pdg_backward_inputs": (_i32, [C.POINTER(PdgParams), C.POINTER(PdgNorm), _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32,
                                   _i32, _i32, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pdg_jvp_ws_bytes": (_sz, [_i64, _i64, _i32]),
    "pdg_jvp": (_i32, [C.POINTER(PdgParams), C.POINTER(PdgNorm), _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _i32, _i32,
                       _vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp]),
    "pdg_jvp_batched_ws_bytes": (_sz, [_i64, _i64, _i32, _i32]),
    "pdg_jvp_batched": (_i32, [C.POINTER(PdgParams), C.POINTER(PdgNorm), _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _i32,
                               _i32, _vp, _vp, _sz, _i32, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp]),
    "pdg_vjp_batched_ws_bytes": (_sz, [_i64, _i64, _i32, _i32]),
    "pdg_vjp_batched": (_i32, [C.POINTER(PdgParams), C.POINTER(PdgNorm), _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _i32,
                               _i32, _vp, _vp, _sz, _i32, _vp, _vp, _vp, _vp, _vp]),
    "pdg_vjp_instances": (_i32, [C.POINTER(PdgParams), C.POINTER(PdgNorm), _vp, _i64, _vp, _i64, _vp, _vp, _i64, _vp,
                                 _i64, _i64, _i32, _i32, _i32, _vp, _i32, _vp, _sz, _i32, _vp, _vp, _vp, _vp, _vp]),
    "pdg_opdiv_plan_bytes": (_sz, [_i64, _i64]),
    "pdg_opdiv_tmp_bytes": (_sz, [_i64, _i64]),
    "pdg_opdiv_plan_build": (_i32, [_vp, _vp, _i64, _vp, _i64, _i64, _vp, _vp, _sz, _vp]),
    "pdg_loss_ws_bytes": (_sz, [_i64, _i64]),
    "pdg_loss": (_i32, [_vp, _vp, C.POINTER(PdgNorm), _vp, _i64, _i64, _vp, _vp, _vp, _i64, _i32, _f, _vp, _vp, _vp]),
    "pdg_loss_backward": (_i32, [_vp, _vp, C.POINTER(PdgNorm), _vp, _i64, _i64, _vp, _vp, _i64, _i32, _f, _vp, _vp,
                                 _vp, _vp]),
    "pdg_grads_check_finite": (_i32, [C.POINTER(C.c_void_p * PDG_NUM_PARAMS), _vp, _vp]),
    "pdg_adam_step": (_i32, [C.POINTER(C.c_void_p * PDG_NUM_PARAMS), C.POINTER(C.c_void_p * PDG_NUM_PARAMS), _vp, _vp,
                             C.POINTER(PdgAdam), _vp, _vp]),
    "pdg_adam_step_counted": (_i32, [C.POINTER(C.c_void_p * PDG_NUM_PARAMS), C.POINTER(C.c_void_p * PDG_NUM_PARAMS), _vp,
                                     _vp, C.POINTER(PdgAdam), _vp, _vp, _vp]),
    "pdg_batch_tmp_bytes": (_sz, [_i64, _i64, _i32, _i64]),
    "pdg_batch_count": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i32, _i32, _vp, _sz, C.POINTER(_i64), _vp]),
    "pdg_labels_tmp_bytes": (_sz, [_i64, _i64, _i32, _i64]),
    "pdg_node_labels": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i32, _vp, _sz, _vp, _vp, _vp]),
    "pdg_batch_fill": (_i32, [_vp, _i64, _i64, _i32, _i64, _i64, _vp, _vp, _vp, _vp]),
    "pdg_periodic_tmp_bytes": (_sz, [_i64, _i64]),
    "pdg_is_periodic": (_i32, [_vp, _vp, _i64, _i64, C.c_double, _vp, _sz, _vp, _vp]),
    "pdg_resident_gather": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _i32, _i64, _i64, _i64,
                                   _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pdg_peer_bytes": (_sz, [_i64, _i32]),
    "pdg_peer_alloc": (_i32, [_i64, _i32, C.POINTER(C.c_void_p), _vp]),
    "pdg_peer_open": (_i32, [_vp, C.POINTER(C.c_void_p)]),
    "pdg_peer_close": (_i32, [_vp]),
    "pdg_peer_free": (_i32, [_vp]),
    "pdg_allreduce_mean": (_i32, [_vp, _i64, C.POINTER(C.c_void_p), _i32, _i32, _i64, _vp, _vp]),
}
_OPTIONAL = set()


def lib():
    """Load (once) and return the CDLL; raises if the library was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `make -C p-div-gnn_b200/csrc` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            try:
                fn = getattr(l, name)
            except AttributeError:
                if name in _OPTIONAL:
                    continue
                raise
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def timing_collect():
    """{kernel class: (total ms, launches)} since the last collect (see pdg_timing_enable)."""
    l = lib()
    n = l.pdg_timing_classes()
    ms, cnt = (C.c_double * n)(), (C.c_longlong * n)()
    check(l.pdg_timing_collect(ms, cnt), "pdg_timing_collect")
    return {l.pdg_timing_class_name(i).decode(): (ms[i], cnt[i]) for i in range(n) if cnt[i]}


def declared_symbols():
    return list(_SIGS.keys())


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f"{what} failed (rc={rc}): {lib().pdg_last_error().decode()}")


def _refuse_legacy_batched(t):
    if torch._C._functorch.is_legacy_batchedtensor(t):
        raise NotImplementedError("pdivgnn_b200: torch.autograd.grad(..., is_grads_batched=True) is not supported (its "
                                  "legacy vmap passes tensors without storage); use torch.func.jacrev or "
                                  "torch.func.vmap over torch.func.vjp, which run all cotangents in one adjoint pass")


def raw(t):
    """The plain tensor under functorch wrappers: inside torch.func transforms (torch.func.jvp), tensors created by the
    transformed function are wrappers without storage of their own; the library reads and writes the wrapped one.
    A vmap BatchedTensor is refused: its storage holds the whole batch while the library would read one tensor.  So is a
    tensor of the legacy vmap behind torch.autograd.grad(..., is_grads_batched=True), which has no storage at all."""
    _refuse_legacy_batched(t)
    while torch._C._functorch.is_functorch_wrapped_tensor(t):
        if torch._C._functorch.is_batchedtensor(t):
            raise RuntimeError("pdivgnn_b200: a vmap BatchedTensor reached the library; its storage holds the whole "
                               "batch, so it cannot be passed as one tensor")
        t = torch._C._functorch.get_unwrapped(t)
        _refuse_legacy_batched(t)
    return t


def is_vmapped(t):
    """True when t carries a torch.func.vmap level (a BatchedTensor under any functorch wrappers)."""
    while torch._C._functorch.is_functorch_wrapped_tensor(t):
        if torch._C._functorch.is_batchedtensor(t):
            return True
        t = torch._C._functorch.get_unwrapped(t)
    return False


def ptr(t):
    return None if t is None else C.c_void_p(raw(t).data_ptr())


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t: torch.Tensor, name: str, dtype=None):
    if not t.is_cuda:
        raise RuntimeError(f"pdivgnn_b200: `{name}` must be a CUDA tensor (got {t.device}); there is no CPU path")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"pdivgnn_b200: `{name}` must be {dtype} (got {t.dtype})")
    return t.contiguous()
