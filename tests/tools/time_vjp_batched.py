"""Cost of K cotangents in one batched adjoint pass (pdg_vjp_batched) against K backward passes (pdg_backward_inputs),
fp32 mode, on the configs[1] batch (32 synthetic meshes x ~1024 nodes, bench.py's seeds) and on one 1 024-node mesh, for
K in {1, 3, 8, 32}.

Both arms read one forward workspace (pdg_forward with PDG_FLAG_SAVE, run once): either K pdg_backward_inputs calls
("loop", each a full training backward with its weight-gradient GEMMs) or one pdg_vjp_batched call ("batched") on the
same K cotangents, all three input gradients.  The arms are alternated
in rounds within one process so that clock and neighbour noise hit both alike.  Also prints the per-kernel-class times
of each arm (pdg_timing_*) and checks that both arms give the same bits.

    python tests/tools/time_vjp_batched.py [rounds=10] [calls per round=10]

Prints the GPU name and power limit, the per-round medians and one JSON line."""
import ctypes as C
import json
import os
import statistics
import sys
from types import SimpleNamespace

R = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, R)
sys.path.insert(0, os.path.join(R, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch  # noqa: E402

import pdg_helpers as H  # noqa: E402
from oracle import pdg_oracle as O  # noqa: E402
from pdivgnn_b200 import _lib, autograd as A, synth  # noqa: E402
from time_jvp import gpu_info  # noqa: E402

ROUNDS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
CALLS = int(sys.argv[2]) if len(sys.argv) > 2 else 10
KS = (1, 3, 8, 32)


def setup(batch, stats):
    L = _lib.lib()
    model = H.make_model(stats, params=O.init_state_dict(seed=69))
    db = H.DeviceBatch(batch)
    n = batch.num_nodes
    plan = A.build_plan(db.edge_index, n)
    e, steps = plan.n_edges, model.message_passing_steps
    types = db.nodes_types.reshape(-1).contiguous()
    ea = db.edge_attr.reshape(-1).contiguous()
    params = [p.detach() for p in A.param_list(model)]
    ps, norm = A._params_struct(params), model._norm_struct()
    flags = _lib.FLAG_SCALE_INPUT | _lib.FLAG_SCALE_OUTPUT | _lib.FLAG_ZERO_CHECK | _lib.FLAG_SAVE
    p = _lib.ptr
    ins = (p(db.mean_stress), p(db.pos), p(types), p(ea), p(plan.buf), n, e, steps, flags, _lib.PREC_FP32)
    ws_bytes = L.pdg_forward_ws_bytes(n, e, steps, flags)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    out = torch.empty(n, 3, device="cuda")
    bb = L.pdg_backward_ws_bytes(n, e, steps)
    bws = torch.empty(bb, dtype=torch.uint8, device="cuda")
    flat = torch.empty(_lib.PDG_PARAM_ELEMS, device="cuda")
    vb = L.pdg_vjp_batched_ws_bytes(n, e, steps, max(KS))
    vws = torch.empty(vb, dtype=torch.uint8, device="cuda")
    g = torch.Generator().manual_seed(1)
    cot = torch.randn((max(KS), n, 3), generator=g).cuda()
    outs = [torch.empty((max(KS),) + sh, device="cuda") for sh in ((n, 3), (n, 2), (e,))]
    st = _lib.stream_ptr()
    _lib.check(L.pdg_forward(C.byref(ps), C.byref(norm), *ins, p(ws), ws_bytes, p(out), st), "pdg_forward")

    def loop(k):
        for i in range(k):
            _lib.check(L.pdg_backward_inputs(C.byref(ps), C.byref(norm), *ins, p(ws), p(bws), bb, p(cot[i]), p(flat),
                                             p(outs[0][i]), p(outs[1][i]), p(outs[2][i]), st), "pdg_backward_inputs")

    def batched(k):
        _lib.check(L.pdg_vjp_batched(C.byref(ps), C.byref(norm), *ins, p(ws), p(vws), vb, k, p(cot), p(outs[0]),
                                     p(outs[1]), p(outs[2]), st), "pdg_vjp_batched")
    return SimpleNamespace(n=n, e=e, loop=loop, batched=batched, outs=outs, keep=(model, db, plan, types, ea, params))


def timed(fn, k):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(CALLS):
        fn(k)
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / CALLS


def by_class(fn, k):
    L = _lib.lib()
    _lib.timing_collect()
    L.pdg_timing_enable(1)
    for _ in range(CALLS):
        fn(k)
    torch.cuda.synchronize()
    cls = _lib.timing_collect()
    L.pdg_timing_enable(0)
    return {c: ms / CALLS for c, (ms, _) in cls.items()}


def main():
    if not torch.cuda.is_available():
        raise SystemExit("time_vjp_batched.py needs a GPU")
    info = gpu_info()
    print("GPU:", info, "| SMs:", _lib.lib().pdg_num_sms())
    _, _, b32, s32 = H.synthetic_batch(32, 1024)
    _, b1, s1 = H.oracle_batch_from_samples([synth.make_rve_mesh(69, 1024)], True)
    result = {"gpu": info, "precision": "fp32", "rounds": ROUNDS, "calls_per_round": CALLS, "shapes": {}}
    for name, (batch, stats) in (("configs1_32x1024", (b32, s32)), ("mesh_1024", (b1, s1))):
        a = setup(batch, stats)
        print(f"== {name}: N {a.n} E {a.e}")
        res = {}
        for k in KS:
            a.loop(k)
            ref = [o[:k].clone() for o in a.outs]
            a.batched(k)
            same = all(torch.equal(r, o[:k]) for r, o in zip(ref, a.outs))
            for _ in range(3):
                a.loop(k)
                a.batched(k)
            torch.cuda.synchronize()
            t = {"loop": [], "batched": []}
            for r in range(ROUNDS):
                order = ("loop", "batched") if r % 2 == 0 else ("batched", "loop")
                for arm in order:
                    t[arm].append(timed(getattr(a, arm), k))
            med = {arm: statistics.median(v) for arm, v in t.items()}
            cls = {arm: by_class(getattr(a, arm), k) for arm in t}
            print(f"K={k}: {k} x pdg_backward_inputs {med['loop']:.3f} ms (min {min(t['loop']):.3f}, max "
                  f"{max(t['loop']):.3f}); pdg_vjp_batched {med['batched']:.3f} ms (min "
                  f"{min(t['batched']):.3f}, max {max(t['batched']):.3f}); ratio {med['batched'] / med['loop']:.3f}; "
                  f"bit-identical {same}")
            for arm in ("loop", "batched"):
                print(f"    {arm}: " + ", ".join(f"{c} {v:.3f}" for c, v in sorted(cls[arm].items(), key=lambda x: -x[1])))
            res[k] = {"ms_median": med, "ms_rounds": t, "ms_per_class": cls, "bit_identical": same}
        result["shapes"][name] = {"nodes": a.n, "edges": a.e, "K": res}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
