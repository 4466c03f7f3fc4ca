"""Cost of per-load input gradients through the batched forward, fp32 mode: K loads (mean_stress of K instances; pos and
edge_attr shared) on one 1 089-node mesh for K in {1, 8, 32, 64}, and on the configs[1] batch (32 synthetic meshes x
~1024 nodes, bench.py's seeds) for K = 3.  One cotangent per instance.  Three arms on the same inputs and cotangents:

  batched   one pdg_forward_batched_saved of K instances + one pdg_vjp_instances (I = K, M = 1): what torch.func.grad of
            a function that vmaps the model costs;
  loop      K x (pdg_forward with PDG_FLAG_SAVE + pdg_backward_inputs): a loop of model(...) + torch.autograd.grad calls;
  loop_vjp  K x (pdg_forward with PDG_FLAG_SAVE + pdg_vjp_batched with K = 1): separates the gain of batching from the
            gain of dropping the weight-gradient GEMMs.

The arms alternate in rounds within one process so that clock and neighbour noise hit them alike; all three must give
the same bits.

    python tests/tools/time_vjp_instances.py [rounds=10] [calls=5] [out.txt=profiles/r10_vjp_instances_timing.txt]

Prints (and writes to out.txt) the GPU name and power limit, the per-round medians and one JSON line."""
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
CALLS = int(sys.argv[2]) if len(sys.argv) > 2 else 5
OUT = sys.argv[3] if len(sys.argv) > 3 else os.path.join(R, "profiles", "r10_vjp_instances_timing.txt")
LINES = []


def say(*a):
    s = " ".join(str(x) for x in a)
    print(s, flush=True)
    LINES.append(s)


def setup(batch, stats, k):
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
    g = torch.Generator().manual_seed(1)
    ms = (db.mean_stress.cpu().unsqueeze(0) * (0.5 + torch.rand(k, 1, 3, generator=g))).cuda().contiguous()
    cot = torch.randn((k, n, 3), generator=g).cuda()
    p, st = _lib.ptr, _lib.stream_ptr()
    one = L.pdg_forward_batched_saved_ws_bytes(n, e, steps, flags, 1)
    bws_ = torch.empty(k * one, dtype=torch.uint8, device="cuda")
    out = torch.empty((k, n, 3), device="cuda")
    vb = L.pdg_vjp_batched_ws_bytes(n, e, steps, k)
    vws = torch.empty(vb, dtype=torch.uint8, device="cuda")
    fb = L.pdg_forward_ws_bytes(n, e, steps, flags)
    fws = torch.empty(fb, dtype=torch.uint8, device="cuda")
    bb = L.pdg_backward_ws_bytes(n, e, steps)
    bws = torch.empty(bb, dtype=torch.uint8, device="cuda")
    vb1 = L.pdg_vjp_batched_ws_bytes(n, e, steps, 1)
    flat = torch.empty(_lib.PDG_PARAM_ELEMS, device="cuda")
    outs = {arm: [torch.empty((k,) + sh, device="cuda") for sh in ((n, 3), (n, 2), (e,))]
            for arm in ("batched", "loop", "loop_vjp")}

    def batched():
        o = outs["batched"]
        _lib.check(L.pdg_forward_batched_saved(C.byref(ps), C.byref(norm), p(ms), n * 3, p(db.pos), 0, p(types), p(ea), 0,
                                               p(plan.buf), n, e, steps, flags, _lib.PREC_FP32, p(bws_), k * one, k, p(out),
                                               st), "pdg_forward_batched_saved")
        _lib.check(L.pdg_vjp_instances(C.byref(ps), C.byref(norm), p(ms), n * 3, p(db.pos), 0, p(types), p(ea), 0,
                                       p(plan.buf), n, e, steps, flags, _lib.PREC_FP32, p(bws_), k, p(vws), vb, 1, p(cot),
                                       p(o[0]), p(o[1]), p(o[2]), st), "pdg_vjp_instances")

    def single_forward(i):
        ins = (p(ms[i]), p(db.pos), p(types), p(ea), p(plan.buf), n, e, steps, flags, _lib.PREC_FP32)
        _lib.check(L.pdg_forward(C.byref(ps), C.byref(norm), *ins, p(fws), fb, p(out[i]), st), "pdg_forward")
        return ins

    def loop():
        o = outs["loop"]
        for i in range(k):
            ins = single_forward(i)
            _lib.check(L.pdg_backward_inputs(C.byref(ps), C.byref(norm), *ins, p(fws), p(bws), bb, p(cot[i]), p(flat),
                                             p(o[0][i]), p(o[1][i]), p(o[2][i]), st), "pdg_backward_inputs")

    def loop_vjp():
        o = outs["loop_vjp"]
        for i in range(k):
            ins = single_forward(i)
            _lib.check(L.pdg_vjp_batched(C.byref(ps), C.byref(norm), *ins, p(fws), p(vws), vb1, 1, p(cot[i]), p(o[0][i]),
                                         p(o[1][i]), p(o[2][i]), st), "pdg_vjp_batched")
    return SimpleNamespace(n=n, e=e, arms={"batched": batched, "loop": loop, "loop_vjp": loop_vjp}, outs=outs,
                           keep=(model, db, plan, types, ea, params, ms, cot))


def timed(fn):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(CALLS):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / CALLS


def main():
    if not torch.cuda.is_available():
        raise SystemExit("time_vjp_instances.py needs a GPU")
    info = gpu_info()
    say("GPU:", info, "| SMs:", _lib.lib().pdg_num_sms())
    _, b1, s1 = H.oracle_batch_from_samples([synth.make_rve_mesh(69, 1024)], True)
    _, _, b32, s32 = H.synthetic_batch(32, 1024)
    result = {"gpu": info, "precision": "fp32", "rounds": ROUNDS, "calls_per_round": CALLS, "runs": []}
    for name, (batch, stats), ks in (("mesh_1089", (b1, s1), (1, 8, 32, 64)), ("configs1_32x1024", (b32, s32), (3,))):
        for k in ks:
            a = setup(batch, stats, k)
            for fn in a.arms.values():
                fn()
            torch.cuda.synchronize()
            same = all(torch.equal(x, y) for arm in ("loop", "loop_vjp")
                       for x, y in zip(a.outs["batched"], a.outs[arm]))
            t = {arm: [] for arm in a.arms}
            for r in range(ROUNDS):
                order = list(a.arms) if r % 2 == 0 else list(a.arms)[::-1]
                for arm in order:
                    t[arm].append(timed(a.arms[arm]))
            med = {arm: statistics.median(v) for arm, v in t.items()}
            say(f"{name} N {a.n} E {a.e} K={k}: batched {med['batched']:.3f} ms (min {min(t['batched']):.3f}, max "
                f"{max(t['batched']):.3f}); loop {med['loop']:.3f} ms (min {min(t['loop']):.3f}); loop_vjp "
                f"{med['loop_vjp']:.3f} ms (min {min(t['loop_vjp']):.3f}); loop / batched "
                f"{med['loop'] / med['batched']:.2f}x, loop_vjp / batched {med['loop_vjp'] / med['batched']:.2f}x; "
                f"bit-identical {same}")
            result["runs"].append({"shape": name, "nodes": a.n, "edges": a.e, "K": k, "ms_median": med, "ms_rounds": t,
                                   "bit_identical": same})
            del a
            torch.cuda.empty_cache()
    say(json.dumps(result))
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as fh:
        fh.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
