"""Cost of K instances of one graph in one batched forward pass (pdg_forward_batched) against K pdg_forward calls, fp32
mode, inference flags (no saved state): one 1 024-node mesh under K = 1, 8, 32 and 64 loads, and the configs[1] batch
(32 synthetic meshes x ~1024 nodes, bench.py's seeds) as one instance under K = 1 and 3 loads.

Both arms compute the same K instances (instance k: the graph's own positions and edge weights, its load scaled and
turned): either K pdg_forward calls ("loop") or one pdg_forward_batched call ("batched").  The arms are alternated in
rounds within one process so that clock and neighbour noise hit both alike.  Also checks that both arms give the same
bits.

    python tests/tools/time_fwd_batched.py [rounds=10] [calls per round=10]

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


def setup(batch, stats, kmax):
    L = _lib.lib()
    model = H.make_model(stats, params=O.init_state_dict(seed=69))
    db = H.DeviceBatch(batch)
    n = batch.num_nodes
    plan = A.build_plan(db.edge_index, n)
    e, steps = plan.n_edges, model.message_passing_steps
    types = db.nodes_types.reshape(-1).contiguous()
    ea = db.edge_attr.reshape(-1).contiguous()
    pos = db.pos.contiguous()
    params = [p.detach() for p in A.param_list(model)]
    ps, norm = A._params_struct(params), model._norm_struct()
    flags = _lib.FLAG_SCALE_INPUT | _lib.FLAG_SCALE_OUTPUT | _lib.FLAG_ZERO_CHECK
    g = torch.Generator().manual_seed(1)
    ms = (db.mean_stress.cpu().unsqueeze(0) * (0.5 + torch.rand(kmax, 1, 3, generator=g))).cuda().contiguous()
    p = _lib.ptr
    ws_bytes = L.pdg_forward_ws_bytes(n, e, steps, flags)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    bb = L.pdg_forward_batched_ws_bytes(n, e, steps, flags, kmax)
    bws = torch.empty(bb, dtype=torch.uint8, device="cuda")
    outs = {"loop": torch.empty((kmax, n, 3), device="cuda"), "batched": torch.empty((kmax, n, 3), device="cuda")}
    st = _lib.stream_ptr()

    def loop(k):
        for i in range(k):
            _lib.check(L.pdg_forward(C.byref(ps), C.byref(norm), p(ms[i]), p(pos), p(types), p(ea), p(plan.buf), n, e,
                                     steps, flags, _lib.PREC_FP32, p(ws), ws_bytes, p(outs["loop"][i]), st), "pdg_forward")

    def batched(k):
        _lib.check(L.pdg_forward_batched(C.byref(ps), C.byref(norm), p(ms), n * 3, p(pos), 0, p(types), p(ea), 0,
                                         p(plan.buf), n, e, steps, flags, _lib.PREC_FP32, p(bws), bb, k,
                                         p(outs["batched"]), st), "pdg_forward_batched")
    return SimpleNamespace(n=n, e=e, loop=loop, batched=batched, outs=outs, keep=(model, db, plan, types, ea, pos, ms,
                                                                                  params))


def timed(fn, k):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(CALLS):
        fn(k)
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / CALLS


def main():
    if not torch.cuda.is_available():
        raise SystemExit("time_fwd_batched.py needs a GPU")
    info = gpu_info()
    print("GPU:", info, "| SMs:", _lib.lib().pdg_num_sms())
    _, b1, s1 = H.oracle_batch_from_samples([synth.make_rve_mesh(69, 1024)], True)
    _, _, b32, s32 = H.synthetic_batch(32, 1024)
    result = {"gpu": info, "precision": "fp32", "rounds": ROUNDS, "calls_per_round": CALLS, "shapes": {}}
    for name, (batch, stats), ks in (("mesh_1024", (b1, s1), (1, 8, 32, 64)),
                                     ("configs1_32x1024", (b32, s32), (1, 3))):
        a = setup(batch, stats, max(ks))
        print(f"== {name}: N {a.n} E {a.e}")
        res = {}
        for k in ks:
            a.loop(k)
            a.batched(k)
            torch.cuda.synchronize()
            same = torch.equal(a.outs["loop"][:k], a.outs["batched"][:k])
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
            print(f"K={k}: {k} x pdg_forward {med['loop']:.3f} ms (min {min(t['loop']):.3f}, max {max(t['loop']):.3f}); "
                  f"pdg_forward_batched {med['batched']:.3f} ms (min {min(t['batched']):.3f}, max "
                  f"{max(t['batched']):.3f}); ratio {med['batched'] / med['loop']:.3f}; bit-identical {same}")
            res[k] = {"ms_median": med, "ms_rounds": t, "bit_identical": same}
        result["shapes"][name] = {"nodes": a.n, "edges": a.e, "K": res}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
