"""Cost of K tangents in one batched tangent pass (pdg_jvp_batched) against K single-tangent passes (pdg_jvp), fp32
mode, on the configs[1] batch (32 synthetic meshes x ~1024 nodes) and on one 1 024-node mesh, for K in {1, 3, 8}.

Each arm is one forward that keeps its state (pdg_forward with PDG_FLAG_SAVE) followed by either K pdg_jvp calls
("loop") or one pdg_jvp_batched call ("batched") on the same K tangents of all three inputs.  The arms are alternated
in rounds within one process so that clock and neighbour noise hit both alike.  Also prints the per-kernel-class times
of each arm (pdg_timing_*) and checks that both arms give the same bits.

    python tests/tools/time_jvp_batched.py [rounds=10] [calls per round=10]

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
KS = (1, 3, 8)


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
    jb = L.pdg_jvp_ws_bytes(n, e, steps)
    jws = torch.empty(max(KS) * jb, dtype=torch.uint8, device="cuda")
    g = torch.Generator().manual_seed(1)
    tan = [torch.randn((max(KS),) + sh, generator=g).cuda() for sh in ((n, 3), (n, 2), (e,))]
    touts = torch.empty(max(KS), n, 3, device="cuda")
    st = _lib.stream_ptr()

    def forward():
        _lib.check(L.pdg_forward(C.byref(ps), C.byref(norm), *ins, p(ws), ws_bytes, p(out), st), "pdg_forward")

    def loop(k):
        forward()
        for i in range(k):
            _lib.check(L.pdg_jvp(C.byref(ps), C.byref(norm), *ins, p(ws), p(jws), jb, p(tan[0][i]), p(tan[1][i]),
                                 p(tan[2][i]), p(touts[i]), st), "pdg_jvp")

    def batched(k):
        forward()
        _lib.check(L.pdg_jvp_batched(C.byref(ps), C.byref(norm), *ins, p(ws), p(jws), k * jb, k, p(tan[0]), n * 3,
                                     p(tan[1]), n * 2, p(tan[2]), e, p(touts), st), "pdg_jvp_batched")
    return SimpleNamespace(n=n, e=e, loop=loop, batched=batched, touts=touts, keep=(model, db, plan, types, ea, params))


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
        raise SystemExit("time_jvp_batched.py needs a GPU")
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
            ref = a.touts[:k].clone()
            a.batched(k)
            same = torch.equal(ref, a.touts[:k])
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
            print(f"K={k}: forward_save + {k} x pdg_jvp {med['loop']:.3f} ms (min {min(t['loop']):.3f}, max "
                  f"{max(t['loop']):.3f}); forward_save + pdg_jvp_batched {med['batched']:.3f} ms (min "
                  f"{min(t['batched']):.3f}, max {max(t['batched']):.3f}); ratio {med['batched'] / med['loop']:.3f}; "
                  f"bit-identical {same}")
            for c in cls["loop"]:
                if c.startswith("jvp_"):
                    print(f"    {c:18s} loop {cls['loop'][c]:8.3f} ms   batched {cls['batched'].get(c, 0.0):8.3f} ms")
            res[k] = {"ms_median": med, "ms_rounds": t, "ms_per_class": cls, "bit_identical": same}
        result["shapes"][name] = {"nodes": a.n, "edges": a.e, "K": res}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
