"""Cost of the forward-mode derivative (pdg_jvp) on the configs[1] batch (32 synthetic meshes x ~1024 nodes), fp32
mode, frozen model: a plain inference forward, a forward that keeps its state (PDG_FLAG_SAVE, what a JVP needs) and a
forward plus one JVP along all three inputs (torch.func.jvp), alternated in rounds within one process so that clock and
neighbour noise hit all three alike.  Also prints the per-kernel-class times of one JVP (pdg_timing_*).

    python tests/tools/time_jvp.py [rounds=10] [calls per round=20]

Prints the GPU name and power limit, the per-round medians and one JSON line."""
import json
import os
import statistics
import subprocess
import sys
from types import SimpleNamespace

R = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, R)
sys.path.insert(0, os.path.join(R, "tests"))
import torch  # noqa: E402

import pdg_helpers as H  # noqa: E402
from oracle import pdg_oracle as O  # noqa: E402
from pdivgnn_b200 import _lib  # noqa: E402

ROUNDS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
CALLS = int(sys.argv[2]) if len(sys.argv) > 2 else 20
KEYS = ("mean_stress", "pos", "edge_attr")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"{torch.cuda.get_device_name()} (nvidia-smi unavailable: {e})"
    return q


def main():
    if not torch.cuda.is_available():
        raise SystemExit("time_jvp.py needs a GPU")
    info = gpu_info()
    print("GPU:", info)
    samples, graphs, batch, stats = H.synthetic_batch(32, 1024)
    db = H.DeviceBatch(batch)
    n, e = batch.num_nodes, batch.edge_index.shape[1]
    print(f"N {n} E {e}")
    model = H.make_model(stats, params=O.init_state_dict(seed=69))
    model.precision = "fp32"
    model.requires_grad_(False)
    g = torch.Generator().manual_seed(1)
    tan = tuple(torch.randn(getattr(batch, k).shape, generator=g).cuda() for k in KEYS)
    x0 = tuple(getattr(db, k) for k in KEYS)
    keep = x0[0].detach().clone().requires_grad_(True)  # a leaf that requires grad: the forward keeps its state

    def f(*xs):
        b = SimpleNamespace(**vars(db))
        for k, x in zip(KEYS, xs):
            setattr(b, k, x)
        return model(b, scale_output=True).local_stress

    def plain():
        with torch.no_grad():
            f(*x0)

    def save():
        f(keep, *x0[1:])

    def jvp():
        torch.func.jvp(f, x0, tan)

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def timed(fn):
        ev[0].record()
        for _ in range(CALLS):
            fn()
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]) / CALLS

    arms = {"forward": plain, "forward_save": save, "forward_jvp": jvp}
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    res = {k: [] for k in arms}
    names = list(arms)
    for r in range(ROUNDS):
        order = names[r % 3:] + names[:r % 3]
        for k in order:
            res[k].append(timed(arms[k]))
    med = {k: statistics.median(v) for k, v in res.items()}
    for k, v in res.items():
        print(f"{k}: {med[k]:.3f} ms (min {min(v):.3f}, max {max(v):.3f})")
    print(f"JVP pass alone (forward_jvp - forward_save): {med['forward_jvp'] - med['forward_save']:.3f} ms; "
          f"forward_jvp / forward = {med['forward_jvp'] / med['forward']:.2f}")
    L = _lib.lib()
    L.pdg_timing_enable(1)
    for _ in range(CALLS):
        jvp()
    torch.cuda.synchronize()
    cls = _lib.timing_collect()
    L.pdg_timing_enable(0)
    print("per call, by kernel class:")
    for k, (ms, cnt) in cls.items():
        print(f"  {k:18s} {ms / CALLS:8.3f} ms  ({cnt // CALLS} launches)")
    print(json.dumps({"gpu": info, "precision": "fp32", "nodes": n, "edges": e, "rounds": ROUNDS, "calls_per_round": CALLS,
                      "ms_median": med, "ms_rounds": res,
                      "ms_per_class": {k: ms / CALLS for k, (ms, _) in cls.items()}}))


if __name__ == "__main__":
    main()
