"""Cost of the input gradients on the configs[1] training step (32 synthetic meshes x ~1024 nodes, fused loss without
divergence, fused Adam), in both precision modes: the step without input gradients and the step with d/d mean_stress,
pos and edge_attr, alternated in rounds within one process so that clock and neighbour noise hit both alike.

    python tests/tools/time_input_grads.py [rounds=10] [steps per round=20]

Prints the GPU name and power limit, the per-round medians and one JSON line per precision mode."""
import json
import os
import statistics
import subprocess
import sys

R = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, R)
sys.path.insert(0, os.path.join(R, "tests"))
import torch  # noqa: E402

import pdg_helpers as H  # noqa: E402
from oracle import pdg_oracle as O  # noqa: E402
import pdivgnn_b200  # noqa: E402
from pdivgnn_b200.optim import FusedAdam  # noqa: E402

ROUNDS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
STEPS = int(sys.argv[2]) if len(sys.argv) > 2 else 20


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"{torch.cuda.get_device_name()} (nvidia-smi unavailable: {e})"
    return q


def main():
    if not torch.cuda.is_available():
        raise SystemExit("time_input_grads.py needs a GPU")
    info = gpu_info()
    print("GPU:", info)
    samples, graphs, batch, stats = H.synthetic_batch(32, 1024)
    sd = O.init_state_dict(seed=69)
    db = H.DeviceBatch(batch)
    n, e = batch.num_nodes, batch.edge_index.shape[1]
    print(f"N {n} E {e}")
    for prec in ("bf16", "fp32"):
        model = H.make_model(stats, params=sd)
        model.precision = prec
        opt = FusedAdam(model.parameters(), lr=1e-3)
        leaves = {k: getattr(db, k).detach().clone() for k in ("mean_stress", "pos", "edge_attr")}

        def step(inputs):
            for k, t in leaves.items():
                t.grad = None
                t.requires_grad_(inputs)
                setattr(db, k, t)
            pred = model(db, scale_output=False).local_stress
            nmse, dv = pdivgnn_b200.nmse_div_loss(pred, db, model, False, 10.0)
            opt.zero_grad(set_to_none=True)
            (nmse + dv).backward()
            opt.step()

        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

        def timed(inputs):
            ev[0].record()
            for _ in range(STEPS):
                step(inputs)
            ev[1].record()
            torch.cuda.synchronize()
            return ev[0].elapsed_time(ev[1]) / STEPS

        for inputs in (False, True):  # warm up both shapes of the backward
            for _ in range(3):
                step(inputs)
        torch.cuda.synchronize()
        base, ig = [], []
        for r in range(ROUNDS):
            order = (False, True) if r % 2 == 0 else (True, False)
            for inputs in order:
                (ig if inputs else base).append(timed(inputs))
        mb, mi = statistics.median(base), statistics.median(ig)
        print(f"{prec}: step without input grads {mb:.3f} ms (min {min(base):.3f}, max {max(base):.3f}); "
              f"with all three {mi:.3f} ms (min {min(ig):.3f}, max {max(ig):.3f}); delta {mi - mb:+.3f} ms "
              f"({(mi / mb - 1) * 100:+.2f} %)")
        print(json.dumps({"precision": prec, "gpu": info, "nodes": n, "edges": e, "rounds": ROUNDS,
                          "steps_per_round": STEPS, "ms_per_step_no_input_grads": mb, "ms_per_step_input_grads": mi,
                          "rounds_no_input_grads": base, "rounds_input_grads": ig}))


if __name__ == "__main__":
    main()
