"""bench.py --dump-outputs on the GPU: the files hold the state after the last timed training step (checked against an
in-process replay of the same seeded training), and the same arguments give the same files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--batch", "2", "--nodes", "256", "--steps", str(steps),
                        "--warmup", "1", "--lean", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "stdout must hold exactly one JSON line"
    line = json.loads(lines[0])
    assert line["steps"] == steps
    return line, {n[:-4]: np.load(os.path.join(out, n)) for n in sorted(os.listdir(out))}


def _replay(n_steps, batch, nodes):
    """bench.py's resident training path rebuilt here: the same seeded batch, model and optimizer, n_steps train steps."""
    import torch
    import pdivgnn_b200
    from pdivgnn_b200 import batcher, synth
    from pdivgnn_b200.optim import FusedAdam
    dev = torch.device("cuda", 0)
    b = batcher.batch_from_host(batcher.host_arrays(synth.make_dataset(batch, nodes, 69), False), dev, True, False)
    torch.manual_seed(69)
    model = pdivgnn_b200.EncodeProcessDecode(1, 10, 128, 6, 3, precision="bf16", **batcher.dataset_stats([b])).to(dev)
    opt = FusedAdam(model.parameters(), lr=1e-3)
    for _ in range(n_steps):
        pred = model(b, scale_output=False, scale_input=True).local_stress
        nmse, div = pdivgnn_b200.nmse_div_loss(pred, b, model, False, 10.0)
        loss = nmse + div
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
    out = {"loss": loss, "nmse": nmse, "div": div, "local_stress": pred}
    for k, p in model.named_parameters():
        out["param." + k], out["grad." + k] = p, p.grad
    return {k: v.detach().cpu().numpy() for k, v in out.items()}


def test_dump_outputs_of_the_timed_step(tmp_path):
    from oracle import pdg_oracle as O
    line, a = _bench(tmp_path / "a", 2)
    _, b = _bench(tmp_path / "b", 2)
    keys = ["loss", "nmse", "div", "local_stress"] + [p + k for p in ("param.", "grad.") for k in O.STATE_KEYS]
    assert sorted(a) == sorted(keys)
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 * 10**6
    assert a["local_stress"].shape == (line["config"]["nodes_per_gpu"], 3)
    assert line["warmup"] == 3 and line["steps"] == 2
    want = _replay(line["warmup"] + line["steps"], 2, 256)  # warm-up and timed steps, nothing after them
    for k in keys:
        assert np.array_equal(a[k], want[k]), k
        assert np.array_equal(a[k], b[k]), k  # same arguments, same outputs
