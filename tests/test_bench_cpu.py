"""The reference arm of bench.py (`--impl reference`: the oracle port timed on the host cores) needs no GPU: run it on a
tiny workload and check the one-line JSON contract the driver parses."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--batch", "2", "--nodes", "128",
                        "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "stdout must hold exactly one JSON line"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "nodes/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("mesh nodes/sec") and d["n_gpus"] == 1 and d["steps"] == 1 and d["scaling"] == "weak"
    assert d["value"] > 0 and abs(d["ms_per_step"] * 1e-3 * d["value"] - d["cpu_baseline"]["value"] * d["ms_per_step"] * 1e-3) < 1e-6
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["config"]["graphs_per_gpu"] == 2 and "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_without_work():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_dump_outputs_limit_dtypes_and_seeded_row_sample(tmp_path):
    """bench.dump_outputs: float32 / float64 files only, small arrays whole, a large one cut to a sorted row sample that
    is the same for the same shapes, and the files together within the limit."""
    import numpy as np
    m = _bench_module()
    rng = np.random.default_rng(3)
    arrays = {"loss": np.float32(1.5), "grad.w": rng.standard_normal((4, 5)).astype(np.float32),
              "ids": np.arange(7, dtype=np.int64), "x64": rng.standard_normal(3), "local_stress": rng.standard_normal((5000, 3))}
    limit = 32 * 1024
    for d in ("a", "b"):
        m.dump_outputs(str(tmp_path / d), arrays, limit)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(k + ".npy" for k in arrays)
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= limit
    got = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    assert got["loss"].dtype == np.float32 and got["loss"] == 1.5 and got["ids"].dtype == np.float32
    assert got["x64"].dtype == np.float64 and np.array_equal(got["x64"], arrays["x64"])
    assert np.array_equal(got["grad.w"], arrays["grad.w"]) and np.array_equal(got["ids"], np.arange(7))
    ls = got["local_stress"]
    assert ls.dtype == np.float64 and ls.shape[1] == 3 and 1000 < ls.shape[0] < 5000
    rows = [int(np.nonzero((arrays["local_stress"] == r).all(axis=1))[0][0]) for r in ls]
    assert rows == sorted(set(rows))  # distinct rows of the full array, in order
    assert np.array_equal(ls, np.load(tmp_path / "b" / "local_stress.npy"))  # the same sample every time
    with pytest.raises(ValueError):
        m.dump_outputs(str(tmp_path / "c"), {"big": np.zeros((10, 1000))}, 2048)


@pytest.mark.parametrize("argv,why", [(["--dump-outputs", "unused", "--config", "4"], "--dump-outputs"),
                                      (["--impl", "reference", "--steps", "0"], "--steps")])
def test_bench_refuses_arguments_it_cannot_honour(argv, why):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True, timeout=300,
                       cwd=ROOT)
    assert r.returncode == 2 and why in r.stderr and r.stdout == "", r.stderr[-2000:]
    assert not os.path.exists(os.path.join(ROOT, "unused"))


def test_reference_arm_times_the_requested_steps_and_dumps_its_last_one(tmp_path, monkeypatch):
    """However slow the host (a clock that advances 1000 s per reading), the reference arm runs exactly --warmup + --steps
    optimizer steps and reports them; --dump-outputs then holds the state an independent replay of that many steps of
    the oracle port reaches.  One thread on both sides: threaded CPU reductions are not bit-reproducible."""
    import numpy as np
    import torch
    from oracle import pdg_oracle as O
    m = _bench_module()
    threads = torch.get_num_threads()
    clock = iter(range(0, 10 ** 9, 1000))
    monkeypatch.setattr(m.time, "perf_counter", lambda: float(next(clock)))
    monkeypatch.setattr(m.os, "cpu_count", lambda: 1)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--batch", "2", "--nodes", "128", "--steps", "3",
                                      "--warmup", "2", "--dump-outputs", str(tmp_path)])
    lines = []
    monkeypatch.setattr(m, "emit", lines.append)
    try:
        m.run_reference(m.parse(), 0)
        assert len(lines) == 1 and lines[0]["steps"] == 3 and lines[0]["warmup"] == 2
        _, batch, stats = m.oracle_case(2, 128)
        params = {k: v.clone().requires_grad_(True) for k, v in O.init_state_dict(seed=69).items()}
        opt = torch.optim.Adam(list(params.values()), lr=1e-3)
        for _ in range(2 + 3):
            total, nmse, div, pred = O.train_loss(params, batch, stats, 10, False, 10.0)
            opt.zero_grad()
            total.backward()
            opt.step()
    finally:
        torch.set_num_threads(threads)
    got = {n[:-4]: np.load(tmp_path / n) for n in os.listdir(tmp_path)}
    want = {"loss": total, "nmse": nmse, "div": div, "local_stress": pred}
    want.update({"param." + k: p for k, p in params.items()})
    want.update({"grad." + k: p.grad for k, p in params.items()})
    assert sorted(got) == sorted(want)
    for k, v in want.items():
        assert got[k].dtype == np.float32 and np.array_equal(got[k], v.detach().numpy()), k


def test_flop_model_counts():
    """bench.flop_model: SURVEY 8d's algorithmic formula (forward = N 1 050 880 + E 2 654 464 at T = 10, training = 3 x) and the
    executed tile-GEMM count of one 128-node / 128-edge graph, by hand."""
    m = _bench_module()
    f = m.flop_model(1000, 5600, 10, "bf16")
    assert f["algorithmic_per_step"] == 3 * (1000 * 1050880 + 5600 * 2654464)
    g = 2 * 128 ** 3  # one tile GEMM
    one = m.flop_model(128, 128, 10, "bf16")["executed_per_step"]
    assert one == g * (10 * (15 + 14) - 6 + 3 + 3 + 3)
    assert m.flop_model(128, 128, 10, "fp32")["executed_per_step"] == g * (10 * (15 + 11) - 3 + 3 + 3 + 3)
    assert m.flop_model(129, 1, 1, "bf16")["executed_per_step"] == g * (2 * 15 + 14 - 6 + 2 * 3 + 3 + 2 * 3)  # padding to whole tiles
    r = m.flops_of(5.0, "bf16", 33273, 193946, 10)
    assert 0.05 < r["tensor_frac_of_executed"] < 1.0 and r["executed_tflops"] < r["reference_equivalent_tflops"]
    r = m.flops_of(23.0, "fp32", 33273, 193946, 10)
    assert 0.1 < r["fp32_pipe_frac_of_executed"] < 1.0
