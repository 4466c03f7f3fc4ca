#!/usr/bin/env python
"""Headline benchmark: mesh nodes / second of the P-GNN training step (fwd + loss + bwd +
Adam) on synthetic periodic 2-D RVE meshes -- BASELINE.json configs[1]
("config_train_no_div.yml ... synthetic meshes batch 32, 1 B200").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 4] [--lean] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for every field.
  value        whole-job nodes/s, inputs resident in HBM, K steps, CUDA events, max over ranks
  e2e          same metric through the public API from HOST buffers: every step copies one
               pinned host batch (coordinates, triangles, fields) to the device, builds the
               graph there, runs fwd+loss+bwd+Adam and reads the loss back
  roofline     dominant kernel, algorithmic HBM bytes / CUDA-event time
  modes        the same two numbers for the OTHER precision mode (fp32 = the reference's precision, 1e-5)
  cpu_baseline the oracle port (pure-torch restatement of the reference) on the host cores, same 32-mesh batch
  gpu_eager_baseline  the same oracle port moved to `cuda` (eager torch, fp32, TF32 off): the reference's own
               execution mode (scripts/gnn_train.py:344, benchmark_gnn_fem.py:81-100), same box, same batch
  configs      the other BASELINE.json configs in short form (B=1 latency, inference sweep, divergence on)
`--impl reference` times that oracle port alone on the SAME batch with the SAME steps / warm-up (the reference
itself needs torch_geometric and cannot be imported here or on the GPU box).
`--config 4` runs BASELINE configs[4] instead: one epoch over >= 10 000 synthetic meshes written to disk in the
reference's dataset format and read back through MeshStressFieldDataset.loader(rank, world).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

B_DEFAULT, NODES_DEFAULT, T_STEPS = 32, 1024, 10


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=B_DEFAULT, help="graphs per GPU")
    ap.add_argument("--nodes", type=int, default=NODES_DEFAULT, help="target nodes per mesh")
    ap.add_argument("--divergence", type=int, default=0, help="1 = configs[3] (divergence regulariser on)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"],
                    help="bf16 = 16-bit tcgen05 MLP tiles (2e-2 tolerance mode); fp32 = FFMA tiles (1e-5 mode)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lean", action="store_true",
                    help="headline numbers only: skip the other precision mode, the GPU-eager baseline and the configs block")
    ap.add_argument("--config", type=int, default=1, choices=[1, 4],
                    help="1 = configs[1] (default line); 4 = configs[4]: epoch over a >= 10k-mesh on-disk dataset, sharded")
    ap.add_argument("--meshes", type=int, default=10240, help="--config 4: dataset size")
    ap.add_argument("--distinct", type=int, default=128, help="--config 4: distinct mesh geometries generated")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed training step returned (loss terms, prediction, "
                         "parameters and gradients after the optimizer step) as DIR/<name>.npy, at most 64 MB in all "
                         "(rank 0; the inputs are seeded, so two builds run with the same arguments can be compared file by file; "
                         "--impl reference writes the same files for the oracle port, after the same number of steps when "
                         "--warmup >= 3; not with --config 4)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.config != 1:
        ap.error("--dump-outputs writes the outputs of the configs[1] training step; --config 4 times whole epochs")
    return args


# ---------------------------------------------------------------------------------------
# oracle arms (the only places bench.py touches oracle/): CPU port and the same port on cuda
# ---------------------------------------------------------------------------------------
def oracle_case(n_graphs, nodes, seed0=69):
    from oracle import pdg_oracle as O
    from pdivgnn_b200 import synth
    samples = synth.make_dataset(n_graphs, nodes, seed0)
    graphs = [O.build_graph(s, True) for s in samples]
    return O, O.collate(graphs), O.dataset_stats(graphs)


def oracle_case_from(samples):
    from oracle import pdg_oracle as O
    graphs = [O.build_graph(s, True) for s in samples]
    return O, O.collate(graphs), O.dataset_stats(graphs)


def oracle_train_rate(n_graphs, nodes, divergence, steps, warmup, device="cpu", dump=None):
    """fwd + loss + bwd + torch.optim.Adam of the oracle port on `device`, max(1, warmup) warm-up steps then `steps` timed
    ones; returns a dict.  With `dump`, writes the last timed step's outputs there (dump_outputs)."""
    O, batch, stats = oracle_case(n_graphs, nodes)
    if device == "cpu":
        torch.set_num_threads(os.cpu_count() or 1)
    else:
        torch.backends.cuda.matmul.allow_tf32 = False  # the reference runs strict fp32 (models.py:194-208)
        torch.backends.cudnn.allow_tf32 = False
        batch = O.batch_to(batch, device)
    sd = O.init_state_dict(seed=69)
    params = {k: v.clone().to(device).requires_grad_(True) for k, v in sd.items()}
    opt = torch.optim.Adam(list(params.values()), lr=1e-3)

    last = {}

    def step():
        total, nmse, div, pred = O.train_loss(params, batch, stats, T_STEPS, bool(divergence), 10.0)
        opt.zero_grad()
        total.backward()
        opt.step()
        last.update(loss=total.detach(), nmse=nmse.detach(), div=div.detach(), local_stress=pred.detach())

    def sync():
        if device != "cpu":
            torch.cuda.synchronize()

    warmup = max(1, warmup)
    for _ in range(warmup):
        step()
    sync()
    if device == "cpu":
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = (time.perf_counter() - t0) / steps
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        dt = e0.elapsed_time(e1) * 1e-3 / steps
    if dump:
        out = {k: v.cpu().numpy() for k, v in last.items()}
        for k, p in params.items():
            out["param." + k] = p.detach().cpu().numpy()
            out["grad." + k] = p.grad.cpu().numpy()
        dump_outputs(dump, out)
    return {"value": batch.num_nodes / dt, "s_per_step": dt, "nodes": int(batch.num_nodes), "graphs": n_graphs,
            "steps": steps, "warmup": warmup, "cores": torch.get_num_threads() if device == "cpu" else None}


def oracle_forward_ms(n_graphs, nodes, device, reps):
    """no-grad forward(scale_output=True) of the oracle port; ms per call (B = 1: BASELINE configs[0])."""
    O, batch, stats = oracle_case(n_graphs, nodes)
    sd = O.init_state_dict(seed=69)
    if device != "cpu":
        batch = O.batch_to(batch, device)
        sd = {k: v.to(device) for k, v in sd.items()}
    with torch.no_grad():
        for _ in range(2):
            O.forward(sd, batch, stats, T_STEPS)
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            O.forward(sd, batch, stats, T_STEPS)
        if device != "cpu":
            torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps * 1e3, int(batch.num_nodes)


_JSON_OUT = None


def guard_stdout():
    """The contract is ONE JSON line on stdout: everything else that writes to fd 1 (NCCL prints its version line
    there on the first communicator) goes to stderr; emit() writes the line to the real stdout."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(folder, arrays, limit=DUMP_LIMIT_BYTES):
    """Write every array as folder/<name>.npy, float64 kept, everything else as float32, at most `limit` bytes of files
    in all.  Arrays are written smallest first; one that no longer fits whole keeps a sample of its rows (along axis 0)
    drawn from a generator seeded with 0 and sorted, so the same shapes always give the same rows."""
    import numpy as np
    header = 1024  # reserved for each .npy header
    os.makedirs(folder, exist_ok=True)
    left = limit
    for name, a in sorted(arrays.items(), key=lambda kv: (np.size(kv[1]), kv[0])):
        a = np.asarray(a)
        a = a if a.dtype == np.float64 else a.astype(np.float32)
        if a.nbytes + header > left:
            rows = max(0, left - header) // (a.nbytes // a.shape[0]) if a.ndim and a.shape[0] else 0
            if rows == 0:
                raise ValueError(f"--dump-outputs: {name} {a.shape} does not fit the {limit}-byte limit")
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], rows, replace=False))]
        path = os.path.join(folder, name + ".npy")
        np.save(path, a)
        left -= os.path.getsize(path)


METRIC = "mesh nodes/sec, P-GNN training step (fwd+loss+bwd+Adam)"


def run_reference(args, rank):
    """The reference's CPU implementation of the path (oracle port, all host threads) on OUR arm's config: the same
    32-mesh batch per step, the same steps and warm-up.  Rank 0 only."""
    if rank != 0:
        return
    r = oracle_train_rate(args.batch, args.nodes, args.divergence, args.steps, args.warmup, "cpu", args.dump_outputs)
    sample = (f"the full configs[1] batch: {r['graphs']} meshes x ~{args.nodes} nodes ({r['nodes']} nodes) per step, "
              f"{r['warmup']} warm-up + {r['steps']} timed steps, {r['s_per_step']:.2f} s/step")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "nodes/s", "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["s_per_step"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": r["value"], "unit": "nodes/s", "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": r["value"], "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "oracle port (pure-torch CPU restatement of the reference path); the reference needs torch_geometric",
    }
    emit(line)


def workload_config(args, world):
    return {"workload": f"configs[1]: P-GNN linear-elastic training step, divergence={'on' if args.divergence else 'off'}, "
                        f"{args.batch} synthetic periodic plate-with-hole meshes x ~{args.nodes} nodes per GPU, "
                        f"latent 128, {T_STEPS} message-passing steps, Adam lr 1e-3",
            "graphs_per_gpu": args.batch, "nodes_per_mesh": args.nodes, "gpus": world,
            "l2_policy": "per-step working set (saved state ~2.2 GB at batch 32) exceeds the 126 MB L2; no flush needed"}


# ---------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------
class Clocks:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.samples, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, l in self.samples:
            if ts < t0 - 0.05 or ts > t1 + 0.05:
                continue
            f = [x.strip() for x in l.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
                for n, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------
# measurement pieces of the product arm
# ---------------------------------------------------------------------------------------
class Arm:
    """One model + optimizer in one precision mode on this rank's data."""

    def __init__(self, precision, stats, dev, world, with_op):
        import pdivgnn_b200
        from pdivgnn_b200 import dist as pdist
        from pdivgnn_b200.optim import FusedAdam
        torch.manual_seed(69)
        self.precision, self.dev, self.world, self.with_op = precision, dev, world, with_op
        self.model = pdivgnn_b200.EncodeProcessDecode(1, T_STEPS, 128, 6, 3, precision=precision, **stats).to(dev)
        if world > 1:
            pdist.broadcast_parameters(self.model)
            pdist.enable_data_parallel(self.model)
        self.opt = FusedAdam(self.model.parameters(), lr=1e-3)  # torch.optim.Adam semantics, one launch (pdg_adam_step)
        self.loss_fn = pdivgnn_b200.nmse_div_loss

    def train_step(self, b):
        pred = self.model(b, scale_output=False, scale_input=True).local_stress
        nmse, dv = self.loss_fn(pred, b, self.model, self.with_op, 10.0)
        loss = nmse + dv
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        self.opt.step()
        # detached: holding `pred` itself would keep the step's autograd state (the saved workspace) alive
        self.last = {"loss": loss.detach(), "nmse": nmse.detach(), "div": dv.detach(), "local_stress": pred.detach()}
        return loss

    def last_outputs(self):
        """What the last train_step handed its caller, as host arrays: the loss terms, the standardised prediction
        (nodes x 3) and every parameter and its gradient after the optimizer step (state_dict names)."""
        out = {k: v.cpu().numpy() for k, v in self.last.items()}
        for k, p in self.model.named_parameters():
            out["param." + k] = p.detach().cpu().numpy()
            out["grad." + k] = p.grad.cpu().numpy()
        return out

    def params_identical_across_ranks(self):
        """SURVEY 8e: identical parameters on all ranks after every step (checked once, after the timed regions)."""
        import torch.distributed as dist
        if self.world == 1:
            return True
        flat = torch.cat([p.detach().reshape(-1) for p in self.model.parameters()])
        ref = flat.clone()
        dist.broadcast(ref, src=0)
        same = torch.tensor([1 if torch.equal(flat, ref) else 0], device=self.dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        return bool(same.item())


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def time_resident(arm, batch, steps, warmup, world):
    from pdivgnn_b200 import _lib
    L = _lib.lib()
    for _ in range(max(3, warmup)):
        arm.train_step(batch)
    barrier(world)
    L.pdg_launch_count(1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    t0 = time.perf_counter()
    ev0.record()
    for _ in range(steps):
        arm.train_step(batch)
    ev1.record()
    barrier(world)
    t1 = time.perf_counter()
    return ev0.elapsed_time(ev1) / steps, t0, t1, int(L.pdg_launch_count(1))


def kernel_pass(arm, batch, steps, world):
    """The same steps again with CUDA events around every kernel class (library hooks).  Kept out of the headline
    region because an event record between two kernels disables their programmatic dependent launch overlap;
    shares are taken against this pass's own step time."""
    from pdivgnn_b200 import _lib
    L = _lib.lib()
    ksteps = max(3, min(steps, 10))
    L.pdg_timing_enable(1)
    _lib.timing_collect()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    k0.record()
    for _ in range(ksteps):
        arm.train_step(batch)
    k1.record()
    barrier(world)
    L.pdg_timing_enable(0)
    return k0.elapsed_time(k1) / ksteps, ksteps, _lib.timing_collect()


def time_e2e(arm, host, steps, warmup, world, with_op):
    """Every step consumes a batch that starts in pinned HOST memory; its copies, device edge construction and plan
    build run on a side stream, in a worker thread, two steps ahead (batcher.DevicePrefetcher), like a DataLoader
    worker.  The loss of every step IS read back (4 bytes, pinned host buffer), one step late: the copy of step j
    is waited for after step j+1 has been enqueued, so the host never drains the GPU queue."""
    from pdivgnn_b200 import batcher
    pf = batcher.DevicePrefetcher(host, arm.dev, True, with_op)
    loss_host = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event() for _ in range(2)]
    seen = []

    def e2e_step(j):
        b = pf.get()
        loss = arm.train_step(b)  # enqueue the whole step ...
        loss_host[j & 1].copy_(loss.detach().reshape(1), non_blocking=True)  # D2H read of the step's loss
        loss_ev[j & 1].record()
        pf.prefetch()             # ... then stage the next host batch underneath it
        if j > 0:
            loss_ev[(j - 1) & 1].synchronize()
            seen.append(float(loss_host[(j - 1) & 1][0]))
        return b.num_nodes

    def drain(j_last):
        loss_ev[j_last & 1].synchronize()
        seen.append(float(loss_host[j_last & 1][0]))

    # warm-up: two full rotations over the host batches, so the caching allocator has seen every batch size
    # (a first-time cudaMalloc / cudaFree inside the timed region would stall the device)
    nw = max(2 * len(host), warmup)
    for j in range(nw):
        e2e_step(j)
    drain(nw - 1)
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    nodes_done = 0
    for j in range(steps):
        nodes_done += e2e_step(j)
    drain(steps - 1)
    e1.record()
    barrier(world)
    pf.close()
    assert len(seen) >= steps and all(v == v for v in seen[-steps:]), "every step's loss must have been read back"
    return e0.elapsed_time(e1) / steps, float(nodes_done) / steps


def reduce_over_ranks(ms, e2e_ms, n_nodes, nodes_e2e, dev, world):
    if world == 1:
        return ms, e2e_ms, float(n_nodes), float(nodes_e2e)
    import torch.distributed as dist
    tt = torch.tensor([ms, e2e_ms, float(n_nodes), float(nodes_e2e)], device=dev, dtype=torch.float64)
    mx, sm = tt.clone(), tt.clone()
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    return float(mx[0]), float(mx[1]), float(sm[2]), float(sm[3])


def algorithmic_bytes(kernel, precision, n_nodes, n_edges):
    """DESIGN.md section 4: bytes one launch has to move for the data types each path stores.
      fp32 path   edge_step_bwd per edge: read e_t, y2_t, ge_{t+1}, y_prev, write ge_t (5 x 512 B) + dhm, dhn rows written
                  (2 x 512 B) + 8 B ids; per node: gathered Pa, Pb, g_agg rows (3 x 512 B) + RA, RB written (2 x 512 B)
                  edge_step per edge: read e_{t-1}, y2_{t-1}, write e_t, y2_t (4 x 512 B) + 8 B ids; per node: Pa, Pb + aggraw
      16-bit path raw edge-MLP outputs (y2, y_prev) are 16-bit rows (256 B), the backward reads e_t as a 16-bit operand-tile
                  image (256 B) written by the forward, dhm / dhn / Pa / Pb / g_agg rows are 16-bit; ge and the e stream fp32:
                  edge_step_bwd per edge: 256 (e image) + 256 (y2_t) + 256 (y_prev) + 512 + 512 (ge read, write)
                  + 2 x 256 (dhm, dhn) + 8; per node 3 x 256 + 2 x 512
                  edge_step (training) per edge: 512 + 256 read, 512 + 256 (image) + 256 (y2) written + 8; per node 2 x 256 + 512"""
    e_pad = (n_edges + 127) // 128 * 128
    if precision == "bf16":
        return {"edge_step_bwd": e_pad * (3 * 256 + 2 * 512 + 2 * 256 + 8) + n_nodes * (3 * 256 + 2 * 512),
                "edge_step": e_pad * (512 + 256 + 512 + 256 + 256 + 8) + n_nodes * (2 * 256 + 512)}.get(kernel)
    return {"edge_step_bwd": e_pad * (5 * 512 + 2 * 512 + 8) + n_nodes * (3 * 512 + 2 * 512),
            "edge_step": e_pad * (4 * 512 + 8) + n_nodes * (2 * 512 + 512)}.get(kernel)


def flop_model(n_nodes, n_edges, steps=10, precision="bf16"):
    """FLOPs of one training step (SURVEY 8d: report both, never quote the reference-equivalent number as utilisation).
      algorithmic  the reference's own Linear layers, 2 m n k each: forward = N (34 304 + 33 536 + T 98 304)
                   + E (33 024 + T 262 144); forward + backward = 3 x forward.
      executed     the 128 x 128 x 128 tile GEMMs the kernels issue after the layer-1 split (Pa / Pb per node, G per edge):
                   per 128-row tile and message-passing step node_pre 2, edge_step 3, node_update 3, node_update_bwd 6,
                   edge_step_bwd 11 in the 16-bit path (G is recomputed for the second evaluation, de / dWe accumulate in two
                   GEMMs each) and 8 in the fp32 path, node_pre_bwd 4 (the last step has no edge update: 1 + 5 fewer, fp32
                   1 + 2); encoders and decoder 1 forward + 2 backward each; rows padded to whole tiles."""
    n_pad = (n_nodes + 127) // 128 * 128
    e_pad = (n_edges + 127) // 128 * 128
    fwd_alg = n_nodes * (34304 + 33536 + steps * 98304) + n_edges * (33024 + steps * 262144)
    per_row = 2 * 128 * 128
    bwd_edge, last_less = (11, 1 + 5) if precision == "bf16" else (8, 1 + 2)
    executed = per_row * (steps * (n_pad * (2 + 3 + 6 + 4) + e_pad * (3 + bwd_edge)) - e_pad * last_less
                          + n_pad * 3 + e_pad * 3 + n_pad * 3)
    return {"algorithmic_per_step": 3 * fwd_alg, "executed_per_step": executed}


def flops_of(ms_per_step, precision, n_nodes, n_edges, steps=10):
    f = flop_model(n_nodes, n_edges, steps, precision)
    out = dict(f)
    out["executed_tflops"] = f["executed_per_step"] / (ms_per_step * 1e-3) / 1e12
    out["reference_equivalent_tflops"] = f["algorithmic_per_step"] / (ms_per_step * 1e-3) / 1e12
    if precision == "bf16":
        peak, src = 1369.5, "fallback 1369.5 TFLOP/s"
        try:
            pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            peak, src = float(pk["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained: the step is a long back-to-back run)"
        except Exception:
            pass
        out.update({"tensor_peak_tflops": peak, "tensor_frac_of_executed": out["executed_tflops"] / peak, "peak_source": src})
    else:
        mhz = 1965.0
        try:
            mhz = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["sm_max_mhz"])
        except Exception:
            pass
        peak = 148 * 128 * 2 * mhz * 1e6 / 1e12  # 148 SMs x 128 fp32 FMA lanes (packed FFMA2 every other cycle per scheduler)
        out.update({"fp32_pipe_peak_tflops": peak, "fp32_pipe_frac_of_executed": out["executed_tflops"] / peak,
                    "note": "fp32 FFMA2 tiles: no tensor-core work; peak = 148 SMs x 128 FMA/clock at the maximum SM clock"})
    return out


def roofline_of(ktimes, ksteps, ms_k, precision, n_nodes, n_edges):
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    if not ktimes:
        return None, {}
    top = max(ktimes.items(), key=lambda kv: kv[1][0])[0]
    dom = top if top in ("edge_step_bwd", "edge_step") else ("edge_step_bwd" if "edge_step_bwd" in ktimes else top)
    traffic_tab = {}
    try:
        traffic_tab = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
    except Exception:
        pass

    def one(kernel):
        tot_ms, cnt = ktimes[kernel]
        alg = algorithmic_bytes(kernel, precision, n_nodes, n_edges)
        if not alg:
            return None
        us = tot_ms / cnt * 1e3
        ach = alg / (us * 1e-6) / 1e9
        return {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                "traffic": traffic_tab.get(f"{kernel}:{precision}"), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg, "us_per_launch": us, "share_of_step": tot_ms / ksteps / ms_k}
    roof = one(dom)
    if roof:
        roof.update({"steps_in_kernel_pass": ksteps, "ms_per_step_kernel_pass": ms_k,
                     "note": ("warp-specialised tcgen05 16-bit tile kernel: bound by L1 gather throughput and epilogue latency, "
                              "not by HBM or the tensor pipe (DESIGN.md section 4b)" if precision == "bf16" else
                              "fp32 FFMA tile path: compute-bound, far from the HBM roof (see DESIGN.md)")})
        # the north star's roofline target is stated for the AGGREGATION kernel (the forward edge kernel): report it too
        if dom != "edge_step" and "edge_step" in ktimes:
            roof["aggregation_kernel"] = one("edge_step")
    kshare = {k: round(v[0] / ksteps / ms_k, 4) for k, v in sorted(ktimes.items(), key=lambda kv: -kv[1][0])}
    return roof, kshare


def configs_block(dev, samples, stats_dev, nodes):
    """BASELINE.json configs 0, 2, 3 in short form on this GPU (16-bit tile mode unless stated).  Forward timings use
    inputs resident in HBM, CUDA events, 3 warm-ups."""
    import pdivgnn_b200
    from pdivgnn_b200 import batcher
    from pdivgnn_b200.optim import FusedAdam
    out = {}

    def fwd_ms(model, b, reps):
        with torch.no_grad():
            for _ in range(3):
                model(b)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                model(b)
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def model_of(prec, graphs=False):
        torch.manual_seed(69)
        return pdivgnn_b200.EncodeProcessDecode(1, T_STEPS, 128, 6, 3, precision=prec, cuda_graphs=graphs, **stats_dev).to(dev)

    # configs[0]: P-DivGNN inference on ONE periodic mesh, batch 1 (the reference's own benchmark shape)
    b1 = batcher.batch_from_host(batcher.host_arrays(samples[:1], False), dev, True, False)
    c0 = {"workload": "configs[0]: inference forward (scale_output=True), one periodic ~1024-node mesh, batch 1",
          "nodes": b1.num_nodes, "edges": int(b1.edge_index.shape[1])}
    for prec in ("bf16", "fp32"):
        m = fwd_ms(model_of(prec), b1, 200)
        mg = fwd_ms(model_of(prec, True), b1, 200)
        c0[prec] = {"ms_per_forward": m, "ms_per_forward_cuda_graph": mg, "nodes_per_s_cuda_graph": b1.num_nodes / (mg * 1e-3)}
    try:
        ms_g, _ = oracle_forward_ms(1, nodes, "cuda", 20)
        ms_c, _ = oracle_forward_ms(1, nodes, "cpu", 5)
        c0["gpu_eager_oracle_ms_per_forward"] = ms_g
        c0["cpu_oracle_ms_per_forward"] = ms_c
        c0["cpu_cores"] = torch.get_num_threads()
    except Exception as ex:  # the baselines must never take the bench line down
        c0["oracle_error"] = repr(ex)[:200]
    out["0"] = c0

    # the reference's own published benchmark (scripts/benchmark_gnn_fem.py:81-100, 485-575; BASELINE.md section 1): forward of
    # ONE periodic mesh per call, 458 ... 25 556 nodes, mean of 5 runs after one warm-up.  Ours: the same protocol with
    # CUDA events (resident inputs), and end to end from HOST arrays the way its orange series counts the graph
    # preprocessing (periodic edges + node labels): H2D + device batcher + device labelling + forward + result D2H.
    from pdivgnn_b200 import synth
    published_ms = {458: 11.6, 1918: 34.5, 5951: 95.4, 12524: 199.0, 19104: 304.0, 25556: 403.0}
    sweep_ref = {}
    for target, pub in published_ms.items():
        smp = [synth.make_rve_mesh(1000 + target, target, 3.0)]
        hst = batcher.host_arrays(smp, False)
        b = batcher.batch_from_host(hst, dev, True, False)
        row = {"nodes": b.num_nodes, "edges": int(b.edge_index.shape[1]), "published_ms": pub}
        for prec in ("bf16", "fp32"):
            m = model_of(prec)
            ms = fwd_ms(m, b, 20)
            row[prec] = {"ms_per_forward": ms, "nodes_per_s": b.num_nodes / (ms * 1e-3)}
            if prec == "bf16":
                pts_h, faces_h, ms_h = smp[0]["pos"], smp[0]["faces"], tuple(float(v) for v in smp[0]["mean_stress"])

                def e2e_once():
                    # benchmark_gnn_fem.convert_mesh_to_graph (:388-415) + the periodicity assert (:195), all on the device
                    bb = batcher.convert_mesh_to_graph(pts_h, faces_h, ms_h, dev, check_periodic=True)
                    with torch.no_grad():
                        return m(bb).local_stress.cpu()
                e2e_once()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(5):
                    e2e_once()
                row["bf16"]["ms_from_host_arrays_incl_graph_build_labels_periodicity_check"] = (time.perf_counter() - t0) / 5 * 1e3
        try:
            O, ob, ost = oracle_case_from(smp)
            sdo = {k: v.to(dev) for k, v in O.init_state_dict(seed=69).items()}
            obd = O.batch_to(ob, dev)
            with torch.no_grad():
                O.forward(sdo, obd, ost, T_STEPS)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(5):
                    O.forward(sdo, obd, ost, T_STEPS)
                torch.cuda.synchronize()
            row["gpu_eager_oracle_ms_per_forward"] = (time.perf_counter() - t0) / 5 * 1e3
        except Exception as ex:
            row["oracle_error"] = repr(ex)[:200]
        sweep_ref[str(target)] = row
        del b
    out["reference_benchmark_sweep"] = {
        "workload": "scripts/benchmark_gnn_fem.py protocol: forward(scale_output=True) of ONE periodic mesh per call, latent 128, "
                    "10 steps; published_ms = docs/benchmark_hyperelast.svg (authors' unnamed GPU, BASELINE.md section 1)",
        "points": sweep_ref}

    # configs[2]: no periodic edges, inference throughput sweep over the batch size
    sweep = {}
    m16 = model_of("bf16")
    for B in (1, 8, 64, 512, 1024):
        sm = [samples[i % len(samples)] for i in range(B)]
        b = batcher.batch_from_host(batcher.host_arrays(sm, False), dev, False, False)
        ms = fwd_ms(m16, b, 50 if B <= 64 else 10)
        sweep[str(B)] = {"nodes": b.num_nodes, "ms_per_forward": ms, "nodes_per_s": b.num_nodes / (ms * 1e-3)}
        del b
    out["2"] = {"workload": "configs[2]: GNN without periodic edges, inference forward, batch 1 .. 1024 graphs "
                            "(the 32 distinct meshes of the headline batch, repeated)", "precision": "bf16", "sweep": sweep}

    # configs[3]: divergence regulariser on (lambda = 10), fwd + loss + bwd + Adam
    c3 = {"workload": "configs[3]: P-DivGNN training step, divergence regulariser on (penalty 10)", "precision": "bf16"}
    for B in (16, 32):
        b = batcher.batch_from_host(batcher.host_arrays(samples[:B], True), dev, True, True)
        model = model_of("bf16")
        opt = FusedAdam(model.parameters(), lr=1e-3)

        def step():
            pred = model(b, scale_output=False, scale_input=True).local_stress
            nmse, dv = pdivgnn_b200.nmse_div_loss(pred, b, model, True, 10.0)
            loss = nmse + dv
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 20
        c3[str(B)] = {"nodes": b.num_nodes, "ms_per_step": ms, "nodes_per_s": b.num_nodes / (ms * 1e-3)}
    out["3"] = c3
    out["4"] = "python bench.py --config 4 [--gpus N under torchrun]: epoch over a >= 10k-mesh on-disk dataset (profiles/)"
    return out


# ---------------------------------------------------------------------------------------
# configs[4]: 10k synthetic meshes on disk -> MeshStressFieldDataset.loader(rank, world) -> train_epoch
# ---------------------------------------------------------------------------------------
def run_config4(args, rank, world, local):
    import shutil
    import tempfile
    import numpy as np
    import torch.distributed as dist
    import pdivgnn_b200
    from pdivgnn_b200 import dist as pdist, engine, io as pio, synth
    from pdivgnn_b200.optim import FusedAdam
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        pdist.init_from_env("nccl")
    folder = os.path.join(tempfile.gettempdir(), f"pdg_cfg4_{args.meshes}_{args.nodes}_{args.distinct}")
    t_gen = time.perf_counter()
    if rank == 0 and not os.path.exists(os.path.join(folder, "dataset.csv")):
        shutil.rmtree(folder, ignore_errors=True)
        base = synth.make_dataset(args.distinct, args.nodes, 69)
        rng = np.random.default_rng(69)
        samples = []
        for i in range(args.meshes):  # every sample: one of the distinct geometries with its own load case and field
            s = dict(base[i % len(base)])
            ms = rng.uniform(-1.0, 1.0, size=3) * 5.0e3
            s["mean_stress"] = ms
            s["stress_field"] = ms[None, :] + 0.3 * 5.0e3 * rng.standard_normal((s["pos"].shape[0], 3))
            samples.append(s)
        pio.write_dataset(samples, folder)
        del samples
    if world > 1:
        dist.barrier()
    t_gen = time.perf_counter() - t_gen
    t_read = time.perf_counter()
    ds = pio.MeshStressFieldDataset(os.path.join(folder, "dataset.csv"), periodic_graph=True, device=dev)
    t_read = time.perf_counter() - t_read
    torch.manual_seed(69)
    model = pdivgnn_b200.EncodeProcessDecode(1, T_STEPS, 128, 6, 3, precision=args.precision, **ds.stats()).to(dev)
    if world > 1:
        pdist.broadcast_parameters(model)
        pdist.enable_data_parallel(model)
    opt = FusedAdam(model.parameters(), lr=1e-3)
    with_op = bool(args.divergence)
    loader = ds.loader(args.batch, shuffle=True, seed=69, with_op_div=with_op, rank=rank, world=world)
    nodes_per_epoch = None

    def epoch():
        return engine.train_epoch(model, loader, opt, with_op, 10.0)

    first = epoch()  # warm-up epoch: allocator, pinned host batches are NOT cached when shuffling (fresh collation every epoch)
    barrier(world)
    clocks = Clocks(local)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    t0 = time.perf_counter()
    e0.record()
    res = epoch()
    e1.record()
    barrier(world)
    t1 = time.perf_counter()
    ms_epoch = e0.elapsed_time(e1)
    clk = clocks.stop(t0, t1)
    # nodes this rank trained on in one epoch (its shard of the epoch's batches)
    my_nodes = sum(int(ds.samples[i]["pos"].shape[0]) for c in loader._batches() for i in c)
    tt = torch.tensor([ms_epoch, float(my_nodes)], device=dev, dtype=torch.float64)
    if world > 1:
        mx, sm = tt.clone(), tt.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms_epoch, tot_nodes = float(mx[0]), float(sm[1])
    else:
        tot_nodes = float(my_nodes)
    same = True
    if world > 1:
        flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
        ref = flat.clone()
        dist.broadcast(ref, src=0)
        ok = torch.tensor([1 if torch.equal(flat, ref) else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        same = bool(ok.item())
    if rank == 0:
        steps = len(loader)
        emit({"metric": "mesh nodes/sec, P-GNN training epoch over an on-disk dataset (fwd+loss+bwd+allreduce+Adam)",
              "value": tot_nodes / (ms_epoch * 1e-3), "unit": "nodes/s", "n_gpus": world, "steps": steps, "warmup": steps,
              "ms_per_step": ms_epoch / steps, "ms_per_epoch": ms_epoch, "higher_is_better": True, "scaling": "strong",
              "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
              "config": {"workload": f"configs[4]: {len(ds)} synthetic meshes x ~{args.nodes} nodes ({args.distinct} distinct geometries, "
                                     f"own load case / field each) written as .vtk + .npz + dataset.csv, read by MeshStressFieldDataset, "
                                     f"sharded by loader(rank, world), batch {args.batch} per GPU, shuffle, divergence="
                                     f"{'on' if with_op else 'off'}; every step collates + pins its host batch, copies it, builds "
                                     f"the graph on the GPU (prefetched on a side stream)", "gpus": world,
                         "graphs_per_gpu": args.batch, "meshes": len(ds)},
              "clocks": clk, "epoch_loss": res["total"], "first_epoch_loss": first["total"],
              "params_identical_across_ranks": same, "dataset_write_s": t_gen, "dataset_read_and_stats_s": t_read,
              "e2e": {"value": tot_nodes / (ms_epoch * 1e-3), "unit": "nodes/s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": 0,
                      "note": "this config IS end to end: every batch starts as host arrays of the dataset"}})
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------
def main():
    args = parse()
    guard_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    if args.config == 4:
        run_config4(args, rank, world, local)
        return
    import torch.distributed as dist
    from pdivgnn_b200 import _lib, batcher, synth
    from pdivgnn_b200 import dist as pdist

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        pdist.init_from_env("nccl")
    L = _lib.lib()

    # ---- data: 4 distinct host batches per rank (e2e rotates through them), first one resident
    n_host = 4
    host, samples0 = [], None
    with_op = bool(args.divergence)
    for j in range(n_host):
        seed0 = 69 + (rank * n_host + j) * args.batch
        smp = synth.make_dataset(args.batch, args.nodes, seed0)
        if j == 0:
            samples0 = smp
        host.append(batcher.host_arrays(smp, with_op))
    resident = batcher.batch_from_host(host[0], dev, True, with_op)
    stats = batcher.dataset_stats([resident])
    n_nodes, n_edges = resident.num_nodes, resident.edge_index.shape[1]

    # ---- headline mode ----------------------------------------------------------------------
    arm = Arm(args.precision, stats, dev, world, with_op)
    clocks = Clocks(local)
    time.sleep(0.25)
    ms, t0, t1, launches = time_resident(arm, resident, args.steps, args.warmup, world)  # launches: timed steps only
    clk = clocks.stop(t0, t1)
    if args.dump_outputs and rank == 0:  # before the passes below train the same model further
        dump_outputs(args.dump_outputs, arm.last_outputs())
    ms_k, ksteps, ktimes = kernel_pass(arm, resident, args.steps, world)
    h2d = batcher.host_bytes(host[0], with_op)
    e2e_ms, nodes_e2e = time_e2e(arm, host, args.steps, args.warmup, world, with_op)
    e2e_retry = None
    again = e2e_ms > 1.15 * ms
    if world > 1:  # the re-measurement has barriers inside: every rank must take the same decision
        flag = torch.tensor([1 if again else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        again = bool(flag.item())
    if again:  # a host-side hiccup (the staging thread lost its core) shows up as an outlier: measure once more, keep both
        e2e_retry = {"first_try_ms_per_step": e2e_ms}
        e2e_ms2, nodes_e2e2 = time_e2e(arm, host, args.steps, args.warmup, world, with_op)
        if e2e_ms2 < e2e_ms:
            e2e_ms, nodes_e2e = e2e_ms2, nodes_e2e2
    same_params = arm.params_identical_across_ranks()
    peer = getattr(arm.model, "_pdg_peer", None)
    if peer is not None and peer.timed_out():
        raise SystemExit("bench.py: a peer did not arrive in pdg_allreduce_mean (status != 0): the run is invalid")
    ms, e2e_ms, tot_nodes, tot_nodes_e2e = reduce_over_ranks(ms, e2e_ms, n_nodes, nodes_e2e, dev, world)
    value = tot_nodes / (ms * 1e-3)
    e2e_value = tot_nodes_e2e / (e2e_ms * 1e-3)

    # ---- the other precision mode, same batch (fewer steps: the fp32 FFMA path is ~7x slower) ----
    modes = None
    if not args.lean:
        other = "fp32" if args.precision == "bf16" else "bf16"
        o_steps = max(5, min(args.steps, 10 if other == "fp32" else args.steps))
        arm2 = Arm(other, stats, dev, world, with_op)
        ms2, _, _, _ = time_resident(arm2, resident, o_steps, 3, world)
        e2e2, nodes2 = time_e2e(arm2, host, o_steps, 3, world, with_op)
        ms2, e2e2, tn2, tne2 = reduce_over_ranks(ms2, e2e2, n_nodes, nodes2, dev, world)
        modes = {other: {"value": tn2 / (ms2 * 1e-3), "ms_per_step": ms2, "steps": o_steps,
                         "e2e": {"value": tne2 / (e2e2 * 1e-3), "ms_per_step": e2e2}},
                 args.precision: {"value": value, "ms_per_step": ms, "steps": args.steps,
                                  "e2e": {"value": e2e_value, "ms_per_step": e2e_ms}},
                 "tolerances": {"bf16": "2e-2 norm-wise relative on fields, loss and per-tensor gradients (tests/test_gpu_bf16.py)",
                                "fp32": "1e-5 on fields / loss; gradients at the reference's own fp32-vs-fp64 noise floor"}}
        del arm2

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    roof, kshare = roofline_of(ktimes, ksteps, ms_k, args.precision, n_nodes, n_edges)

    try:
        flops = flops_of(ms, args.precision, n_nodes, n_edges, T_STEPS)
    except Exception as ex:  # bookkeeping must never take the bench line down
        flops = {"error": repr(ex)[:200]}
    cpu = gpu_eager = cfgs = None
    if not args.no_cpu_baseline and world == 1:
        r = oracle_train_rate(args.batch, args.nodes, args.divergence, 3, 1, "cpu")
        cpu = {"value": r["value"], "unit": "nodes/s", "cores": r["cores"], "kind": "port",
               "sample": f"the same configs[1] batch ({r['graphs']} meshes x ~{args.nodes} nodes = {r['nodes']} nodes per step), "
                         f"1 warm-up + 3 steps, {r['s_per_step']:.2f} s/step, oracle port (pure torch)"}
    if not args.lean and world == 1:
        try:
            r = oracle_train_rate(args.batch, args.nodes, args.divergence, 10, 3, "cuda")
            gpu_eager = {"value": r["value"], "unit": "nodes/s", "ms_per_step": r["s_per_step"] * 1e3, "steps": r["steps"],
                         "warmup": r["warmup"], "kind": "oracle port on cuda: eager torch ops, fp32, allow_tf32=False, "
                         "torch.optim.Adam -- the reference's own execution mode (gnn_train.py:344) without PyG's Python overhead",
                         "speedup_of_value": value / r["value"], "speedup_of_e2e": e2e_value / r["value"],
                         "speedup_of_fp32_mode": (modes["fp32"]["value"] / r["value"]) if modes and "fp32" in modes else None}
        except Exception as ex:
            gpu_eager = {"error": repr(ex)[:300]}
        try:
            cfgs = configs_block(dev, samples0, stats, args.nodes)
        except Exception as ex:
            cfgs = {"error": repr(ex)[:300]}

    line = {
        "metric": METRIC, "value": value, "unit": "nodes/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {**workload_config(args, world), "nodes_per_gpu": n_nodes, "edges_per_gpu": n_edges,
                   "precision_mode": ("16-bit MLP-tile operands on tcgen05 (fp16 tiles, scaled gradients), fp32 accumulate / "
                                      "LayerNorm / latents (tolerance 2e-2; measured 1e-3 on fields, <= 1.5e-2 per gradient tensor)"
                                      if args.precision == "bf16" else "fp32 FFMA tiles (tolerance 1e-5)")},
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "nodes/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms, **({"remeasured": e2e_retry} if e2e_retry else {})},
        "gpu_launches": int(launches),
        "roofline": roof, "flops": flops, "cpu_baseline": cpu, "gpu_eager_baseline": gpu_eager, "modes": modes,
        "params_identical_across_ranks": same_params,
        "allreduce": (None if world == 1 else ("p2p: pdg_allreduce_mean over NVLink peer memory (one kernel)"
                                               if getattr(arm.model, "_pdg_peer", None) is not None else "nccl all_reduce(AVG)")),
        "kernel_share_of_step": kshare, "configs": cfgs,
        "published_reference_gpu_forward_nodes_per_s": 63000,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
