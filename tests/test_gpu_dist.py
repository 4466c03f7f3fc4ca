"""Two NCCL ranks on two GPUs (skipped on a 1-GPU box): SURVEY 8e's correctness check on hardware.

  * the gradient every rank holds after backward == the MEAN of the per-shard oracle gradients (each rank's
    graph-LayerNorm statistics are those of its own shard: the reference run with batch B_local, SURVEY H6);
  * parameters are bit-identical on all ranks after 3 optimizer steps;
  * rank 0's loss / gradient with world = 2 on ITS shard equals a single-process run on that shard up to the
    all-reduce (checked through the oracle comparison).
"""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, precision, out):
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    for p in (os.path.dirname(here), here):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist
    import pdg_helpers as H
    from oracle import pdg_oracle as O
    import pdivgnn_b200
    from pdivgnn_b200 import dist as pd
    from pdivgnn_b200.optim import FusedAdam
    pd.init_from_env("nccl")
    dev = torch.device("cuda", rank)
    # shards: 3 meshes each, different seeds; statistics of the WHOLE set (both shards) like a real dataset
    shards = [H.synthetic_batch(3, 300, seed0=69 + 10 * r) for r in range(world)]
    stats = O.dataset_stats([g for s in shards for g in s[1]])
    sd = O.init_state_dict(seed=69)
    model = H.make_model(stats, params=sd, device=dev)
    model.precision = precision
    pd.broadcast_parameters(model)
    pd.enable_data_parallel(model)
    db = H.DeviceBatch(shards[rank][2], device=dev)
    pred = model(db, scale_output=False).local_stress
    nmse, div = pdivgnn_b200.nmse_div_loss(pred, db, model, True, 10.0)
    (nmse + div).backward()
    grads = {k: p.grad.detach().cpu() for k, p in model.named_parameters()}
    # oracle: mean over shards of the per-shard gradients (fp64 yard-stick, fp32 = the reference's arithmetic)
    per64 = [O.loss_and_grads(sd, s[2], stats, 10, True, 10.0, dtype=torch.float64)[4] for s in shards]
    per32 = [O.loss_and_grads(sd, s[2], stats, 10, True, 10.0, dtype=torch.float32)[4] for s in shards]
    worst = 0.0
    ok = True
    for k in O.STATE_KEYS:
        m64 = sum(g[k] for g in per64) / world
        m32 = sum(g[k].double() for g in per32) / world
        ours, ref = H.rel_err(grads[k], m64), H.rel_err(m32, m64)
        tol = (max(1e-5, 4 * ref[0]), max(1e-5, 3 * ref[1])) if precision == "fp32" else (2e-2, 2e-2)
        ok = ok and ours[0] <= tol[0] and ours[1] <= tol[1]
        worst = max(worst, ours[0])
    # 3 optimizer steps, then bit-identical parameters everywhere
    opt = FusedAdam(model.parameters(), lr=1e-3)
    for _ in range(3):
        pred = model(db, scale_output=False).local_stress
        nmse, div = pdivgnn_b200.nmse_div_loss(pred, db, model, True, 10.0)
        opt.zero_grad(set_to_none=True)
        (nmse + div).backward()
        opt.step()
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    same = all(torch.equal(g, gathered[0]) for g in gathered)
    moved = not torch.equal(flat.cpu(), torch.cat([sd[k].reshape(-1) for k in O.STATE_KEYS]))
    out[rank] = (bool(ok), float(worst), bool(same), bool(moved))
    dist.destroy_process_group()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_two_nccl_ranks_average_gradients_and_stay_in_sync(precision):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world, port = 2, _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, port, precision, out), nprocs=world, join=True)
    for r in range(world):
        ok, worst, same, moved = out[r]
        print(f"rank {r} [{precision}]: averaged gradient vs mean of per-shard oracle gradients, worst rel-Linf {worst:.2e}; "
              f"params identical across ranks after 3 steps: {same}")
        assert ok, (r, worst)
        assert same and moved


def _peer_worker(rank, world, port, out):
    import sys
    import time
    here = os.path.dirname(os.path.abspath(__file__))
    for p in (os.path.dirname(here), here):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist
    from pdivgnn_b200 import _lib, dist as pd
    pd.init_from_env("nccl")
    dev = torch.device("cuda", rank)
    n = _lib.PDG_PARAM_ELEMS
    pa = pd.PeerAllreduce(n, dev)
    ok, bit_equal = pa.self_test(), True
    g = torch.Generator().manual_seed(7 + rank)
    for it in range(9):  # odd and even sequence numbers (double-buffered exchange area), ranks arriving at different times
        x = (torch.randn(n, generator=g) * (10.0 ** (it % 4 - 2))).to(dev)
        ref = x.double()
        dist.all_reduce(ref, op=dist.ReduceOp.SUM)
        ref = (ref / world).float()
        if rank == it % world:
            time.sleep(0.05)
        y = pa(x.clone())
        ok = ok and torch.allclose(y, ref, rtol=2e-6, atol=1e-7)
        ys = [torch.empty_like(y) for _ in range(world)]
        dist.all_gather(ys, y)
        bit_equal = bit_equal and all(torch.equal(ys[0], t) for t in ys)  # rank-order sums: identical everywhere
    out[rank] = (bool(ok), bool(bit_equal), pa.timed_out())
    pa.close()
    dist.destroy_process_group()


def test_peer_memory_allreduce_matches_nccl_and_is_rank_identical():
    """pdg_allreduce_mean (NVLink peer memory, one kernel) vs NCCL on two ranks: same means (fp32 rounding), bit-identical
    results on both ranks (needed for identical parameters without a broadcast), no timeout."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world, port = 2, _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_peer_worker, args=(world, port, out), nprocs=world, join=True)
    for r in range(world):
        ok, same, timed_out = out[r]
        assert ok and same and not timed_out, (r, ok, same, timed_out)
