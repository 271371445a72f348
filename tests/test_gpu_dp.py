"""Data parallelism over graph batches on the PRODUCT path (BASELINE configs[2]; SURVEY.md sections 4.8, 8e): the
gradients of N ranks, each running the repo's `Block` on its share of the graphs and all-reducing the flat bucket of
pfs-neural-net_b200/dp.py, equal the gradients of one GPU running all graphs.

  * test_dp_gradients_equal_single_gpu_sum: one GPU, the ranks emulated one after the other (always runs);
  * test_dp_two_gpus_nccl: two processes, two GPUs, NCCL all-reduce (skipped on a one-GPU machine)."""
import os
import socket

import pytest
import torch

from oracle import block_oracle as bo

pytestmark = pytest.mark.gpu
F, S, T, G = 10, 60, 12, 4


def _problem(dev):
    from pfs_neural_net_b200 import gnn
    state = bo.random_block_state(F, seed=4)
    blk = gnn.Block(F)
    blk.load_state_dict(state, strict=True)
    blk = blk.to(dev).train()
    ei = bo.complete_bipartite(S, T).to(dev)
    g = torch.Generator().manual_seed(9)
    ins = [torch.randn(G, n, F, generator=g).to(dev) for n in (S, T, S * T, 1)]
    ups = [torch.randn(G, n, F, generator=g).to(dev) for n in (S, T, S * T, 1)]
    return blk, ei, ins, ups


def _run(blk, ei, ins, ups, graphs):
    for p in blk.parameters():
        p.grad = None
    xs = [t[graphs].clone().requires_grad_(True) for t in ins]
    _, o_s, o_t, o_e, o_u = blk((ei, *xs))
    torch.autograd.backward([o_s, o_t, o_e, o_u], [u[graphs] for u in ups])
    return [x.grad for x in xs]


def _close(a, b, what, floor=0.0):
    scale = max(b.abs().max().item(), floor, 1e-30)
    err = (a - b).abs().max().item()
    assert err <= 2e-5 * scale, (what, err, scale)


def _floors(named, grads):
    """a bias in front of a train-mode BatchNorm has an analytically zero gradient (fp32 noise): judge it on the scale of
    its weight's gradient, like the parity tests do"""
    mags = {n: g.abs().max().item() for (n, _), g in zip(named, grads)}
    return {n: mags.get(n[:-4] + "weight", 0.0) if n.endswith("bias") else 0.0 for n in mags}


def test_dp_gradients_equal_single_gpu_sum():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from pfs_neural_net_b200 import dp
    dev = torch.device("cuda:0")
    blk, ei, ins, ups = _problem(dev)
    state0 = {k: v.clone() for k, v in blk.state_dict().items()}
    xg_full = _run(blk, ei, ins, ups, list(range(G)))
    full = [p.grad.clone() for p in blk.parameters()]
    world = 2
    total = torch.zeros(sum(p.numel() for p in blk.parameters()), device=dev)
    xg_parts = {}
    for rank in range(world):
        blk.load_state_dict(state0)                               # every rank starts from the same buffers
        mine = dp.shard_graphs(G, rank, world)
        xg = _run(blk, ei, ins, ups, mine)
        bucket = dp.GradBucket(blk.parameters())
        bucket.pack()                                             # what the all-reduce would sum
        total += bucket.flat
        for j, g in enumerate(mine):
            xg_parts[g] = [t[j] for t in xg]
    off = 0
    floors = _floors(list(blk.named_parameters()), full)
    for (name, p), ref in zip(blk.named_parameters(), full):
        _close(total[off:off + p.numel()].view_as(p), ref, name, floors[name])
        off += p.numel()
    for g in range(G):                                            # input gradients are per graph: unchanged by the split
        for t_full, t_part in zip(xg_full, xg_parts[g]):
            _close(t_part, t_full[g], "input gradient of graph %d" % g)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, out):
    import torch.distributed as dist
    from pfs_neural_net_b200 import dp
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    blk, ei, ins, ups = _problem(dev)
    dp.broadcast_parameters(blk)
    state0 = {k: v.clone() for k, v in blk.state_dict().items()}
    _run(blk, ei, ins, ups, dp.shard_graphs(G, rank, world))
    bucket = dp.GradBucket(blk.parameters())
    bucket.all_reduce()
    reduced = [p.grad.clone() for p in blk.parameters()]
    ok = all(p.grad.data_ptr() == v.data_ptr() for p, v in zip(bucket.params, bucket.views))   # views, no copy back
    blk.load_state_dict(state0)
    _run(blk, ei, ins, ups, list(range(G)))
    named = list(blk.named_parameters())
    floors = _floors(named, [p.grad for _, p in named])
    for (name, p), r in zip(named, reduced):
        scale = max(p.grad.abs().max().item(), floors[name], 1e-30)
        ok &= (r - p.grad).abs().max().item() <= 2e-5 * scale
    out[rank] = bool(ok)
    dist.destroy_process_group()


def test_dp_two_gpus_nccl():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    import torch.multiprocessing as mp
    world = 2
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_nccl_worker, args=(world, _free_port(), out), nprocs=world, join=True)
        assert dict(out) == {0: True, 1: True}
