"""Fibre-range sharding of ONE large graph over the ranks of a process group (BASELINE config C4;
SURVEY.md section 8e "Fibre-range edge sharding").

Rank r owns a contiguous range of fibres and all their edges (the dense layout is fibre-major, so
that is a contiguous slab of x_e); x_t, u and the weights are replicated.  Every fibre-side
statistic is then local, and the layer needs one exchange per reduction over "all edges / all
fibres": the BatchNorm statistics of the edge and source models, the class aggregate of the target
model (the tensor the north star names), the class-table gradients and the fibre-local parts of the
weight gradients.  They are all small fp32 tensors, all-reduced (sum) over NCCL/NVLink on the
compute stream; with no group active every function here is the identity.

Usage:   with shard.fibre_sharded(group):  y = block((edge_index_local, x_s_local, x_t, x_e_local, u))
"""
import contextlib

import torch
import torch.distributed as dist

_state = {"group": None, "active": False, "replicated": 0, "bytes": 0, "calls": 0, "counts": {}}


def active():
    return _state["active"] and _state["replicated"] == 0


@contextlib.contextmanager
def fibre_sharded(group=None):
    """Run the enclosed module calls (forward AND the backward they record) as one fibre shard."""
    if not dist.is_initialized():
        raise RuntimeError("fibre_sharded() needs torch.distributed to be initialised")
    prev = (_state["group"], _state["active"])
    _state["group"], _state["active"] = group, True
    try:
        yield
    finally:
        _state["group"], _state["active"] = prev


@contextlib.contextmanager
def replicated():
    """Rows that every shard holds in full (classes, the global row): reductions stay local."""
    _state["replicated"] += 1
    try:
        yield
    finally:
        _state["replicated"] -= 1


def group_key():
    """Hashable identity of the active process group (for per-partition caches)."""
    return id(_state["group"]) if _state["active"] else None


def world_size():
    return dist.get_world_size(_state["group"]) if _state["active"] else 1


def rank():
    return dist.get_rank(_state["group"]) if _state["active"] else 0


def allreduce_sum(t):
    """Sum of a (small, fp32) tensor over the shards; identity when not sharded."""
    if not active():
        return t
    t = t.contiguous()
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=_state["group"])
    _state["bytes"] += t.numel() * t.element_size()
    _state["calls"] += 1
    return t


def allreduce_packed(tensors):
    """Sum several small fp32 tensors over the shards with ONE collective (they travel as one flat buffer);
    returns new tensors of the same shapes.  Identity when not sharded."""
    if not active():
        return list(tensors)
    tensors = [t.contiguous() for t in tensors]
    if len(tensors) == 1:
        return [allreduce_sum(tensors[0])]
    flat = torch.cat([t.reshape(-1).float() for t in tensors])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=_state["group"])
    _state["bytes"] += flat.numel() * 4
    _state["calls"] += 1
    out, o = [], 0
    for t in tensors:
        out.append(flat[o:o + t.numel()].view(t.shape).to(t.dtype))
        o += t.numel()
    return out


def exchange_rows(row):
    """Every shard's `row` (a 1-D tensor of n values), stacked in rank order as a [world, n] tensor of its dtype that is
    bitwise the same on every rank: each rank fills its own row of a zero buffer and ONE all-reduce (sum) completes it --
    adding zeros is exact, and all-reduce is the one collective every backend offers for CUDA tensors.  Not sharded:
    the row as a [1, n] tensor."""
    row = row.reshape(-1)
    if not active():
        return row.reshape(1, -1)
    world = dist.get_world_size(_state["group"])
    buf = torch.zeros(world, row.numel(), dtype=row.dtype, device=row.device)
    buf[dist.get_rank(_state["group"])] = row
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=_state["group"])
    _state["bytes"] += buf.numel() * buf.element_size()
    _state["calls"] += 1
    return buf


def shard_counts(n_local, kind=None):
    """Per-shard values of a host-known integer (rows or edges of this shard), as a tuple indexed by rank.  The
    exchange (the only host synchronisation of the sharded path) runs ONCE per distinct local value inside a
    fibre_sharded() scope family: shard sizes are properties of the partition, not of the step.  The cache is keyed by
    (group, local value), and a miss is a collective, so all ranks must miss together: run a partition with other shard
    sizes (another graph) in a group of its own when some rank's local value could repeat an earlier one.
    `kind` (e.g. "edges") counts under a cache key of its own, so a rank whose edge count equals its fibre count (or
    any count of another kind cached earlier) still misses together with the other ranks."""
    if not active():
        return (int(n_local),)
    key = (id(_state["group"]), int(n_local)) if kind is None else (id(_state["group"]), kind, int(n_local))
    hit = _state["counts"].get(key)
    if hit is None:
        world, rank = dist.get_world_size(_state["group"]), dist.get_rank(_state["group"])
        slots = torch.zeros(world, dtype=torch.int64)
        slots[rank] = int(n_local)
        if dist.get_backend(_state["group"]) == "nccl":
            slots = slots.cuda()
        dist.all_reduce(slots, op=dist.ReduceOp.SUM, group=_state["group"])      # gather as a sum of one-hot rows
        hit = tuple(int(v) for v in slots.tolist())
        _state["counts"][key] = hit
        _state["calls"] += 1
        _state["bytes"] += 8 * world
    return hit


def total_count(n_local, kind=None):
    """Sum of a per-shard integer over the shards (host int, cached like shard_counts, under `kind`)."""
    return sum(shard_counts(n_local, kind))


def allreduce_moments(n, mean, m2):
    """Combine per-shard (count, mean, sum of squared deviations) into the global ones (Chan et al.);
    returns (n_total as float, mean, m2).  ONE collective and no host synchronisation per call: the shards' counts
    are cached (shard_counts), the (mean, M2) pairs are all-gathered and merged locally in rank order, so every
    rank computes bit-identical results."""
    if not active():
        return n, mean, m2
    counts = shard_counts(int(n))
    F = mean.numel()
    allp = exchange_rows(torch.cat([mean.reshape(-1), m2.reshape(-1)]).float()).double()       # [world, 2F]
    cnt = torch.tensor(counts, dtype=torch.float64, device=mean.device)[:, None]
    n_tot = float(sum(counts))
    # sum of n, n*mean, and m2 + n*mean^2 would cancel; merge the moments exactly:
    # M2 = sum_r [ m2_r + n_r (mean_r - mean)^2 ]
    g_mean = (allp[:, :F] * cnt).sum(0) / n_tot
    dev = (allp[:, F:] + cnt * (allp[:, :F] - g_mean) ** 2).sum(0)
    return n_tot, g_mean.float().view(mean.shape), dev.float().view(m2.shape)


def partition_fibres(edge_index, S, world, rank):
    """Fibre-range partition of a GENERAL edge list (BASELINE config C5 sharded; the dense C4 graph is a slab of the
    canonical order and needs no index work).  Rank r owns the fibres [S*r/world, S*(r+1)/world) and every edge
    whose source lies in that range, in the order the edge list has them.
    Returns (local edge_index [2, E_r] with fibres renumbered from 0, fibre slice, positions of the kept edges in
    the global edge list -- use them to slice x_e / to scatter results back, and pass them as the `edge_ids` of
    loss.loss_function / TrainStep to train the sharded edge list)."""
    f0, f1 = (S * rank) // world, (S * (rank + 1)) // world
    src = edge_index[0]
    keep = torch.nonzero((src >= f0) & (src < f1)).flatten()
    local = torch.stack([src[keep] - f0, edge_index[1][keep]]).contiguous()
    return local, slice(f0, f1), keep


def traffic():
    """(collective calls, bytes) since the last reset -- bench.py reports them."""
    return _state["calls"], _state["bytes"]


def reset_traffic():
    _state["calls"] = _state["bytes"] = 0
