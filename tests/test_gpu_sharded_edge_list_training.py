"""Training an edge list whose fibres are sharded over the ranks (shard.fibre_sharded() with the `edge_ids` of
shard.partition_fibres): the per-rank edge-list records, one exchange and the rank-order merge against the fp64 oracle of
the whole edge list, its bitwise contracts (one rank = the unsharded edge-list call, every rank agrees, run to run), its
launches and collectives, the default noise, a graph whose rank-0 slab is canonical, and 3 Adam steps of a bf16 GNN on 2
ranks against the same steps on the whole graph.
With at least as many CUDA devices as ranks, every rank has its own GPU and NCCL; otherwise all ranks share cuda:0 and
exchange through gloo, as in tests/test_gpu_sharded_training.py, so a 1-GPU box runs every test."""
import os
import socket
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import block_oracle as bo
from tests import edge_loss_oracle as elo
from tests.test_gpu_edge_list_loss import edge_list

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _class_info(T, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([0.5 + 3 * torch.rand(T, generator=g), 50 + 400 * torch.rand(T, generator=g)], 1)


def _times(E, S, seed):
    g = torch.Generator().manual_seed(seed)
    return 2 * (42.0 * S / E) * torch.rand(E, generator=g), torch.rand(E, generator=g)


# (kind, S, T, p, dup): a shuffled sparse graph (fibre 1 and class T/2 without edges), a class-permuted complete graph, and
# long class segments with duplicate runs at T = 600
CASES = [("sparse", 300, 40, 0.1, 0.1), ("class", 64, 12, 1.0, 0.0), ("sparse", 40, 600, 0.5, 0.1)]


def _case(i):
    kind, S, T, p, dup = CASES[i]
    ei = edge_list(kind, S, T, seed=S + T, p=p, dup=dup)
    time, noise = _times(ei.shape[1], S, seed=i + 5)
    return ei, time, noise, _class_info(T, seed=T), S, T


def _bounds(S, world):
    """uneven fibre ranges: [0,1), [1,S/2), [S/2,S) for 3 ranks; equal parts otherwise (as shard.partition_fibres)"""
    if world == 3:
        return [0, 1, S // 2, S]
    return [S * r // world for r in range(world + 1)]


def _partition(ei, f0, f1):
    """shard.partition_fibres for the fibre range [f0, f1): local edge_index and the global positions of its edges"""
    keep = torch.nonzero((ei[0] >= f0) & (ei[0] < f1)).flatten()
    return torch.stack([ei[0][keep] - f0, ei[1][keep]]).contiguous(), keep


def _outputs(pl, time, ci, S, T, noise=None, edge_index=None, edge_ids=None):
    """loss_from_times forward + backward on a leaf copy of `time`; every output the contracts name, on the CPU"""
    t = time.detach().clone().requires_grad_(True)
    loss, sc, n_prime, fibre_time, time2 = pl.loss_from_times(t, ci, S, T, noise=noise, edge_index=edge_index,
                                                               edge_ids=edge_ids)
    saved = loss.grad_fn.saved_tensors        # time, noise, hours, counts, time2, fibre_time, class_mean, class_coef, cell_time
    loss.backward()
    torch.cuda.synchronize()
    out = dict(loss=loss, scalars=sc, n_prime=n_prime, fibre_time=fibre_time, time2=time2, class_mean=saved[6],
               class_coef=saved[7], noise=saved[1], g_time=t.grad)
    return {k: v.detach().cpu() for k, v in out.items()}


def _golden_job(rank, world, dev, out):
    from pfs_neural_net_b200 import loss as pl, shard
    res = []
    for i in range(len(CASES)):
        ei, time, noise, ci, S, T = _case(i)
        b = _bounds(S, world)
        f0, f1 = b[rank], b[rank + 1]
        local, keep = _partition(ei, f0, f1)
        assert local.shape[1] > 0, (i, rank)
        args = (time[keep].to(dev), ci.to(dev), f1 - f0, T)
        kw = dict(noise=noise[keep].to(dev), edge_index=local.to(dev), edge_ids=keep.to(dev))
        with shard.fibre_sharded(dist.new_group(list(range(world)))):     # a partition of its own: its own count cache
            r = _outputs(pl, *args, **kw)
            r2 = _outputs(pl, *args, **kw)
        r["rerun_equal"] = all(torch.equal(r[k], r2[k]) for k in r)
        r["keep"], r["f0"], r["f1"] = keep, f0, f1
        res.append(r)
    # the default noise: the whole edge list's draw, this rank's edges -- bitwise the single-GPU draw
    ei, time, _, ci, S, T = _case(0)
    b = _bounds(S, world)
    local, keep = _partition(ei, b[rank], b[rank + 1])
    torch.manual_seed(7)
    single = _outputs(pl, time.to(dev), ci.to(dev), S, T, edge_index=ei.to(dev))["noise"]
    torch.manual_seed(7)
    with shard.fibre_sharded(dist.new_group(list(range(world)))):
        mine = _outputs(pl, time[keep].to(dev), ci.to(dev), b[rank + 1] - b[rank], T, edge_index=local.to(dev),
                        edge_ids=keep.to(dev))["noise"]
    out[rank] = dict(cases=res, noise_equal=torch.equal(mine, single[keep]))


def _one_rank_job(rank, world, dev, out):
    """one-rank group: bitwise the unsharded edge-list call; launches and collectives per call"""
    from pfs_neural_net_b200 import _abi, loss as pl, shard
    lib = _abi.load_library()
    equal = []
    for i in range(len(CASES)):
        ei, time, noise, ci, S, T = _case(i)
        ei, time, noise, ci = ei.to(dev), time.to(dev), noise.to(dev), ci.to(dev)
        ref = _outputs(pl, time, ci, S, T, noise, edge_index=ei)
        ids = torch.arange(ei.shape[1], device=dev)
        with shard.fibre_sharded(dist.new_group([0])):
            r = _outputs(pl, time, ci, S, T, noise, edge_index=ei, edge_ids=ids)
            _outputs(pl, time, ci, S, T, noise, edge_index=ei, edge_ids=ids)       # counts, topology, edge_ids cached
            t = time.detach().clone().requires_grad_(True)
            torch.cuda.synchronize()
            shard.reset_traffic()
            n0 = lib.pfs_launch_count()
            loss = pl.loss_from_times(t, ci, S, T, noise=noise, edge_index=ei, edge_ids=ids)[0]
            torch.cuda.synchronize()
            fwd = (shard.traffic()[0], lib.pfs_launch_count() - n0)
            shard.reset_traffic()
            n0 = lib.pfs_launch_count()
            loss.backward()
            torch.cuda.synchronize()
            bwd = (shard.traffic()[0], lib.pfs_launch_count() - n0)
        equal.append(({k: torch.equal(r[k], ref[k]) for k in r}, fwd, bwd))
    out[rank] = equal


# a graph whose rank-0 slab (fibres [0, S/3)) is complete and in canonical order, the other fibres sparse
S_MIX, T_MIX = 90, 16


def _mixed_graph():
    g = torch.Generator().manual_seed(21)
    third = S_MIX // 3
    dense = bo.complete_bipartite(third, T_MIX)
    e = torch.nonzero(torch.rand((S_MIX - third) * T_MIX, generator=g) < 0.2).flatten() + third * T_MIX
    e = e[torch.randperm(e.numel(), generator=g)]
    return torch.cat([dense, torch.stack([e // T_MIX, e % T_MIX])], 1)


def _mixed_job(rank, world, dev, out):
    """loss_function with edge_ids takes the edge-list path on every rank, the canonical rank 0 included"""
    from pfs_neural_net_b200 import _abi, loss as pl, shard
    from pfs_neural_net_b200.topology import get_topology
    ei = _mixed_graph()
    time, noise = _times(ei.shape[1], S_MIX, seed=22)
    ci = _class_info(T_MIX, seed=23).to(dev)
    local, sl, keep = shard.partition_fibres(ei, S_MIX, world, rank)
    S = sl.stop - sl.start
    local, keep = local.to(dev), keep.to(dev)
    x = time[keep.cpu()].to(dev).reshape(-1, 1).requires_grad_(True)
    graph = types.SimpleNamespace(edge_index=local, x_e=x, x_t=ci, x_s=torch.zeros(S, 1, device=dev))
    times = types.SimpleNamespace(edge_prediction=lambda x_e, scale: x_e)      # the edge times are the inputs
    lib = _abi.load_library()
    with shard.fibre_sharded():
        lib.pfs_profile_enable(1)
        try:
            loss, util, _, n_prime, fibre_time, time2, variance = pl.loss_function(
                times, graph, ci, noise=noise[keep.cpu()].to(dev), finaloutput=True, edge_ids=keep)
            loss.backward()
            kernels = {k: v[0] for k, v in _abi.profile_report().items() if k.startswith("k_loss")}
        finally:
            lib.pfs_profile_enable(0)
    out[rank] = dict(canonical=get_topology(local, S, T_MIX).canonical, kernels=kernels, loss=loss.detach().cpu(),
                     util=util.detach().cpu(), n_prime=n_prime.detach().cpu(), fibre_time=torch.from_numpy(fibre_time),
                     time2=time2.detach().cpu(), variance=variance.detach().cpu(), g_time=x.grad.reshape(-1).cpu(),
                     keep=keep.cpu(), f0=sl.start, f1=sl.stop)


# ------------------------------------------------------------------------------------------------ end to end
S_E2E, T_E2E, F_E2E = 128, 64, 32


def _e2e_inputs():
    ei = edge_list("sparse", S_E2E, T_E2E, seed=31, p=0.3, dup=0.0, empty=False)
    g = torch.Generator().manual_seed(11)
    class_info = torch.stack([0.5 + 3 * torch.rand(T_E2E, generator=g), 20 + 100 * torch.rand(T_E2E, generator=g)], 1)
    x_e = torch.randn(ei.shape[1], F_E2E, generator=g)
    torch.manual_seed(0)
    from pfs_neural_net_b200 import gnn as pg
    state = pg.GNN(B=2, Fdim=F_E2E, T=T_E2E, F_s=1, F_t=2).to(torch.bfloat16).state_dict()
    return ei, class_info, x_e, state


def _graph(pg, ei, f0, f1, keep, class_info, x_e, dev):
    gr = pg.BipartiteData.__new__(pg.BipartiteData)
    gr.edge_index = ei.to(dev)
    gr.x_s = torch.arange(f0, f1, dtype=torch.float32).reshape(f1 - f0, 1).bfloat16().to(dev)
    gr.x_t = class_info.bfloat16().to(dev)
    gr.x_e = x_e[keep].bfloat16().to(dev)
    gr.x_u = torch.zeros(1, F_E2E).bfloat16().to(dev)
    gr.num_nodes = T_E2E
    return gr


def _train(pg, pl, state, graph, class_info, dev, edge_ids=None, perm=None, steps=3):
    """the hand-written loop of reference src/train.py:136-141.  Returns per step [loss, totutils, variance], the first
    step's parameter gradients and the final state.  `perm`: the graph is the whole edge list permuted by `perm`, and each
    edge gets the noise the unpermuted whole graph draws for it."""
    model = pg.GNN(B=2, Fdim=F_E2E, T=T_E2E, F_s=1, F_t=2).to(torch.bfloat16)
    model.load_state_dict(state, strict=True)
    model = model.to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    sharp = torch.full((1,), 0.5, device=dev)
    terms, grads = [], None
    for i in range(steps):
        torch.manual_seed(100 + i)                       # the softfloor draw of step i, alike on every rank
        noise = None if perm is None else torch.rand(perm.numel(), device=dev)[perm.to(dev)]
        opt.zero_grad(set_to_none=True)
        out = model(graph)
        loss, totutils, _, _, _, _, variance = pl.loss_function(model, out, class_info, sharpness=sharp, finaloutput=True,
                                                                edge_ids=edge_ids, noise=noise)
        loss.backward()
        if i == 0:
            grads = {k: p.grad.detach().float().cpu() for k, p in model.named_parameters() if p.grad is not None}
        terms.append(torch.stack([loss.detach().double().cpu(), totutils.detach().double().cpu(),
                                  variance.detach().double().cpu()]))
        opt.step()
    torch.cuda.synchronize()
    final = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
    return terms, grads, final


def _e2e_job(rank, world, dev, out):
    from pfs_neural_net_b200 import _abi, gnn as pg, loss as pl, shard
    from pfs_neural_net_b200.train_step import TrainStep
    ei, class_info, x_e, state = _e2e_inputs()
    ci = class_info.to(dev)
    local, sl, keep = shard.partition_fibres(ei, S_E2E, world, rank)
    graph = _graph(pg, local, sl.start, sl.stop, keep, class_info, x_e, dev)
    ids = keep.to(dev)
    res = {}
    with shard.fibre_sharded():
        res["scal"], res["grads"], res["final"] = _train(pg, pl, state, graph, ci, dev, edge_ids=ids)
        # TrainStep(use_graph=False, edge_ids=...) inside the scope: the loss of the hand-written loop's first step
        model = pg.GNN(B=2, Fdim=F_E2E, T=T_E2E, F_s=1, F_t=2).to(torch.bfloat16)
        model.load_state_dict(state, strict=True)
        model = model.to(dev).train()
        step = TrainStep(model, graph, ci, torch.optim.Adam(model.parameters(), lr=1e-3), use_graph=False, edge_ids=ids)
        torch.manual_seed(100)
        loss, _ = step(0.5)
        res["trainstep_loss"] = loss.detach().cpu()
        refused = {}
        try:                                                # the edge list without its edge ids
            pl.loss_function(model, model(graph), ci)
        except _abi.PfsError as e:
            refused["no_edge_ids"] = "canonical dense edge order" in str(e)
        try:
            pl.loss_function(model, model(graph), ci, edge_ids=ids[:-1])
        except _abi.PfsError as e:
            refused["length"] = "entries" in str(e)
    try:                                                    # outside the scope there is no shard
        pl.loss_function(model, model(graph), ci, edge_ids=ids)
    except _abi.PfsError as e:
        refused["outside"] = "fibre_sharded" in str(e)
    res["refused"] = refused
    out[rank] = res
    if rank == 0:
        full = _graph(pg, ei, 0, S_E2E, torch.arange(ei.shape[1]), class_info, x_e, dev)
        out["full"] = dict(zip(("scal", "grads", "final"), _train(pg, pl, state, full, ci, dev)))
        # the whole graph with its edge list permuted: the same function summed in another order, the yardstick of the
        # bf16 rounding a different reduction order brings
        perm = torch.randperm(ei.shape[1], generator=torch.Generator().manual_seed(5))
        full = _graph(pg, ei[:, perm], 0, S_E2E, perm, class_info, x_e, dev)
        out["perm"] = dict(zip(("scal", "grads", "final"), _train(pg, pl, state, full, ci, dev, perm=perm)))


# ------------------------------------------------------------------------------------------------ harness
_JOBS = {"golden": _golden_job, "one_rank": _one_rank_job, "mixed": _mixed_job, "e2e": _e2e_job}


def _worker(rank, world, port, out, job, ngpu):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank if ngpu >= world else 0)
    torch.cuda.set_device(dev)
    if ngpu >= world:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        _JOBS[job](rank, world, dev, out)
        torch.cuda.synchronize(dev)
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _spawn(job, world):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(world, _free_port(), out, job, torch.cuda.device_count()), nprocs=world, join=True)
        return dict(out)


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _oracle(time, noise, ci, ei, S, T):
    t64 = time.double().requires_grad_(True)
    r = elo.loss_terms_edges(t64, noise.double(), ci.double(), ei, S, T)
    r["loss"].backward()
    r["g_time"] = t64.grad
    r["scale"] = max(abs(r["loss"].item()), 2000.0 * abs(r["totutils"].item()), r["fiber_penalty"].item(),
                     r["variance"].item())
    return r


def _check_local_rows(m, r, keep, f0, f1):
    """the rank's fibre and edge rows, judged on the scale of the whole graph's rows"""
    assert (m["fibre_time"].double() - r["fiber_time"][f0:f1].detach()).abs().max().item() \
        < 1e-4 * r["fiber_time"].abs().max().item()
    assert (m["time2"].double() - r["time"][keep].detach()).abs().max().item() < 1e-4 * r["time"].abs().max().item()
    assert (m["g_time"].double() - r["g_time"][keep]).abs().max().item() < 1e-4 * r["g_time"].abs().max().item()


def test_sharded_edge_list_loss_over_three_ranks_matches_the_oracle():
    world = 3
    out = _spawn("golden", world)
    for i in range(len(CASES)):
        ei, time, noise, ci, S, T = _case(i)
        r = _oracle(time, noise, ci, ei, S, T)
        for rank in range(world):
            m = out[rank]["cases"][i]
            sc = m["scalars"]
            assert m["rerun_equal"], (i, rank)
            assert _rel(sc[1], r["totutils"]) < 1e-4 or r["totutils"].item() == 0.0, (i, rank)
            assert _rel(m["n_prime"], r["n_prime"]) < 1e-4, (i, rank)
            assert _rel(sc[4], r["variance"]) < 1e-4, (i, rank)
            assert _rel(sc[2], r["class_penalty"]) < 1e-4 or r["class_penalty"].abs().item() < 1e-6, (i, rank)
            assert _rel(sc[3], r["fiber_penalty"]) < 1e-4, (i, rank)
            assert abs(m["loss"].item() - r["loss"].item()) < 1e-4 * r["scale"], (i, rank)
            _check_local_rows(m, r, m["keep"], m["f0"], m["f1"])
        for rank in range(1, world):                       # every rank holds bitwise the same global results
            for k in ("loss", "scalars", "n_prime", "class_mean", "class_coef"):
                assert torch.equal(out[rank]["cases"][i][k], out[0]["cases"][i][k]), (i, rank, k)
    for rank in range(world):
        assert out[rank]["noise_equal"], rank


def test_one_rank_group_is_the_unsharded_edge_list_call():
    out = _spawn("one_rank", 1)[0]
    for i, (eq, fwd, bwd) in enumerate(out):
        assert all(eq.values()), (i, eq)
        assert fwd == (1, 5), (i, fwd)                     # one exchange; 4 launches + the merge
        assert bwd == (0, 1), (i, bwd)


def test_every_rank_takes_the_edge_list_path_when_one_slab_is_canonical():
    world = 3
    out = _spawn("mixed", world)
    assert out[0]["canonical"] and not out[1]["canonical"] and not out[2]["canonical"]
    ei = _mixed_graph()
    time, noise = _times(ei.shape[1], S_MIX, seed=22)
    r = _oracle(time, noise, _class_info(T_MIX, seed=23), ei, S_MIX, T_MIX)
    expect = {k: 1 for k in ("k_loss_list_edge_fwd", "k_loss_list_fibre_sums", "k_loss_list_class",
                             "k_loss_list_shard_record", "k_loss_shard_merge", "k_loss_list_edge_bwd")}
    for rank in range(world):
        m = out[rank]
        assert m["kernels"] == expect, (rank, m["kernels"])
        assert abs(m["loss"].item() - r["loss"].item()) < 1e-4 * r["scale"], rank
        assert _rel(m["util"], r["totutils"]) < 1e-4, rank
        assert _rel(m["n_prime"], r["n_prime"]) < 1e-4, rank
        assert _rel(m["variance"], r["variance"]) < 1e-4, rank
        _check_local_rows(m, r, m["keep"], m["f0"], m["f1"])
        assert torch.equal(m["loss"], out[0]["loss"]), rank


def test_two_rank_training_of_an_edge_list_matches_the_whole_graph():
    world = 2
    out = _spawn("e2e", world)
    full, perm = out["full"], out["perm"]
    verbose = os.environ.get("PFS_SHARD_TEST_VERBOSE")
    for r in range(world):
        o = out[r]
        assert o["refused"] == dict(no_edge_ids=True, length=True, outside=True), o["refused"]
        assert o["trainstep_loss"].item() == o["scal"][0][0].item(), (o["trainstep_loss"], o["scal"][0])
        for i, (a, b) in enumerate(zip(o["scal"], full["scal"])):
            # the loss is a difference of large terms: judged on the scale of its largest term (of the whole graph)
            scale = max(abs(b[0].item()), 2000.0 * abs(b[1].item()), abs(b[2].item()))
            assert abs(a[0].item() - b[0].item()) / scale < 2e-2, (r, i)
        g, gf = o["grads"], full["grads"]
        assert sorted(g) == sorted(gf) and any(k.startswith("encoder_s.") for k in gf)
        for k in gf:
            # the scale rules of tests/test_gpu_sharded_training.py: analytically zero biases are judged on their weight's
            # gradient, and the global model's first weight on its bias's
            scale_key = k[:-4] + "weight" if k.endswith("bias") else k
            zero_grad = k.endswith(("edge_model.2.bias", "node_mlp_2.2.bias"))
            part_zero = k.endswith("s_model.node_mlp_1.2.bias")
            if k.endswith("global_model.0.weight"):
                scale_key, zero_grad = k[:-6] + "bias", True
            den = max(gf[k].abs().max().item(),
                      (1.0 if zero_grad else 0.1 if part_zero else 1e-3) * gf[scale_key].abs().max().item())
            err = (g[k] - gf[k]).abs().max().item() / den
            err_perm = (perm["grads"][k] - gf[k]).abs().max().item() / den
            if verbose:
                print("rank %d %-40s err %.3e  permuted whole graph %.3e" % (r, k, err, err_perm))
                continue
            # bf16 sums in another order move the gradients too: the shards may differ from the whole graph by 3 %, or
            # by up to twice what the permuted whole graph differs by
            assert err < max(3e-2, 2 * err_perm), (r, k, err, err_perm)
    for k in out[0]["final"]:                               # every rank ends with the same model
        assert torch.equal(out[0]["final"][k], out[1]["final"][k]), k
