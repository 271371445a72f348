"""Training one graph whose fibres are sharded over the ranks (shard.fibre_sharded()): the sharded loss (per-rank records,
one exchange, a rank-order merge) against the fp64 oracle of the whole graph, its bitwise contracts (one rank = the
unsharded call, every rank agrees, run to run), its collectives and launches, the default noise, and 3 Adam steps of a
bf16 GNN on 2 ranks against the same steps on the whole graph.
With at least as many CUDA devices as ranks, every rank has its own GPU and NCCL; otherwise all ranks share cuda:0
and exchange through gloo, as in tests/test_gpu_wide_shard.py, so a 1-GPU box runs every test."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import block_oracle as bo
from oracle import loss_oracle as lo
from tests.util import golden_loss_cases

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _cases():
    return [c for c in golden_loss_cases() if c["time"].dtype == torch.float64]


def _bounds(S, world):
    """uneven fibre ranges: [0,1), [1,S/2), [S/2,S) for 3 ranks; equal halves for 2; everything for 1"""
    if world == 3:
        return [0, 1, S // 2, S]
    return [S * r // world for r in range(world + 1)]


def _kw(c):
    return dict(nfields=c["nfields"], total_time=c["total_time"], wutils=c["wutils"], wvar=c["wvar"])


def _loss_outputs(pl, time, class_info, S, T, kw, noise=None):
    """loss_from_times forward + backward on a leaf copy of `time`; every output the contracts name, on the CPU"""
    t = time.detach().clone().requires_grad_(True)
    loss, sc, n_prime, fibre_time, time2 = pl.loss_from_times(t, class_info, S, T, noise=noise, **kw)
    saved = loss.grad_fn.saved_tensors                     # time, noise, hours, counts, time2, fibre_time, class_mean, class_coef
    loss.backward()
    torch.cuda.synchronize()
    out = dict(loss=loss, scalars=sc, n_prime=n_prime, fibre_time=fibre_time, time2=time2, class_mean=saved[6],
               class_coef=saved[7], noise=saved[1], g_time=t.grad)
    return {k: v.detach().cpu() for k, v in out.items()}


def _golden_job(rank, world, dev, out):
    from pfs_neural_net_b200 import loss as pl, shard
    res = []
    # every graph is a partition of its own: its own group, so the cached shard sizes of one graph never answer for
    # another (rank 0 holds 1 fibre of every graph, the other ranks' counts change)
    groups = []
    for c in _cases():
        S, T = c["S"], c["T"]
        b = _bounds(S, world)
        f0, f1 = b[rank], b[rank + 1]
        time = c["time"].float().reshape(S, T)[f0:f1].reshape(-1).to(dev)
        noise = c["noise"].float().reshape(S, T)[f0:f1].reshape(-1).to(dev)
        ci = c["class_info"].float().to(dev)
        groups.append(dist.new_group(list(range(world))))
        with shard.fibre_sharded(groups[-1]):
            r = _loss_outputs(pl, time, ci, f1 - f0, T, _kw(c), noise)
            r2 = _loss_outputs(pl, time, ci, f1 - f0, T, _kw(c), noise)
        r["rerun_equal"] = all(torch.equal(r[k], r2[k]) for k in r)
        r["f0"], r["f1"] = f0, f1
        res.append(r)
    # the default noise: the whole graph's draw, this rank's slice -- bitwise the single-GPU draw
    S, T = 100, 7
    b = _bounds(S, world)
    f0, f1 = b[rank], b[rank + 1]
    g = torch.Generator().manual_seed(9)
    ci = torch.stack([0.5 + 3 * torch.rand(T, generator=g), 50 + 400 * torch.rand(T, generator=g)], 1).to(dev)
    full = (torch.rand(S * T, generator=g) * 6).to(dev)
    torch.manual_seed(7)
    single = _loss_outputs(pl, full, ci, S, T, {})["noise"]
    torch.manual_seed(7)
    groups.append(dist.new_group(list(range(world))))
    with shard.fibre_sharded(groups[-1]):
        mine = _loss_outputs(pl, full[f0 * T:f1 * T], ci, f1 - f0, T, {})["noise"]
    out[rank] = dict(cases=res, noise_equal=torch.equal(mine, single[f0 * T:f1 * T]))


def _one_rank_job(rank, world, dev, out):
    """one-rank group: the sharded loss is bitwise the unsharded call; collectives and launches per call"""
    from pfs_neural_net_b200 import _abi, loss as pl, shard
    lib = _abi.load_library()
    g = torch.Generator().manual_seed(4)
    cases = [(c["time"].float(), c["noise"].float(), c["class_info"].float(), c["S"], c["T"], _kw(c)) for c in _cases()]
    S, T = 700, 1100                                       # several row blocks, more classes than threads
    cases.append((torch.rand(S * T, generator=g) * 0.2, torch.rand(S * T, generator=g),
                  torch.stack([0.5 + 3 * torch.rand(T, generator=g), 50 + 400 * torch.rand(T, generator=g)], 1), S, T, {}))
    equal = []
    for time, noise, ci, S, T, kw in cases:
        time, noise, ci = time.to(dev), noise.to(dev), ci.to(dev)
        ref = _loss_outputs(pl, time, ci, S, T, kw, noise)
        with shard.fibre_sharded():
            r = _loss_outputs(pl, time, ci, S, T, kw, noise)
        equal.append({k: torch.equal(r[k], ref[k]) for k in r})
    time, noise, ci, S, T, kw = (x.to(dev) if torch.is_tensor(x) else x for x in cases[-1])
    with shard.fibre_sharded():
        _loss_outputs(pl, time, ci, S, T, kw, noise)       # fills the shard-size cache
        t = time.detach().clone().requires_grad_(True)
        torch.cuda.synchronize()
        shard.reset_traffic()
        n0 = lib.pfs_launch_count()
        loss = pl.loss_from_times(t, ci, S, T, noise=noise, **kw)[0]
        torch.cuda.synchronize()
        fwd = (shard.traffic()[0], lib.pfs_launch_count() - n0)
        shard.reset_traffic()
        n0 = lib.pfs_launch_count()
        loss.backward()
        torch.cuda.synchronize()
        bwd = (shard.traffic()[0], lib.pfs_launch_count() - n0)
    out[rank] = dict(equal=equal, fwd=fwd, bwd=bwd)


# ------------------------------------------------------------------------------------------------ end to end
S_E2E, T_E2E, F_E2E = 128, 64, 32


def _e2e_inputs():
    g = torch.Generator().manual_seed(11)
    class_info = torch.stack([0.5 + 3 * torch.rand(T_E2E, generator=g), 20 + 100 * torch.rand(T_E2E, generator=g)], 1)
    x_e = torch.randn(S_E2E * T_E2E, F_E2E, generator=g)
    torch.manual_seed(0)
    from pfs_neural_net_b200 import gnn as pg
    state = pg.GNN(B=2, Fdim=F_E2E, T=T_E2E, F_s=1, F_t=2).to(torch.bfloat16).state_dict()
    return class_info, x_e, state


def _graph(pg, f0, f1, class_info, x_e, dev):
    n = f1 - f0
    gr = pg.BipartiteData.__new__(pg.BipartiteData)
    gr.edge_index = bo.complete_bipartite(n, T_E2E).to(dev)
    gr.x_s = torch.arange(f0, f1, dtype=torch.float32).reshape(n, 1).bfloat16().to(dev)
    gr.x_t = class_info.bfloat16().to(dev)
    gr.x_e = x_e[f0 * T_E2E:f1 * T_E2E].bfloat16().to(dev)
    gr.x_u = torch.zeros(1, F_E2E).bfloat16().to(dev)
    gr.num_nodes = T_E2E
    return gr


def _train(pg, pl, state, graph, class_info, dev, steps=3):
    """the hand-written loop of reference src/train.py:136-141.  Returns per step [loss, totutils, variance, fibre
    penalty of the fibres the rank holds], the first step's parameter gradients and the final state."""
    model = pg.GNN(B=2, Fdim=F_E2E, T=T_E2E, F_s=1, F_t=2).to(torch.bfloat16)
    model.load_state_dict(state, strict=True)
    model = model.to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    sharp = torch.full((1,), 0.5, device=dev)
    terms, grads = [], None
    for i in range(steps):
        torch.manual_seed(100 + i)                       # the softfloor draw of step i, alike on every rank
        opt.zero_grad(set_to_none=True)
        out = model(graph)
        loss, totutils, _, _, fibre_time, _, variance = pl.loss_function(model, out, class_info, sharpness=sharp,
                                                                         finaloutput=True)
        loss.backward()
        if i == 0:
            # decoder_s (node_prediction) is not part of the loss: no gradient, on one device as on the shards
            grads = {k: p.grad.detach().float().cpu() for k, p in model.named_parameters() if p.grad is not None}
        ot = torch.from_numpy(fibre_time).double() - 42
        fpen = torch.where(ot > 0, ot, 0.1 * ot).pow(2).sum()
        terms.append(torch.stack([loss.detach().double().cpu(), totutils.detach().double().cpu(),
                                  variance.detach().double().cpu(), fpen]))
        opt.step()
    torch.cuda.synchronize()
    final = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
    return terms, grads, final


def _e2e_job(rank, world, dev, out):
    from pfs_neural_net_b200 import gnn as pg, loss as pl, shard
    from pfs_neural_net_b200.train_step import TrainStep
    class_info, x_e, state = _e2e_inputs()
    ci = class_info.to(dev)
    f0, f1 = S_E2E * rank // world, S_E2E * (rank + 1) // world
    local = _graph(pg, f0, f1, class_info, x_e, dev)
    res = {}
    with shard.fibre_sharded():
        res["scal"], res["grads"], res["final"] = _train(pg, pl, state, local, ci, dev)
        # TrainStep(use_graph=False) inside the scope: the loss of the hand-written loop's first step
        model = pg.GNN(B=2, Fdim=F_E2E, T=T_E2E, F_s=1, F_t=2).to(torch.bfloat16)
        model.load_state_dict(state, strict=True)
        model = model.to(dev).train()
        step = TrainStep(model, local, ci, torch.optim.Adam(model.parameters(), lr=1e-3), use_graph=False)
        torch.manual_seed(100)
        loss, _ = step(0.5)
        res["trainstep_loss"] = loss.detach().cpu()
        # refusals
        refused = {}
        try:
            TrainStep(model, local, ci, torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True), use_graph=True)
        except ValueError:
            refused["capture"] = True
        blk = pg.Block(10).to(dev).train()
        nf = f1 - f0
        try:
            blk((bo.complete_bipartite(nf, 12).to(dev), torch.randn(nf, 10, device=dev), torch.randn(12, 10, device=dev),
                 torch.randn(nf * 12, 10, device=dev), torch.randn(1, 10, device=dev)))
        except Exception as e:
            refused["fp32_block"] = type(e).__name__ == "PfsError"
        try:
            model.decoder_e.float()
            model.edge_prediction(torch.randn(nf * 12, F_E2E, device=dev))
        except Exception as e:
            refused["fp32_head"] = type(e).__name__ == "PfsError"
        try:
            pl.loss_from_times(torch.rand(2, nf * T_E2E, device=dev), ci, nf, T_E2E)
        except Exception as e:
            refused["batch"] = type(e).__name__ == "PfsError"
        res["refused"] = refused
    out[rank] = res
    if rank == 0:
        full = _graph(pg, 0, S_E2E, class_info, x_e, dev)
        out["full"] = dict(zip(("scal", "grads", "final"), _train(pg, pl, state, full, ci, dev)))


# ------------------------------------------------------------------------------------------------ harness
_JOBS = {"golden": _golden_job, "one_rank": _one_rank_job, "e2e": _e2e_job}


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


def test_golden_loss_sharded_over_three_ranks():
    world = 3
    out = _spawn("golden", world)
    for ci, c in enumerate(_cases()):
        S, T = c["S"], c["T"]
        t64 = c["time"].float().double().requires_grad_(True)
        r = lo.loss_terms(t64, c["noise"].float().double(), c["class_info"].float().double(), bo.complete_bipartite(S, T), S, T,
                          **_kw(c))
        r["loss"].backward()
        scale = max(abs(r["loss"].item()), c["wutils"] * abs(r["totutils"].item()), r["fiber_penalty"].item(),
                    r["variance"].item())
        for rank in range(world):
            m = out[rank]["cases"][ci]
            f0, f1 = m["f0"], m["f1"]
            sc = m["scalars"]
            assert m["rerun_equal"], (ci, rank)
            assert _rel(sc[1], r["totutils"]) < 1e-4, (ci, rank)
            assert _rel(m["n_prime"], r["n_prime"]) < 1e-4, (ci, rank)
            assert _rel(sc[4], r["variance"]) < 1e-4, (ci, rank)
            assert _rel(sc[2], r["class_penalty"]) < 1e-4 or r["class_penalty"].abs().item() < 1e-6
            assert _rel(sc[3], r["fiber_penalty"]) < 1e-4, (ci, rank)
            assert abs(m["loss"].item() - r["loss"].item()) < 1e-4 * scale, (ci, rank)
            # the local rows, judged on the scale of the whole graph's rows
            assert (m["fibre_time"].double() - r["fiber_time"][f0:f1].detach()).abs().max().item() \
                < 1e-4 * r["fiber_time"].abs().max().item(), (ci, rank)
            E = slice(f0 * T, f1 * T)
            assert (m["time2"].double() - r["time"][E].detach()).abs().max().item() < 1e-4 * r["time"].abs().max().item()
            assert (m["g_time"].double() - t64.grad[E]).abs().max().item() < 1e-4 * t64.grad.abs().max().item(), (ci, rank)
        for rank in range(1, world):                       # every rank holds bitwise the same global results
            for k in ("loss", "scalars", "n_prime", "class_mean", "class_coef"):
                assert torch.equal(out[rank]["cases"][ci][k], out[0]["cases"][ci][k]), (ci, rank, k)
    for rank in range(world):
        assert out[rank]["noise_equal"], rank


def test_one_rank_group_is_the_unsharded_call():
    out = _spawn("one_rank", 1)[0]
    for i, eq in enumerate(out["equal"]):
        assert all(eq.values()), (i, eq)
    assert out["fwd"] == (1, 5), out["fwd"]                 # one exchange, 5 launches
    assert out["bwd"] == (0, 1), out["bwd"]


def test_two_rank_training_matches_the_whole_graph():
    world = 2
    out = _spawn("e2e", world)
    full = out["full"]
    verbose = os.environ.get("PFS_SHARD_TEST_VERBOSE")
    for r in range(world):
        o = out[r]
        assert o["refused"] == dict(capture=True, fp32_block=True, fp32_head=True, batch=True), o["refused"]
        assert o["trainstep_loss"].item() == o["scal"][0][0].item(), (o["trainstep_loss"], o["scal"][0])
        for i, (a, b) in enumerate(zip(o["scal"], full["scal"])):
            # the loss is a difference of large terms: judged on the scale of its largest term (of the whole graph)
            scale = max(abs(b[0].item()), 2000.0 * abs(b[1].item()), abs(b[2].item()), abs(b[3].item()))
            err = abs(a[0].item() - b[0].item()) / scale
            if verbose:
                print("rank %d step %d loss %.6e vs %.6e  err %.3e" % (r, i, a[0].item(), b[0].item(), err))
            assert err < 2e-2, (r, i, err)
        g, gf = o["grads"], full["grads"]
        assert sorted(g) == sorted(gf) and any(k.startswith("encoder_s.") for k in gf)
        for k in gf:
            scale_key = k[:-4] + "weight" if k.endswith("bias") else k
            zero_grad = k.endswith(("edge_model.2.bias", "node_mlp_2.2.bias"))
            part_zero = k.endswith("s_model.node_mlp_1.2.bias")
            # the input of the global model's first layer is [u, mean of x_s, mean of x_t]: u = 0 here, and the means
            # pool BatchNorm outputs (zero mean over their rows, beta = 0 at init), so it is bf16 rounding noise and the
            # weight gradient dh^T input is ~1e-3 of the bias gradient dh (measured: |g_W| 1.2, |g_b| 867): judged on the
            # scale of the bias gradient, like the analytically zero biases on the weight's
            if k.endswith("global_model.0.weight"):
                scale_key, zero_grad = k[:-6] + "bias", True
            den = max(gf[k].abs().max().item(),
                      (1.0 if zero_grad else 0.1 if part_zero else 1e-3) * gf[scale_key].abs().max().item())
            err = (g[k] - gf[k]).abs().max().item() / den
            if verbose:
                a_, b_ = g[k].flatten().double(), gf[k].flatten().double()
                cos = torch.nn.functional.cosine_similarity(a_, b_, dim=0).item()
                print("rank %d %-40s err %.3e  |g| %.3e  |g_full| %.3e  cos %.4f" % (r, k, err, a_.norm(), b_.norm(), cos))
                continue
            assert err < 3e-2, (r, k, err)
    for k in out[0]["final"]:                               # every rank ends with the same model
        assert torch.equal(out[0]["final"][k], out[1]["final"][k]), k
