"""The training loss on a general edge list (loss_from_times(..., edge_index=...), loss_function on a non-canonical graph)
on the GPU:

  * against the fp64 oracle `tests/edge_loss_oracle.loss_terms_edges` at the loss tests' norm-wise 1e-4 (outputs and the gradient w.r.t. the edge
    times): class-permuted and shuffled complete graphs, sparse graphs with fibres and classes without edges and duplicate
    edges, T = 1, S = 2, T = 600 (fibres of more than 256 edges), and class segments long enough that duplicate runs cross
    the chunks of the class pass;
  * the determinism contract: a G = 4 batch is bitwise 4 single-graph calls, permuting the graphs permutes the results
    bitwise, and at the C5a size (100 000 x 512, 10 %) the results repeat bitwise; permuting the edge list changes them
    only within fp32 tolerance;
  * launches: 4 forward and 1 backward for G = 1 and G = 16; a canonical graph keeps the 5 launches of the dense kernels
    and its results;
  * loss_function through the model (fp32 Fdim 10, a collated batch, bf16 Fdim 16 on the wide time head), TrainStep
    eager against graph replay, and the refusal of a non-canonical graph inside shard.fibre_sharded()."""
import contextlib
import copy

import pytest
import torch
import torch.distributed as dist

from oracle import block_oracle as bo
from tests import edge_loss_oracle as elo
from tests.test_gpu_batched_training import _param_grads_match


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _class_info(T, G=None, seed=1):
    g = torch.Generator().manual_seed(seed)
    lead = () if G is None else (G,)
    return torch.stack([0.5 + 3 * torch.rand(lead + (T,), generator=g), 50 + 400 * torch.rand(lead + (T,), generator=g)], -1)


def edge_list(kind, S, T, seed=0, p=0.1, dup=0.1, empty=True):
    """[2, E] int64 (CPU).  "class": the complete graph, classes permuted within each fibre (like graphs/graph-0.pt);
    "shuffle": the complete graph in random order; "sparse": each pair an edge with probability p, a fraction `dup`
    of the edges listed again, with `empty` fibre 1 and class T // 2 without edges (when S > 2, T > 1), shuffled."""
    g = torch.Generator().manual_seed(seed)
    if kind == "class":
        perm = torch.cat([k * T + torch.randperm(T, generator=g) for k in range(S)])
        return bo.complete_bipartite(S, T)[:, perm]
    if kind == "shuffle":
        return bo.complete_bipartite(S, T)[:, torch.randperm(S * T, generator=g)]
    e = torch.nonzero(torch.rand(S * T, generator=g) < p).flatten()
    k, i = e // T, e % T
    keep = torch.ones_like(e, dtype=torch.bool)
    if empty and S > 2:
        keep &= k != 1
    if empty and T > 1:
        keep &= i != T // 2
    e = e[keep]
    e = torch.cat([e, e[torch.rand(e.numel(), generator=g) < dup]])
    e = e[torch.randperm(e.numel(), generator=g)]
    return torch.stack([e // T, e % T])


def _times(G, E, T, seed=2, mean_degree=None):
    g = torch.Generator().manual_seed(seed)
    scale = 42.0 / (mean_degree or T)                 # fibre times around TOTAL_TIME
    lead = () if G is None else (G,)
    return 2 * scale * torch.rand(lead + (E,), generator=g), torch.rand(lead + (E,), generator=g)


def _run(time, noise, ci, ei, S, T, dev):
    from pfs_neural_net_b200 import loss as pl
    t = time.to(dev).requires_grad_(True)
    out = pl.loss_from_times(t, ci.to(dev), S, T, noise=noise.to(dev), edge_index=ei.to(dev))
    out[0].sum().backward()
    return [o.detach() for o in out] + [t.grad]


def _check_oracle(res, time, noise, ci, ei, S, T):
    loss, sc, n_prime, fibre_time, time2, g_time = res
    t64 = time.double().requires_grad_(True)
    r = elo.loss_terms_edges(t64, noise.double(), ci.double(), ei, S, T)
    r["loss"].backward()
    assert _rel(sc[1], r["totutils"]) < 1e-4 or r["totutils"].item() == 0.0
    assert _rel(n_prime, r["n_prime"]) < 1e-4
    assert _rel(fibre_time, r["fiber_time"]) < 1e-4
    assert _rel(time2, r["time"]) < 1e-4
    assert _rel(sc[4], r["variance"]) < 1e-4
    assert _rel(sc[2], r["class_penalty"]) < 1e-4 or r["class_penalty"].abs().item() < 1e-6
    assert _rel(sc[3], r["fiber_penalty"]) < 1e-4
    scale = max(abs(r["loss"].item()), 2000.0 * abs(r["totutils"].item()), r["fiber_penalty"].item(), r["variance"].item())
    assert abs(loss.item() - r["loss"].item()) < 1e-4 * scale
    assert _rel(g_time, t64.grad) < 1e-4


CASES = [("class", 64, 12, 0.1), ("shuffle", 50, 20, 0.1), ("sparse", 300, 40, 0.1), ("sparse", 200, 1, 0.3),
         ("shuffle", 2, 1, 0.1), ("sparse", 2, 7, 0.6), ("shuffle", 40, 600, 0.1), ("sparse", 40, 600, 0.5),
         ("sparse", 20000, 3, 0.5)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,S,T,p", CASES)
def test_edge_list_loss_matches_the_fp64_oracle(kind, S, T, p):
    dev = _dev()
    ei = edge_list(kind, S, T, seed=S + T, p=p, dup=0.3 if S == 20000 else 0.1)
    E = ei.shape[1]
    ci = _class_info(T, seed=T)
    time, noise = _times(None, E, T, mean_degree=max(1.0, E / S))
    res = _run(time, noise, ci, ei, S, T, dev)
    assert res[3].shape == (S,) and res[4].shape == (E,) and res[5].shape == (E,) and res[2].shape == (T,)
    if kind == "sparse" and S > 2 and T > 1:
        assert res[3][1].item() == 0.0 and res[2][T // 2].item() == 0.0          # the fibre and the class without edges
    _check_oracle(res, time, noise, ci, ei, S, T)
    # [E, 1] times are one graph, like the canonical path's
    from pfs_neural_net_b200 import loss as pl
    again = pl.loss_from_times(time.to(dev).reshape(E, 1), ci.to(dev), S, T, noise=noise.to(dev), edge_index=ei.to(dev))
    assert torch.equal(again[0], res[0]) and torch.equal(again[4], res[4])


@pytest.mark.gpu
@pytest.mark.parametrize("tables", ["per_graph", "shared"])
def test_batched_edge_list_loss_is_bitwise_single_graph_calls(tables):
    dev = _dev()
    G, S, T = 4, 700, 30
    ei = edge_list("sparse", S, T, seed=5, p=0.2)
    E = ei.shape[1]
    ci = _class_info(T, G if tables == "per_graph" else None, seed=3)
    time, noise = _times(G, E, T, seed=4, mean_degree=E / S)
    batched = _run(time, noise, ci, ei, S, T, dev)
    assert batched[0].shape == (G,) and batched[4].shape == (G, E) and batched[3].shape == (G, S)
    single = [_run(time[g], noise[g], ci[g] if ci.dim() == 3 else ci, ei, S, T, dev) for g in range(G)]
    single = [torch.stack(k) for k in zip(*single)]
    names = ("loss", "scalars", "n_prime", "fibre_time", "time2", "time.grad")
    for n, a, b in zip(names, batched, single):
        assert torch.equal(a, b), n
    for n, a, b in zip(names, batched, _run(time, noise, ci, ei, S, T, dev)):
        assert torch.equal(a, b), n
    perm = torch.tensor([2, 0, 3, 1])
    permuted = _run(time[perm], noise[perm], ci[perm] if ci.dim() == 3 else ci, ei, S, T, dev)
    for n, a, b in zip(names, permuted, batched):
        assert torch.equal(a, b[perm.to(dev)]), n
    _check_oracle([x[1] for x in single], time[1], noise[1], ci[1] if ci.dim() == 3 else ci, ei, S, T)


@pytest.mark.gpu
def test_c5a_size_is_bitwise_repeatable_and_edge_order_changes_only_rounding():
    dev = _dev()
    S, T = 100000, 512
    gsp = torch.Generator().manual_seed(7)                     # bench.py --workload c5a's edge list
    e = torch.nonzero(torch.rand(S * T, generator=gsp) < 0.1).flatten()
    e = e[torch.randperm(e.numel(), generator=gsp)]
    ei = torch.stack([e // T, e % T]).to(dev)
    E = ei.shape[1]
    ci = _class_info(T, seed=11)
    time, noise = _times(None, E, T, seed=12, mean_degree=E / S)
    a = _run(time, noise, ci, ei, S, T, dev)
    b = _run(time, noise, ci, ei, S, T, dev)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    perm = torch.randperm(E, generator=torch.Generator().manual_seed(13))
    c = _run(time[perm], noise[perm], ci, ei[:, perm.to(dev)], S, T, dev)
    pd = perm.to(dev)
    assert torch.equal(c[4], a[4][pd])                          # per-edge arithmetic does not depend on the order
    for x, y in ((c[1][1:5], a[1][1:5]), (c[2], a[2]), (c[3], a[3]), (c[5], a[5][pd])):
        assert _rel(x, y) < 1e-4
    scale = max(abs(a[0].item()), 2000.0 * abs(a[1][1].item()), a[1][3].item(), a[1][4].item())
    assert abs(c[0].item() - a[0].item()) < 1e-5 * scale


@pytest.mark.gpu
def test_launch_counts():
    from pfs_neural_net_b200 import _abi, loss as pl
    dev = _dev()
    lib = _abi.load_library()
    S, T = 300, 40
    ei = edge_list("sparse", S, T, seed=1).to(dev)
    E = ei.shape[1]
    for G in (1, 16):
        time, noise = _times(G, E, T)
        ci = _class_info(T, G).to(dev)
        for _ in range(2):                                      # the second call finds the topology cached
            t = time.to(dev).requires_grad_(True)
            nz = noise.to(dev)
            torch.cuda.synchronize()
            n0 = lib.pfs_launch_count()
            loss = pl.loss_from_times(t, ci, S, T, noise=nz, edge_index=ei)[0]
            torch.cuda.synchronize()
            n1 = lib.pfs_launch_count()
            loss.sum().backward()
            torch.cuda.synchronize()
            n2 = lib.pfs_launch_count()
        assert (n1 - n0, n2 - n1) == (4, 1), (G, n1 - n0, n2 - n1)
    # a canonical graph: loss_function runs the dense kernels, one launch each, and none of the edge-list kernels
    from pfs_neural_net_b200 import gnn as pg
    torch.manual_seed(0)
    Sc, Tc, F = 64, 12, 10
    model = pg.GNN(B=1, Fdim=F, T=Tc, F_s=1, F_t=2).to(dev).train()
    g = torch.Generator().manual_seed(1)
    ci = _class_info(Tc).to(dev)
    graph = pg.BipartiteData(bo.complete_bipartite(Sc, Tc), torch.rand(Sc, 1, generator=g), ci.cpu(),
                             2 + 8 * torch.rand(Sc * Tc, F, generator=g), torch.zeros(1, F))
    out = model(graph)
    noise = torch.rand(Sc * Tc, device=dev)
    torch.cuda.synchronize()
    lib.pfs_profile_enable(1)
    try:
        loss, _ = pl.loss_function(model, out, ci, noise=noise)
        loss.backward()
        kernels = _abi.profile_report()
    finally:
        lib.pfs_profile_enable(0)
    loss_kernels = {k: v[0] for k, v in kernels.items() if k.startswith("k_loss")}
    assert loss_kernels == {k: 1 for k in ("k_loss_edge_fwd", "k_loss_fibre_sums", "k_loss_class_partial", "k_loss_scalars",
                                           "k_loss_edge_bwd")}, kernels
    time = model.edge_prediction(out.x_e, scale=42.0 / Tc).squeeze(-1).detach()
    assert torch.equal(loss.detach(), pl.loss_from_times(time, ci, Sc, Tc, noise=noise)[0])


def _sparse_graph(S, T, F, ei, seed=1, dtype=torch.float32):
    from pfs_neural_net_b200 import gnn as pg
    g = torch.Generator().manual_seed(seed)
    return pg.BipartiteData(ei, torch.arange(S, dtype=torch.float32).reshape(-1, 1) / S + torch.rand(S, 1, generator=g),
                            _class_info(T, seed=seed + 100), (2 + 8 * torch.rand(ei.shape[1], F, generator=g)).to(dtype),
                            torch.zeros(1, F))


@pytest.mark.gpu
def test_loss_function_through_the_model_on_a_sparse_graph():
    """parameter gradients against the same model with the loss computed by the fp64 oracle"""
    from pfs_neural_net_b200 import gnn as pg, loss as pl
    dev = _dev()
    S, T, F = 200, 24, 10
    ei = edge_list("sparse", S, T, seed=3, p=0.3, empty=False)
    graph = _sparse_graph(S, T, F, ei)
    ci = graph.x_t.to(dev)
    torch.manual_seed(0)
    model = pg.GNN(B=2, Fdim=F, T=T, F_s=1, F_t=2).to(dev).train()
    ref = copy.deepcopy(model)
    noise = torch.rand(ei.shape[1], generator=torch.Generator().manual_seed(4)).to(dev)
    loss, util = pl.loss_function(model, model(graph), ci, noise=noise)
    loss.backward()
    out = ref(graph)
    t = ref.edge_prediction(out.x_e, scale=42.0 / T).squeeze(-1)
    r = elo.loss_terms_edges(t.double(), noise.double(), ci.double(), ei.to(dev), S, T)
    r["loss"].backward()
    scale = max(abs(r["loss"].item()), 2000.0 * abs(r["totutils"].item()))
    assert abs(loss.item() - r["loss"].item()) < 1e-4 * scale
    assert _rel(util, r["totutils"]) < 1e-4
    _param_grads_match(model, ref)


@pytest.mark.gpu
def test_loss_function_on_a_collated_sparse_batch_against_the_oracle():
    """the summed loss of a collated batch: parameter gradients against the same model with the G losses computed by the
    fp64 oracle (the same batched forward, so both see bitwise the same edge times)"""
    from pfs_neural_net_b200 import gnn as pg, loss as pl
    dev = _dev()
    G, S, T, F = 3, 150, 16, 10
    ei = edge_list("sparse", S, T, seed=6, p=0.3, empty=False)
    graphs = [_sparse_graph(S, T, F, ei, seed=10 + k) for k in range(G)]
    ci = torch.stack([gr.x_t for gr in graphs]).to(dev)
    noise = torch.rand(G, ei.shape[1], generator=torch.Generator().manual_seed(9)).to(dev)
    batch = pg.Loader.collate(graphs)
    torch.manual_seed(0)
    model = pg.GNN(B=2, Fdim=F, T=T, F_s=1, F_t=2).to(dev).train()
    ref = copy.deepcopy(model)
    loss, util = pl.loss_function(model, model(batch), ci, noise=noise)
    loss.backward()
    t = ref.edge_prediction(ref(batch).x_e, scale=42.0 / T).squeeze(-1)
    rs = [elo.loss_terms_edges(t[g].double(), noise[g].double(), ci[g].double(), ei.to(dev), S, T) for g in range(G)]
    sum(r["loss"] for r in rs).backward()
    assert util.shape == (G,)
    assert _rel(util, torch.stack([r["totutils"] for r in rs])) < 1e-4
    scale = max(max(abs(r["loss"].item()) for r in rs), 2000.0 * util.max().item())
    assert abs(loss.item() - sum(r["loss"].item() for r in rs)) < 1e-4 * G * scale
    _param_grads_match(model, ref)


@pytest.mark.gpu
def test_loss_function_bf16_wide_time_head_on_a_sparse_graph():
    from pfs_neural_net_b200 import gnn as pg, loss as pl
    dev = _dev()
    S, T, F = 120, 16, 16
    ei = edge_list("sparse", S, T, seed=8, p=0.4, dup=0.0, empty=False)
    graph = _sparse_graph(S, T, F, ei, dtype=torch.bfloat16)
    graph.x_s, graph.x_t, graph.x_u = graph.x_s.bfloat16(), graph.x_t.bfloat16(), graph.x_u.bfloat16()
    ci = _class_info(T, seed=108).to(dev)
    torch.manual_seed(0)
    model = pg.GNN(B=1, Fdim=F, T=T, F_s=1, F_t=2).to(torch.bfloat16).to(dev).train()
    ref = copy.deepcopy(model)
    noise = torch.rand(ei.shape[1], generator=torch.Generator().manual_seed(4)).to(dev)
    loss, util = pl.loss_function(model, model(graph), ci, noise=noise)
    loss.backward()
    out = ref(graph)
    t = ref.edge_prediction(out.x_e, scale=42.0 / T).squeeze(-1)
    r = elo.loss_terms_edges(t.double(), noise.double(), ci.double(), ei.to(dev), S, T)
    r["loss"].backward()
    scale = max(abs(r["loss"].item()), 2000.0 * abs(r["totutils"].item()))
    assert abs(loss.item() - r["loss"].item()) < 1e-4 * scale
    for (n, p), (_, q) in zip(model.named_parameters(), ref.named_parameters()):
        if q.grad is None:
            continue
        a, b = p.grad.double(), q.grad.double()
        assert (a - b).norm().item() <= 2e-2 * max(b.norm().item(), 1e-6), n     # upstream gradient rounded to bf16


@pytest.mark.gpu
def test_train_step_on_a_sparse_graph_replays_like_eager():
    """3 Adam steps eager against graph replay, then load() of a second graph with the same edge_index"""
    from pfs_neural_net_b200 import gnn as pg
    from pfs_neural_net_b200.train_step import TrainStep
    dev = _dev()
    S, T, F = 300, 20, 10
    ei = edge_list("sparse", S, T, seed=2, p=0.3, empty=False).to(dev)
    runs = []
    for use_graph in (False, True):
        a, b = _sparse_graph(S, T, F, ei, seed=1), _sparse_graph(S, T, F, ei, seed=2)
        for gr in (a, b):
            gr.edge_index = ei
        ci_a, ci_b = a.x_t.clone(), b.x_t.clone()
        torch.manual_seed(0)
        model = pg.GNN(B=2, Fdim=F, T=T, F_s=1, F_t=2).to(dev).train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
        step = TrainStep(model, a, ci_a, opt, use_graph=use_graph, warmup=2)
        out = []
        for i in range(3):
            torch.manual_seed(100 + i)
            loss, util = step(0.5 + 0.1 * i)
            out.append((float(loss), float(util)))
        if use_graph:
            step.load(b, ci_b)
        else:
            step = TrainStep(model, b, ci_b, opt, use_graph=False)
        torch.manual_seed(200)
        loss, util = step(0.8)
        out.append((float(loss), float(util)))
        runs.append((out, {k: v.clone() for k, v in model.state_dict().items()}))
    (la, sa), (lb, sb) = runs
    for (x, ux), (y, uy) in zip(la, lb):
        assert abs(x - y) <= 1e-5 * max(1.0, abs(x)), (la, lb)
        assert abs(ux - uy) <= 1e-6 * max(1.0, abs(ux)), (la, lb)
    assert abs(la[3][0] - la[2][0]) > 1e-4 * abs(la[2][0])
    for k in sa:
        assert torch.allclose(sa[k].float(), sb[k].float(), rtol=1e-5, atol=1e-6), k


@contextlib.contextmanager
def _one_rank_group():
    dist.init_process_group("gloo", store=dist.HashStore(), rank=0, world_size=1)
    try:
        yield
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_a_non_canonical_graph_is_refused_inside_fibre_sharded():
    from pfs_neural_net_b200 import _abi, gnn as pg, loss as pl, shard
    dev = _dev()
    S, T, F = 40, 12, 32
    ei = edge_list("class", S, T, seed=1)
    graph = _sparse_graph(S, T, F, ei)
    graph.edge_index = graph.edge_index.to(dev)
    model = pg.GNN(B=1, Fdim=F, T=T, F_s=1, F_t=2).to(dev)
    with _one_rank_group(), shard.fibre_sharded():
        with pytest.raises(_abi.PfsError, match="canonical dense edge order"):
            pl.loss_function(model, graph, graph.x_t.to(dev))


def test_edge_list_shape_errors_are_reported_on_the_host():
    """wrong time, noise or class-table shapes raise before any device work (time on the CPU, so no GPU is needed
    when the edge list is never read)"""
    from pfs_neural_net_b200 import _abi, loss as _l
    S, T, E = 8, 4, 20
    edges = dict(E=E)
    time, noise = _times(3, E, T)
    for ci, nz, what in ((_class_info(T, 4), noise, "class_info"), (_class_info(T + 1), noise, "class_info"),
                         (_class_info(T, 3), noise[:, :-1], "noise"), (_class_info(T, 3), noise[:2], "noise")):
        with pytest.raises(_abi.PfsError, match=what):
            _l._batched_loss(time, ci, S, T, 10, {}, nz, edges)
    with pytest.raises(_abi.PfsError, match="batch of edge times"):
        _l._batched_loss(time[:, :-1], _class_info(T), S, T, 10, {}, noise, edges)
