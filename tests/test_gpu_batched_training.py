"""The training loss and the training step over a leading graph dimension (G graphs that share one edge_index).

  * loss_from_times on [G, E] edge times against the fp64 oracle, graph by graph (per-graph and shared class tables,
    and 300 classes for the class-chunk loop of k_loss_class_partial);
  * the determinism contract: a batched call, forward and gradient, is bitwise G single-graph calls, run-to-run
    identical, and permuting the graphs permutes the results bitwise; five launches per forward + backward whatever G;
  * loss_function on a collated batch: parameter gradients of the summed loss equal those of the graphs run one after
    the other ("sum"), 1/G of that ("mean");
  * TrainStep on a batch: eager == graph replay, construction changes nothing, an epoch driven by load() and replay
    matches eager steps on the same batches, load() refuses another topology or other shapes.
Shape errors are checked on the host, so those tests run without a GPU."""
import copy
import os
import subprocess
import sys

import pytest
import torch

from oracle import block_oracle as bo
from oracle import loss_oracle as lo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _class_info(T, G=None, seed=1):
    """[T, 2] (G None) or [G, T, 2]: hours in [0.5, 3.5), galaxy counts in [50, 450) as in the loss tests."""
    g = torch.Generator().manual_seed(seed)
    lead = () if G is None else (G,)
    return torch.stack([0.5 + 3 * torch.rand(lead + (T,), generator=g), 50 + 400 * torch.rand(lead + (T,), generator=g)], -1)


def _times(G, S, T, seed=2):
    g = torch.Generator().manual_seed(seed)
    scale = 42.0 / T                                   # the time head's scale: fibre times around TOTAL_TIME
    return 2 * scale * torch.rand(G, S * T, generator=g), torch.rand(G, S * T, generator=g)


def _batched(time, noise, ci, S, T, dev):
    from pfs_neural_net_b200 import loss as pl
    t = time.to(dev).requires_grad_(True)
    out = pl.loss_from_times(t, ci.to(dev), S, T, noise=noise.to(dev))
    out[0].sum().backward()
    return [o.detach() for o in out] + [t.grad]


def _single(time, noise, ci, S, T, dev):
    """the same graphs one call each: results stacked along a leading G"""
    from pfs_neural_net_b200 import loss as pl
    outs = []
    for g in range(time.shape[0]):
        t = time[g].to(dev).requires_grad_(True)
        out = pl.loss_from_times(t, (ci[g] if ci.dim() == 3 else ci).to(dev), S, T, noise=noise[g].to(dev))
        out[0].backward()
        outs.append([o.detach() for o in out] + [t.grad])
    return [torch.stack(k) for k in zip(*outs)]


@pytest.mark.gpu
@pytest.mark.parametrize("T,tables", [(12, "per_graph"), (12, "shared"), (300, "per_graph")])
def test_batched_loss_matches_the_oracle_graph_by_graph(T, tables):
    dev = _dev()
    G, S = 5, 64
    ci = _class_info(T, G if tables == "per_graph" else None)
    time, noise = _times(G, S, T)
    loss, sc, n_prime, fibre_time, time2, g_time = _batched(time, noise, ci, S, T, dev)
    assert loss.shape == (G,) and sc.shape == (G, 8) and n_prime.shape == (G, T) and fibre_time.shape == (G, S)
    assert time2.shape == (G, S * T) and g_time.shape == (G, S * T)
    ei = bo.complete_bipartite(S, T)
    for g in range(G):
        t64 = time[g].double().requires_grad_(True)
        r = lo.loss_terms(t64, noise[g].double(), (ci[g] if ci.dim() == 3 else ci).double(), ei, S, T)
        r["loss"].backward()
        assert _rel(sc[g, 1], r["totutils"]) < 1e-4, g
        assert _rel(n_prime[g], r["n_prime"]) < 1e-4, g
        assert _rel(fibre_time[g], r["fiber_time"]) < 1e-4, g
        assert _rel(time2[g], r["time"]) < 1e-4, g
        assert _rel(sc[g, 4], r["variance"]) < 1e-4, g
        assert _rel(sc[g, 2], r["class_penalty"]) < 1e-4 or r["class_penalty"].abs().item() < 1e-6, g
        assert _rel(sc[g, 3], r["fiber_penalty"]) < 1e-4, g
        scale = max(abs(r["loss"].item()), 2000.0 * abs(r["totutils"].item()), r["fiber_penalty"].item(), r["variance"].item())
        assert abs(loss[g].item() - r["loss"].item()) < 1e-4 * scale, g
        assert _rel(g_time[g], t64.grad) < 1e-4, g


@pytest.mark.gpu
@pytest.mark.parametrize("tables", ["per_graph", "shared"])
def test_batched_loss_is_bitwise_single_graph_calls(tables):
    """600 fibres: three row blocks per graph in k_loss_class_partial"""
    dev = _dev()
    G, S, T = 6, 600, 12
    ci = _class_info(T, G if tables == "per_graph" else None, seed=3)
    time, noise = _times(G, S, T, seed=4)
    batched = _batched(time, noise, ci, S, T, dev)
    single = _single(time, noise, ci, S, T, dev)
    names = ("loss", "scalars", "n_prime", "fibre_time", "time2", "time.grad")
    for n, a, b in zip(names, batched, single):
        assert torch.equal(a, b), n
    for n, a, b in zip(names, batched, _batched(time, noise, ci, S, T, dev)):      # run to run
        assert torch.equal(a, b), n
    perm = torch.tensor([4, 1, 5, 0, 3, 2])
    permuted = _batched(time[perm], noise[perm], ci[perm] if ci.dim() == 3 else ci, S, T, dev)
    for n, a, b in zip(names, permuted, batched):
        assert torch.equal(a, b[perm.to(dev)]), n


@pytest.mark.gpu
def test_loss_launches_do_not_grow_with_the_batch():
    from pfs_neural_net_b200 import _abi
    dev = _dev()
    lib = _abi.load_library()
    S, T = 64, 12
    counts = {}
    for G in (1, 16):
        time, noise = _times(G, S, T)
        _batched(time, noise, _class_info(T, G), S, T, dev)              # warm-up
        torch.cuda.synchronize()
        n0 = lib.pfs_launch_count()
        _batched(time, noise, _class_info(T, G), S, T, dev)
        torch.cuda.synchronize()
        counts[G] = lib.pfs_launch_count() - n0
    assert counts[1] == counts[16] == 5, counts


def _graphs(G, S, T, F, seed=1):
    from pfs_neural_net_b200 import gnn as pg
    g = torch.Generator().manual_seed(seed)
    ei = bo.complete_bipartite(S, T)
    return [pg.BipartiteData(ei, torch.arange(S, dtype=torch.float32).reshape(-1, 1) + torch.rand(S, 1, generator=g),
                             _class_info(T, seed=seed * 100 + k), 2 + 8 * torch.rand(S * T, F, generator=g),
                             torch.zeros(1, F)) for k in range(G)]


def _param_grads_match(model, ref, factor=1.0):
    """the tolerance of tests/test_gpu_parity.py::test_loader_collate_batches_graphs_like_sequential_runs, with its rule
    for analytically zero gradients applied to both parameters of a layer: a layer's weight and bias are judged on the
    larger of their two gradient scales.  A bias in front of a train-mode BatchNorm has zero gradient, and so has the
    first weight of the GlobalModel while the norms' shift is zero (it reads the per-graph means of BatchNorm outputs,
    which equal that shift); what both carry is fp32 rounding noise of the layer's gradient flow."""
    refs = dict(ref.named_parameters())
    for (n, p), (_, q) in zip(model.named_parameters(), ref.named_parameters()):
        if q.grad is None:
            assert p.grad is None, n
            continue
        qg = q.grad * factor
        scale = max(qg.abs().max().item(), 1e-6)
        for own, sibling in (("bias", "weight"), ("weight", "bias")):
            other = refs.get(n[:-len(own)] + sibling) if n.endswith(own) else None
            if other is not None and other.grad is not None:
                scale = max(scale, other.grad.abs().max().item() * factor)
        assert (p.grad - qg).abs().max().item() < 2e-3 * scale + 1e-5 * factor, n


@pytest.mark.gpu
def test_loss_function_on_a_collated_batch_sums_the_graphs():
    from pfs_neural_net_b200 import _abi, gnn as pg, loss as pl
    dev = _dev()
    G, S, T, F = 3, 64, 12, 10
    torch.manual_seed(0)
    model = pg.GNN(B=2, Fdim=F, T=T, F_s=1, F_t=2).to(dev).train()
    ref, mean_model = copy.deepcopy(model), copy.deepcopy(model)
    graphs = _graphs(G, S, T, F)
    class_info = torch.stack([gr.x_t for gr in graphs]).to(dev)
    noise = torch.rand(G, S * T, generator=torch.Generator().manual_seed(9)).to(dev)
    losses, utils = [], []
    for k, gr in enumerate(graphs):
        l, u = pl.loss_function(ref, ref(gr), class_info[k], noise=noise[k])
        l.backward()
        losses.append(l.item())
        utils.append(u.item())
    batch = pg.Loader.collate(graphs)
    loss, util = pl.loss_function(model, model(batch), class_info, noise=noise)
    loss.backward()
    assert loss.dim() == 0 and util.shape == (G,)
    # the loss is a difference of large terms: judge it on the scale of the utility term, as tests/test_gpu_loss.py does
    assert abs(loss.item() - sum(losses)) < 1e-4 * G * max(max(abs(x) for x in losses), 2000.0 * max(utils))
    assert _rel(util, torch.tensor(utils)) < 1e-4
    _param_grads_match(model, ref)
    loss_m, _ = pl.loss_function(mean_model, mean_model(batch), class_info, noise=noise, reduction="mean")
    loss_m.backward()
    assert abs(loss_m.item() - loss.item() / G) < 1e-6 * abs(loss.item())
    _param_grads_match(mean_model, ref, 1.0 / G)
    # every per-graph diagnostic of finaloutput carries the leading G; a shared class table works too
    full = pl.loss_function(model, model(batch), class_info[0], noise=noise, finaloutput=True)
    assert len(full) == 7 and full[1].shape == (G,) and full[2].shape == (G, T) and full[3].shape == (G, T)
    assert full[4].shape == (G, S) and full[5].shape == (G, S * T) and full[6].shape == (G,)
    out = model(batch)
    with pytest.raises(_abi.PfsError):
        pl.loss_function(model, out, class_info[:2], noise=noise)                 # G does not match
    with pytest.raises(_abi.PfsError):
        pl.loss_function(model, out, class_info, noise=noise[:, :-1])            # noise of another shape
    with pytest.raises(ValueError):
        pl.loss_function(model, out, class_info, noise=noise, reduction="max")


def test_batched_loss_shape_errors_are_reported_on_the_host():
    from pfs_neural_net_b200 import _abi, loss as pl
    G, S, T = 3, 8, 4
    time, noise = _times(G, S, T)
    for ci, nz, what in ((_class_info(T, G + 1), noise, "class_info"), (_class_info(T + 1), noise, "class_info"),
                         (torch.zeros(T), noise, "class_info"), (_class_info(T, G), noise[:, :-1], "noise"),
                         (_class_info(T, G), noise[:2], "noise")):
        with pytest.raises(_abi.PfsError, match=what):
            pl.loss_from_times(time, ci, S, T, noise=nz)
    with pytest.raises(_abi.PfsError, match="batch of edge times"):
        pl.loss_from_times(time.reshape(G, S, T), _class_info(T), S, T)        # 3-D is [G, E, 1] only
    with pytest.raises(_abi.PfsError, match="CUDA"):                          # right shapes: no CPU fallback
        pl.loss_from_times(time, _class_info(T, G), S, T, noise=noise)


def _train_setup(dev, G=4, S=200, T=12, F=10, seed=1):
    from pfs_neural_net_b200 import gnn as pg
    torch.manual_seed(0)
    model = pg.GNN(B=2, Fdim=F, T=T, F_s=1, F_t=2).to(dev).train()
    graphs = _graphs(G, S, T, F, seed=seed)
    batch = pg.Loader.collate(graphs)
    return model, batch, batch.x_t.clone()


def _clone_batch(batch):
    from pfs_neural_net_b200 import gnn as pg
    return pg.BipartiteData(batch.edge_index, batch.x_s.clone(), batch.x_t.clone(), batch.x_e.clone(), batch.x_u.clone())


@pytest.mark.gpu
def test_batched_train_step_graph_replay_matches_eager():
    from pfs_neural_net_b200.train_step import TrainStep
    dev = _dev()
    runs = []
    for use_graph in (False, True):
        model, batch, ci = _train_setup(dev)
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
        step = TrainStep(model, batch, ci, opt, use_graph=use_graph, warmup=2)
        out = []
        for i in range(5):
            torch.manual_seed(100 + i)
            loss, util = step(0.5 + 0.1 * i)
            assert loss.dim() == 0 and util.shape == (4,)
            out.append((float(loss), util.detach().cpu().clone()))
        runs.append((out, {k: v.clone() for k, v in model.state_dict().items()}))
    (la, sa), (lb, sb) = runs
    for (a, ua), (b, ub) in zip(la, lb):
        assert abs(a - b) <= 1e-5 * max(1.0, abs(a)), (la, lb)
        assert torch.allclose(ua, ub, rtol=1e-6, atol=1e-6), (ua, ub)
    for k in sa:
        assert torch.allclose(sa[k].float(), sb[k].float(), rtol=1e-5, atol=1e-6), k
    assert len({round(l[0], 3) for l in lb}) > 1


@pytest.mark.gpu
def test_constructing_a_batched_train_step_changes_nothing():
    from pfs_neural_net_b200.train_step import TrainStep
    dev = _dev()
    model, batch, ci = _train_setup(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
    before = copy.deepcopy(model.state_dict())
    inputs = [t.clone() for t in (batch.x_s, batch.x_t, batch.x_e, batch.x_u, ci)]
    torch.manual_seed(5)
    rng = torch.cuda.get_rng_state(dev).clone()
    TrainStep(model, batch, ci, opt, use_graph=True, warmup=2)
    for k, v in model.state_dict().items():
        assert torch.equal(v, before[k]), k
    assert torch.equal(torch.cuda.get_rng_state(dev), rng)
    for a, b in zip(inputs, (batch.x_s, batch.x_t, batch.x_e, batch.x_u, ci)):
        assert torch.equal(a, b)
    for st in opt.state.values():
        for k, v in st.items():
            if torch.is_tensor(v):
                assert float(v.abs().max()) == 0.0, k


@pytest.mark.gpu
def test_epoch_of_loaded_batches_replays_like_eager_steps():
    """two batches, two epochs: load() + replay of one captured step == eager steps on each batch"""
    from pfs_neural_net_b200.train_step import TrainStep
    dev = _dev()
    runs = []
    for use_graph in (False, True):
        model, a, ci_a = _train_setup(dev, seed=1)
        _, b, ci_b = _train_setup(dev, seed=2)
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
        if use_graph:
            step = TrainStep(model, _clone_batch(a), ci_a.clone(), opt, use_graph=True, warmup=2)
            run = lambda batch, ci, s: (step.load(batch, ci), step(s))[1]
        else:
            steps = {id(a): TrainStep(model, a, ci_a, opt, use_graph=False), id(b): TrainStep(model, b, ci_b, opt, use_graph=False)}
            run = lambda batch, ci, s: steps[id(batch)](s)
        out = []
        for i, (batch, ci) in enumerate([(a, ci_a), (b, ci_b)] * 2):
            torch.manual_seed(200 + i)
            loss, util = run(batch, ci, 0.5 + 0.1 * i)
            out.append((float(loss), util.detach().cpu().clone()))
        runs.append((out, {k: v.clone() for k, v in model.state_dict().items()}))
    (la, sa), (lb, sb) = runs
    for (x, ux), (y, uy) in zip(la, lb):
        assert abs(x - y) <= 1e-5 * max(1.0, abs(x)), (la, lb)
        assert torch.allclose(ux, uy, rtol=1e-6, atol=1e-6), (ux, uy)
    assert abs(la[0][0] - la[1][0]) > 1e-3 * abs(la[0][0])         # the two batches are different work
    for k in sa:
        assert torch.allclose(sa[k].float(), sb[k].float(), rtol=1e-5, atol=1e-6), k


@pytest.mark.gpu
def test_load_refuses_another_topology_or_other_shapes():
    from pfs_neural_net_b200 import gnn as pg
    from pfs_neural_net_b200.train_step import TrainStep
    dev = _dev()
    model, batch, ci = _train_setup(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
    step = TrainStep(model, batch, ci, opt, use_graph=False)
    other = _clone_batch(batch)
    other.edge_index = batch.edge_index.flip(1).contiguous()
    with pytest.raises(ValueError, match="edge_index"):
        step.load(other)
    _, small, ci_small = _train_setup(dev, G=3)
    with pytest.raises(ValueError):
        step.load(small)
    with pytest.raises(ValueError):
        step.load(_clone_batch(batch), ci_small)
    kept = batch.x_e.clone()
    step.load(pg.BipartiteData(batch.edge_index, batch.x_s, batch.x_t, batch.x_e * 2, batch.x_u))
    assert torch.equal(batch.x_e, kept * 2)                          # copied into the step's own input tensors


def test_batched_train_bench_runs_up_to_the_device():
    """tools/batched_train_bench.py parses its arguments and builds its inputs without a GPU, then stops with a message"""
    if torch.cuda.is_available():
        pytest.skip("on a GPU the script runs the whole measurement")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "batched_train_bench.py"), "--graphs", "1,2", "--steps", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "needs a CUDA device" in r.stderr, r.stderr[-2000:]
