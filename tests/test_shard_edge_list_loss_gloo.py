"""Host-side and algorithmic parts of the loss of an edge list sharded over fibre ranges, on CPU: an fp64 mirror of the
per-shard record (k_loss_list_class's totals over the local fibres, zero cells folded in with the local S, and
k_loss_list_shard_record) and of the rank-order merge of k_loss_shard_merge, against the fp64 oracle of the whole edge
list; the C ABI's refusals of the new entry points; the checks of `edge_ids`; edge counts cached apart from fibre counts
over two gloo ranks; and tools/sharded_train_bench.py --graph c5 stopping cleanly without a GPU.  The kernels themselves
are checked in tests/test_gpu_sharded_edge_list_training.py."""
import ctypes as ct
import datetime
import os
import socket
import subprocess
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle.block_oracle import segment_sum
from oracle.loss_oracle import softfloor
from pfs_neural_net_b200 import _abi, shard
from tests import edge_loss_oracle as elo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _edge_terms(time, noise, ci, edge_index, sharpness=0.5):
    """galaxies and time2 per edge, as the oracle computes them"""
    h = ci[:, 0][edge_index[1]]
    gal = torch.clamp(softfloor(time / h, noise, sharpness), min=0.0)
    return gal, gal * h


def _record(gal, time2, local, S, T, total_time=42.0):
    """the record of one shard: its S local fibres, fibre-penalty sum, and per class the sum of galaxies and the mean and
    M2 of the cells over the S local fibres -- the present cells reduced first, the S - count zero cells folded in with
    the pairwise update, as k_loss_list_class does"""
    src, tgt = local[0], local[1]
    cells = segment_sum(time2, src * T + tgt, S * T).reshape(S, T)
    present = segment_sum(torch.ones_like(time2), src * T + tgt, S * T).reshape(S, T) > 0
    cnt = present.sum(0).double()
    mc = torch.where(cnt > 0, (cells * present).sum(0) / cnt.clamp(min=1), torch.zeros_like(cnt))
    m2c = ((cells - mc) ** 2 * present).sum(0)
    mean = mc * cnt / S
    m2 = m2c + cnt * (S - cnt) / S * mc * mc
    ft = segment_sum(time2, src, S)
    ot = ft - total_time
    fpen = torch.where(ot > 0, ot, 0.1 * ot).pow(2).sum()
    return dict(n=float(S), fpen=fpen, gal=segment_sum(gal, tgt, T), mean=mean, m2=m2)


def _merge(records):
    """k_loss_shard_merge: sums added, (n, mean, M2) by the pairwise update in rank order"""
    r0 = records[0]
    n, mean, m2, gal, fpen = r0["n"], r0["mean"], r0["m2"], r0["gal"], r0["fpen"]
    for r in records[1:]:
        nb = r["n"]
        nab = n + nb
        d = r["mean"] - mean
        gal = gal + r["gal"]
        mean = mean + d * nb / nab
        m2 = m2 + r["m2"] + d * d * n * nb / nab
        fpen = fpen + r["fpen"]
        n = nab
    return n, gal, mean, m2, fpen


def _graph(kind, S, T, seed):
    """[2, E] edge lists: "sparse" (10 %, duplicates, fibre 2 without edges, shuffled), "class_gap" (complete, then class
    3 dropped on the fibres [S/2, S): classes without edges on some ranks), "offset" (complete, shuffled)"""
    g = torch.Generator().manual_seed(seed)
    if kind == "sparse":
        e = torch.nonzero(torch.rand(S * T, generator=g) < 0.1).flatten()
        e = e[e // T != 2]
        e = torch.cat([e, e[torch.rand(e.numel(), generator=g) < 0.2]])
    else:
        e = torch.arange(S * T)
        if kind == "class_gap":
            e = e[~((e % T == 3) & (e // T >= S // 2))]
    e = e[torch.randperm(e.numel(), generator=g)]
    return torch.stack([e // T, e % T])


@pytest.mark.parametrize("kind,S,T,bounds", [
    ("sparse", 60, 9, [0, 1, 30, 60]),
    ("sparse", 60, 9, [0, 17, 18, 60]),
    ("class_gap", 40, 7, [0, 1, 20, 40]),
    ("class_gap", 40, 7, [0, 40]),
    ("offset", 50, 5, [0, 1, 25, 49, 50]),
])
def test_record_and_merge_match_the_edge_list_oracle(kind, S, T, bounds):
    g = torch.Generator().manual_seed(S + T)
    ei = _graph(kind, S, T, seed=S * T)
    E = ei.shape[1]
    ci = torch.stack([0.5 + 3 * torch.rand(T, generator=g, dtype=torch.float64),
                      50 + 400 * torch.rand(T, generator=g, dtype=torch.float64)], 1)
    if kind == "offset":                       # |mean| >> std: every cell near 1000 T_i
        time = ci[:, 0][ei[1]] * (1000 + 3 * torch.randn(E, generator=g, dtype=torch.float64))
    else:
        time = 2 * (42.0 * S / E) * torch.rand(E, generator=g, dtype=torch.float64)
    noise = torch.rand(E, generator=g, dtype=torch.float64)
    r = elo.loss_terms_edges(time, noise, ci, ei, S, T)
    gal, time2 = _edge_terms(time, noise, ci, ei)
    records = []
    for f0, f1 in zip(bounds[:-1], bounds[1:]):
        keep = torch.nonzero((ei[0] >= f0) & (ei[0] < f1)).flatten()
        local = torch.stack([ei[0][keep] - f0, ei[1][keep]])
        records.append(_record(gal[keep], time2[keep], local, f1 - f0, T))
    n, n_prime, mean, m2, fpen = _merge(records)
    assert n == S
    assert torch.allclose(n_prime, r["n_prime"], rtol=1e-12, atol=1e-12)
    assert torch.allclose(mean, r["cells"].mean(0), rtol=1e-12, atol=1e-9)
    var = torch.clamp(m2, min=0) / (S - 1)
    assert torch.allclose(var, torch.var(r["cells"], dim=0), rtol=1e-9, atol=1e-9)
    assert abs(var.sum().item() - r["variance"].item()) <= 1e-9 * r["variance"].item()
    assert abs(fpen.item() - r["fiber_penalty"].item()) <= 1e-12 * max(r["fiber_penalty"].item(), 1.0)
    N = ci[:, 1] / 10
    cmin = (n_prime / N).min()
    loss = -2000.0 * cmin + fpen + 0.1 * torch.relu(n_prime - N).pow(2).sum() - var.sum()
    scale = max(abs(r["loss"].item()), 2000.0 * abs(r["totutils"].item()), r["variance"].item())
    assert abs(loss.item() - r["loss"].item()) <= 1e-12 * scale


def _lib():
    if not os.path.exists(_abi.LIB_PATH):
        _abi.build_library()
    return _abi.load_library()


@pytest.mark.parametrize("entry", ["pfs_loss_list_shard_fwd", "pfs_loss_list_shard_bwd"])
def test_abi_refuses_list_shard_calls_it_cannot_serve(entry):
    """argument checks run before any CUDA call, so they answer without a GPU"""
    lib = _lib()
    fn = getattr(lib, entry)

    def args():
        a = _abi.LossArgs()
        for k in ("time", "noise", "hours", "counts", "galaxies", "time2", "fibre_time", "n_prime", "class_mean",
                  "class_coef", "scalars", "workspace", "shard_record", "g_time", "csr_rowptr", "csr_eid", "csr_src",
                  "csr_tgt", "csc_colptr", "csc_q", "cell_time"):
            setattr(a, k, 256)                   # never dereferenced: every call below fails its argument check
        a.S, a.T, a.S_total, a.E, a.G = 10, 12, 20, 30, 2
        return a

    a = args()
    assert fn(ct.byref(a)) == -1 and b"one graph per call" in lib.pfs_last_error()
    for E in (0, -1):
        a = args()
        a.E = E
        assert fn(ct.byref(a)) == -1 and b"must be > 0" in lib.pfs_last_error(), E
    a = args()
    a.S_total = 0
    assert fn(ct.byref(a)) == -1 and b"S_total" in lib.pfs_last_error()
    a = args()
    a.G, a.S = 1, 21
    assert fn(ct.byref(a)) == -1 and b"shard sizes" in lib.pfs_last_error()
    a = args()
    a.G, a.S_total, a.S = 0, 1, 1                # the graph needs 2 fibres over all shards
    assert fn(ct.byref(a)) == -1 and b"shard sizes" in lib.pfs_last_error()
    for k in ("csr_eid", "csc_q", "cell_time"):
        a = args()
        a.G = 0
        setattr(a, k, None)
        assert fn(ct.byref(a)) == -1 and b"needs csr_rowptr" in lib.pfs_last_error(), k
    a = args()
    a.G = 0
    a.time = None
    assert fn(ct.byref(a)) == -1 and b"null pointer" in lib.pfs_last_error()
    if entry.endswith("fwd"):
        a = args()
        a.G = 0
        a.shard_record = None
        assert fn(ct.byref(a)) == -1 and b"null pointer" in lib.pfs_last_error()
    # the unsharded entry points keep refusing an edge list with S_total
    a = args()
    a.G = 0
    assert lib.pfs_loss_fwd(ct.byref(a)) == -1
    assert lib.pfs_loss_bwd(ct.byref(a)) == -1 and b"cannot be fibre-sharded" in lib.pfs_last_error()


def test_edge_ids_are_refused_outside_the_scope():
    """the refusal comes before any device work, so it answers without a GPU"""
    from pfs_neural_net_b200 import loss as pl
    S, T = 6, 3
    ei = _graph("offset", S, T, seed=1)
    time = torch.rand(S * T)
    ci = torch.stack([torch.ones(T), 100 * torch.ones(T)], 1)
    with pytest.raises(_abi.PfsError, match="only taken inside shard.fibre_sharded"):
        pl.loss_from_times(time, ci, S, T, noise=torch.rand(S * T), edge_index=ei, edge_ids=torch.arange(S * T))


def test_edge_ids_checks():
    """dtype, shape, device, length and range; the range is read once per tensor"""
    from pfs_neural_net_b200 import loss as pl
    cpu = torch.device("cpu")
    E, E_total = 5, 12
    ok = torch.tensor([0, 3, 4, 9, 11])
    pl._check_edge_ids(ok, E, E_total, cpu)
    assert any(v is ok for v in pl._EDGE_IDS_CHECKED.values())
    pl._check_edge_ids(ok, E, E_total, cpu)
    for bad, what in ((ok.int(), "1-D int64"), (ok.float(), "1-D int64"), (ok.reshape(1, 5), "1-D int64"),
                      (ok.tolist(), "1-D int64"), (ok[:4], "4 entries for 5 local edges"),
                      (torch.cat([ok, ok[:1]]), "6 entries"), (torch.tensor([0, 3, 4, 9, 12]), "out of range"),
                      (torch.tensor([-1, 3, 4, 9, 10]), "out of range")):
        with pytest.raises(_abi.PfsError, match=what):
            pl._check_edge_ids(bad, E, E_total, cpu)
    if torch.cuda.is_available():
        with pytest.raises(_abi.PfsError, match="1-D int64"):
            pl._check_edge_ids(ok, E, E_total, torch.device("cuda:0"))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _count_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=60))
    fibres, edges = (5, 5) if rank == 0 else (5, 9)   # rank 0's edge count equals its fibre count
    with shard.fibre_sharded():
        shard.reset_traffic()
        S_total = shard.total_count(fibres)
        E_total = shard.total_count(edges, kind="edges")
        per_rank = shard.shard_counts(edges, kind="edges")
        first = shard.traffic()[0]
        again = (shard.total_count(fibres), shard.total_count(edges, kind="edges"), shard.shard_counts(fibres))
        out[rank] = dict(S_total=S_total, E_total=E_total, per_rank=per_rank, first=first, again=again,
                         calls=shard.traffic()[0])
    dist.destroy_process_group()


def test_edge_counts_are_cached_apart_from_fibre_counts():
    world = 2
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_count_worker, args=(world, _free_port(), out), nprocs=world, join=True)
        out = dict(out)
    for r in range(world):
        o = out[r]
        assert (o["S_total"], o["E_total"], o["per_rank"]) == (10, 14, (5, 9)), o
        assert o["first"] == 2 and o["calls"] == 2, o      # one exchange per kind, then every count is cached
        assert o["again"] == (10, 14, (5, 5)), o


def test_sharded_train_bench_c5_runs_up_to_the_device():
    """tools/sharded_train_bench.py --graph c5 parses its arguments without a GPU, then stops with a message"""
    if torch.cuda.is_available():
        pytest.skip("on a GPU the script runs the whole measurement")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sharded_train_bench.py"), "--graph", "c5",
                        "--steps", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "needs a CUDA device" in r.stderr, r.stderr[-2000:]
