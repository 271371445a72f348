"""The loss on a general edge list, on the CPU: `tests/edge_loss_oracle.loss_terms_edges` (the fp64 restatement of the
cell-matrix definition, DESIGN.md section 8b) against `loss_terms` (pinned to the unmodified reference) on the complete
graph in canonical, class-permuted and shuffled order, and against a direct dense-matrix computation on a small graph
with duplicate edges, a fibre without edges and a class without edges.  Also: the C ABI's refusals of edge-list calls it
cannot serve (argument checks run before any CUDA call), and tools/sparse_train_bench.py stopping without a GPU."""
import contextlib
import ctypes as ct
import os
import subprocess
import sys

import pytest
import torch
import torch.distributed as dist

from oracle import block_oracle as bo
from oracle import loss_oracle as lo
from tests import edge_loss_oracle as elo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("loss", "totutils", "class_penalty", "fiber_penalty", "variance", "n_prime", "fiber_time")


def _inputs(S, T, seed=0):
    g = torch.Generator().manual_seed(seed)
    ci = torch.stack([0.5 + 3 * torch.rand(T, generator=g, dtype=torch.float64),
                      50 + 400 * torch.rand(T, generator=g, dtype=torch.float64)], -1)
    time = 2 * (42.0 / T) * torch.rand(S * T, generator=g, dtype=torch.float64)
    return time, torch.rand(S * T, generator=g, dtype=torch.float64), ci


def permuted_complete(S, T, mode, seed=0):
    """the complete graph in another order: "class" permutes the classes within each fibre (fibre-major, like the
    reference's graphs/graph-0.pt), "shuffle" permutes all edges"""
    g = torch.Generator().manual_seed(seed)
    ei = bo.complete_bipartite(S, T)
    if mode == "class":
        perm = torch.cat([k * T + torch.randperm(T, generator=g) for k in range(S)])
    else:
        perm = torch.randperm(S * T, generator=g)
    return ei[:, perm]


def _close(a, b, tol):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return (a - b).abs().max().item() <= tol * max(b.abs().max().item(), 1.0)


def _both(time, noise, ci, ei, S, T, oracle):
    t = time.clone().requires_grad_(True)
    r = oracle(t, noise, ci, ei, S, T)
    r["loss"].backward()
    return r, t.grad


@pytest.mark.parametrize("S,T", [(40, 12), (7, 1), (2, 5)])
def test_edge_oracle_is_the_reference_loss_on_the_canonical_graph(S, T):
    time, noise, ci = _inputs(S, T)
    ei = bo.complete_bipartite(S, T)
    a, ga = _both(time, noise, ci, ei, S, T, elo.loss_terms_edges)
    b, gb = _both(time, noise, ci, ei, S, T, lo.loss_terms)
    for k in KEYS + ("time",):
        assert _close(a[k], b[k], 1e-12), k
    assert _close(ga, gb, 1e-12)


@pytest.mark.parametrize("mode", ["class", "shuffle"])
def test_edge_oracle_on_a_permuted_complete_graph_is_the_reference_loss_unpermuted(mode):
    S, T = 30, 9
    time, noise, ci = _inputs(S, T, seed=1)
    ei = permuted_complete(S, T, mode, seed=2)
    canon = ei[0] * T + ei[1]                    # canonical position of every listed edge
    assert not torch.equal(canon, torch.arange(S * T))
    t_c, n_c = torch.empty_like(time), torch.empty_like(noise)
    t_c[canon], n_c[canon] = time, noise
    a, ga = _both(time, noise, ci, ei, S, T, elo.loss_terms_edges)
    b, gb = _both(t_c, n_c, ci, bo.complete_bipartite(S, T), S, T, lo.loss_terms)
    for k in KEYS:
        assert _close(a[k], b[k], 1e-12), k
    assert _close(a["time"], b["time"][canon], 1e-12)
    assert _close(ga, gb[canon], 1e-12)


def test_edge_oracle_with_duplicates_and_empty_rows_against_the_dense_matrix():
    """5 fibres x 4 classes: fibre 3 has no edge, class 2 has none, (0, 1) and (4, 3) appear twice"""
    S, T = 5, 4
    src = torch.tensor([0, 1, 0, 4, 2, 0, 4, 1, 4, 2])
    tgt = torch.tensor([1, 0, 3, 3, 1, 1, 0, 3, 3, 0])
    ei = torch.stack([src, tgt])
    E = ei.shape[1]
    g = torch.Generator().manual_seed(3)
    ci = torch.tensor([[1.0, 30.0], [2.5, 80.0], [0.7, 40.0], [1.9, 120.0]], dtype=torch.float64)
    time = 8 * torch.rand(E, generator=g, dtype=torch.float64)
    noise = torch.rand(E, generator=g, dtype=torch.float64)
    r = elo.loss_terms_edges(time, noise, ci, ei, S, T)
    # direct computation, one edge and one matrix entry at a time
    sharp, wutils, wvar, pclass, pfiber, total = 0.5, 2000.0, 1.0, 0.1, 1.0, 42.0
    gal = [max(0.0, lo.softfloor(time[e:e + 1] / ci[tgt[e], 0], noise[e:e + 1], sharp).item()) for e in range(E)]
    t2 = [gal[e] * ci[tgt[e], 0].item() for e in range(E)]
    M = [[0.0] * T for _ in range(S)]
    n_prime, ft = [0.0] * T, [0.0] * S
    for e in range(E):
        M[src[e]][tgt[e]] += t2[e]
        n_prime[tgt[e]] += gal[e]
        ft[src[e]] += t2[e]
    var = 0.0
    for i in range(T):
        col = [M[k][i] for k in range(S)]
        m = sum(col) / S
        var += sum((x - m) ** 2 for x in col) / (S - 1)
    N = [ci[i, 1].item() / 10 for i in range(T)]
    util = min(n_prime[i] / N[i] for i in range(T))
    cpen = pclass * sum(max(0.0, n_prime[i] - N[i]) ** 2 for i in range(T))
    fpen = pfiber * sum((x - total if x > total else 0.1 * (x - total)) ** 2 for x in ft)
    assert n_prime[2] == 0.0 and ft[3] == 0.0 and util == 0.0     # the empty class is the minimum
    assert _close(r["cells"], torch.tensor(M, dtype=torch.float64), 1e-12)
    assert _close(r["n_prime"], torch.tensor(n_prime, dtype=torch.float64), 1e-12)
    assert _close(r["fiber_time"], torch.tensor(ft, dtype=torch.float64), 1e-12)
    for k, v in (("variance", var), ("totutils", util), ("class_penalty", cpen), ("fiber_penalty", fpen),
                 ("loss", -wutils * util + fpen + cpen - wvar * var)):
        assert abs(r[k].item() - v) <= 1e-12 * max(1.0, abs(v)), k


def _lib():
    from pfs_neural_net_b200 import _abi
    if not os.path.exists(_abi.LIB_PATH):
        _abi.build_library()
    return _abi.load_library()


def test_abi_refuses_edge_list_calls_it_cannot_serve():
    """argument checks run before any CUDA call, so they answer without a GPU"""
    from pfs_neural_net_b200 import _abi
    lib = _lib()
    a = _abi.LossArgs()
    for k in ("time", "noise", "hours", "counts", "galaxies", "time2", "fibre_time", "n_prime", "class_mean", "class_coef",
              "scalars", "workspace", "shard_record", "shard_records", "g_time", "csr_rowptr", "csr_eid", "csr_src",
              "csr_tgt", "csc_colptr", "csc_q", "cell_time"):
        setattr(a, k, 256)                       # never dereferenced: every call below fails its argument check
    a.S, a.T, a.E, a.world = 20, 12, 100, 2
    a.S_total = 40                               # sharding an edge list
    for fn in (lib.pfs_loss_fwd, lib.pfs_loss_bwd, lib.pfs_loss_shard_fwd, lib.pfs_loss_shard_merge):
        assert fn(ct.byref(a)) == -1, fn
    assert lib.pfs_loss_shard_fwd(ct.byref(a)) == -1 and b"cannot be fibre-sharded" in lib.pfs_last_error()
    a.S_total = 0
    for k in ("csr_eid", "csc_q", "cell_time"):  # E set and an array NULL
        setattr(a, k, None)
        assert lib.pfs_loss_fwd(ct.byref(a)) == -1 and b"needs csr_rowptr" in lib.pfs_last_error(), k
        assert lib.pfs_loss_bwd(ct.byref(a)) == -1 and b"needs csr_rowptr" in lib.pfs_last_error(), k
        setattr(a, k, 256)
    a.E = -1
    assert lib.pfs_loss_fwd(ct.byref(a)) == -1 and b"negative edge count" in lib.pfs_last_error()
    a.E = 0                                      # edge arrays without E
    assert lib.pfs_loss_fwd(ct.byref(a)) == -1 and b"E (edges per graph) is 0" in lib.pfs_last_error()
    a.E, a.S = 100, 1                            # bad sizes
    assert lib.pfs_loss_fwd(ct.byref(a)) == -1 and b"edge-list sizes" in lib.pfs_last_error()
    a.S, a.T = 20, 0
    assert lib.pfs_loss_bwd(ct.byref(a)) == -1 and b"edge-list sizes" in lib.pfs_last_error()
    a.T, a.G = 12, 1 << 28                       # G*T >= 2^31 CTAs of the class pass
    assert lib.pfs_loss_fwd(ct.byref(a)) == -1 and b"G*T" in lib.pfs_last_error()
    a.G, a.workspace_bytes = 1, lib.pfs_loss_list_workspace_bytes(12) - 1
    assert lib.pfs_loss_fwd(ct.byref(a)) == -4 and b"workspace too small" in lib.pfs_last_error()     # PFS_ERR_WORKSPACE


@contextlib.contextmanager
def one_rank_group():
    """a one-process gloo group on an in-process store (no sockets)"""
    dist.init_process_group("gloo", store=dist.HashStore(), rank=0, world_size=1)
    try:
        yield
    finally:
        dist.destroy_process_group()


def test_loss_from_times_refuses_an_edge_list_inside_a_sharded_scope():
    """the refusal comes before any device work, so it answers without a GPU"""
    from pfs_neural_net_b200 import _abi, loss as pl, shard
    S, T = 6, 3
    time, noise, ci = _inputs(S, T)
    ei = permuted_complete(S, T, "class")
    with one_rank_group(), shard.fibre_sharded():
        with pytest.raises(_abi.PfsError, match="edge list cannot be fibre-sharded"):
            pl.loss_from_times(time.float(), ci.float(), S, T, noise=noise.float(), edge_index=ei)


def test_sparse_train_bench_runs_up_to_the_device():
    """tools/sparse_train_bench.py parses its arguments without a GPU, then stops with a message"""
    if torch.cuda.is_available():
        pytest.skip("on a GPU the script runs the whole measurement")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sparse_train_bench.py"), "--iters", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "needs a CUDA device" in r.stderr, r.stderr[-2000:]
