"""Host-side and algorithmic parts of the fibre-sharded loss, on CPU: the per-shard record and its rank-order merge
(an fp64 mirror of k_loss_shard_record / k_loss_shard_merge) against two-pass statistics of the whole column,
shard.exchange_rows over 2 and 3 gloo ranks, the C ABI's refusals of a sharded call it cannot serve, and
tools/sharded_train_bench.py stopping cleanly without a GPU.  The kernels themselves are checked in
tests/test_gpu_sharded_training.py."""
import ctypes as ct
import os
import socket
import subprocess
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from pfs_neural_net_b200 import _abi, shard

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _record(x):
    """the record of one shard's [n, T] column block as k_loss_shard_record builds it from shifted sums"""
    n = x.shape[0]
    d = x - x[0]
    s1, s2 = d.sum(0), (d * d).sum(0)
    return n, x[0] + s1 / n, s2 - s1 * s1 / n


def _merge(records):
    """rank-order pairwise update of k_loss_shard_merge"""
    n, mean, m2 = records[0]
    for nb, mb, m2b in records[1:]:
        nab = n + nb
        d = mb - mean
        mean = mean + d * nb / nab
        m2 = m2 + m2b + d * d * n * nb / nab
        n = nab
    return n, mean, m2


@pytest.mark.parametrize("bounds", [[0, 1, 500, 1000], [0, 380, 1000], [0, 999, 1000], [0, 1000]])
def test_record_merge_matches_two_pass_statistics(bounds):
    g = torch.Generator().manual_seed(3)
    full = (torch.randn(1000, 6, generator=g, dtype=torch.float64) * 3 + 4e4).float().double()   # |mean| >> std
    n, mean, m2 = _merge([_record(full[a:b]) for a, b in zip(bounds[:-1], bounds[1:])])
    ref_mean = full.mean(0)
    ref_m2 = ((full - ref_mean) ** 2).sum(0)
    assert n == 1000
    assert torch.allclose(mean, ref_mean, rtol=1e-14, atol=0)
    assert torch.allclose(m2, ref_m2, rtol=1e-10, atol=0)
    # the variance the loss takes: M2 / (S_total - 1), as torch.var
    assert torch.allclose(m2 / (n - 1), torch.var(full, dim=0), rtol=1e-10)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    row = torch.arange(5, dtype=torch.float64) + 10 * rank + 0.1
    ok = torch.equal(shard.exchange_rows(row), row.reshape(1, -1))            # outside the scope: no exchange
    with shard.fibre_sharded():
        shard.reset_traffic()
        rows = shard.exchange_rows(row)
        ok &= shard.traffic() == (1, world * 5 * 8)
        ok &= rows.dtype == torch.float64 and rows.shape == (world, 5)
        ok &= all(torch.equal(rows[r], torch.arange(5, dtype=torch.float64) + 10 * r + 0.1) for r in range(world))
        ok &= shard.rank() == rank
        f32 = shard.exchange_rows(row.float())
        ok &= f32.dtype == torch.float32 and torch.equal(f32, rows.float())
    out[rank] = bool(ok)
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_exchange_rows(world):
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
        assert dict(out) == {r: True for r in range(world)}


def _lib():
    if not os.path.exists(_abi.LIB_PATH):
        _abi.build_library()
    return _abi.load_library()


def test_abi_refuses_sharded_calls_it_cannot_serve():
    """argument checks run before any CUDA call, so they answer without a GPU"""
    lib = _lib()
    a = _abi.LossArgs()
    for k in ("time", "noise", "hours", "counts", "galaxies", "time2", "fibre_time", "n_prime", "class_mean", "class_coef",
              "scalars", "workspace", "shard_record", "shard_records", "g_time"):
        setattr(a, k, 256)                       # never dereferenced: every call below fails its argument check
    a.T, a.world = 12, 2
    a.S, a.S_total, a.G = 10, 20, 2
    assert lib.pfs_loss_shard_fwd(ct.byref(a)) == -1 and b"one graph per call" in lib.pfs_last_error()
    assert lib.pfs_loss_shard_merge(ct.byref(a)) == -1
    assert lib.pfs_loss_bwd(ct.byref(a)) == -1
    a.G = 0
    assert lib.pfs_loss_fwd(ct.byref(a)) == -1 and b"S_total is set" in lib.pfs_last_error()
    a.S, a.S_total = 1, 1                        # the graph needs 2 fibres over all shards
    assert lib.pfs_loss_shard_fwd(ct.byref(a)) == -1 and b"shard sizes" in lib.pfs_last_error()
    a.S, a.S_total = 1, 0                        # a single fibre is a shard, not a graph
    assert lib.pfs_loss_bwd(ct.byref(a)) == -1 and b"at least 2 fibres" in lib.pfs_last_error()
    assert lib.pfs_loss_shard_fwd(ct.byref(a)) == -1 and b"S_total" in lib.pfs_last_error()


def test_sharded_train_bench_runs_up_to_the_device():
    """tools/sharded_train_bench.py parses its arguments without a GPU, then stops with a message"""
    if torch.cuda.is_available():
        pytest.skip("on a GPU the script runs the whole measurement")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sharded_train_bench.py"), "--steps", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "needs a CUDA device" in r.stderr, r.stderr[-2000:]
