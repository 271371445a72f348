"""Fibres with more than PFS_TILE_EDGES (256) edges on the fp32 path: split tiles.

A fibre of d > 256 edges is cut into ceil(d / 256) consecutive tiles of its own with balanced chunk sizes.  The SModel
edge pass writes one chunk record per split tile (n, sum m, sum m^2 and the 2nd-4th central sums about the chunk mean),
merged per fibre in slot order in fp64 (pairwise update of the central moments); the fibre sums of the EdgeModel and
TModel backward are partial rows per split tile, added in slot order.

CPU part: an fp64 mirror of the chunk record and the merge against direct two-pass moments, and the tile table the
packer must produce, stated as literal tables.  GPU part: every module and the whole Block against the fp64 oracle
(metric of tests/test_gpu_parity.py), determinism, the tile table read back from the device, GNN + loss with 300
classes, and invariants of the complete 12 500 x 512 graph at Fdim 10.
"""
import contextlib
import math

import pytest
import torch

TILE = 256


# ----------------------------------------------------------------------------------------------------------------
# CPU: chunk records and their merge (mirror of k_source_edge_fwd's split branch and k_split_moments, in fp64)
# ----------------------------------------------------------------------------------------------------------------
def chunk_record(x):
    """(n, sum m, sum m^2, M2, M3, M4) of one chunk; M_k about the chunk mean (two passes, as the kernel does)."""
    n = x.numel()
    s1 = x.sum().item()
    mean = s1 / n
    d = x - mean
    return n, s1, (x * x).sum().item(), (d ** 2).sum().item(), (d ** 3).sum().item(), (d ** 4).sum().item()


def merge_records(records):
    """The fibre's moment row [mean, E[m^2], c2, c3, c4] from its chunk records, combined in order."""
    n = mean = sq = m2 = m3 = m4 = 0.0
    for nb, b1, bsq, b2, b3, b4 in records:
        mb = b1 / nb
        sq += bsq
        if n == 0.0:
            n, mean, m2, m3, m4 = float(nb), mb, b2, b3, b4
            continue
        na, nn = n, n + nb
        d = mb - mean
        dn = d / nn
        dn2 = dn * dn
        m4 += b4 + d * dn2 * dn * na * nb * (na * na - na * nb + nb * nb) + 6.0 * dn2 * (na * na * b2 + nb * nb * m2) + \
            4.0 * dn * (na * b3 - nb * m3)
        m3 += b3 + d * dn2 * na * nb * (na - nb) + 3.0 * dn * (na * b2 - nb * m2)
        m2 += b2 + d * dn * na * nb
        mean += dn * nb
        n = nn
    return [mean, sq / n, m2 / n, m3 / n, m4 / n]


def direct_moments(x):
    mean = math.fsum(x.tolist()) / x.numel()
    d = x - mean
    return [mean, (x * x).mean().item(), (d ** 2).mean().item(), (d ** 3).mean().item(), (d ** 4).mean().item()]


def _check_merge(x, sizes):
    assert sum(sizes) == x.numel()
    recs, q = [], 0
    for s in sizes:
        recs.append(chunk_record(x[q:q + s]))
        q += s
    got, ref = merge_records(recs), direct_moments(x)
    std = max(ref[2] ** 0.5, 1e-300)
    # each moment on its natural scale: the mean and E[m^2] against their own size, c_k against std^k
    scales = [max(abs(ref[0]), std), abs(ref[1]), std ** 2, std ** 3, std ** 4]
    for k, (a, b, s) in enumerate(zip(got, ref, scales)):
        if s == 0.0:
            assert a == b, (k, a, b)
        else:
            assert abs(a - b) <= 1e-12 * s, (k, a, b, sizes)


@pytest.mark.parametrize("chunk", [1, 128, 256])
def test_merge_of_equal_chunks_matches_two_pass_moments(chunk):
    g = torch.Generator().manual_seed(chunk)
    x = torch.randn(chunk * 7, generator=g, dtype=torch.float64) * 3 + 0.5
    _check_merge(x, [chunk] * 7)


def test_merge_of_random_splits_matches_two_pass_moments():
    g = torch.Generator().manual_seed(11)
    for trial in range(50):
        n = int(torch.randint(2, 3000, (1,), generator=g))
        x = torch.randn(n, generator=g, dtype=torch.float64).exp()         # skewed, heavy right tail
        cuts = sorted(set(torch.randint(1, n, (int(torch.randint(1, 12, (1,), generator=g)),), generator=g).tolist()))
        bounds = [0] + cuts + [n]
        _check_merge(x, [b - a for a, b in zip(bounds[:-1], bounds[1:])])


def test_merge_of_an_all_equal_fibre_has_no_spread():
    x = torch.full((700,), 1.25, dtype=torch.float64)
    recs = [chunk_record(x[:234]), chunk_record(x[234:467]), chunk_record(x[467:])]
    assert merge_records(recs) == [1.25, 1.5625, 0.0, 0.0, 0.0]


def test_merge_keeps_the_spread_when_the_mean_dominates():
    g = torch.Generator().manual_seed(5)
    x = 1e3 + torch.randn(5000, generator=g, dtype=torch.float64)       # |mean| / std = 1e3
    _check_merge(x, balanced_chunks(5000))
    _check_merge(x, [1, 4998, 1])


# ----------------------------------------------------------------------------------------------------------------
# CPU: the tile table of pfs_build_split_tiles
# ----------------------------------------------------------------------------------------------------------------
def balanced_chunks(d):
    k = -(-d // TILE)
    base, rem = divmod(d, k)
    return [base + (1 if c < rem else 0) for c in range(k)]


def pack_split_tiles(degrees):
    """Expected table for a degree sequence: whole fibres packed greedily into tiles of <= 256 edges and <= 256 fibres
    (as pfs_build_topology packs them), a fibre of more than 256 edges in balanced chunks on tiles of its own."""
    tile_fibre, tile_q, tile_slot, split_fibre, split_ptr = [], [], [], [], []
    q = cur = nf = nslot = 0
    open_ = False
    for f, d in enumerate(degrees):
        if d > TILE:
            split_fibre.append(f)
            split_ptr.append(nslot)
            for c in balanced_chunks(d):
                tile_fibre.append(f)
                tile_q.append(q)
                tile_slot.append(nslot)
                nslot += 1
                q += c
            open_ = False
            continue
        if not open_ or (cur + d > TILE and cur > 0) or nf >= TILE:
            tile_fibre.append(f)
            tile_q.append(q)
            tile_slot.append(-1)
            cur = nf = 0
            open_ = True
        cur += d
        nf += 1
        q += d
    tile_fibre.append(len(degrees))
    tile_q.append(q)
    split_ptr.append(nslot)
    return dict(tile_fibre=tile_fibre, tile_q=tile_q, tile_slot=tile_slot, split_fibre=split_fibre, split_ptr=split_ptr)


TILE_TABLES = {
    "256": ([256], dict(tile_fibre=[0, 1], tile_q=[0, 256], tile_slot=[-1], split_fibre=[], split_ptr=[0])),
    "257": ([257], dict(tile_fibre=[0, 0, 1], tile_q=[0, 129, 257], tile_slot=[0, 1], split_fibre=[0], split_ptr=[0, 2])),
    "512": ([512], dict(tile_fibre=[0, 0, 1], tile_q=[0, 256, 512], tile_slot=[0, 1], split_fibre=[0], split_ptr=[0, 2])),
    "513": ([513], dict(tile_fibre=[0, 0, 0, 1], tile_q=[0, 171, 342, 513], tile_slot=[0, 1, 2], split_fibre=[0],
                        split_ptr=[0, 3])),
    "5000": ([5000], dict(tile_fibre=[0] * 20 + [1], tile_q=list(range(0, 5001, 250)), tile_slot=list(range(20)),
                          split_fibre=[0], split_ptr=[0, 20])),
    # empty fibres, split fibres next to whole-fibre tiles, the last fibre split
    "mixed": ([3, 0, 257, 0, 100, 200, 513],
              dict(tile_fibre=[0, 2, 2, 3, 5, 6, 6, 6, 7], tile_q=[0, 3, 132, 260, 360, 560, 731, 902, 1073],
                   tile_slot=[-1, 0, 1, -1, -1, 2, 3, 4], split_fibre=[2, 6], split_ptr=[0, 2, 5])),
    "split_first_then_whole": ([300, 256, 1, 0, 0],
                               dict(tile_fibre=[0, 0, 1, 2, 5], tile_q=[0, 150, 300, 556, 557], tile_slot=[0, 1, -1, -1],
                                    split_fibre=[0], split_ptr=[0, 2])),
}


@pytest.mark.parametrize("name", sorted(TILE_TABLES))
def test_tile_table_of_the_packer(name):
    degrees, table = TILE_TABLES[name]
    assert pack_split_tiles(degrees) == table


def test_tile_table_invariants_on_a_heavy_tailed_sequence():
    g = torch.Generator().manual_seed(3)
    degrees = (torch.rand(3000, generator=g) ** 6 * 4000).long().tolist()
    degrees[::97] = [0] * len(degrees[::97])
    t = pack_split_tiles(degrees)
    sizes = [b - a for a, b in zip(t["tile_q"][:-1], t["tile_q"][1:])]
    assert all(0 <= s <= TILE for s in sizes) and t["tile_q"][-1] == sum(degrees)
    for i, f in enumerate(t["split_fibre"]):
        chunks = [sizes[k] for k, s in enumerate(t["tile_slot"]) if t["split_ptr"][i] <= s < t["split_ptr"][i + 1]]
        assert chunks == balanced_chunks(degrees[f]) and min(chunks) >= TILE // 2
    assert len(t["tile_fibre"]) <= len(degrees) + sum(degrees) // TILE + 2


# ----------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------
def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def edge_index_from_degrees(degrees, T, gen, distinct=True, lo=0):
    """Shuffled edge list in which fibre f has degrees[f] edges to classes in [lo, T) (distinct, or drawn with
    repetition: duplicate edges, so a fibre can have more edges than there are classes)."""
    src, tgt = [], []
    for f, d in enumerate(degrees):
        cls = lo + (torch.randperm(T - lo, generator=gen)[:d] if distinct else torch.randint(0, T - lo, (d,), generator=gen))
        src.append(torch.full((d,), f, dtype=torch.long))
        tgt.append(cls)
    e = torch.stack([torch.cat(src), torch.cat(tgt)])
    return e[:, torch.randperm(e.shape[1], generator=gen)].contiguous()


# sparse graph with mixed degrees (T = 600 classes, the first 7 never used; the fibres of thousands of edges repeat
# classes): whole-fibre tiles, empty fibres and split fibres side by side
MIXED_DEGREES = [40, 257, 0, 512, 120, 513, 3000, 0, 256, 60, 2600, 90]


def high_degree_case(seed, F=10, S=12, T=300, kind="dense", training=True, normed=True):
    from tests.test_gpu_parity import make_case
    if kind in ("dense", "shuffled", "class_major"):
        return make_case(seed, F=F, S=S, T=T, kind=kind, training=training, normed=normed)
    gen = torch.Generator().manual_seed(seed)
    if kind == "mixed":
        degrees = MIXED_DEGREES
        ei = edge_index_from_degrees(degrees, T, gen, distinct=False, lo=7)
    elif kind == "duplicates":                                  # degree > 256 with few classes (Fdim 16 tail limit)
        degrees = [300, 700, 257, 20, 513, 90]
        ei = edge_index_from_degrees(degrees, T, gen, distinct=False)
    else:
        raise ValueError(kind)
    case = make_case(seed, F=F, S=len(degrees), T=T, kind="dense", training=training, normed=normed)
    E = ei.shape[1]
    case.update(kind=kind, edge_index=ei, x_e=torch.randn(E, F, generator=gen, dtype=torch.float64))
    return case


CASES = {
    "complete_T300_F10": dict(seed=1),
    "complete_T600_F4": dict(seed=2, F=4, S=16, T=600),
    "complete_T600_F8": dict(seed=3, F=8, S=16, T=600),
    "shuffled_T300_F10": dict(seed=4, kind="shuffled"),
    "class_major_T300_F10": dict(seed=5, kind="class_major"),
    "mixed_degrees_F10": dict(seed=6, kind="mixed", T=600),
    "duplicates_F16": dict(seed=7, F=16, kind="duplicates", T=120),
    "eval_T300_F10": dict(seed=8, training=False),
    "unnormed_T300_F10": dict(seed=9, normed=False),
}


def _max_degree(case):
    return int(torch.bincount(case["edge_index"][0]).max())


@contextlib.contextmanager
def _noise_allowance(case):
    """600 classes: the TModel tail adds its per-class terms in fp32 one after the other in one CTA, so its parameter
    gradients and grad u sit at 2-3x the error of the fp32 oracle (which sums blockwise).  The tail is the same code with
    or without split tiles; those cases are judged with the wider allowance tests/test_gpu_parity.py uses for its
    ill-conditioned cases."""
    from tests import test_gpu_parity as tp
    old = tp._conditioning[0]
    tp._conditioning[0] = "ill" if case["T"] > 512 else "well"
    try:
        yield
    finally:
        tp._conditioning[0] = old


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["edge_model", "s_model", "t_model"])
@pytest.mark.parametrize("case_name", sorted(CASES))
def test_module_parity_on_split_fibres(name, case_name):
    from tests.test_gpu_parity import check_input_grads, check_param_grads, check_tensor, nerr, oracle_module, ours_module
    dev = _cuda()
    case = high_degree_case(**CASES[case_name])
    assert _max_degree(case) > TILE
    o_ref, gin_ref, gp_ref, buf_ref = oracle_module(name, case)
    o_32, gin_32, gp_32, _ = oracle_module(name, case, torch.float32)
    o, gin, gp, buf = ours_module(name, case, dev)
    with _noise_allowance(case):
        check_tensor("forward", o, o_ref, o_32)
        check_input_grads(gin, gin_ref, gin_32)
        check_param_grads(gp, gp_ref, gp_32)
    if case["training"] and case["normed"]:
        for k, v in buf_ref.items():
            if k.endswith("num_batches_tracked"):
                assert int(buf[k]) == int(v)
            else:
                assert nerr(buf[k], v) < 1e-4, k


def _block_oracle(case):
    from oracle import block_oracle as bo
    from tests.util import run_oracle_block
    return run_oracle_block(bo, case, torch.float64), run_oracle_block(bo, case, torch.float32)


def _check_block(case, ours, refs, G=1):
    from tests.test_gpu_parity import check_input_grads, check_param_grads, check_tensor, nerr
    (outs, gin, gparam, buffers), ((o64, g64, p64, b64), (o32, g32, p32, _)) = ours, refs
    names = ("x_s", "x_t", "x_e", "u")
    with _noise_allowance(case):
        for i in range(G):
            pick = (lambda t: t[i]) if G > 1 else (lambda t: t)
            for k in names:
                check_tensor(k, pick(outs[k]), o64[k], o32[k])
            check_input_grads([pick(gin[k]) for k in names], [g64[k] for k in names], [g32[k] for k in names])
        if G == 1:
            check_param_grads(gparam, p64, p32)
        else:      # the same graph G times: parameter gradients are G times the single-graph ones
            check_param_grads({k: v / G for k, v in gparam.items()}, p64, p32)
    if case["training"] and case.get("normed", True) and G == 1:
        for k, v in b64.items():
            if k.endswith("num_batches_tracked"):
                assert int(buffers[k]) == int(v), k
            else:
                assert nerr(buffers[k], v) < 1e-4, k


@pytest.mark.gpu
@pytest.mark.parametrize("case_name", sorted(CASES))
def test_block_parity_on_split_fibres(case_name):
    """The whole Block: the EdgeModel norm deferred into the SModel edge pass and the x_e' gradients added up inside the
    backward kernels run on split tiles too."""
    from tests.test_gpu_parity import run_ours_block
    dev = _cuda()
    case = high_degree_case(**CASES[case_name])
    _check_block(case, run_ours_block(case, dev), _block_oracle(case))


@pytest.mark.gpu
def test_block_parity_on_split_fibres_two_graphs():
    from tests.test_gpu_parity import run_ours_block
    dev = _cuda()
    case = high_degree_case(seed=21, kind="mixed", T=600)
    _check_block(case, run_ours_block(case, dev, G=2), _block_oracle(case), G=2)


@pytest.mark.gpu
def test_split_fibres_are_bitwise_deterministic():
    from tests.test_gpu_parity import run_ours_block
    dev = _cuda()
    ei = high_degree_case(seed=31, kind="mixed", T=600)["edge_index"]
    for seed in (31, 32):                  # one edge_index, inputs and weights of two seeds
        case = high_degree_case(seed=seed, kind="mixed", T=600)
        case["edge_index"] = ei
        a = run_ours_block(case, dev)
        b = run_ours_block(case, dev)
        for x, y in zip(a[:3], b[:3]):
            for k in x:
                assert torch.equal(x[k], y[k]), (seed, k)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(TILE_TABLES))
def test_device_tile_table_equals_the_expected_table(name):
    from pfs_neural_net_b200 import topology
    dev = _cuda()
    degrees, table = TILE_TABLES[name]
    T = max(degrees) + 1
    ei = edge_index_from_degrees(degrees, T, torch.Generator().manual_seed(1)).to(dev)
    topo = topology.Topology(ei, len(degrees), T)
    t = topo.struct(1, 10)
    if max(degrees) <= TILE:           # whole fibres only: the table of pfs_build_topology, no split fields
        assert t.nsplit == 0 and not t.tile_q and topo._split is None
        assert topo.csr()["tile_fibre"][:topo.ntiles + 1].tolist() == table["tile_fibre"]
        return
    got = {k: v.tolist() for k, v in topo.split_tiles().items() if torch.is_tensor(v)}
    assert got == table
    assert (t.ntiles, t.nsplit, t.nslots) == (len(table["tile_slot"]), len(table["split_fibre"]), table["split_ptr"][-1])


@pytest.mark.gpu
def test_device_tile_table_heavy_tailed():
    from pfs_neural_net_b200 import topology
    dev = _cuda()
    g = torch.Generator().manual_seed(9)
    degrees = (torch.rand(4000, generator=g) ** 6 * 3000).long().tolist()
    degrees[5::101] = [0] * len(degrees[5::101])
    ei = edge_index_from_degrees(degrees, 3000, g).to(dev)
    topo = topology.Topology(ei, len(degrees), 3000)
    got = {k: v.tolist() for k, v in topo.split_tiles().items() if torch.is_tensor(v)}
    assert got == pack_split_tiles(degrees)


@pytest.mark.gpu
def test_gnn_and_loss_with_300_classes():
    """train.py with NCLASSES = 300: GNN forward, loss.loss_function and backward on the complete 40 x 300 graph
    against oracle/loss_oracle.py (loss, edge times, parameter gradients)."""
    from oracle import block_oracle as bo
    from oracle import loss_oracle as lo
    from pfs_neural_net_b200 import gnn as pg, loss as pl
    from tests.test_gpu_parity import check_param_grads, check_tensor
    dev = _cuda()
    S, T, F, B = 40, 300, 10, 2
    torch.manual_seed(0)
    model = pg.GNN(B=B, Fdim=F, T=T, F_s=1, F_t=2).to(dev).train()
    g = torch.Generator().manual_seed(1)
    class_info = torch.stack([0.5 + 3 * torch.rand(T, generator=g), 50 + 400 * torch.rand(T, generator=g)], 1)
    ei = bo.complete_bipartite(S, T)
    x_s = torch.arange(S, dtype=torch.float32).reshape(-1, 1)
    x_e = 2 + 8 * torch.rand(S * T, F, generator=g)
    u = torch.zeros(1, F)
    noise = torch.rand(S * T, generator=g)
    state = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    graph = pg.BipartiteData(ei.to(dev), x_s.to(dev), class_info.to(dev), x_e.to(dev), u.to(dev))
    out = model(graph)
    time = model.edge_prediction(out.x_e, scale=42 / T).squeeze(-1)
    loss, utils = pl.loss_function(model, out, class_info.to(dev), noise=noise.to(dev))
    loss.backward()
    mine = {k: p.grad for k, p in model.named_parameters() if p.grad is not None}

    def oracle(dtype):
        sd = bo.cast_state(state, dtype)
        params = {k: v.clone().requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running" not in k}
        full = dict(sd)
        full.update(params)
        xs, xt, xe, uu = bo.gnn_forward(full, B, ei, x_s.to(dtype), class_info.to(dtype), x_e.to(dtype), u.to(dtype),
                                        training=True, buffers={})
        tm = bo.edge_prediction(full, xe, 42 / T).squeeze(-1)
        r = lo.loss_terms(tm, noise.to(dtype), class_info.to(dtype), ei, S, T)
        r["loss"].backward()
        return r, tm.detach(), {k: p.grad for k, p in params.items() if p.grad is not None}

    r64, t64, p64 = oracle(torch.float64)
    r32, t32, p32 = oracle(torch.float32)
    check_tensor("time", time, t64, t32)
    scale = max(abs(r64["loss"].item()), 2000.0 * abs(r64["totutils"].item()), r64["fiber_penalty"].item(),
                r64["variance"].item())
    err32 = abs(r32["loss"].item() - r64["loss"].item())
    assert abs(loss.item() - r64["loss"].item()) <= max(1e-4 * scale, 3 * err32)
    assert abs(utils.item() - r64["totutils"].item()) <= max(1e-4 * abs(r64["totutils"].item()),
                                                             3 * abs(r32["totutils"].item() - r64["totutils"].item()))
    check_param_grads(mine, p64, p32)


# ----------------------------------------------------------------------------------------------------------------
# full size: the complete 12 500 x 512 graph at Fdim 10 (every fibre split in two), invariants only
# ----------------------------------------------------------------------------------------------------------------
def _full_block(F, dev):
    from pfs_neural_net_b200 import gnn
    torch.manual_seed(0)
    blk = gnn.Block(F)
    g = torch.Generator().manual_seed(1)
    for m in blk.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.weight.data = 0.5 + torch.rand(m.weight.shape, generator=g)
            m.bias.data = 2 * torch.rand(m.bias.shape, generator=g) - 1
    return blk.to(dev).train()


def _run(blk, state, ei, ins, ups):
    blk.load_state_dict(state)
    for p in blk.parameters():
        p.grad = None
    xs = [t.detach().clone().requires_grad_(True) for t in ins]
    _, o_s, o_t, o_e, o_u = blk((ei, *xs))
    torch.autograd.backward([o_s, o_t, o_e, o_u], ups)
    torch.cuda.synchronize()
    return [o.detach() for o in (o_s, o_t, o_e, o_u)], [x.grad for x in xs], \
        {k: p.grad.clone() for k, p in blk.named_parameters()}


def _close(a, b, tol, what):
    err = (a.double() - b.double()).abs().max().item() / max(b.double().abs().max().item(), 1e-30)
    assert err < tol, (what, err)


def _close_params(a, b, what, tol=1e-3):
    """parameter gradients norm-wise; a bias in front of a train-mode BatchNorm (analytically zero) on its weight's scale"""
    for k in b:
        scale = max(b[k].abs().max().item(), b[k[:-4] + "weight"].abs().max().item() if k.endswith("bias") else 0.0)
        err = (a[k].double() - b[k].double()).abs().max().item() / max(scale, 1e-30)
        assert err < tol, (what, k, err)


@pytest.mark.gpu
def test_full_size_complete_512_classes_fp32():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    if torch.cuda.get_device_properties(0).total_memory < 20 * 2 ** 30:
        pytest.skip("needs 20 GB of device memory")
    dev = torch.device("cuda:0")
    S, T, F = 12500, 512, 10
    E = S * T
    blk = _full_block(F, dev)
    state = {k: v.clone() for k, v in blk.state_dict().items()}
    ei = torch.cartesian_prod(torch.arange(S), torch.arange(T)).T.contiguous().to(dev)
    gen = torch.Generator(device=dev).manual_seed(3)
    ins = [torch.randn(S, F, generator=gen, device=dev), torch.randn(T, F, generator=gen, device=dev),
           torch.randn(E, F, generator=gen, device=dev), torch.randn(1, F, generator=gen, device=dev)]
    ups = [torch.randn(t.shape, generator=gen, device=dev) for t in ins]
    out1, gin1, gp1 = _run(blk, state, ei, ins, ups)
    for t in out1 + gin1 + list(gp1.values()):
        assert torch.isfinite(t).all()
    # run to run: bit-exact
    out2, gin2, gp2 = _run(blk, state, ei, ins, ups)
    for a, b in zip(out1 + gin1, out2 + gin2):
        assert torch.equal(a, b)
    for k in gp1:
        assert torch.equal(gp1[k], gp2[k]), k
    del out2, gin2, gp2
    # relabelled fibres: x_s' and the edge rows permute along, x_t', u' and the parameter gradients stay (sums over
    # fibres reassociated)
    perm = torch.randperm(S, generator=torch.Generator().manual_seed(4)).to(dev)
    eperm = (perm[:, None] * T + torch.arange(T, device=dev)[None, :]).reshape(-1)
    ins_p = [ins[0][perm].contiguous(), ins[1], ins[2][eperm].contiguous(), ins[3]]
    ups_p = [ups[0][perm].contiguous(), ups[1], ups[2][eperm].contiguous(), ups[3]]
    out3, gin3, gp3 = _run(blk, state, ei, ins_p, ups_p)
    _close(out3[0], out1[0][perm], 1e-4, "x_s")
    _close(out3[2], out1[2][eperm], 1e-4, "x_e")
    _close(out3[1], out1[1], 1e-4, "x_t")
    _close(out3[3], out1[3], 1e-4, "u")
    _close(gin3[0], gin1[0][perm], 1e-3, "grad x_s")
    _close(gin3[2], gin1[2][eperm], 1e-3, "grad x_e")
    _close(gin3[1], gin1[1], 1e-3, "grad x_t")
    _close_params(gp3, gp1, "fibre permutation")
    del out3, gin3, gp3
    # edge order: a shuffled edge list against the fibre-major one (CSR path on both).  The edges of a fibre are then
    # visited in another order and fall into other chunks, so the fp32 sums of the fibre moments change in their last
    # bits.  The reference's var = E[m^2] - mean^2 (kept as is) cancels in fp32 where a message feature has |mean| >>
    # std, and the std / skew / kurtosis backward amplifies that in the gradients; the outputs stay at 1e-4.  The
    # gradient bounds are those of the same check on the bf16 path (tests/test_gpu_full_size.py).
    order = torch.randperm(E, generator=torch.Generator().manual_seed(5)).to(dev)
    ei_s = ei[:, order].contiguous()
    ins_s = [ins[0], ins[1], ins[2][order].contiguous(), ins[3]]
    ups_s = [ups[0], ups[1], ups[2][order].contiguous(), ups[3]]
    out4, gin4, gp4 = _run(blk, state, ei_s, ins_s, ups_s)
    _close(out4[0], out1[0], 1e-4, "x_s")
    _close(out4[2], out1[2][order], 1e-4, "x_e")
    _close(out4[1], out1[1], 1e-4, "x_t")
    _close(out4[3], out1[3], 1e-4, "u")
    _close(gin4[0], gin1[0], 6e-2, "grad x_s")
    _close(gin4[2], gin1[2][order], 6e-2, "grad x_e")
    _close(gin4[1], gin1[1], 6e-2, "grad x_t")
    _close_params(gp4, gp1, "edge order", 5e-2)
