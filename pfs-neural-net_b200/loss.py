"""The training loss of the reference (`softfloor` + `loss_function`, reference src/train.py:21-80) on
the B200 kernels `pfs_loss_fwd` / `pfs_loss_bwd` (SURVEY.md section 8f, row N1): the step right after the
message-passing path, consuming `GNN.edge_prediction`'s times.

`loss_function(gnn, graph, class_info, ...)` keeps the reference's argument meaning and return values
(`(loss, totutils)`, or the 7-tuple of `finaloutput=True`); the module-level globals the reference
reads (`gnn`, NFIBERS, NCLASSES, NFIELDS, TOTAL_TIME, wutils, wvar; src/config.py:16-28) are explicit
arguments with the reference's values as defaults.  The uniform noise of `softfloor` is drawn with
`torch.rand_like` exactly where the reference draws it (so a seeded run consumes the generator the
same way) or can be passed in.  fp32; no CPU fallback.

The edge order is the canonical dense one (e = k*T + i, which the reference reshapes to [NFIBERS, NCLASSES]) or any
edge list: `loss_from_times(..., edge_index=...)`, and `loss_function` on a graph whose `edge_index` is not canonical
(a class-permuted file such as the reference's graphs/graph-0.pt, or a sparse visibility graph).  On an edge list the
variance runs over the fibre x class matrix of cells c_ki = sum of time2 over the edges (k, i), 0 where fibre k has no
edge to class i (DESIGN.md section 8b): on any permutation of the complete graph that is the reference loss of the
un-permuted graph.

Both functions also take a batch of G graphs that share one `edge_index` (the leading graph dimension of
`Loader.collate`): edge times [G, E], one class table [T, 2] for all graphs or one per graph [G, T, 2].  Each
graph gets its own loss, computed exactly as a call on that graph alone would compute it (bitwise), in the same
five kernel launches whatever G is.

Inside `shard.fibre_sharded()` (one graph whose fibres are split over the ranks, DESIGN.md section 7) both functions
compute the loss of the WHOLE graph on every rank from the rank's own fibres: each rank reduces its fibres to a record
of 2 + 3T doubles, one all-reduce makes every record visible to every rank, and a merge in rank order gives every rank
bitwise the same class statistics, scalars and loss.  The gradient w.r.t. the local edge times is that of the global
loss, so the Blocks' gradient all-reduces sum the parts of one function.  The graph is a slab of the canonical order, or
an edge list split by `shard.partition_fibres` whose `edge_ids` (the global positions of the rank's edges) are passed in:
every cell c_ki lies on the rank that owns fibre k, so the records need no other exchange.
"""
import collections
import ctypes as ct

import torch

from . import _abi
from . import shard as _shard

NOISELEVEL = 0.3          # softfloor default (reference src/train.py:21)


class LossFunction(torch.autograd.Function):
    """loss(time): forward = pfs_loss_fwd, backward = pfs_loss_bwd (gradient w.r.t. the edge times only).

    G = 0: one graph (time [S*T], hours / counts [T]; the loss is a scalar).  G >= 1: a batch (time [G, S*T], hours /
    counts [T] shared or [G, T]; the loss is [G] and every other output gains the leading G).
    S_total > 0: this rank's S fibres of a graph of S_total fibres sharded over the active group (G = 0): the forward is
    pfs_loss_shard_fwd, the record exchange (shard.exchange_rows) and pfs_loss_shard_merge.
    edges: None (canonical order, E = S*T) or an edge list {"E": edges per graph, and the int32 CSR / CSC arrays of
    Topology.csr()}; the forward saves the per-edge cell values for the backward.  An edge list with S_total > 0 is this
    rank's edges of a sharded edge list: pfs_loss_list_shard_fwd, the exchange and pfs_loss_shard_merge, and the backward
    pfs_loss_list_shard_bwd."""

    @staticmethod
    def forward(ctx, time, noise, hours, counts, G, S, T, consts, S_total, edges=None):
        for t, n in ((time, "time"), (noise, "noise"), (hours, "hours"), (counts, "counts")):
            if not t.is_cuda:
                raise _abi.PfsError("pfs_b200 loss needs CUDA tensors, %s is on %s (no CPU fallback)" % (n, t.device))
            if t.dtype != torch.float32:
                raise _abi.PfsError("pfs_b200 loss is fp32, %s is %s" % (n, t.dtype))
        time, noise, hours, counts = (t.contiguous() for t in (time, noise, hours, counts))
        E = S * T if edges is None else edges["E"]
        nt = max(G, 1) * T if hours.dim() == 2 else T
        if time.numel() != max(G, 1) * E or noise.numel() != time.numel() or hours.numel() != nt or counts.numel() != nt:
            raise _abi.PfsError("loss: expected %d edge times / noise values and %d class rows" % (max(G, 1) * E, nt))
        dev = time.device
        f32 = dict(dtype=torch.float32, device=dev)
        lib = _abi.load_library()
        a = _abi.LossArgs()
        a.S, a.T, a.G, a.class_tables = S, T, G, int(hours.dim() == 2)
        lead = (G,) if G else ()
        out = dict(galaxies=torch.empty(lead + (E,), **f32), time2=torch.empty(lead + (E,), **f32),
                   fibre_time=torch.empty(lead + (S,), **f32), n_prime=torch.empty(lead + (T,), **f32),
                   class_mean=torch.empty(lead + (T,), **f32), class_coef=torch.empty(lead + (T,), **f32),
                   scalars=torch.zeros(lead + (8,), **f32))
        if edges is None:
            ws = torch.empty(max(G, 1) * lib.pfs_loss_workspace_bytes(S, T), dtype=torch.uint8, device=dev)
        else:
            out["cell_time"] = torch.empty(lead + (E,), **f32)
            ws = torch.empty(max(G, 1) * lib.pfs_loss_list_workspace_bytes(T), dtype=torch.uint8, device=dev)
            _set_edges(a, edges)
        for k, v in dict(time=time, noise=noise, hours=hours, counts=counts, **out).items():
            setattr(a, k, v.data_ptr())
        sharp_dev = consts.get("sharpness_dev")
        for k, v in consts.items():
            if k != "sharpness_dev":
                setattr(a, k, float(v))
        a.sharpness_dev = _abi.ptr(sharp_dev)
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        with torch.cuda.device(dev):
            a.stream = torch.cuda.current_stream(dev).cuda_stream
            if S_total:
                record = torch.empty(2 + 3 * T, dtype=torch.float64, device=dev)
                a.S_total, a.world, a.shard_record = S_total, _shard.world_size(), record.data_ptr()
                fwd = "pfs_loss_shard_fwd" if edges is None else "pfs_loss_list_shard_fwd"
                _abi.check(getattr(lib, fwd)(ct.byref(a)), fwd)
                records = _shard.exchange_rows(record)                  # [world, 2 + 3T], rank order, on every rank
                a.shard_records = records.data_ptr()
                if edges is not None:                 # the merge reads the records alone: E = 0, no edge arrays
                    a.E = 0
                    for k in _EDGE_ARRAYS + ("cell_time",):
                        setattr(a, k, None)
                _abi.check(lib.pfs_loss_shard_merge(ct.byref(a)), "pfs_loss_shard_merge")
            else:
                _abi.check(lib.pfs_loss_fwd(ct.byref(a)), "pfs_loss_fwd")
        ctx.G, ctx.S, ctx.T, ctx.S_total, ctx.consts, ctx.edges = G, S, T, S_total, dict(consts), edges
        ctx.save_for_backward(time, noise, hours, counts, out["time2"], out["fibre_time"], out["class_mean"], out["class_coef"],
                              out.get("cell_time"))
        sc = out["scalars"]
        ctx.mark_non_differentiable(sc, out["n_prime"], out["fibre_time"], out["time2"])
        return sc[..., 0].clone(), sc, out["n_prime"], out["fibre_time"], out["time2"]

    @staticmethod
    def backward(ctx, g_loss, *_):
        time, noise, hours, counts, time2, fibre_time, class_mean, class_coef, cell_time = ctx.saved_tensors
        dev = time.device
        g_time = torch.empty_like(time)
        gl = g_loss.detach().to(torch.float32).reshape(-1).contiguous()
        a = _abi.LossArgs()
        a.S, a.T, a.G, a.class_tables, a.S_total = ctx.S, ctx.T, ctx.G, int(hours.dim() == 2), ctx.S_total
        for k, v in dict(time=time, noise=noise, hours=hours, counts=counts, time2=time2, fibre_time=fibre_time,
                         class_mean=class_mean, class_coef=class_coef, g_loss=gl, g_time=g_time).items():
            setattr(a, k, v.data_ptr())
        if ctx.edges is not None:
            _set_edges(a, ctx.edges)
            a.cell_time = cell_time.data_ptr()
        for k, v in ctx.consts.items():
            if k != "sharpness_dev":
                setattr(a, k, float(v))
        a.sharpness_dev = _abi.ptr(ctx.consts.get("sharpness_dev"))
        with torch.cuda.device(dev):
            a.stream = torch.cuda.current_stream(dev).cuda_stream
            bwd = "pfs_loss_list_shard_bwd" if ctx.edges is not None and ctx.S_total else "pfs_loss_bwd"
            _abi.check(getattr(_abi.load_library(), bwd)(ct.byref(a)), bwd)
        return g_time, None, None, None, None, None, None, None, None, None


_EDGE_ARRAYS = ("csr_rowptr", "csr_eid", "csr_src", "csr_tgt", "csc_colptr", "csc_q")


def _set_edges(a, edges):
    a.E = edges["E"]
    for k in _EDGE_ARRAYS:
        setattr(a, k, edges[k].data_ptr())


def _edge_list(edge_index, S, T):
    """the LossFunction `edges` of an edge_index [2, E]: the cached CSR / CSC arrays of its Topology (built once per
    edge_index, in the first call; a captured step finds them cached)"""
    from .topology import get_topology
    topo = get_topology(edge_index, S, T)
    arrays = topo.csr()
    return dict(E=topo.E, **{k: arrays[k] for k in _EDGE_ARRAYS})


_EDGE_IDS_CHECKED = collections.OrderedDict()


def _check_edge_ids(edge_ids, E, E_total, device):
    """`edge_ids` of a sharded edge list: 1-D int64 on `device`, one per local edge, every value in [0, E_total).  The
    range is read once per tensor (one host synchronisation) and remembered, like a Topology: an index out of range would
    fault the device in the noise gather."""
    if not torch.is_tensor(edge_ids) or edge_ids.dtype != torch.int64 or edge_ids.dim() != 1 or edge_ids.device != device:
        raise _abi.PfsError("loss: edge_ids are the global positions of this rank's edges, a 1-D int64 tensor on %s; got %s"
                            % (device, (edge_ids.dtype, tuple(edge_ids.shape), str(edge_ids.device))
                               if torch.is_tensor(edge_ids) else type(edge_ids).__name__))
    if edge_ids.numel() != E:
        raise _abi.PfsError("loss: edge_ids has %d entries for %d local edges" % (edge_ids.numel(), E))
    key = (edge_ids.data_ptr(), edge_ids._version, E, E_total, str(device))
    if key in _EDGE_IDS_CHECKED:
        _EDGE_IDS_CHECKED.move_to_end(key)
        return
    lo, hi = torch.stack([edge_ids.min(), edge_ids.max()]).tolist()
    if lo < 0 or hi >= E_total:
        raise _abi.PfsError("loss: edge_ids out of range [%d, %d] for %d edges over all shards" % (lo, hi, E_total))
    _EDGE_IDS_CHECKED[key] = edge_ids             # keeps the tensor alive, so its address cannot be recycled under the key
    while len(_EDGE_IDS_CHECKED) > 16:
        _EDGE_IDS_CHECKED.popitem(last=False)


def _graph_rows(x, E):
    """[G, E] view of a batch given as [G, E] or [G, E, 1]; None when `x` is not a batch of E-edge graphs."""
    if x.dim() == 3 and x.shape[2] == 1:
        x = x.squeeze(2)
    return x if x.dim() == 2 and x.shape[1] == E else None


def _batched_loss(time, class_info, S, T, nfields, consts, noise, edges=None):
    E = S * T if edges is None else edges["E"]
    t = _graph_rows(time, E)
    if t is None:
        raise _abi.PfsError("loss: a batch of edge times is [G, %d] or [G, %d, 1], got %s" % (E, E, tuple(time.shape)))
    G = t.shape[0]
    if G < 1:
        raise _abi.PfsError("loss: empty batch of graphs")
    if class_info.dim() not in (2, 3) or tuple(class_info.shape[-2:-1]) != (T,) or class_info.shape[-1] < 2 or \
            (class_info.dim() == 3 and class_info.shape[0] != G):
        raise _abi.PfsError("loss: class_info is [%d, 2] (shared) or [%d, %d, 2] (per graph), got %s"
                            % (T, G, T, tuple(class_info.shape)))
    if t.dtype != torch.float32:
        t = t.float()
    if noise is None:
        noise = torch.rand_like(t)                # one draw for the whole batch, see loss_from_times
    else:
        n = _graph_rows(noise, E)
        if n is None or n.shape[0] != G:
            raise _abi.PfsError("loss: noise has the shape of the edge times [%d, %d], got %s" % (G, E, tuple(noise.shape)))
        noise = n
    hours = class_info[..., 0].to(torch.float32)
    counts = (class_info[..., 1] / nfields).to(torch.float32)
    return LossFunction.apply(t, noise.to(torch.float32), hours, counts, G, S, T, consts, 0, edges)


def loss_from_times(time, class_info, nfibers, nclasses, nfields=10, total_time=42, wutils=2000.0, wvar=1.0, pclass=0.1,
                    pfiber=1.0, sharpness=0.5, noise=None, edge_index=None, edge_ids=None):
    """Loss terms from the edge times [E] (or [E,1]); returns (loss, scalars, n_prime, fibre_time, time2) where
    scalars = [loss, totutils, class_penalty, fibre_penalty, variance, #minima, 0, 0].

    A batch of G graphs: `time` [G, E] (or [G, E, 1]), `class_info` [T, 2] for all graphs or [G, T, 2]; returns
    losses [G] (differentiable), scalars [G, 8], n_prime [G, T], fibre_time [G, S], time2 [G, E].  Graph g's results
    are bitwise those of a single-graph call on time[g] with the same noise.  `noise` has the shape of `time`; when
    it is omitted it is drawn by ONE torch.rand_like over the whole batch, which is not the random stream of G
    separate single-graph calls (those draw E values each, interleaved with whatever else uses the generator):
    pass `noise` to reproduce them.

    Inside `shard.fibre_sharded()`: `time` holds this rank's `nfibers` fibres (a contiguous fibre range, canonical order)
    of one graph; the loss, scalars and n_prime are those of the whole graph (bitwise the same on every rank),
    fibre_time and time2 the local rows.  Without `noise` the whole graph's S_total * T draws are made by one
    torch.rand and this rank takes its slice [f0 * T, f1 * T), so a run seeded alike on every rank draws bitwise the
    noise of the single-GPU run and no two shards share draws.  A batch of graphs is refused.

    `edge_index` [2, E] (int64, on the device): the edges in any order, edge e = (fibre edge_index[0, e], class
    edge_index[1, e]); `time` is [E], [E, 1], [G, E] or [G, E, 1] in that order, and so are `noise` and time2.  None:
    the canonical dense order e = k*T + i.

    `edge_ids` [E] (int64, on the device; only inside `shard.fibre_sharded()`): this rank's edges of an edge list sharded
    over fibre ranges are `edge_index` (local fibres numbered from 0, `nfibers` of them) and their positions in the whole
    graph's edge list are `edge_ids` -- the second and third values of `shard.partition_fibres`.  As for the canonical
    sharded graph, the loss, scalars and n_prime are those of the whole graph (bitwise the same on every rank), fibre_time
    the local rows and time2 the local edges in local order.  Without `noise` the whole edge list's draws are made by one
    torch.rand and this rank takes [edge_ids], so a run seeded alike on every rank draws bitwise the noise of the
    single-GPU run.  Every rank of the group must pass `edge_ids` (or none may): the path decides which collectives run.
    Inside the scope an edge list without `edge_ids` is refused; outside it, `edge_ids` is."""
    consts = dict(total_time=total_time, wutils=wutils, wvar=wvar, pclass=pclass, pfiber=pfiber, noiselevel=NOISELEVEL)
    if torch.is_tensor(sharpness):                # device scalar: the value is read by the kernels (CUDA-graph replays)
        consts.update(sharpness=0.0, sharpness_dev=sharpness.to(torch.float32).reshape(1))
    else:
        consts.update(sharpness=sharpness)
    nfibers, nclasses = int(nfibers), int(nclasses)
    sharded = _shard.active()
    edges = None
    if edge_ids is not None:
        if not sharded:
            raise _abi.PfsError("loss: edge_ids (the global positions of a shard's edges) are only taken inside "
                                "shard.fibre_sharded(); outside it there is no shard")
        if edge_index is None:
            raise _abi.PfsError("loss: edge_ids are the global positions of the edges of edge_index, which is missing")
    if edge_index is not None:
        if sharded and edge_ids is None:
            raise _abi.PfsError("loss: an edge list cannot be fibre-sharded without the global positions of its edges: the "
                                "canonical sharded loss splits the order e = k*T + i into contiguous fibre ranges; pass "
                                "edge_ids from shard.partition_fibres")
        edges = _edge_list(edge_index, nfibers, nclasses)
    E = nfibers * nclasses if edges is None else edges["E"]
    if time.dim() == 3 or (time.dim() == 2 and time.shape[1] == E):
        if sharded:
            raise _abi.PfsError("loss: a fibre-sharded graph is one graph per call, not a batch of %d" % time.shape[0])
        return _batched_loss(time, class_info, nfibers, nclasses, nfields, consts, noise, edges)
    time = time.reshape(-1)
    if time.dtype != torch.float32:
        time = time.float()                       # bf16 head output: dtype plumbing, the loss itself is fp32
    S_total = _shard.total_count(nfibers) if sharded else 0      # cached: no host synchronisation per step
    if edge_ids is not None:
        E_total = _shard.total_count(E, kind="edges")                # cached apart from the fibre counts
        _check_edge_ids(edge_ids, E, E_total, time.device)
    if noise is None:
        if edge_ids is not None:                  # the whole edge list's draw, this rank's edges
            noise = torch.rand(E_total, dtype=torch.float32, device=time.device)[edge_ids]
        elif sharded:                             # the whole graph's draw, this rank's slice
            f0 = sum(_shard.shard_counts(nfibers)[:_shard.rank()])       # cached like S_total
            noise = torch.rand(S_total * nclasses, dtype=torch.float32, device=time.device)
            noise = noise[f0 * nclasses:(f0 + nfibers) * nclasses]
        else:
            noise = torch.rand_like(time)         # the draw of softfloor, reference src/train.py:22
    hours = class_info[:, 0].to(torch.float32)
    counts = (class_info[:, 1] / nfields).to(torch.float32)
    return LossFunction.apply(time, noise.reshape(-1).to(torch.float32), hours, counts, 0, nfibers, nclasses, consts,
                              S_total, edges)


def loss_function(gnn, graph, class_info, pclass=0.1, pfiber=1.0, sharpness=0.5, finaloutput=False, *, nfibers=None,
                  nclasses=None, nfields=10, total_time=42, wutils=2000.0, wvar=1.0, noise=None, reduction="sum",
                  edge_ids=None):
    """reference src/train.py:29-80 with its globals as arguments (`gnn` first; NFIBERS / NCLASSES default to the
    graph's node counts).

    On a collated batch (`Loader.collate`: x_e [G, E, F]) `class_info` is [T, 2] or [G, T, 2] and `noise` [G, E];
    returns (loss, utilities [G]) where loss is the sum of the G per-graph losses (`reduction="sum"`: the parameter
    gradients are those of the G single-graph losses backpropagated one after the other, as the Block sums them over
    graphs) or their mean (`"mean"`).  With `finaloutput=True` every per-graph diagnostic carries the leading G.

    Inside `shard.fibre_sharded()`, `edge_ids` (the third value of `shard.partition_fibres`) makes the graph this rank's
    part of an edge list sharded over fibre ranges: the loss takes the edge-list path of `loss_from_times` even where the
    rank's local edge_index happens to be canonical (a complete slab of a sparse graph), so every rank of the group runs
    the same collectives."""
    from .topology import get_topology
    if reduction not in ("sum", "mean"):
        raise ValueError("loss_function: reduction is 'sum' or 'mean', got %r" % (reduction,))
    batched = graph.x_e.dim() == 3
    nclasses = int(nclasses if nclasses is not None else graph.x_t.shape[-2])
    nfibers = int(nfibers if nfibers is not None else graph.x_s.shape[-2])
    topo = get_topology(graph.edge_index, nfibers, nclasses)
    edge_index = None
    if edge_ids is not None:
        edge_index = graph.edge_index           # one shard of an edge list, canonical or not (loss_from_times checks)
    elif not topo.canonical:
        if _shard.active():
            raise _abi.PfsError("loss: a fibre-sharded graph needs the canonical dense edge order e = k*T + i, because the "
                                "sharded loss splits that order into contiguous fibre ranges; this graph's edge_index is "
                                "not canonical (pass edge_ids from shard.partition_fibres to train an edge list)")
        edge_index = graph.edge_index           # any edge list: the cell-matrix loss of DESIGN.md section 8b
    time = gnn.edge_prediction(graph.x_e, scale=total_time / nclasses).squeeze(-1)
    loss, sc, n_prime, fibre_time, time2 = loss_from_times(time, class_info, nfibers, nclasses, nfields, total_time, wutils,
                                                            wvar, pclass, pfiber, sharpness, noise, edge_index, edge_ids)
    if batched:
        loss = loss.sum() if reduction == "sum" else loss.mean()
    if not finaloutput:
        return loss, sc[..., 1]
    counts = class_info[..., 1] / nfields
    comp = (n_prime / counts).detach().cpu().numpy()
    return loss, sc[..., 1], comp, n_prime, fibre_time.detach().cpu().numpy(), time2, sc[..., 4]
