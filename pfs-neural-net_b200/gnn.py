"""Drop-in replacement for the reference's `src/gnn.py` module surface, running on B200 kernels.

Same class names, constructor signatures, child-module names and parameter registration order as
reference src/gnn.py:7-325, so `train.py` (`from gnn import GNN, BipartiteData`) and the shipped
checkpoints (`params/model_gnn_0.pth`, `models/model_gnn_0.pth`) load with `strict=True` and Adam's
index-keyed state lands on the right tensors.  What differs is what runs underneath: every update
module's forward/backward is one call into libpfs_b200.so (hand-written sm_100a CUDA; see
functional.py and include/pfs_b200.h).  There is no torch_scatter / torch_geometric dependency and
no CPU fallback: calling a module on CPU tensors raises.

Extension over the reference: every module also accepts a leading graph dimension
(x_s [G,S,F], x_t [G,T,F], x_e [G,E,F], u [G,1,F] or [G,F]) for G independent graphs that share
`edge_index` and weights -- BatchNorm statistics stay per graph (the reference runs one graph per
step) and parameter gradients are summed over the graphs.
"""
import torch
import torch.nn.functional as Fn

from . import _abi
from . import functional as pf
from . import shard as _shard
from . import wide as pw
from .topology import get_topology

# same device pick as reference src/config.py:4-9 (captured at import by BipartiteData there)
if torch.cuda.is_available():
    device = torch.device('cuda')
else:
    device = torch.device('cpu')


class BipartiteData:
    """Attribute bag of reference src/gnn.py:7-47 (there a torch_geometric `Data`): edge_index [2,E]
    (row 0 = fibre, row 1 = class), x_s, x_t, x_e, x_u; every tensor is moved to `device`."""

    def __init__(self, edge_index=None, x_s=None, x_t=None, x_e=None, x_u=None):
        if edge_index is not None:
            self.edge_index = edge_index.to(device)
        if x_s is not None:
            self.x_s = x_s.to(device)
        if x_t is not None:
            self.x_t = x_t.to(device)
            self.num_nodes = len(self.x_t)
        if x_e is not None:
            self.x_e = x_e.to(device)
        if x_u is not None:
            self.x_u = x_u.to(device)

    def __inc__(self, key, value, *args):
        # reference src/gnn.py:32-47: batching offsets for edge_index
        if key == 'edge_index':
            return torch.tensor([[self.x_s.size(0)], [self.x_t.size(0)]]).to(device)
        return 0

    def to(self, dev, *args, **kwargs):
        for k, v in list(self.__dict__.items()):
            if torch.is_tensor(v):
                setattr(self, k, v.to(dev, *args, **kwargs))
        return self

    def keys(self):
        return [k for k, v in self.__dict__.items() if torch.is_tensor(v)]


class Loader(torch.utils.data.Dataset):
    """List wrapper of reference src/gnn.py:49-63."""

    def __init__(self, graphs_list=None):
        self.graphs_list = graphs_list

    def __len__(self):
        return len(self.graphs_list)

    def __getitem__(self, idx):
        return self.graphs_list[idx]

    @staticmethod
    def collate(graphs):
        """Batch graphs that share one `edge_index` into leading-dimension tensors x_s [G,S,F], x_t [G,T,F],
        x_e [G,E,F], x_u [G,1,F] -- the form every module of this file accepts (SURVEY.md section 8f row N4).  Unlike
        the reference's PyG collation (`__inc__`, src/gnn.py:32-47, which concatenates nodes and cannot carry one
        global row per graph through `u.expand`, src/gnn.py:100), every graph keeps its own global features and its
        own BatchNorm statistics, exactly as if the graphs were run one after the other."""
        if not graphs:
            raise ValueError("no graphs to collate")
        ei = graphs[0].edge_index
        for g in graphs[1:]:
            if g.edge_index.shape != ei.shape or not torch.equal(g.edge_index, ei):
                raise ValueError("collate() batches graphs with identical edge_index; shard different topologies "
                                 "over separate calls")
        out = BipartiteData.__new__(BipartiteData)
        out.edge_index = ei
        for k in ("x_s", "x_t", "x_e", "x_u"):
            setattr(out, k, torch.stack([getattr(g, k) for g in graphs]))
        out.num_nodes = graphs[0].x_t.shape[0]
        return out

    def batches(self, batch_size):
        """Collated batches in list order (the last one may be smaller)."""
        for i in range(0, len(self.graphs_list), batch_size):
            yield Loader.collate(self.graphs_list[i:i + batch_size])


class MLP(torch.nn.Sequential):
    """Linear -> LeakyReLU(0.1) -> Linear with children '0', '1', '2' (reference src/gnn.py:65-71)."""

    def __init__(self, D1, D2, D3):
        super(MLP, self).__init__(torch.nn.Linear(D1, D2), torch.nn.LeakyReLU(0.1), torch.nn.Linear(D2, D3))


def _batched(x_s, x_t, edge_attr, u):
    """Normalise the reference's 2-D calling convention to [G, rows, F]; returns the flag to undo it."""
    single = x_s.dim() == 2
    if single:
        x_s, x_t, edge_attr = x_s.unsqueeze(0), x_t.unsqueeze(0), edge_attr.unsqueeze(0)
        if u.shape[0] != 1:
            raise RuntimeError("global features with %d rows cannot be expanded over one graph "
                               "(reference src/gnn.py:100 fails the same way)" % u.shape[0])
        u = u.reshape(1, -1)
    else:
        u = u.reshape(x_s.shape[0], -1)
    return single, x_s, x_t, edge_attr, u


def _wide_args(x_s, x_t, edge_attr, u):
    """bf16 tensors of one graph for the wide (tensor-core) path, or None for the fp32 kernels."""
    if not pw.supported(edge_attr.shape[-1], edge_attr.dtype):
        return None
    if x_s.dim() != 2:
        raise RuntimeError("the bf16 wide path takes one graph per call (2-D tensors); batch graphs with dp.py")
    if u.shape[0] != 1:
        raise RuntimeError("global features with %d rows cannot be expanded over one graph "
                           "(reference src/gnn.py:100 fails the same way)" % u.shape[0])
    return x_s, x_t, edge_attr, u.reshape(1, -1)


def _refuse_sharded_narrow(what):
    """The fp32 kernels reduce over the fibres of the call only: inside a fibre-sharding scope they would return per-shard
    BatchNorm statistics and class sums."""
    if _shard.active():
        raise _abi.PfsError("%s: a fibre-sharded graph runs on the bf16 wide path (Fdim >= 32, bf16 tensors); the fp32 "
                            "kernels are not sharded" % what)


class _SumGradsOverShards(torch.autograd.Function):
    """Identity on a module's parameters whose backward sums their gradients over the fibre shards in ONE all-reduce:
    the parameters of a fibre-local module (encoder_s, decoder_s) see only the rank's own fibres."""

    @staticmethod
    def forward(ctx, *params):
        return tuple(p.view_as(p) for p in params)

    @staticmethod
    def backward(ctx, *grads):
        return tuple(_shard.allreduce_packed(list(grads)))


def _fibre_local(module, x):
    """module(x) for a module applied to the rank's own fibres; inside an active fibre-sharding scope its parameter
    gradients are summed over the shards, so every rank's .grad is the global gradient."""
    if not _shard.active():
        return module(x)
    names, params = zip(*module.named_parameters())
    routed = _SumGradsOverShards.apply(*params)
    return torch.func.functional_call(module, dict(zip(names, routed)), (x,))


def _norm_tensors(mod):
    norm = mod.norm if isinstance(mod.norm, torch.nn.Module) else None
    if norm is None:
        return False, None, None, None, None, None
    return True, norm.weight, norm.bias, norm.running_mean, norm.running_var, norm.num_batches_tracked


class EdgeModel(MLP):
    """Edge update (reference src/gnn.py:73-101).  `norm` is registered after the Sequential's three
    layers exactly as in the reference, where that makes it BOTH the Sequential's 4th child and the
    explicit post-norm: the BatchNorm is applied twice per forward (SURVEY.md section 0.2); the kernels
    reproduce that in closed form, including the two running-statistics updates."""

    def __init__(self, Fdim=10, normed=True):
        F_message = 4 * Fdim
        super(EdgeModel, self).__init__(F_message, F_message, Fdim)
        self.norm = torch.nn.BatchNorm1d(Fdim) if normed else (lambda x: x)

    def forward(self, x_s, x_t, edge_index, edge_attr, u):
        wide = _wide_args(x_s, x_t, edge_attr, u)
        if wide is not None:
            topo = get_topology(edge_index, x_s.shape[0], x_t.shape[0])
            normed, gamma, beta, rm, rv, nbt = _norm_tensors(self)
            return pw.WideEdgeFunction.apply(topo, self.training, normed, *wide, self[0].weight, self[0].bias,
                                             self[2].weight, self[2].bias, gamma, beta, rm, rv, nbt)
        _refuse_sharded_narrow("EdgeModel (fp32)")
        single, x_s, x_t, edge_attr, u = _batched(x_s, x_t, edge_attr, u)
        topo = get_topology(edge_index, x_s.shape[1], x_t.shape[1])
        normed, gamma, beta, rm, rv, nbt = _norm_tensors(self)
        out = pf.EdgeFunction.apply(topo, self.training, normed, x_s, x_t, edge_attr, u, self[0].weight, self[0].bias,
                                    self[2].weight, self[2].bias, gamma, beta, rm, rv, nbt, getattr(self, "_defer", None))
        return out[0] if single else out


class SModel(torch.nn.Module):
    """Source-node (fibre) update (reference src/gnn.py:104-154)."""

    def __init__(self, Fdim=10, normed=True):
        super(SModel, self).__init__()
        F_message = 2 * Fdim
        self.node_mlp_1 = MLP(F_message, F_message, F_message)
        F_message2 = 4 * F_message + 2 * Fdim
        self.node_mlp_2 = MLP(F_message2, F_message2, Fdim)
        self.norm = torch.nn.BatchNorm1d(Fdim) if normed else (lambda x: x)

    def forward(self, x_s, x_t, edge_index, edge_attr, u):
        wide = _wide_args(x_s, x_t, edge_attr, u)
        if wide is not None:
            topo = get_topology(edge_index, x_s.shape[0], x_t.shape[0])
            normed, gamma, beta, rm, rv, nbt = _norm_tensors(self)
            m1, m2 = self.node_mlp_1, self.node_mlp_2
            return pw.WideSourceFunction.apply(topo, self.training, normed, *wide, m1[0].weight, m1[0].bias, m1[2].weight,
                               m1[2].bias, m2[0].weight, m2[0].bias, m2[2].weight, m2[2].bias, gamma, beta, rm, rv, nbt)
        _refuse_sharded_narrow("SModel (fp32)")
        single, x_s, x_t, edge_attr, u = _batched(x_s, x_t, edge_attr, u)
        topo = get_topology(edge_index, x_s.shape[1], x_t.shape[1])
        normed, gamma, beta, rm, rv, nbt = _norm_tensors(self)
        m1, m2 = self.node_mlp_1, self.node_mlp_2
        out = pf.SourceFunction.apply(topo, self.training, normed, x_s, x_t, edge_attr, u, m1[0].weight, m1[0].bias,
                                      m1[2].weight, m1[2].bias, m2[0].weight, m2[0].bias, m2[2].weight, m2[2].bias,
                                      gamma, beta, rm, rv, nbt, getattr(self, "_xe_bus", None),
                                      getattr(self, "_edge_affine", None))
        return out[0] if single else out


class TModel(torch.nn.Module):
    """Target-node (class) update (reference src/gnn.py:157-192)."""

    def __init__(self, Fdim=10, normed=True):
        super(TModel, self).__init__()
        F_message = 2 * Fdim
        self.node_mlp_1 = MLP(F_message, F_message, F_message)
        F_message2 = 4 * Fdim
        self.node_mlp_2 = MLP(F_message2, F_message2, Fdim)
        self.norm = torch.nn.BatchNorm1d(Fdim) if normed else (lambda x: x)

    def forward(self, x_s, x_t, edge_index, edge_attr, u):
        wide = _wide_args(x_s, x_t, edge_attr, u)
        if wide is not None:
            topo = get_topology(edge_index, x_s.shape[0], x_t.shape[0])
            normed, gamma, beta, rm, rv, nbt = _norm_tensors(self)
            m1, m2 = self.node_mlp_1, self.node_mlp_2
            return pw.WideTargetFunction.apply(topo, self.training, normed, *wide, m1[0].weight, m1[0].bias, m1[2].weight,
                               m1[2].bias, m2[0].weight, m2[0].bias, m2[2].weight, m2[2].bias, gamma, beta, rm, rv, nbt)
        _refuse_sharded_narrow("TModel (fp32)")
        single, x_s, x_t, edge_attr, u = _batched(x_s, x_t, edge_attr, u)
        topo = get_topology(edge_index, x_s.shape[1], x_t.shape[1])
        normed, gamma, beta, rm, rv, nbt = _norm_tensors(self)
        m1, m2 = self.node_mlp_1, self.node_mlp_2
        out = pf.TargetFunction.apply(topo, self.training, normed, x_s, x_t, edge_attr, u, m1[0].weight, m1[0].bias,
                                      m1[2].weight, m1[2].bias, m2[0].weight, m2[0].bias, m2[2].weight, m2[2].bias,
                                      gamma, beta, rm, rv, nbt, getattr(self, "_xe_bus", None))
        return out[0] if single else out


class GlobalModel(MLP):
    """Graph-level update (reference src/gnn.py:195-223); the RMSNorm is applied twice for the same
    Sequential-child reason as EdgeModel's BatchNorm."""

    def __init__(self, Fdim=10, normed=True):
        F_message = 3 * Fdim
        super(GlobalModel, self).__init__(F_message, F_message, Fdim)
        self.norm = torch.nn.RMSNorm(Fdim) if normed else (lambda x: x)

    def forward(self, x_s, x_t, edge_index, edge_attr, u):
        if pw.supported(x_s.shape[-1], x_s.dtype):
            if x_s.dim() != 2:
                raise RuntimeError("the bf16 wide path takes one graph per call (2-D tensors)")
            normed = isinstance(self.norm, torch.nn.Module)
            # nn.RMSNorm(eps=None) uses finfo(input dtype).eps (reference src/gnn.py:203 run in bf16)
            return pw.WideGlobalFunction.apply(normed, x_s, x_t, u, self[0].weight, self[0].bias, self[2].weight,
                                               self[2].bias, self.norm.weight if normed else None,
                                               float(torch.finfo(u.dtype).eps))
        _refuse_sharded_narrow("GlobalModel (fp32)")
        single = x_s.dim() == 2
        if single:
            x_s, x_t = x_s.unsqueeze(0), x_t.unsqueeze(0)
        lead = u.shape[:-1]
        u2 = u.reshape(x_s.shape[0], -1)
        normed = isinstance(self.norm, torch.nn.Module)
        out = pf.GlobalFunction.apply(normed, x_s, x_t, u2, self[0].weight, self[0].bias, self[2].weight,
                                      self[2].bias, self.norm.weight if normed else None)
        return out.reshape(*lead, out.shape[-1])


class Block(torch.nn.Module):
    """One message-passing layer: edge -> source -> target -> global, each stage consuming the previous
    stage's outputs (reference src/gnn.py:226-259).  I/O is the 5-tuple so Blocks chain in Sequential."""

    def __init__(self, Fdim=10, e_model=True, s_model=True, t_model=True, u_model=True, normed=True):
        super(Block, self).__init__()
        if e_model:
            self.edge_model = EdgeModel(Fdim, normed=normed)
        if s_model:
            self.s_model = SModel(Fdim, normed=normed)
        if t_model:
            self.t_model = TModel(Fdim, normed=normed)
        if u_model:
            self.global_model = GlobalModel(Fdim, normed=normed)

    def forward(self, args):
        edge_index, x_s, x_t, x_e, x_u = args
        # fp32 path: the EdgeModel leaves its BatchNorm affine to the SModel's edge pass, which normalises x_e' in place
        # while it reads it (one pass over [G, E, F] and one launch less); nothing in between looks at x_e'
        defer = None
        if (hasattr(self, "edge_model") and hasattr(self, "s_model") and x_e.is_cuda and x_e.dtype == torch.float32):
            defer = {}
        # fp32 path: the three gradients of x_e' (SModel, TModel, the output) are added up inside the backward
        # kernels instead of by autograd (functional.XeGradBus); the values are the same sum
        bus = None
        if (torch.is_grad_enabled() and x_e.is_cuda and x_e.dtype == torch.float32
                and hasattr(self, "s_model") and hasattr(self, "t_model")):
            bus = pf.XeGradBus()
        if hasattr(self, "edge_model"):
            self.edge_model._defer = defer
            try:
                x_e = self.edge_model(x_s, x_t, edge_index, x_e, x_u)
            finally:
                self.edge_model._defer = None
        edge_affine = defer.pop("affine", None) if defer else None
        x_e_s = x_e_t = x_e
        if bus is not None and x_e.requires_grad:
            x_e_s, x_e_t, x_e = pf.XeFanout.apply(x_e, bus)
        else:
            bus = None
        try:
            if hasattr(self, "s_model"):
                self.s_model._xe_bus = bus
                self.s_model._edge_affine = edge_affine
                x_s = self.s_model(x_s, x_t, edge_index, x_e_s, x_u)
            if hasattr(self, "t_model"):
                self.t_model._xe_bus = bus
                x_t = self.t_model(x_s, x_t, edge_index, x_e_t, x_u)
        finally:
            if hasattr(self, "s_model"):
                self.s_model._xe_bus = None
                self.s_model._edge_affine = None
            if hasattr(self, "t_model"):
                self.t_model._xe_bus = None
        if hasattr(self, "global_model"):
            x_u = self.global_model(x_s, x_t, edge_index, x_e, x_u)
        if bus is not None:
            x_e = pf.XeOutTap.apply(x_e, bus)
        return edge_index, x_s, x_t, x_e, x_u


class GNN(torch.nn.Module):
    """Encoders, B Blocks, decoders (reference src/gnn.py:261-325); registration order matches
    src/gnn.py:270-278 (encoder_s, encoder_t, mpb, decoder_e, decoder_s)."""

    def __init__(self, B=4, Fdim=16, T=12, F_s=1, F_t=1, normed=True):
        super(GNN, self).__init__()
        self.encoder_s = MLP(F_s, Fdim, Fdim)
        self.encoder_t = MLP(F_t, Fdim, Fdim)
        self.mpb = torch.nn.Sequential(*(Block(Fdim, normed=normed) for b in range(B)))
        self.decoder_e = MLP(Fdim, Fdim, 1)
        self.decoder_s = MLP(Fdim, Fdim, T)
        self._last_edge_index = None
        self._head_checked = None

    def forward(self, graph):
        x_s, x_t = graph.x_s, graph.x_t
        edge_index, x_e, x_u = graph.edge_index, graph.x_e, graph.x_u
        # per-node encoders stay in PyTorch (SURVEY.md section 2 row 2).  Fibre-sharded, encoder_s sees the local fibres
        # and its gradients are summed over the shards; encoder_t's already are global (replicated classes, global g_x_t)
        x_s = _fibre_local(self.encoder_s, x_s)
        x_t = self.encoder_t(x_t)
        _, x_s, x_t, x_e, x_u = self.mpb((edge_index, x_s, x_t, x_e, x_u))
        self._last_edge_index = edge_index
        return BipartiteData(edge_index, x_s, x_t, x_e, x_u)

    def _head_classes(self, x_e, class_hours, edge_index):
        """int64 class index of every edge for the integer times: row 1 of the graph's `edge_index` (the last forward's,
        or the one passed).  The time head itself never looks at the topology, so no CSR is built and the class count
        comes from `class_hours`, not from the model."""
        if edge_index is None:
            edge_index = self._last_edge_index
        if edge_index is None:
            raise RuntimeError("integer_times needs the graph's edge_index (run forward first or pass it)")
        E, T = x_e.shape[-2], class_hours.shape[0]
        if edge_index.dim() != 2 or edge_index.shape[0] != 2 or edge_index.shape[1] != E:
            raise ValueError("edge_index %s does not match x_e with %d edges" % (tuple(edge_index.shape), E))
        key = (edge_index.data_ptr(), edge_index._version, E, T)
        if self._head_checked != key:                    # one range check (a host sync) per edge_index tensor
            tgt = edge_index[1]
            if int(tgt.min()) < 0 or int(tgt.max()) >= T:
                raise IndexError("edge_index names classes outside class_hours (%d entries)" % T)
            self._head_checked = key
        return edge_index[1].contiguous()

    def edge_prediction(self, x_e, scale=1, edge_index=None):
        """softplus(decoder_e(x_e)) * scale, [E, 1] (reference src/gnn.py:307-312; `round` is the
        identity there, see `round`).  The time head does not depend on the topology."""
        d = self.decoder_e
        if pw.supported(x_e.shape[-1], x_e.dtype):
            if x_e.dim() != 2:
                raise RuntimeError("the bf16 wide path takes one graph per call (2-D tensors)")
            return pw.WideTimeHeadFunction.apply(scale, x_e, d[0].weight, d[0].bias, d[2].weight, d[2].bias).unsqueeze(-1)
        _refuse_sharded_narrow("the time head (fp32)")
        single = x_e.dim() == 2
        xe3 = x_e.unsqueeze(0) if single else x_e
        topo = _FlatTopology(xe3.shape[1], x_e.device)
        time = pf.TimeHeadFunction.apply(topo, scale, xe3, d[0].weight, d[0].bias, d[2].weight, d[2].bias)
        time = time.unsqueeze(-1)
        return time[0] if single else time

    def integer_times(self, x_e, class_hours, scale=1, edge_index=None):
        """(time, visits, time_int): visits = round-half-even(time / T_i[tgt]), time_int = visits * T_i.
        This is the "rounded integer time" this build defines (DESIGN.md; reference src/train.py:257)."""
        d = self.decoder_e
        tgt = self._head_classes(x_e, class_hours, edge_index)
        if pw.supported(x_e.shape[-1], x_e.dtype):
            if x_e.dim() != 2:
                raise RuntimeError("the bf16 wide path takes one graph per call (2-D tensors)")
            return pw.integer_times(tgt.to(torch.int32), x_e, d[0].weight, d[0].bias, d[2].weight, d[2].bias, scale, class_hours)
        single = x_e.dim() == 2
        xe3 = x_e.unsqueeze(0) if single else x_e
        topo = _FlatTopology(xe3.shape[1], x_e.device, dense=False)
        out = pf.integer_times(topo, xe3, d[0].weight, d[0].bias, d[2].weight, d[2].bias, scale,
                               class_hours.to(torch.float32), edge_tgt=tgt)
        return tuple(o[0] for o in out) if single else out

    def node_prediction(self, x_s, scale=1):
        pred = _fibre_local(self.decoder_s, x_s)
        time = torch.softmax(pred, dim=-1) * scale
        return self.round(time)

    def round(self, x):
        # reference src/gnn.py:321-325 tests `self.train` (a bound method, always truthy), so it never
        # rounds, in train or eval mode; kept bit-compatible.  Use integer_times() for integers.
        return x


class _FlatTopology:
    """Topology stand-in for per-edge ops that never look at src/tgt (the time head)."""

    def __init__(self, E, dev, dense=True):
        self.E, self.S, self.T, self.dense, self.device = int(E), int(E), 1, dense, dev
        self._ws = None

    def struct(self, G, F):
        t = _abi.TopologyStruct()
        t.layout, t.G, t.F, t.S, t.T, t.E = _abi.PFS_LAYOUT_DENSE, int(G), int(F), self.S, 1, self.E
        return t

    def workspace(self, G, F):
        if self._ws is None:
            self._ws = torch.empty(4 * 1024 * (F * F + 2 * F + 1) + 4096, dtype=torch.uint8, device=self.device)
        return self._ws
