"""autograd Functions that lower the reference's update modules onto the C ABI (include/pfs_b200.h).

One Function per module of reference src/gnn.py (EdgeModel :73-101, SModel :104-154, TModel :157-192,
GlobalModel :195-223, time head :307-312).  Each `forward` / `backward` is ONE library call on the
current CUDA stream; PyTorch only owns the memory.  Tensors are batched [G, rows, F] (G graphs that
share topology and weights, independent BatchNorm statistics); the module wrappers in gnn.py add and
remove the leading dimension for the reference's 2-D calling convention.
"""
import ctypes as ct

import torch

from . import _abi

BN_EPS = 1e-5
BN_MOMENTUM = 0.1
RMS_EPS = float(torch.finfo(torch.float32).eps)    # nn.RMSNorm(eps=None), reference src/gnn.py:203


def _dev_check(*tensors):
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise _abi.PfsError("pfs_b200 kernels need CUDA tensors, got %s (there is no CPU fallback)" % t.device)
        if t.dtype != torch.float32:
            raise _abi.PfsError("pfs_b200 kernels are fp32, got %s" % t.dtype)
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise _abi.PfsError("tensors on different devices: %s vs %s" % (t.device, dev))
    return dev


def _c(t):
    return None if t is None else t.contiguous()


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def _fill_common(a, topo, G, F, named):
    a.topo = topo.struct(G, F)
    ws = topo.workspace(G, F)
    a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    for k, v in named.items():
        setattr(a, k, _abi.ptr(v))
    return ws


def _check_shapes(topo, x_s, x_t, x_e, u):
    G, S, F = x_s.shape
    if x_t.shape != (G, topo.T, F) or x_e.shape != (G, topo.E, F) or u.shape != (G, F) or S != topo.S:
        raise _abi.PfsError("shape mismatch: x_s %s x_t %s x_e %s u %s for a %dx%d graph with %d edges"
                            % (tuple(x_s.shape), tuple(x_t.shape), tuple(x_e.shape), tuple(u.shape),
                               topo.S, topo.T, topo.E))
    return G, F


class XeGradBus:
    """Lets the backward kernels of a Block add up the three gradients of the updated edge embedding x_e'
    (it feeds SModel, TModel and the Block output) instead of autograd: 2 x 3 passes over [G, E, F] per step.

    Opportunistic and order-independent: whoever runs later fuses what is already there into its own store
    (`g_x_e_add` of pfs_target_bwd / pfs_source_bwd) and marks it used; `XeFanout.backward` adds whatever was not
    fused, so every combination of used / unused branches gives the same sum.  In a training step autograd runs
    the output tap first, then TModel, then SModel, and nothing is left for it to add."""
    __slots__ = ("g_o", "g_t", "o_used", "t_used")

    def __init__(self):
        self.clear()

    def clear(self):
        self.g_o = self.g_t = None
        self.o_used = self.t_used = False

    def addend_for_target(self, like):
        if (self.g_o is not None and not self.o_used and self.g_o.numel() == like.numel()
                and self.g_o.dtype == torch.float32 and self.g_o.device == like.device):
            self.o_used = True
            return self.g_o.contiguous()
        return None

    def addend_for_source(self, like):
        if self.g_t is not None and not self.t_used and self.g_t.numel() == like.numel():
            self.t_used = True
            return self.g_t
        return self.addend_for_target(like)


class XeFanout(torch.autograd.Function):
    """x_e' -> (for SModel, for TModel, for the output); backward adds the parts the kernels have not fused."""

    @staticmethod
    def forward(ctx, x, bus):
        ctx.bus = bus
        ctx.set_materialize_grads(False)
        return x.view_as(x), x.view_as(x), x.view_as(x)

    @staticmethod
    def backward(ctx, g_s, g_t, g_o):
        bus = ctx.bus
        parts = []
        if g_s is not None:
            parts.append(g_s)
        if g_t is not None and not bus.t_used:
            parts.append(g_t)
        if g_o is not None and not bus.o_used:
            parts.append(g_o)
        bus.clear()
        if not parts:
            return None, None
        total = parts[0]
        for q in parts[1:]:
            total = total + q
        return total, None


class XeOutTap(torch.autograd.Function):
    """Identity on the Block's x_e' output: its backward runs before the modules' and shows them the upstream
    gradient."""

    @staticmethod
    def forward(ctx, x, bus):
        ctx.bus = bus
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        ctx.bus.g_o = g
        return g, None


class EdgeFunction(torch.autograd.Function):
    """EdgeModel (reference src/gnn.py:73-101) -> pfs_edge_fwd / pfs_edge_bwd."""

    @staticmethod
    def forward(ctx, topo, training, normed, x_s, x_t, x_e, u, w1, b1, w2, b2, gamma, beta, rm, rv, nbt, defer=None):
        """`defer`: a dict handed in by Block.forward.  When the module is normed the BatchNorm affine is NOT applied here:
        the returned tensor holds the pre-norm z, defer["affine"] the per-graph (scale, shift), and the next consumer
        (SourceFunction with edge_affine=...) normalises the rows in place while it reads them."""
        dev = _dev_check(x_s, x_t, x_e, u, w1, b1, w2, b2, gamma, beta, rm, rv)
        x_s, x_t, x_e, u, w1, b1, w2, b2, gamma, beta = (_c(t) for t in (x_s, x_t, x_e, u, w1, b1, w2, b2, gamma, beta))
        G, F = _check_shapes(topo, x_s, x_t, x_e, u)
        lib = _abi.load_library()
        out = torch.empty_like(x_e)
        bn_save = torch.empty(G, 4, F, device=dev, dtype=torch.float32) if normed else None
        # node tables of the first-layer split, kept for the backward when one will follow (it then skips their recomputation)
        keep = any(ctx.needs_input_grad)
        tab_s = torch.empty(G, topo.S, 4 * F, device=dev, dtype=torch.float32) if keep else None
        tab_t = torch.empty(G, topo.T, 4 * F, device=dev, dtype=torch.float32) if keep else None
        a = _abi.EdgeArgs()
        ws = _fill_common(a, topo, G, F, dict(x_s=x_s, x_t=x_t, x_e=x_e, u=u, w1=w1, b1=b1, w2=w2, b2=b2, gamma=gamma,
                                              beta=beta, running_mean=rm, running_var=rv, num_batches_tracked=nbt,
                                              x_e_out=out, bn_save=bn_save, table_s=tab_s, table_t=tab_t))
        a.training, a.normed, a.eps, a.momentum = int(training), int(normed), BN_EPS, BN_MOMENTUM
        deferred = defer is not None and bool(normed)
        a.defer_affine = int(deferred)
        with torch.cuda.device(dev):
            a.stream = _stream(dev)
            _abi.check(lib.pfs_edge_fwd(ct.byref(a)), "pfs_edge_fwd")
        if deferred:
            defer["affine"] = bn_save
        ctx.topo, ctx.training, ctx.normed = topo, training, normed
        ctx.buffers = (rm, rv)
        ctx.save_for_backward(x_s, x_t, x_e, u, w1, b1, w2, b2, gamma, beta, out, bn_save, tab_s, tab_t)
        del ws
        return out

    @staticmethod
    def backward(ctx, g):
        x_s, x_t, x_e, u, w1, b1, w2, b2, gamma, beta, out, bn_save, tab_s, tab_t = ctx.saved_tensors
        topo, dev = ctx.topo, x_e.device
        G, F = x_s.shape[0], x_s.shape[2]
        lib = _abi.load_library()
        g = g.contiguous()
        gr = dict(g_x_s=torch.empty_like(x_s), g_x_t=torch.empty_like(x_t), g_x_e=torch.empty_like(x_e),
                  g_u=torch.empty_like(u), g_w1=torch.empty_like(w1), g_b1=torch.empty_like(b1),
                  g_w2=torch.empty_like(w2), g_b2=torch.empty_like(b2),
                  g_gamma=torch.empty_like(gamma) if ctx.normed else None,
                  g_beta=torch.empty_like(beta) if ctx.normed else None)
        a = _abi.EdgeArgs()
        rm, rv = ctx.buffers
        named = dict(x_s=x_s, x_t=x_t, x_e=x_e, u=u, w1=w1, b1=b1, w2=w2, b2=b2, gamma=gamma, beta=beta,
                     running_mean=rm, running_var=rv, x_e_out=out, bn_save=bn_save, g_out=g, table_s=tab_s, table_t=tab_t)
        named.update(gr)
        ws = _fill_common(a, topo, G, F, named)
        a.training, a.normed, a.eps, a.momentum = int(ctx.training), int(ctx.normed), BN_EPS, BN_MOMENTUM
        with torch.cuda.device(dev):
            a.stream = _stream(dev)
            _abi.check(lib.pfs_edge_bwd(ct.byref(a)), "pfs_edge_bwd")
        del ws
        return (None, None, None, gr["g_x_s"], gr["g_x_t"], gr["g_x_e"], gr["g_u"], gr["g_w1"], gr["g_b1"],
                gr["g_w2"], gr["g_b2"], gr["g_gamma"], gr["g_beta"], None, None, None, None)


class SourceFunction(torch.autograd.Function):
    """SModel (reference src/gnn.py:104-154) -> pfs_source_fwd / pfs_source_bwd."""

    @staticmethod
    def forward(ctx, topo, training, normed, x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta, rm, rv, nbt, bus=None,
                edge_affine=None):
        """`edge_affine`: bn_save of an EdgeFunction run with a deferred norm -- x_e then holds the pre-norm z and is
        normalised IN PLACE by the edge pass of this call (every row is read and written by the same thread)."""
        dev = _dev_check(x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta, rm, rv)
        if edge_affine is not None and not x_e.is_contiguous():
            raise _abi.PfsError("deferred edge norm needs a contiguous x_e")
        (x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta) = (
            _c(t) for t in (x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta))
        G, F = _check_shapes(topo, x_s, x_t, x_e, u)
        lib = _abi.load_library()
        f32 = dict(device=dev, dtype=torch.float32)
        out = torch.empty_like(x_s)
        moments = torch.empty(G, topo.S, 5, 2 * F, **f32)
        hidden = torch.empty(G, topo.S, 10 * F, **f32)
        y_pre = torch.empty(G, topo.S, F, **f32)
        bn_save = torch.empty(G, 4, F, **f32) if normed else None
        a = _abi.SourceArgs()
        ws = _fill_common(a, topo, G, F, dict(
            x_s=x_s, x_t=x_t, x_e=x_e, u=u, w1=w1, b1=b1, w2=w2, b2=b2, w3=w3, b3=b3, w4=w4, b4=b4, gamma=gamma,
            beta=beta, running_mean=rm, running_var=rv, num_batches_tracked=nbt, x_s_out=out, moments=moments,
            hidden=hidden, y_pre=y_pre, bn_save=bn_save,
            x_e_affine=edge_affine, x_e_norm_out=x_e if edge_affine is not None else None))
        a.training, a.normed, a.eps, a.momentum = int(training), int(normed), BN_EPS, BN_MOMENTUM
        with torch.cuda.device(dev):
            a.stream = _stream(dev)
            _abi.check(lib.pfs_source_fwd(ct.byref(a)), "pfs_source_fwd")
        ctx.topo, ctx.training, ctx.normed = topo, training, normed
        ctx.bus = bus
        ctx.buffers = (rm, rv)
        ctx.save_for_backward(x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta, moments, hidden, y_pre,
                              bn_save)
        del ws
        return out

    @staticmethod
    def backward(ctx, g):
        (x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta, moments, hidden, y_pre,
         bn_save) = ctx.saved_tensors
        topo, dev = ctx.topo, x_e.device
        G, F = x_s.shape[0], x_s.shape[2]
        lib = _abi.load_library()
        g = g.contiguous()
        gr = dict(g_x_s=torch.empty_like(x_s), g_x_t=torch.empty_like(x_t), g_x_e=torch.empty_like(x_e),
                  g_u=torch.empty_like(u), g_w1=torch.empty_like(w1), g_b1=torch.empty_like(b1),
                  g_w2=torch.empty_like(w2), g_b2=torch.empty_like(b2), g_w3=torch.empty_like(w3),
                  g_b3=torch.empty_like(b3), g_w4=torch.empty_like(w4), g_b4=torch.empty_like(b4),
                  g_gamma=torch.empty_like(gamma) if ctx.normed else None,
                  g_beta=torch.empty_like(beta) if ctx.normed else None)
        rm, rv = ctx.buffers
        named = dict(x_s=x_s, x_t=x_t, x_e=x_e, u=u, w1=w1, b1=b1, w2=w2, b2=b2, w3=w3, b3=b3, w4=w4, b4=b4,
                     gamma=gamma, beta=beta, running_mean=rm, running_var=rv, moments=moments, hidden=hidden,
                     y_pre=y_pre, bn_save=bn_save, g_out=g)
        add = ctx.bus.addend_for_source(x_e) if ctx.bus is not None else None
        named.update(gr, g_x_e_add=add)
        a = _abi.SourceArgs()
        ws = _fill_common(a, topo, G, F, named)
        a.training, a.normed, a.eps, a.momentum = int(ctx.training), int(ctx.normed), BN_EPS, BN_MOMENTUM
        with torch.cuda.device(dev):
            a.stream = _stream(dev)
            _abi.check(lib.pfs_source_bwd(ct.byref(a)), "pfs_source_bwd")
        del ws
        return (None, None, None, gr["g_x_s"], gr["g_x_t"], gr["g_x_e"], gr["g_u"], gr["g_w1"], gr["g_b1"],
                gr["g_w2"], gr["g_b2"], gr["g_w3"], gr["g_b3"], gr["g_w4"], gr["g_b4"], gr["g_gamma"], gr["g_beta"],
                None, None, None, None, None)


class TargetFunction(torch.autograd.Function):
    """TModel (reference src/gnn.py:157-192) -> pfs_target_fwd / pfs_target_bwd."""

    @staticmethod
    def forward(ctx, topo, training, normed, x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta, rm, rv, nbt, bus=None):
        dev = _dev_check(x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta, rm, rv)
        (x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta) = (
            _c(t) for t in (x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta))
        G, F = _check_shapes(topo, x_s, x_t, x_e, u)
        lib = _abi.load_library()
        f32 = dict(device=dev, dtype=torch.float32)
        out = torch.empty_like(x_t)
        act_sum = torch.empty(G, topo.T, 2 * F, **f32)
        y_pre = torch.empty(G, topo.T, F, **f32)
        bn_save = torch.empty(G, 4, F, **f32) if normed else None
        keep = any(ctx.needs_input_grad)
        tab_s = torch.empty(G, topo.S, 2 * F, **f32) if keep else None
        a = _abi.TargetArgs()
        ws = _fill_common(a, topo, G, F, dict(
            x_s=x_s, x_t=x_t, x_e=x_e, u=u, w1=w1, b1=b1, w2=w2, b2=b2, w3=w3, b3=b3, w4=w4, b4=b4, gamma=gamma,
            beta=beta, running_mean=rm, running_var=rv, num_batches_tracked=nbt, x_t_out=out, act_sum=act_sum,
            y_pre=y_pre, bn_save=bn_save, table_s=tab_s))
        a.training, a.normed, a.eps, a.momentum = int(training), int(normed), BN_EPS, BN_MOMENTUM
        with torch.cuda.device(dev):
            a.stream = _stream(dev)
            _abi.check(lib.pfs_target_fwd(ct.byref(a)), "pfs_target_fwd")
        ctx.topo, ctx.training, ctx.normed = topo, training, normed
        ctx.bus = bus
        ctx.buffers = (rm, rv)
        ctx.save_for_backward(x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta, act_sum, y_pre, bn_save, tab_s)
        del ws
        return out

    @staticmethod
    def backward(ctx, g):
        (x_s, x_t, x_e, u, w1, b1, w2, b2, w3, b3, w4, b4, gamma, beta, act_sum, y_pre, bn_save, tab_s) = ctx.saved_tensors
        topo, dev = ctx.topo, x_e.device
        G, F = x_s.shape[0], x_s.shape[2]
        lib = _abi.load_library()
        g = g.contiguous()
        gr = dict(g_x_s=torch.empty_like(x_s), g_x_t=torch.empty_like(x_t), g_x_e=torch.empty_like(x_e),
                  g_u=torch.empty_like(u), g_w1=torch.empty_like(w1), g_b1=torch.empty_like(b1),
                  g_w2=torch.empty_like(w2), g_b2=torch.empty_like(b2), g_w3=torch.empty_like(w3),
                  g_b3=torch.empty_like(b3), g_w4=torch.empty_like(w4), g_b4=torch.empty_like(b4),
                  g_gamma=torch.empty_like(gamma) if ctx.normed else None,
                  g_beta=torch.empty_like(beta) if ctx.normed else None)
        rm, rv = ctx.buffers
        named = dict(x_s=x_s, x_t=x_t, x_e=x_e, u=u, w1=w1, b1=b1, w2=w2, b2=b2, w3=w3, b3=b3, w4=w4, b4=b4,
                     gamma=gamma, beta=beta, running_mean=rm, running_var=rv, act_sum=act_sum, y_pre=y_pre,
                     bn_save=bn_save, g_out=g, table_s=tab_s)
        add = ctx.bus.addend_for_target(x_e) if ctx.bus is not None else None
        named.update(gr, g_x_e_add=add)
        a = _abi.TargetArgs()
        ws = _fill_common(a, topo, G, F, named)
        a.training, a.normed, a.eps, a.momentum = int(ctx.training), int(ctx.normed), BN_EPS, BN_MOMENTUM
        with torch.cuda.device(dev):
            a.stream = _stream(dev)
            _abi.check(lib.pfs_target_bwd(ct.byref(a)), "pfs_target_bwd")
        del ws
        if ctx.bus is not None:
            ctx.bus.g_t = gr["g_x_e"]
        return (None, None, None, gr["g_x_s"], gr["g_x_t"], gr["g_x_e"], gr["g_u"], gr["g_w1"], gr["g_b1"],
                gr["g_w2"], gr["g_b2"], gr["g_w3"], gr["g_b3"], gr["g_w4"], gr["g_b4"], gr["g_gamma"], gr["g_beta"],
                None, None, None, None)


_global_ws = {}


def _global_workspace(dev, G, F):
    key = (str(dev), G, F)
    ws = _global_ws.get(key)
    if ws is None:
        ws = torch.empty(4 * G * (12 * F * F + 5 * F) + 4096, dtype=torch.uint8, device=dev)
        _global_ws[key] = ws
    return ws


class GlobalFunction(torch.autograd.Function):
    """GlobalModel (reference src/gnn.py:195-223) -> pfs_global_fwd / pfs_global_bwd."""

    @staticmethod
    def forward(ctx, normed, x_s, x_t, u, w1, b1, w2, b2, rms_w):
        dev = _dev_check(x_s, x_t, u, w1, b1, w2, b2, rms_w)
        x_s, x_t, u, w1, b1, w2, b2, rms_w = (_c(t) for t in (x_s, x_t, u, w1, b1, w2, b2, rms_w))
        G, S, F = x_s.shape
        T = x_t.shape[1]
        if x_t.shape != (G, T, F) or u.shape != (G, F):
            raise _abi.PfsError("global model: shape mismatch x_s %s x_t %s u %s"
                                % (tuple(x_s.shape), tuple(x_t.shape), tuple(u.shape)))
        lib = _abi.load_library()
        out = torch.empty_like(u)
        a = _abi.GlobalArgs()
        a.G, a.F, a.S, a.T, a.normed, a.rms_eps = G, F, S, T, int(normed), RMS_EPS
        for k, v in dict(x_s=x_s, x_t=x_t, u=u, w1=w1, b1=b1, w2=w2, b2=b2, rms_weight=rms_w, u_out=out).items():
            setattr(a, k, _abi.ptr(v))
        with torch.cuda.device(dev):
            a.stream = _stream(dev)
            _abi.check(lib.pfs_global_fwd(ct.byref(a)), "pfs_global_fwd")
        ctx.normed = normed
        ctx.save_for_backward(x_s, x_t, u, w1, b1, w2, b2, rms_w)
        return out

    @staticmethod
    def backward(ctx, g):
        x_s, x_t, u, w1, b1, w2, b2, rms_w = ctx.saved_tensors
        dev = u.device
        G, S, F = x_s.shape
        T = x_t.shape[1]
        lib = _abi.load_library()
        g = g.contiguous()
        gr = dict(g_x_s=torch.empty_like(x_s), g_x_t=torch.empty_like(x_t), g_u=torch.empty_like(u),
                  g_w1=torch.empty_like(w1), g_b1=torch.empty_like(b1), g_w2=torch.empty_like(w2),
                  g_b2=torch.empty_like(b2), g_rms_weight=torch.empty_like(rms_w) if ctx.normed else None)
        ws = _global_workspace(dev, G, F)
        a = _abi.GlobalArgs()
        a.G, a.F, a.S, a.T, a.normed, a.rms_eps = G, F, S, T, int(ctx.normed), RMS_EPS
        named = dict(x_s=x_s, x_t=x_t, u=u, w1=w1, b1=b1, w2=w2, b2=b2, rms_weight=rms_w, g_out=g)
        named.update(gr)
        for k, v in named.items():
            setattr(a, k, _abi.ptr(v))
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        with torch.cuda.device(dev):
            a.stream = _stream(dev)
            _abi.check(lib.pfs_global_bwd(ct.byref(a)), "pfs_global_bwd")
        return (None, gr["g_x_s"], gr["g_x_t"], gr["g_u"], gr["g_w1"], gr["g_b1"], gr["g_w2"], gr["g_b2"],
                gr["g_rms_weight"])


class TimeHeadFunction(torch.autograd.Function):
    """GNN.edge_prediction (reference src/gnn.py:307-312) -> pfs_time_head_fwd / pfs_time_head_bwd."""

    @staticmethod
    def forward(ctx, topo, scale, x_e, w1, b1, w2, b2):
        dev = _dev_check(x_e, w1, b1, w2, b2)
        x_e, w1, b1, w2, b2 = (_c(t) for t in (x_e, w1, b1, w2, b2))
        G, E, F = x_e.shape
        lib = _abi.load_library()
        time = torch.empty(G, E, device=dev, dtype=torch.float32)
        a = _abi.HeadArgs()
        ws = _fill_common(a, topo, G, F, dict(x_e=x_e, w1=w1, b1=b1, w2=w2, b2=b2, time=time))
        a.scale = float(scale)
        with torch.cuda.device(dev):
            a.stream = _stream(dev)
            _abi.check(lib.pfs_time_head_fwd(ct.byref(a)), "pfs_time_head_fwd")
        ctx.topo, ctx.scale = topo, float(scale)
        ctx.save_for_backward(x_e, w1, b1, w2, b2)
        del ws
        return time

    @staticmethod
    def backward(ctx, g):
        x_e, w1, b1, w2, b2 = ctx.saved_tensors
        dev = x_e.device
        G, E, F = x_e.shape
        lib = _abi.load_library()
        g = g.contiguous()
        gr = dict(g_x_e=torch.empty_like(x_e), g_w1=torch.empty_like(w1), g_b1=torch.empty_like(b1),
                  g_w2=torch.empty_like(w2), g_b2=torch.empty_like(b2))
        named = dict(x_e=x_e, w1=w1, b1=b1, w2=w2, b2=b2, g_time=g)
        named.update(gr)
        a = _abi.HeadArgs()
        ws = _fill_common(a, ctx.topo, G, F, named)
        a.scale = ctx.scale
        with torch.cuda.device(dev):
            a.stream = _stream(dev)
            _abi.check(lib.pfs_time_head_bwd(ct.byref(a)), "pfs_time_head_bwd")
        del ws
        return None, None, gr["g_x_e"], gr["g_w1"], gr["g_b1"], gr["g_w2"], gr["g_b2"]


def integer_times(topo, x_e, w1, b1, w2, b2, scale, class_hours, edge_tgt=None):
    """Fused time head + integer times (no gradient): returns (time, visits, time_int), each [G, E].
    visits = rint(time / hours[tgt]) (round-half-even like torch.round), time_int = visits * hours[tgt]
    -- the definition adopted in DESIGN.md for "rounded integer times" (reference src/train.py:257)."""
    dev = _dev_check(x_e, w1, b1, w2, b2, class_hours)
    x_e, w1, b1, w2, b2, class_hours = (_c(t.detach()) for t in (x_e, w1, b1, w2, b2, class_hours))
    G, E, F = x_e.shape
    lib = _abi.load_library()
    time, visits, time_int = (torch.empty(G, E, device=dev, dtype=torch.float32) for _ in range(3))
    if not topo.dense and edge_tgt is None:
        edge_tgt = topo.edge_index[1].contiguous()
    a = _abi.HeadArgs()
    ws = _fill_common(a, topo, G, F, dict(x_e=x_e, w1=w1, b1=b1, w2=w2, b2=b2, class_hours=class_hours, time=time,
                                          visits=visits, time_int=time_int,
                                          edge_tgt=None if topo.dense else edge_tgt))
    a.scale = float(scale)
    with torch.cuda.device(dev):
        a.stream = _stream(dev)
        _abi.check(lib.pfs_time_head_fwd(ct.byref(a)), "pfs_time_head_fwd")
    del ws
    return time, visits, time_int
