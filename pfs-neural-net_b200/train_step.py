"""One optimisation step of the reference training loop (reference src/train.py:136-141: zero_grad, forward,
loss_function, backward, optimizer.step) as a replayable CUDA graph (SURVEY.md section 8f, row N2).

At the reference's sizes (2000 x 12 fibre-class pairs, 3 Blocks) the step is launch-bound: ~200 kernel launches,
each a few microseconds of GPU work.  Capturing the whole step -- the torch encoders, the Block kernels of
libpfs_b200.so (their weight uploads into the constant bank are memcpy nodes), the time head, the loss kernels and
a capturable Adam -- removes the per-launch host cost; the sharpness schedule (src/train.py:139) is fed through a
device scalar so a replay sees the new value.  The graph inputs (node / edge features, class table) are static, as in
the reference, where only the weights change between epochs.

The warm-up and capture passes execute real steps; everything they touch -- parameters, BatchNorm buffers (running
statistics AND num_batches_tracked), Adam moments and step counters, the CUDA generator -- is snapshotted before and
restored afterwards IN PLACE (the captured graph keeps the addresses), so the first user-visible step starts from the
state the caller handed in, like reference src/train.py:133 or a resumed checkpoint (:126-132).

The graph may be a collated batch of G graphs that share one `edge_index` (`Loader.collate`, x_e [G, E, F]) with a
class table [T, 2] for all of them or [G, T, 2]: the step then trains on the sum of the G per-graph losses (the
parameter gradients of the G graphs stepped one after the other, summed) and returns the G utilities.  `load()`
copies the next batch of the same shapes and topology into the step's input tensors, so an epoch over
`Loader.batches(G)` replays the one captured graph.

Inside `shard.fibre_sharded()` (one graph split over the ranks by fibre ranges) the step runs eager only
(`use_graph=False`): its all-reduces are not captured into a CUDA graph.
"""
import torch

from . import loss as _loss
from . import shard as _shard


class TrainStep:
    def __init__(self, model, graph, class_info, optimizer, *, pclass=0.1, pfiber=1.0, nfields=10, total_time=42,
                 wutils=2000.0, wvar=1.0, use_graph=True, warmup=3, noise=None):
        """`noise`: optional static device tensor [E] (a batch: [G, E]) of softfloor draws in [0, 1) (reference
        src/train.py:22); the caller refills it (copy_) before a step to control the draw.  None: torch.rand_like per
        step, as the reference.  The tensors of `graph` and `class_info` are the step's static inputs: `load()`
        overwrites them in place."""
        self.model, self.graph, self.class_info, self.opt = model, graph, class_info, optimizer
        self.kw = dict(pclass=pclass, pfiber=pfiber, nfields=nfields, total_time=total_time, wutils=wutils, wvar=wvar)
        dev = class_info.device
        self.sharp = torch.zeros(1, dtype=torch.float32, device=dev)
        self.noise = noise
        self.loss = self.utility = None
        self._graph = None
        if use_graph:
            if _shard.active():
                raise ValueError("TrainStep: a fibre-sharded step all-reduces between ranks and runs eager "
                                 "(use_graph=False); collectives are not captured into a CUDA graph")
            for g in optimizer.param_groups:
                if not g.get("capturable", False):
                    raise ValueError("CUDA-graph capture needs torch.optim.Adam(..., capturable=True)")
            snap = self._snapshot(dev)
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):                       # warm-up: workspaces, topology, Adam state
                for _ in range(warmup):
                    self._eager()
            torch.cuda.current_stream(dev).wait_stream(side)
            self.opt.zero_grad(set_to_none=True)
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph):
                self._eager()
            self._restore(snap, dev)

    def _snapshot(self, dev):
        model_sd = {k: v.detach().clone() for k, v in self.model.state_dict().items()}
        opt_sd = {p: {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in st.items()}
                  for p, st in self.opt.state.items()}
        return model_sd, opt_sd, torch.cuda.get_rng_state(dev)

    def _restore(self, snap, dev):
        model_sd, opt_sd, rng = snap
        with torch.no_grad():
            for k, v in self.model.state_dict().items():
                v.copy_(model_sd[k])
            for p, st in self.opt.state.items():
                old = opt_sd.get(p)
                for k, v in st.items():
                    if torch.is_tensor(v):
                        if old is not None and k in old:
                            v.copy_(old[k])
                        else:
                            v.zero_()                           # state created by the warm-up: back to "never stepped"
        torch.cuda.set_rng_state(rng, dev)
        torch.cuda.synchronize(dev)

    def _eager(self):
        self.opt.zero_grad(set_to_none=True)
        out = self.model(self.graph)
        self.loss, self.utility = _loss.loss_function(self.model, out, self.class_info, sharpness=self.sharp,
                                                      noise=self.noise, **self.kw)
        self.loss.backward()
        self.opt.step()

    def load(self, batch, class_info=None):
        """Copies the node, edge and global features of `batch` (and `class_info`, if given) into the step's input
        tensors in place, for the next call.  The batch must have the shapes of the step's graph and its `edge_index`:
        the captured kernels hold that topology.  A batch of another size (the short last batch of `Loader.batches`)
        needs a step of its own."""
        mine = self.graph
        ei = batch.edge_index
        if ei is not mine.edge_index and (ei.shape != mine.edge_index.shape or not torch.equal(ei, mine.edge_index.to(ei.device))):
            raise ValueError("TrainStep.load: the batch's edge_index differs from the one the step was built on")
        pairs = [(getattr(mine, k), getattr(batch, k), k) for k in ("x_s", "x_t", "x_e", "x_u")]
        if class_info is not None:
            pairs.append((self.class_info, class_info, "class_info"))
        for dst, src, k in pairs:
            if src.shape != dst.shape:
                raise ValueError("TrainStep.load: %s is %s, the step was built for %s" % (k, tuple(src.shape), tuple(dst.shape)))
        with torch.no_grad():
            for dst, src, _ in pairs:
                if src is not dst:
                    dst.copy_(src)

    def __call__(self, sharpness):
        """Runs one step at this sharpness; returns (loss, utility) as device tensors (no host synchronisation): scalars,
        or for a batch the summed loss and the utilities [G]."""
        self.sharp.fill_(float(sharpness))
        if self._graph is not None:
            self._graph.replay()
        else:
            self._eager()
        return self.loss, self.utility
