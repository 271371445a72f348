#!/usr/bin/env python
"""bench.py -- edges/sec, forward+backward, per GNN layer (`Block`) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[2], "C3"): a batch of 256 synthetic complete bipartite graphs of
2394 fibres x 12 classes (28 728 edges each), Fdim 10, fp32, train mode; one step = one `Block`
forward + backward w.r.t. all four outputs (upstream gradients linspace(0.5, 1.5)), every parameter
gets a gradient.  configs[1] (ONE such graph) needs ~1 us of HBM time, below a kernel-launch latency,
so the throughput configuration is the 256-graph batch (SURVEY.md section 0.7); the single graph is a
parity-test case (tests/test_gpu_parity.py::test_full_size_graph_c2).

N > 1 (launched by torchrun, one rank per GPU): data parallel over graph batches as BASELINE configs[2]
states it -- the batch of 256 graphs is split 256/N per GPU (STRONG scaling), weights replicated, one
NCCL all-reduce of the flat gradient bucket per step.  The step (forward, backward, bucket pack,
all-reduce) is captured once as a CUDA graph and replayed: at 32 graphs per GPU the ~40 kernel launches
of a step would otherwise be bound by the host.  The weak-scaling run (256 graphs per GPU) of round 1 is
kept as the extra key `weak`.  Extra keys of the default run: `c2` (BASELINE configs[1], ONE graph, with
and without an L2 flush between steps) and `c4` (a 3-step record of BASELINE configs[3], Fdim 128 bf16,
fibre-sharded over the N GPUs).

Printed JSON line: see the keys at the bottom.  `value` = edges of all ranks / device time (CUDA
events, max over ranks, inputs resident in HBM); `e2e` = the same through the nn.Module API with
pinned HOST inputs copied in every step and the loss read back; `roofline` = dominant kernel,
algorithmic bytes / CUDA-event duration against the measured HBM copy bandwidth (the binding
ceiling of these small-width MLPs is the FP32 FMA pipe, reported beside it in `fma`);
`cpu_baseline` = the oracle port of the reference path on this box's host cores.
"""
import argparse
import json
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "edges_per_sec_fwd_bwd_per_gnn_layer"
UNIT = "edges/s"

# algorithmic bytes each kernel must move, in units of F*4 bytes (one fp32 feature row):
# per edge (E) and per fibre (S); DESIGN.md section 6 derives them from SURVEY.md section 8(d).
KERNEL_ROWS = {
    "k_edge_fwd": (2, 0), "k_edge_bwd": (3, 0), "k_edge_bwd2": (3, 0), "k_edge_bn_bwd_stats": (2, 0), "k_affine_rows": (2, 0),
    "k_source_edge_fwd": (1, 10), "k_source_edge_bwd": (2, 18), "k_target_edge_fwd": (1, 2),
    "k_target_edge_bwd": (2, 2), "k_source_node_fwd": (0, 22), "k_source_node_bwd": (0, 32),
    "k_source_node_fwd_mma": (0, 22), "k_source_node_bwd_mma": (0, 32),
}
# DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) come from profiles/ncu_traffic.json, written by
# tools/ncu_traffic.py from an `ncu --set full` capture of the default C3 workload and stamped with the commit the
# capture was taken at; a kernel that is not in the file reports traffic null
def kernel_traffic():
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


# executed multiply-accumulates per edge / per fibre, forward + backward, in units of F^2 (DESIGN.md 6)
MAC_PER_EDGE_F2 = 60
MAC_PER_FIBRE_F2 = 318


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--graphs", type=int, default=256, help="graphs of the whole batch (split over the GPUs)")
    ap.add_argument("--no-graph", action="store_true", help="c3: launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-extras", action="store_true", help="c3: skip the weak / c2 / c4 extra records")
    ap.add_argument("--fibres", type=int, default=2394)
    ap.add_argument("--classes", type=int, default=12)
    ap.add_argument("--fdim", type=int, default=10)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work budget of the cpu_baseline sample")
    ap.add_argument("--workload", default="c3", choices=["c3", "c4", "c5", "c5a", "n1", "train"],
                    help="c3: 256 x 2394x12 graphs, Fdim 10 fp32 (headline); c4: one 12500*N x 512 graph, Fdim 128 bf16, "
                         "fibre-sharded over the N GPUs; c5: 10%% sparse 100000x512 edge list, Fdim 128 bf16 (CSR/CSC path); "
                         "c5a: the same edge list at Fdim 10 fp32 through the narrow kernels; "
                         "n1: the training loss (softfloor + loss_function) forward+backward on 612864 x 12 edge times; "
                         "train: the reference's whole training step (2000 x 12, 3 Blocks, loss, Adam) as a CUDA graph")
    ap.add_argument("--wide-fibres", type=int, default=12500, help="c4: fibres per GPU")
    ap.add_argument("--wide-classes", type=int, default=512)
    ap.add_argument("--wide-fdim", type=int, default=128)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="c3 / c5a: after the timed steps, write the outputs and gradients of the last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("c3", "c5a")):
        ap.error("--dump-outputs writes what the GPU path of c3 / c5a computes")
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(p.get("sm_max_mhz", 1965.0))
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


# ---------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi fields through NVML) running during the timed region
# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index, period=0.05):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    self.nv, "nvmlDeviceGetCurrentClocksEventReasons") else self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------------------------------------
# CPU reference arm: the oracle port of the reference path on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_reference_graph_step(bo, state, ei, ins, ups):
    """One Block forward + backward of the CPU arm: the UNMODIFIED reference `Block` (reference src/gnn.py:226-259, imported
    through oracle/ref_loader from /root/reference or its verbatim copy under baseline/_ref/) when it is present, else the
    oracle port.  Returns the kind that ran."""
    blk = _reference_block(state)
    xs = [t.clone().requires_grad_(True) for t in ins]
    if blk is not None:
        for p in blk.parameters():
            p.grad = None
        outs = blk((ei, xs[0], xs[1], xs[2], xs[3]))[1:]
        torch.autograd.backward(list(outs), [u for u in ups])
        return "reference"
    params = {k: v.clone().requires_grad_(True) for k, v in state.items() if v.is_floating_point() and "running" not in k}
    full = dict(state)
    full.update(params)
    outs = bo.block(full, "", ei, *xs, training=True, buffers={})
    torch.autograd.backward(list(outs), [u for u in ups])
    return "port"


_REF_BLOCKS = {}


def _reference_block(state):
    """The reference's own Block with `state` loaded (cached per state dict), or None when the reference is not on this box."""
    key = id(state)
    if key not in _REF_BLOCKS:
        blk = None
        try:
            from oracle import ref_loader
            if ref_loader.reference_available() and os.environ.get("PFS_CPU_ARM", "") != "port":
                ref = ref_loader.load_reference_gnn()
                F = state["edge_model.2.weight"].shape[0]
                blk = ref.Block(F)
                blk.load_state_dict({k: v.clone() for k, v in state.items()}, strict=True)
                blk.train()
        except Exception as e:                      # an importable port beats a broken vendored copy
            sys.stderr.write("bench: unmodified reference not usable (%r), timing the oracle port\n" % (e,))
            blk = None
        _REF_BLOCKS[key] = blk
    return _REF_BLOCKS[key]


CPU_KIND = {"kind": "port"}     # what the last CPU-arm run actually executed ("reference" = the unmodified Block)


def cpu_reference(args, seconds, steps=None, warmup=1):
    """Times the reference path on the host cores, reference-style threading (src/train.py:15-19): the UNMODIFIED
    reference Block through the shim when its sources are on this box (/root/reference, or the verbatim copy build()
    vendors under baseline/_ref/), else the oracle port (the two time the same within noise: VERDICT round 1).
    Returns (edges_per_s, cores, sample description, seconds per graph); CPU_KIND["kind"] says which one ran."""
    from oracle import block_oracle as bo
    ncores = os.cpu_count() or 1
    torch.set_num_threads(ncores)
    F, S, T = args.fdim, args.fibres, args.classes
    E = S * T
    state = bo.random_block_state(F, seed=0)
    ei = bo.complete_bipartite(S, T)
    g = torch.Generator().manual_seed(1234)
    ins = [torch.randn(S, F, generator=g), torch.randn(T, F, generator=g), torch.randn(E, F, generator=g),
           torch.randn(1, F, generator=g)]
    ups = [torch.linspace(0.5, 1.5, t.numel()).reshape(t.shape) for t in
           (ins[0], ins[1], ins[2], ins[3])]
    for _ in range(warmup):
        cpu_reference_graph_step(bo, state, ei, ins, ups)
    times = []
    t_begin = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        CPU_KIND["kind"] = cpu_reference_graph_step(bo, state, ei, ins, ups)
        times.append(time.perf_counter() - t0)
        if steps is not None:
            if len(times) >= steps:
                break
        elif time.perf_counter() - t_begin >= seconds and len(times) >= 3:
            break
    total = sum(times)
    return E * len(times) / total, ncores, ("%d forward+backward passes of one %dx%d graph (Fdim %d, fp32), one after the other as the "
                                            "reference runs its graphs; the batch is %d such graphs; %.1f s of CPU work"
                                            % (len(times), S, T, F, args.graphs, total)), total / len(times)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step_graphs = 8
    w_graphs = max(1, args.warmup)
    t0 = time.perf_counter()
    eps, ncores, sample, sec_per_graph = cpu_reference(args, seconds=0, steps=per_step_graphs * args.steps, warmup=w_graphs)
    ms_per_step = sec_per_graph * per_step_graphs * 1e3
    line = {
        "impl": "reference", "metric": METRIC, "value": eps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C3: batch of %d complete bipartite %dx%d graphs, Fdim %d, one Block fwd+bwd, train mode (CPU: each "
                               "step is a bounded sample of %d graphs of the batch, one after the other on all host cores)"
                               % (args.graphs, args.fibres, args.classes, args.fdim, per_step_graphs),
                   "global_graphs": args.graphs, "fibres": args.fibres, "classes": args.classes, "fdim": args.fdim},
        "cpu_baseline": {"value": eps, "unit": UNIT, "cores": ncores, "kind": CPU_KIND["kind"], "sample": sample},
        "e2e": {"value": eps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# end-to-end leg shared by all workloads
# ---------------------------------------------------------------------------------------------
def pipelined_e2e(dev, host, sets, steppers, timed, k):
    """Every step copies ITS inputs from pinned host memory and returns its result to the host.  The copies run on a
    second stream into one of two device input sets (sets[i] is read by steppers[i], a callable returning the step's
    device scalar), so the H2D of step i+1 overlaps the kernels of step i; the result goes back through a pinned buffer
    and is read one step late (an event per step), so the host never stalls the device inside the timed region.  All k
    copies-in and k reads-back happen inside it.  Returns ms per step."""
    copy_stream = torch.cuda.Stream(dev)
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    loss_host = [torch.zeros(1).pin_memory() for _ in range(2)]
    loss_ready = [torch.cuda.Event() for _ in range(2)]
    losses = []

    def issue_copy(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])          # the step that last used this slot is done with it
            for d, h in zip(sets[slot], host):
                d.copy_(h, non_blocking=True)
            copied[slot].record(copy_stream)

    def run(n):
        cur = torch.cuda.current_stream(dev)
        for ev in consumed:
            ev.record(cur)
        issue_copy(0)
        for i in range(n):
            slot = i & 1
            if i + 1 < n:
                issue_copy(slot ^ 1)                          # next step's inputs (copied afresh every step)
            cur.wait_event(copied[slot])
            loss = steppers[slot]()
            consumed[slot].record(cur)
            loss_host[slot].copy_(loss.detach().float().reshape(1), non_blocking=True)   # device -> host result
            loss_ready[slot].record(cur)
            if i > 0:                                         # read the previous step's result on the host
                loss_ready[slot ^ 1].synchronize()
                losses.append(float(loss_host[slot ^ 1][0]))
        last = (n - 1) & 1
        loss_ready[last].synchronize()
        losses.append(float(loss_host[last][0]))

    run(2)
    ms = timed(lambda: run(k), 1)
    return ms / k


E2E_NOTE = ("H2D of step i+1 on a copy stream overlaps the kernels of step i; loss read back one step late through a "
            "pinned buffer")


# ---------------------------------------------------------------------------------------------
# the B200 arm
# ---------------------------------------------------------------------------------------------
def build_block(F, dev):
    from pfs_neural_net_b200 import gnn
    torch.manual_seed(0)
    blk = gnn.Block(F)
    g = torch.Generator().manual_seed(1)
    for m in blk.modules():
        if isinstance(m, torch.nn.BatchNorm1d):     # non-trivial affine so the double norm matters
            m.weight.data = 0.5 + torch.rand(m.weight.shape, generator=g)
            m.bias.data = 2 * torch.rand(m.bias.shape, generator=g) - 1
    return blk.to(dev).train()


def numa_bind(local_rank):
    """Bind this rank to the CPUs of its GPU's NUMA node before any pinned buffer is allocated (first touch then puts
    the buffers on that node): with every rank on node 0 the host->device feed of 8 GPUs collapsed in round 1."""
    info = {"node": None}
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        info["pci"] = bdf
        info["node"] = node
        if node >= 0:
            with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
                cpus = set()
                for part in f.read().strip().split(","):
                    lo, _, hi = part.partition("-")
                    cpus.update(range(int(lo), int(hi or lo) + 1))
            cpus &= os.sched_getaffinity(0)
            if cpus:
                os.sched_setaffinity(0, cpus)
                info["cpus_bound"] = len(cpus)
    except Exception as e:          # best effort: an unknown topology leaves the affinity alone
        info["error"] = str(e)[:80]
    return info


class BlockStepper:
    """One data-parallel step of the layer: Block forward + backward w.r.t. all four outputs on static inputs, then
    the flat-bucket all-reduce; optionally captured as a CUDA graph (the NCCL all-reduce is a node of the graph)."""

    def __init__(self, blk, ei, xs, ups, bucket, dev, use_graph, warmup=3, pool=None, keep_results=False):
        self.blk, self.ei, self.xs, self.ups, self.bucket, self.dev = blk, ei, xs, ups, bucket, dev
        self.out = None
        self.keep_results = keep_results
        self.results = None
        self.graph = None
        if use_graph:
            cur = torch.cuda.current_stream(dev)
            side = torch.cuda.Stream(dev)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                for _ in range(warmup):
                    self.eager()
            cur.wait_stream(side)
            torch.cuda.synchronize(dev)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, pool=pool):
                self.eager()
        else:
            for _ in range(warmup):
                self.eager()

    def eager(self):
        for p in self.blk.parameters():
            p.grad = None
        xs = [x.detach().requires_grad_(True) for x in self.xs]
        _, o_s, o_t, o_e, o_u = self.blk((self.ei, xs[0], xs[1], xs[2], xs[3]))
        torch.autograd.backward([o_s, o_t, o_e, o_u], self.ups)
        self.bucket.all_reduce()
        self.out = o_u.detach().sum()        # the step's result (what the end-to-end leg reads back); no autograd graph kept
        if self.keep_results:
            # what a caller of the step receives; a graph replay rewrites these tensors in place.  Off by default: the
            # tensors it keeps alive would change how the timed step's memory is laid out
            self.results = {n: o.detach() for n, o in zip(("x_s", "x_t", "x_e", "u"), (o_s, o_t, o_e, o_u))}
            self.results.update({"grad_" + n: x.grad for n, x in zip(("x_s", "x_t", "x_e", "u"), xs)})
            self.results.update({"grad_" + n: p.grad for n, p in self.blk.named_parameters() if p.grad is not None})
        return self.out

    def __call__(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self.eager()
        return self.out


DUMP_ARRAY_BYTES = 7 << 20       # eight arrays scale with the graphs (four outputs, four input gradients): 56 MB of the 64


def dump_outputs(path, arrays):
    """Write every array as path/<name>.npy in float32.  An array larger than DUMP_ARRAY_BYTES is reduced to a fixed,
    seeded sample of its rows (leading dimensions flattened, rows kept whole and in order): the same rows on every run
    with the same arguments, so that the files of two builds can be compared element for element."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() * 4 > DUMP_ARRAY_BYTES:
            rows = t.reshape(-1, t.shape[-1] if t.dim() > 1 else 1)
            keep = max(1, DUMP_ARRAY_BYTES // (4 * rows.shape[1]))
            idx = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = rows[idx.to(rows.device)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def make_inputs(G, S, T, E, F, dev, seed):
    gen = torch.Generator(device=dev).manual_seed(seed)
    shapes = [(G, S, F), (G, T, F), (G, E, F), (G, 1, F)]
    ins = [torch.randn(s, generator=gen, device=dev) for s in shapes]
    ups = [torch.linspace(0.5, 1.5, s[1] * s[2], device=dev).reshape(1, s[1], s[2]).expand(s).contiguous() for s in shapes]
    return ins, ups


def run_ours(args):
    import torch.distributed as dist
    from pfs_neural_net_b200 import _abi, dp
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the message-passing layer has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = numa_bind(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _abi.load_library()
    S, T, F = args.fibres, args.classes, args.fdim
    E = S * T
    G_total = args.graphs
    G = max(1, G_total // world)                 # BASELINE configs[2]: the batch is split over the GPUs
    blk = build_block(F, dev)
    bucket = dp.GradBucket(blk.parameters())
    if world > 1:
        dp.broadcast_parameters(blk)
    if args.workload == "c5a":
        # BASELINE configs[4]: general sparse edge_index, 10% density, shuffled (SURVEY.md 8d "C5")
        G, G_total, S, T = 1, world, 100000, 512
        gsp = torch.Generator().manual_seed(7)
        e = torch.nonzero(torch.rand(S * T, generator=gsp) < 0.1).flatten()
        e = e[torch.randperm(e.numel(), generator=gsp)]
        ei = torch.stack([e // T, e % T]).contiguous().to(dev)
        E = int(e.numel())
    else:
        ei = torch.cartesian_prod(torch.arange(S), torch.arange(T)).T.contiguous().to(dev)   # reference src/train.py:94
    use_graph = not args.no_graph
    ins, ups = make_inputs(G, S, T, E, F, dev, 1234 + rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    # kernels of one step (counted on an eager step: a graph replay launches the same kernels without host calls)
    keep = bool(args.dump_outputs)
    eager = BlockStepper(blk, ei, ins, ups, bucket, dev, use_graph=False, warmup=max(args.warmup, 3),
                         keep_results=keep and not use_graph)
    n0 = lib.pfs_launch_count()
    eager()
    launches_per_step = int(lib.pfs_launch_count() - n0)
    stepper = BlockStepper(blk, ei, ins, ups, bucket, dev, use_graph=True, warmup=1, keep_results=keep) if use_graph else eager
    for _ in range(max(args.warmup, 3)):
        stepper()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms = timed(stepper, args.steps)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, stepper.results)
    ms_per_step = ms / args.steps
    edges_total = float(E) * G * world
    value = edges_total / (ms_per_step * 1e-3)

    # ---- per-kernel durations (CUDA events on the launch stream), eager steps ------------------------
    hbm_gbs, peak_src, sm_max = measured_peaks()
    roofline, kernels = None, None
    if not args.no_profile:
        lib.pfs_profile_enable(1)
        torch.cuda.synchronize(dev)
        for _ in range(args.steps):
            eager()
        torch.cuda.synchronize(dev)
        rep = _abi.profile_report()
        lib.pfs_profile_enable(0)
        tot = sum(v[1] for v in rep.values())
        kernels = {k: {"launches": v[0], "ms_per_step": v[1] / args.steps, "share": v[1] / tot}
                   for k, v in sorted(rep.items(), key=lambda kv: -kv[1][1])[:None if os.environ.get("PFS_BENCH_ALL_KERNELS") else 12]}
        cand = [k for k in rep if k in KERNEL_ROWS]
        if cand:
            top = max(cand, key=lambda k: rep[k][1])
            n, tms = rep[top]
            per_e, per_s = KERNEL_ROWS[top]
            bytes_per_launch = 4.0 * F * (per_e * E + per_s * S) * G
            dur_s = tms / n * 1e-3
            achieved = bytes_per_launch / dur_s / 1e9
            tr = kernel_traffic()
            same = args.workload == "c3" and (G, S, T, F) == (256, 2394, 12, 10)
            roofline = {"kernel": top, "bound": "hbm", "achieved": achieved, "peak": hbm_gbs, "unit": "GB/s",
                        "frac": achieved / hbm_gbs,
                        "traffic": tr.get("kernels", {}).get(top) if same else None,
                        "traffic_source": ("ncu --set full capture at commit %s (%s)" % (tr.get("commit"), tr.get("file")))
                        if same and tr else None, "peak_source": peak_src,
                        "avg_launch_ms": tms / n, "algorithmic_bytes_per_launch": bytes_per_launch,
                        "share_of_step": tms / tot, "binding": "fp32_fma (see fma)"}
    step_bytes = ((5.0 * F * 4 + (16 if args.workload == "c5a" else 0)) * E + 6.0 * (S + T) * F * 4) * G
    flops = 2.0 * F * F * (MAC_PER_EDGE_F2 * E + MAC_PER_FIBRE_F2 * S) * G
    clk = (clocks.get("sm_mhz") or sm_max)
    fma_peak = 148 * 128 * 2 * sm_max * 1e6 / 1e12
    fma = {"executed_tflops": flops / (ms_per_step * 1e-3) / 1e12, "peak_tflops_at_max_clock": fma_peak,
           "frac": flops / (ms_per_step * 1e-3) / 1e12 / fma_peak,
           "frac_at_measured_clock": flops / (ms_per_step * 1e-3) / 1e12 / (148 * 128 * 2 * clk * 1e6 / 1e12)}
    step_roofline = {"bound": "hbm", "achieved": step_bytes / (ms_per_step * 1e-3) / 1e9, "peak": hbm_gbs,
                     "unit": "GB/s", "frac": step_bytes / (ms_per_step * 1e-3) / 1e9 / hbm_gbs,
                     "algorithmic_bytes_per_step": step_bytes}

    # ---- end to end: pinned host inputs in, result out, every step ---------------------------------------
    # two input sets, each with its own captured step: the H2D copy of step i+1 (copy stream) overlaps step i
    e2e = None
    if not args.no_e2e:
        host = [x.detach().cpu().pin_memory() for x in ins]
        h2d = sum(h.numel() * h.element_size() for h in host)
        sets = [ins, [torch.empty_like(x) for x in ins]]
        pool = stepper.graph.pool() if use_graph else None
        steppers = [stepper, BlockStepper(blk, ei, sets[1], ups, bucket, dev, use_graph=use_graph, warmup=1, pool=pool)]
        ms_e = pipelined_e2e(dev, host, sets, steppers, timed, args.steps)
        e2e = {"value": edges_total / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
               "ms_per_step": ms_e, "pipelined": E2E_NOTE, "h2d_gbs_per_gpu": h2d / (ms_e * 1e-3) / 1e9,
               "result_read_back": "sum of the updated global features (4 bytes), as a training loop reads its loss"}
        del steppers, sets, host

    extras = {}
    if args.workload == "c3" and not args.no_extras:
        # ---- weak scaling (round 1's definition: 256 graphs per GPU), N > 1 only; at N = 1 it IS the headline ----
        if world > 1:
            stepper = eager = None
            torch.cuda.empty_cache()
            ins_w, ups_w = make_inputs(G_total, S, T, E, F, dev, 1234 + rank)
            st_w = BlockStepper(blk, ei, ins_w, ups_w, bucket, dev, use_graph=use_graph, warmup=3)
            ms_w = timed(st_w, args.steps) / args.steps
            extras["weak"] = {"graphs_per_gpu": G_total, "ms_per_step": ms_w, "value": float(E) * G_total * world / (ms_w * 1e-3),
                              "unit": UNIT, "scaling": "weak"}
            del st_w, ins_w, ups_w
            torch.cuda.empty_cache()
        # ---- C2: BASELINE configs[1], ONE 2394x12 graph (SURVEY.md 8d: latency-bound by construction) ----
        if world == 1:
            extras["c2"] = c2_record(args, blk, ei, bucket, dev, lib, hbm_gbs)

    # ---- CPU baseline (rank 0, N = 1) ------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.workload == "c3":
        eps, ncores, sample, _ = cpu_reference(args, seconds=args.cpu_seconds)
        cpu = {"value": eps, "unit": UNIT, "cores": ncores, "kind": CPU_KIND["kind"], "sample": sample}

    # ---- C4 (Fdim 128, bf16, tcgen05 path): a short record inside the driver-run line ----------------------
    if args.workload == "c3" and not args.no_extras:
        stepper = eager = ins = ups = None            # release the C3 tensors and the captured graph's pool
        torch.cuda.empty_cache()
        try:
            extras["c4"] = wide_record(args, "c4", world, rank, local_rank, dev, steps=3, warmup=3, with_e2e=False,
                                       with_cpu=False, with_profile=True)
        except Exception as e:                       # the headline line must survive a failure of the extra
            extras["c4"] = {"error": repr(e)[:200]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if args.workload == "c3" else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": ("C3: batch of %d complete bipartite %dx%d graphs split over %d GPU(s) (%d per GPU), Fdim %d, "
                                    "one Block fwd+bwd, train mode" % (G * world, S, T, world, G, F)) if args.workload == "c3" else
                                   ("C5a: 10%% Bernoulli edge list of %d x %d (%d edges, shuffled; CSR/CSC segmented "
                                    "reductions), Fdim %d fp32, one Block fwd+bwd" % (S, T, E, F)),
                       "graphs_per_gpu": G, "global_graphs": G * world, "fibres": S, "classes": T, "fdim": F,
                       "edges_per_step": edges_total, "parallelism": "dp%d" % world,
                       "launch": "one CUDA-graph replay per step (forward, backward, bucket pack, NCCL all-reduce)" if use_graph
                       else "eager launches",
                       "l2": "inputs larger than L2 (x_e %.0f MB per step per GPU)" % (G * E * F * 4 / 1e6)
                       if G * E * F * 4 > 126e6 else
                       "x_e is %.0f MB per GPU, below the 126 MB L2: every step reads the inputs the previous step left "
                       "in L2 (see c2 for the flushed variant of one graph)" % (G * E * F * 4 / 1e6)},
            "roofline": roofline, "step_roofline": step_roofline, "fma": fma, "kernels": kernels,
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches_per_step * args.steps,
            "gpu_launches_per_step": launches_per_step, "clocks": clocks, "numa": numa,
        }
        line.update(extras)
        print(json.dumps(line), flush=True)
    # NCCL does not let go of a communicator while a captured CUDA graph still holds its collectives: release every
    # stepper (and with it the graph) before the process group goes away
    stepper = eager = None
    import gc
    gc.collect()
    if world > 1:
        torch.cuda.synchronize(dev)
        shutdown_process_group()


def shutdown_process_group():
    """destroy_process_group with a watchdog: the record is already printed, so a teardown that does not return within
    a minute (a communicator still referenced by a CUDA graph, a peer that died) ends the process with status 0 instead
    of hanging the launcher."""
    import threading
    import torch.distributed as dist
    t = threading.Timer(60.0, lambda: os._exit(0))
    t.daemon = True
    t.start()
    dist.destroy_process_group()
    t.cancel()


def c2_record(args, blk, ei, bucket, dev, lib, hbm_gbs):
    """BASELINE configs[1]: one complete 2394x12 graph, Fdim 10, one Block forward+backward; graph replay and eager,
    with the inputs left in L2 by the previous step and with an L2 flush (a 512 MB write) before every step."""
    S, T, F = args.fibres, args.classes, args.fdim
    E = S * T
    ins, ups = make_inputs(1, S, T, E, F, dev, 4321)
    out = {"workload": "C2: one complete bipartite %dx%d graph, Fdim %d, fp32, one Block fwd+bwd" % (S, T, F), "edges": E}
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    n = 50
    for mode in ("graph", "eager"):
        st = BlockStepper(blk, ei, ins, ups, bucket, dev, use_graph=(mode == "graph"), warmup=3)
        for _ in range(5):
            st()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            st()
        e1.record()
        torch.cuda.synchronize(dev)
        warm = e0.elapsed_time(e1) / n
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(20)]
        for a, b in evs:
            flush.zero_()                      # evicts the inputs and the workspace from the 126 MB L2
            a.record()
            st()
            b.record()
        torch.cuda.synchronize(dev)
        cold = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
        out[mode] = {"ms_per_step": warm, "edges_per_s": E / (warm * 1e-3), "ms_per_step_l2_flushed": cold,
                     "edges_per_s_l2_flushed": E / (cold * 1e-3)}
        del st
    alg = (5.0 * F * 4) * E + 6.0 * (S + T) * F * 4
    out["hbm_frac_l2_flushed"] = alg / (out["graph"]["ms_per_step_l2_flushed"] * 1e-3) / 1e9 / hbm_gbs
    out["note"] = ("6.3 MB of algorithmic traffic = ~1 us of HBM time: the step is bound by the dependent chain of its kernels "
                   "(launch / drain latency), not by bandwidth or FLOPs")
    return out


# ---------------------------------------------------------------------------------------------
# wide workloads (C4 / C5b): one large graph, Fdim 128, bf16, tensor-core path
# ---------------------------------------------------------------------------------------------
WIDE_MAC_PER_EDGE_F2 = 48     # executed: fwd 16 F^2 (five GEMMs), bwd 32 F^2 (input + weight gradients), DESIGN.md 6
WIDE_MAC_PER_FIBRE_F2 = 318


def wide_graph(args, workload, rank, world, dev):
    """(edge_index of this rank's shard, S_local, T, E_local, description)."""
    T, S = args.wide_classes, args.wide_fibres
    if workload == "c4":
        ei = torch.cartesian_prod(torch.arange(S), torch.arange(T)).T.contiguous().to(dev)
        return ei, S, T, S * T, "C4: complete bipartite %d x %d (fibre range of %d per GPU), Fdim %d, bf16" % (
            S * world, T, S, args.wide_fdim)
    S = 100000 if args.wide_fibres == 12500 else args.wide_fibres
    g = torch.Generator().manual_seed(7)
    keep = torch.rand(S * T, generator=g) < 0.1
    e = torch.nonzero(keep).flatten()
    e = e[torch.randperm(e.numel(), generator=g)]
    ei = torch.stack([e // T, e % T]).contiguous()
    desc = "C5b: 10%% Bernoulli edge list of %d x %d (%d edges), shuffled, Fdim %d, bf16 (CSR/CSC path)" % (
        S, T, int(e.numel()), args.wide_fdim)
    if world > 1:
        # the SAME graph split by fibre range over the ranks (strong scaling): every rank keeps the edges of its fibres
        from pfs_neural_net_b200 import shard
        ei, sl, pos = shard.partition_fibres(ei, S, world, rank)
        S = sl.stop - sl.start
        desc += ", fibre-range sharded: rank %d holds %d fibres / %d edges" % (rank, S, int(pos.numel()))
    return ei.to(dev), S, T, int(ei.shape[1]), desc


def cpu_reference_wide(args, S_sub, seconds):
    """The reference Block (unmodified when present, else the oracle port: cpu_reference_graph_step) on the host cores, fp32,
    on a fibre sub-range of the wide graph (linear in fibres)."""
    from oracle import block_oracle as bo
    ncores = os.cpu_count() or 1
    torch.set_num_threads(ncores)
    F, T = args.wide_fdim, args.wide_classes
    E = S_sub * T
    state = bo.random_block_state(F, seed=0)
    ei = bo.complete_bipartite(S_sub, T)
    g = torch.Generator().manual_seed(1234)
    ins = [torch.randn(S_sub, F, generator=g), torch.randn(T, F, generator=g), torch.randn(E, F, generator=g),
           torch.randn(1, F, generator=g)]
    ups = [torch.linspace(0.5, 1.5, t.numel()).reshape(t.shape) for t in ins]
    cpu_reference_graph_step(bo, state, ei, ins, ups)
    times, t_begin = [], time.perf_counter()
    while len(times) < 2 or time.perf_counter() - t_begin < seconds:
        t0 = time.perf_counter()
        CPU_KIND["kind"] = cpu_reference_graph_step(bo, state, ei, ins, ups)
        times.append(time.perf_counter() - t0)
    total = sum(times)
    return E * len(times) / total, ncores, "%d steps on a %d-fibre sub-range (%d edges, Fdim %d, fp32) of the graph, %.1f s; " \
        "throughput is linear in fibres" % (len(times), S_sub, E, F, total)


def run_wide(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            t0 = time.perf_counter()
            eps, ncores, sample = cpu_reference_wide(args, 48, seconds=max(5.0, 2.0 * args.steps))
            print(json.dumps({
                "impl": "reference", "metric": METRIC, "value": eps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": {"workload": args.workload + " (CPU oracle port, sub-range)"},
                "cpu_baseline": {"value": eps, "unit": UNIT, "cores": ncores, "kind": CPU_KIND["kind"], "sample": sample},
                "e2e": {"value": eps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "wall_s": time.perf_counter() - t0}))
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the message-passing layer has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_bind(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rec = wide_record(args, args.workload, world, rank, local_rank, dev, steps=args.steps, warmup=args.warmup,
                      with_e2e=not args.no_e2e, with_cpu=not args.no_cpu_baseline, with_profile=not args.no_profile)
    if rank == 0:
        print(json.dumps(rec), flush=True)
    if world > 1:
        torch.cuda.synchronize(dev)
        shutdown_process_group()


def wide_record(args, workload, world, rank, local_rank, dev, steps, warmup, with_e2e, with_cpu, with_profile):
    """One bench record of a wide workload (c4: one fibre slab of the complete graph per rank, weak scaling; c5: the
    sparse graph partitioned by fibre range, strong scaling); the process group, if any, is already initialised.  Returns the record on every rank (rank 0 prints it)."""
    import torch.distributed as dist
    from pfs_neural_net_b200 import _abi, gnn, shard
    sharded = world > 1                     # c4: a fibre slab of the complete graph per rank; c5: partition_fibres
    lib = _abi.load_library()
    F = args.wide_fdim
    ei, S, T, E, desc = wide_graph(args, workload, rank, world, dev)
    torch.manual_seed(0)
    blk = gnn.Block(F)
    g = torch.Generator().manual_seed(1)
    for m in blk.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.weight.data = 0.5 + torch.rand(m.weight.shape, generator=g)
            m.bias.data = 2 * torch.rand(m.bias.shape, generator=g) - 1
    blk = blk.to(torch.bfloat16).to(dev).train()
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    gen_rep = torch.Generator(device=dev).manual_seed(99)            # replicated tensors: same on every rank
    bf = torch.bfloat16
    ins = [torch.randn(S, F, generator=gen, device=dev).to(bf), torch.randn(T, F, generator=gen_rep, device=dev).to(bf),
           torch.randn(E, F, generator=gen, device=dev).to(bf), torch.randn(1, F, generator=gen_rep, device=dev).to(bf)]
    ups = [torch.linspace(0.5, 1.5, t.shape[1], device=dev).to(bf).expand(t.shape).contiguous() for t in ins]
    ctx = (lambda: shard.fibre_sharded()) if sharded else (lambda: __import__("contextlib").nullcontext())

    def step(xs):
        for p in blk.parameters():
            p.grad = None
        xs = [x.requires_grad_(True) for x in xs]
        with ctx():
            _, o_s, o_t, o_e, o_u = blk((ei, xs[0], xs[1], xs[2], xs[3]))
            torch.autograd.backward([o_s, o_t, o_e, o_u], ups)
        return o_u

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = lib.pfs_launch_count()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        launches = lib.pfs_launch_count() - n0
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms, launches

    detached = [x.detach() for x in ins]
    for _ in range(max(warmup, 3)):
        step([x.detach() for x in detached])
    shard.reset_traffic()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms, launches = timed(lambda: step([x.detach() for x in detached]), steps)
    clocks = sampler.stop()
    coll_calls, coll_bytes = shard.traffic()
    ms_per_step = ms / steps
    if world > 1 and workload == "c5":      # shard sizes differ: the job's edges are the sum over the ranks
        t = torch.tensor([float(E)], device=dev, dtype=torch.float64)
        dist.all_reduce(t)
        edges_total = float(t.item())
    else:
        edges_total = float(E) * world
    value = edges_total / (ms_per_step * 1e-3)
    hbm_gbs, peak_src, sm_max = measured_peaks()
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            tensor_peak = float(json.load(f)["bf16_tflops_sustained"])
        tpeak_src = "measured sustained bf16 matmul (MEASURED_PEAKS.json)"
    except Exception:
        tensor_peak, tpeak_src = 1387.0, "fallback (B200_PROFILING.md)"
    flops = 2.0 * F * F * (WIDE_MAC_PER_EDGE_F2 * E + WIDE_MAC_PER_FIBRE_F2 * S)
    kernels, roofline = None, None
    if with_profile:
        lib.pfs_profile_enable(1)
        torch.cuda.synchronize(dev)
        nprof = min(steps, 5)
        for _ in range(nprof):
            step([x.detach() for x in detached])
        torch.cuda.synchronize(dev)
        rep = _abi.profile_report()
        lib.pfs_profile_enable(0)
        tot = sum(v[1] for v in rep.values())
        kernels = {k: {"launches": v[0], "ms_per_step": v[1] / nprof, "share": v[1] / tot}
                   for k, v in sorted(rep.items(), key=lambda kv: -kv[1][1])[:12]}
        gemm_ms = sum(v[1] for k, v in rep.items() if k.startswith("k_wide_gemm")) / nprof
        achieved = flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None
        roofline = {"kernel": "k_wide_gemm_nt + k_wide_gemm_tn (all tcgen05 GEMM launches of the step)", "bound": "tensor",
                    "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s",
                    "frac": achieved / tensor_peak if achieved else None, "traffic": None, "peak_source": tpeak_src,
                    "gemm_ms_per_step": gemm_ms, "share_of_step": gemm_ms * nprof / tot,
                    "executed_flops_per_step": flops}
    step_bytes = (5.0 * F * 2 + (0 if workload == "c4" else 16)) * E + 6.0 * (S + T) * F * 2
    step_roofline = {"bound": "hbm", "achieved": step_bytes / (ms_per_step * 1e-3) / 1e9, "peak": hbm_gbs, "unit": "GB/s",
                     "frac": step_bytes / (ms_per_step * 1e-3) / 1e9 / hbm_gbs, "algorithmic_bytes_per_step": step_bytes}
    tensor = {"executed_tflops": flops / (ms_per_step * 1e-3) / 1e12, "peak_tflops": tensor_peak,
              "frac": flops / (ms_per_step * 1e-3) / 1e12 / tensor_peak, "peak_source": tpeak_src}
    e2e = None
    if with_e2e:
        host = [x.detach().cpu().pin_memory() for x in ins]
        h2d = sum(h.numel() * h.element_size() for h in host)

        def e2e_step(dbuf):
            for p in blk.parameters():
                p.grad = None
            xs = [d.detach().requires_grad_(True) for d in dbuf]
            with ctx():
                _, o_s, o_t, o_e, o_u = blk((ei, xs[0], xs[1], xs[2], xs[3]))
                torch.autograd.backward([o_s, o_t, o_e, o_u], ups)
            return o_u.float().sum()

        sets = [detached, [torch.empty_like(x) for x in detached]]
        ms_e = pipelined_e2e(dev, host, sets, [lambda: e2e_step(sets[0]), lambda: e2e_step(sets[1])],
                             lambda fn, k: timed(fn, k)[0], steps)
        e2e = {"value": edges_total / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
               "ms_per_step": ms_e, "pipelined": E2E_NOTE}
    cpu = None
    if rank == 0 and world == 1 and with_cpu:
        eps, ncores, sample = cpu_reference_wide(args, 48, seconds=args.cpu_seconds)
        cpu = {"value": eps, "unit": UNIT, "cores": ncores, "kind": CPU_KIND["kind"], "sample": sample}
    return {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if workload == "c5" else "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": desc, "fibres_per_gpu": S, "classes": T, "fdim": F, "edges_per_step": edges_total,
                   "parallelism": ("fibre-sharded x%d (class-side all-reduces: %d calls, %d bytes per step)"
                                   % (world, coll_calls // max(steps, 1), coll_bytes // max(steps, 1)))
                   if sharded else "single GPU",
                   "l2": "inputs larger than L2 (x_e %.0f MB per step)" % (E * F * 2 / 1e6)},
        "roofline": roofline, "step_roofline": step_roofline, "tensor": tensor, "kernels": kernels, "cpu_baseline": cpu,
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks}


# ---------------------------------------------------------------------------------------------
# N1: the training loss that follows the path (reference src/train.py:21-80), forward + backward
# ---------------------------------------------------------------------------------------------
def complete_bipartite(S, T):
    """canonical dense edge order of reference src/train.py:94"""
    return torch.cartesian_prod(torch.arange(S), torch.arange(T)).T.contiguous()


def run_loss(args):
    S, T = args.fibres * args.graphs, args.classes            # one graph with the edge count of the C3 batch
    E = S * T
    g = torch.Generator().manual_seed(1)
    class_info = torch.stack([0.5 + 3 * torch.rand(T, generator=g), 50 + 400 * torch.rand(T, generator=g)], 1)
    if args.impl == "reference":
        from oracle import loss_oracle as lo                    # CPU arm only
        Sc = 20000
        ncores = os.cpu_count() or 1
        torch.set_num_threads(ncores)
        ei = complete_bipartite(Sc, T)
        time_c, noise_c = 6 * torch.rand(Sc * T, generator=g), torch.rand(Sc * T, generator=g)
        ts = []
        for _ in range(args.warmup + args.steps):
            tt = time_c.clone().requires_grad_(True)
            t0 = time.perf_counter()
            lo.loss_terms(tt, noise_c, class_info, ei, Sc, T)["loss"].backward()
            ts.append(time.perf_counter() - t0)
        ts = ts[args.warmup:]
        eps = Sc * T * len(ts) / sum(ts)
        print(json.dumps({"impl": "reference", "metric": "edges_per_sec_loss_fwd_bwd", "value": eps, "unit": UNIT, "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(ts) / len(ts), "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": "N1 loss fwd+bwd, CPU oracle port on %d x %d edge times" % (Sc, T)},
                          "cpu_baseline": {"value": eps, "unit": UNIT, "cores": ncores, "kind": "port", "sample": "%d steps" % len(ts)},
                          "e2e": {"value": eps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return
    from pfs_neural_net_b200 import _abi, loss as pl
    dev = torch.device("cuda", 0)
    lib = _abi.load_library()
    ci = class_info.to(dev)
    gen = torch.Generator(device=dev).manual_seed(2)
    time_d = 6 * torch.rand(E, generator=gen, device=dev)
    noise = torch.rand(E, generator=gen, device=dev)

    def step():
        t = time_d.detach().requires_grad_(True)
        loss = pl.loss_from_times(t, ci, S, T, noise=noise)[0]
        loss.backward()
        return loss

    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = lib.pfs_launch_count()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize(dev)
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    launches = lib.pfs_launch_count() - n0
    hbm_gbs, peak_src, _ = measured_peaks()
    alg = 12.0 * E                                            # read time + noise, write g_time
    print(json.dumps({"metric": "edges_per_sec_loss_fwd_bwd", "value": E / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "f32", "data": "synthetic",
                      "config": {"workload": "N1: training loss (softfloor + loss_function) forward+backward on %d x %d edge times"
                                             % (S, T), "l2": "inputs larger than L2 (%.0f MB per tensor)" % (E * 4 / 1e6)},
                      "roofline": {"kernel": "whole loss step (5 kernels)", "bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9,
                                   "peak": hbm_gbs, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / hbm_gbs, "traffic": None,
                                   "peak_source": peak_src, "algorithmic_bytes_per_step": alg},
                      "gpu_launches": int(launches), "clocks": clocks}))


# ---------------------------------------------------------------------------------------------
# N2: the reference's whole training step (src/train.py:136-141) at its own sizes (src/config.py:16-23)
# ---------------------------------------------------------------------------------------------
PUBLISHED_TRAIN_ITS = 65.86      # it/s, 1x A100, reference slurm/slurm-2561734.out:1 (BASELINE.md section 1)


def run_train(args):
    S, T, F, B = 2000, 12, 10, 3
    g = torch.Generator().manual_seed(1)
    class_info = torch.stack([0.5 + 3 * torch.rand(T, generator=g), 50 + 400 * torch.rand(T, generator=g)], 1)
    x_s = torch.arange(S, dtype=torch.float32).reshape(-1, 1)
    x_e = 2 + 8 * torch.rand(S * T, F, generator=g)
    ei = complete_bipartite(S, T)
    desc = "reference training step: %d x %d graph, Fdim %d, %d Blocks, loss_function, Adam (src/train.py:136-141)" % (S, T, F, B)
    if args.impl == "reference":
        from oracle import block_oracle as bo, loss_oracle as lo      # CPU arm only
        ncores = os.cpu_count() or 1
        torch.set_num_threads(ncores)
        torch.manual_seed(0)
        state = {}
        for b in range(B):
            state.update({"mpb.%d.%s" % (b, k): v for k, v in bo.random_block_state(F, seed=b).items()})
        lin = lambda o, i: ((torch.rand(o, i) * 2 - 1) / i ** 0.5, (torch.rand(o) * 2 - 1) / i ** 0.5)
        for name, (d1, d2, d3) in (("encoder_s.", (1, F, F)), ("encoder_t.", (2, F, F)), ("decoder_e.", (F, F, 1))):
            state[name + "0.weight"], state[name + "0.bias"] = lin(d2, d1)
            state[name + "2.weight"], state[name + "2.bias"] = lin(d3, d2)
        params = {k: v.clone().requires_grad_(True) for k, v in state.items() if v.is_floating_point() and "running" not in k}
        opt = torch.optim.Adam(params.values(), lr=1e-3)
        full = dict(state)
        full.update(params)
        ts = []
        for it in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            opt.zero_grad()
            xs, xt, xe, u = bo.gnn_forward(full, B, ei, x_s, class_info, x_e, torch.zeros(1, F), training=True, buffers={})
            tm = bo.edge_prediction(full, xe, 42 / T).squeeze(-1)
            lo.loss_terms(tm, torch.rand_like(tm), class_info, ei, S, T)["loss"].backward()
            opt.step()
            ts.append(time.perf_counter() - t0)
        ts = ts[args.warmup:]
        its = len(ts) / sum(ts)
        print(json.dumps({"impl": "reference", "metric": "train_steps_per_sec", "value": its, "unit": "it/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / its, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": its / PUBLISHED_TRAIN_ITS, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": desc + " -- CPU oracle port"},
                          "cpu_baseline": {"value": its, "unit": "it/s", "cores": ncores, "kind": "port", "sample": "%d steps" % len(ts)},
                          "e2e": {"value": its, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return
    from pfs_neural_net_b200 import _abi, gnn as pg
    from pfs_neural_net_b200.train_step import TrainStep
    dev = torch.device("cuda", 0)
    lib = _abi.load_library()
    res = {}
    for mode in ("eager", "graph"):
        torch.manual_seed(0)
        model = pg.GNN(B=B, Fdim=F, T=T, F_s=1, F_t=2).to(dev).train()
        graph = pg.BipartiteData(ei, x_s, class_info, x_e, torch.zeros(1, F))
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
        step = TrainStep(model, graph, class_info.to(dev), opt, use_graph=(mode == "graph"))
        for i in range(max(3, args.warmup)):
            step(0.5)
        torch.cuda.synchronize(dev)
        n0 = lib.pfs_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler = ClockSampler(0)
        sampler.start()
        e0.record()
        for i in range(args.steps):
            loss, util = step(0.5 + 0.5 * i / args.steps)
        e1.record()
        torch.cuda.synchronize(dev)
        clocks = sampler.stop()
        res[mode] = dict(ms=e0.elapsed_time(e1) / args.steps, launches=(lib.pfs_launch_count() - n0) / args.steps,
                         loss=float(loss.detach()), clocks=clocks)
    ms = res["graph"]["ms"]
    # end to end: the host reads the loss of every step (the reference's loss.item(), src/train.py:143)
    t_e2e0 = torch.cuda.Event(enable_timing=True); t_e2e1 = torch.cuda.Event(enable_timing=True)
    t_e2e0.record()
    for i in range(args.steps):
        loss, util = step(0.5)
        float(loss.detach())
    t_e2e1.record()
    torch.cuda.synchronize(dev)
    ms_e = t_e2e0.elapsed_time(t_e2e1) / args.steps
    print(json.dumps({"metric": "train_steps_per_sec", "value": 1e3 / ms, "unit": "it/s", "n_gpus": 1, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": (1e3 / ms) / PUBLISHED_TRAIN_ITS, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": desc + ", one CUDA-graph replay per step",
                                 "baseline": "published 65.86 it/s on 1x A100 (reference slurm/slurm-2561734.out:1)",
                                 "eager_ms_per_step": res["eager"]["ms"], "kernels_per_step_in_library": res["eager"]["launches"],
                                 "edge_layers_per_s": S * T * B * 1e3 / ms},
                      "e2e": {"value": 1e3 / ms_e, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 4,
                              "ms_per_step": ms_e, "note": "inputs are the static training graph (never re-copied, as in the "
                                                           "reference); the loss is read back every step"},
                      "gpu_launches": int(res["eager"]["launches"] * args.steps), "clocks": res["graph"]["clocks"]}))


def main():
    args = parse_args()
    if args.workload == "n1":
        return run_loss(args)
    if args.workload == "train":
        return run_train(args)
    if args.workload in ("c4", "c5"):
        run_wide(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
