"""Time the training loss and the training step on the sparse C5a edge list.

The graph is the one of bench.py --workload c5a: 100 000 fibres x 512 classes, each fibre-class pair an edge with
probability 0.1 (seeded), the edge list shuffled; about 5.12 M edges.  One process, one GPU.  Reports:
  * the loss alone, forward + backward (loss_from_times with edge_index), on that edge list, and beside it the canonical
    loss on a complete 10 000 x 512 graph of about the same E: ms (CUDA events over --iters calls after --warmup),
    library launches per call, the bytes the kernels must move (from the shapes, `loss_bytes`), and the share of
    the HBM bandwidth those bytes over that time imply;
  * the whole training step of GNN(B=3, Fdim=10, T=512) in fp32 on the C5a graph, eager and as a captured TrainStep:
    ms per step, and the standalone loss time over the step time;
  * the card's name and power limit, read in the same run.
Writes one JSON line to stdout (and to --out if given).

  python tools/sparse_train_bench.py --iters 50 --steps 10 --warmup 3
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

S, T, F, B = 100000, 512, 10, 3        # bench.py --workload c5a (BASELINE configs[4]) and the GNN of the step
S_DENSE = 10000                        # complete S_DENSE x T graph: the same E as the 10 % C5a graph
HBM_BYTES_PER_S = 7.7e12               # B200 data sheet (one GPU of an HGX B200)


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in out.split(",")]
    except Exception as e:           # the numbers still stand; the card's settings are then unknown
        info["power_limit"] = "unknown (%s)" % str(e)[:60]
    return info


def c5a_edge_index():
    """bench.py --workload c5a's edge list (CPU, int64 [2, E])"""
    gsp = torch.Generator().manual_seed(7)
    e = torch.nonzero(torch.rand(S * T, generator=gsp) < 0.1).flatten()
    e = e[torch.randperm(e.numel(), generator=gsp)]
    return torch.stack([e // T, e % T]).contiguous()


def loss_bytes(E, S_, T_, edge_list):
    """bytes one forward + backward must move, fp32 / int32, each array once per kernel that reads or writes it.
    Canonical: edge pass (time, noise in; galaxies, time2 out) 16 E, fibre sums 4 E, class partials 8 E, backward (time,
    noise, time2 in; g_time out) 16 E.  Edge list: edge pass 24 E (+ csr_eid, csr_tgt), fibre sums 8 E + 8 S (csr_eid,
    time2, rowptr, fibre_time), class pass 24 E (csc_q, csr_src, csr_eid, time2, galaxies in; cell_time out), backward
    28 E (csr_eid, csr_tgt, csr_src, time, noise, cell_time in; g_time out).  The O(T) tail is left out."""
    if edge_list:
        return 84 * E + 12 * S_
    return 44 * E + 4 * S_


def time_loss(ei, S_, T_, iters, warmup, dev, lib):
    from pfs_neural_net_b200 import loss as pl
    E = ei.shape[1] if ei is not None else S_ * T_
    gen = torch.Generator(device=dev).manual_seed(2)
    time_d = (2 * 42.0 / 51.2) * torch.rand(E, generator=gen, device=dev)   # C5a: fibre times around TOTAL_TIME
    noise = torch.rand(E, generator=gen, device=dev)
    ci = torch.stack([0.5 + 3 * torch.rand(T_, generator=gen, device=dev),
                      50 + 400 * torch.rand(T_, generator=gen, device=dev)], -1)
    kw = dict(noise=noise, edge_index=ei) if ei is not None else dict(noise=noise)

    def call():
        t = time_d.detach().requires_grad_(True)
        pl.loss_from_times(t, ci, S_, T_, **kw)[0].backward()

    for _ in range(warmup):
        call()
    torch.cuda.synchronize(dev)
    n0 = lib.pfs_launch_count()
    call()
    torch.cuda.synchronize(dev)
    launches = int(lib.pfs_launch_count() - n0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        call()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / iters
    nbytes = loss_bytes(E, S_, T_, ei is not None)
    return dict(S=S_, T=T_, E=E, ms=ms, launches=launches, bytes=nbytes, bytes_per_s=nbytes / (ms * 1e-3),
                hbm_share=nbytes / (ms * 1e-3) / HBM_BYTES_PER_S)


def time_step(ei, steps, warmup, dev):
    from pfs_neural_net_b200 import gnn as pg
    from pfs_neural_net_b200.train_step import TrainStep
    E = ei.shape[1]
    g = torch.Generator().manual_seed(3)
    graph = pg.BipartiteData.__new__(pg.BipartiteData)
    graph.edge_index = ei
    graph.x_s = (torch.arange(S, dtype=torch.float32).reshape(-1, 1) / S).to(dev)
    graph.x_t = torch.stack([0.5 + 3 * torch.rand(T, generator=g), 50 + 400 * torch.rand(T, generator=g)], -1).to(dev)
    graph.x_e = (2 + 8 * torch.rand(E, F, generator=g)).to(dev)
    graph.x_u = torch.zeros(1, F, device=dev)
    graph.num_nodes = T
    class_info = graph.x_t.clone()
    res = {}
    for mode in ("eager", "graph"):
        torch.manual_seed(0)
        model = pg.GNN(B=B, Fdim=F, T=T, F_s=1, F_t=2).to(dev).train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
        step = TrainStep(model, graph, class_info, opt, use_graph=(mode == "graph"))
        for _ in range(warmup):
            step(0.5)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            loss, util = step(0.5 + 0.5 * i / steps)
        e1.record()
        torch.cuda.synchronize(dev)
        res[mode] = dict(ms_per_step=e0.elapsed_time(e1) / steps, loss=float(loss.detach()),
                         finite=bool(torch.isfinite(loss.detach())))
        del step, model, opt
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50, help="timed loss calls")
    ap.add_argument("--steps", type=int, default=10, help="timed training steps per mode")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    ei = c5a_edge_index()                                     # inputs are built the same way with or without a GPU
    if not torch.cuda.is_available():
        sys.exit("sparse_train_bench.py needs a CUDA device: it measures the loss and the step on the GPU "
                 "(there is no CPU fallback)")
    from pfs_neural_net_b200 import _abi
    dev = torch.device("cuda", 0)
    lib = _abi.load_library()
    ei = ei.to(dev)
    rec = {"card": card(), "graph": "C5a: %d x %d, 10 %% Bernoulli, shuffled, seed 7, E = %d" % (S, T, ei.shape[1]),
           "iters": args.iters, "steps": args.steps, "warmup": args.warmup, "hbm_peak_bytes_per_s": HBM_BYTES_PER_S}
    rec["loss_edge_list"] = time_loss(ei, S, T, args.iters, args.warmup, dev, lib)
    rec["loss_canonical"] = time_loss(None, S_DENSE, T, args.iters, args.warmup, dev, lib)
    for k in ("loss_edge_list", "loss_canonical"):
        r = rec[k]
        print("%-15s %6d x %d, E %8d: %7.3f ms fwd+bwd, %d launches, %.3e B, %.2f TB/s = %.1f %% of HBM peak"
              % (k, r["S"], r["T"], r["E"], r["ms"], r["launches"], r["bytes"], r["bytes_per_s"] / 1e12,
                 100 * r["hbm_share"]), file=sys.stderr)
    rec["train_step"] = time_step(ei, args.steps, args.warmup, dev)
    for mode, r in rec["train_step"].items():
        r["loss_share"] = rec["loss_edge_list"]["ms"] / r["ms_per_step"]
        print("train step %-5s GNN(B=%d, Fdim=%d, T=%d) fp32: %8.3f ms/step, loss fwd+bwd %.1f %% of it"
              % (mode, B, F, T, r["ms_per_step"], 100 * r["loss_share"]), file=sys.stderr)
    print("card: %s" % rec["card"], file=sys.stderr)
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
