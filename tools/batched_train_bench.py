"""Time the reference's training step on a batch of G graphs per step, and the loss alone batched against a loop.

The step is the one of bench.py --workload train (reference src/train.py:136-141 at its sizes: a complete 2000 x 12
graph, Fdim 10, 3 Blocks, loss_function, Adam with capturable=True, one CUDA-graph replay per step), run on a collated
batch of G such graphs (same edge_index, own features and class table each) and the summed loss.  For each G:
  ms per step (CUDA events over replays after warm-up), graph-steps per second (G graphs trained per step),
  edge-layers per second (G * 24 000 edges * 3 Blocks per step), library launches per step (pfs_launch_count over one
  eager step).
Then the loss alone (loss_from_times forward + backward) on 256 graphs: one batched call against a Python loop of 256
single-graph calls, CUDA events around each.
The card's name and power limit are read in the same run and printed with the numbers.  Writes one JSON line to
stdout (and to --out if given).

  python tools/batched_train_bench.py --graphs 1,8,64,256 --steps 20 --warmup 5
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

S, T, F, B = 2000, 12, 10, 3          # reference src/config.py:16-23 (bench.py --workload train)


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in out.split(",")]
    except Exception as e:           # the numbers still stand; the card's settings are then unknown
        info["power_limit"] = "unknown (%s)" % str(e)[:60]
    return info


def make_batch(G, seed=1):
    """G complete S x T graphs as Loader.collate lays them out (CPU tensors): x_s [G,S,1], x_t = class table [G,T,2],
    x_e [G,S*T,F], x_u [G,1,F]; the inputs of bench.py --workload train, with a class table and edge features per graph."""
    g = torch.Generator().manual_seed(seed)
    ei = torch.cartesian_prod(torch.arange(S), torch.arange(T)).T.contiguous()          # reference src/train.py:94
    class_info = torch.stack([0.5 + 3 * torch.rand(G, T, generator=g), 50 + 400 * torch.rand(G, T, generator=g)], -1)
    x_s = torch.arange(S, dtype=torch.float32).reshape(1, S, 1).expand(G, S, 1).contiguous()
    x_e = 2 + 8 * torch.rand(G, S * T, F, generator=g)
    return ei, x_s, class_info, x_e, torch.zeros(G, 1, F)


def to_batch(tensors, dev):
    from pfs_neural_net_b200 import gnn as pg
    out = pg.BipartiteData.__new__(pg.BipartiteData)
    out.edge_index, out.x_s, out.x_t, out.x_e, out.x_u = (t.to(dev) for t in tensors)
    out.num_nodes = T
    return out


def time_step(G, tensors, steps, warmup, dev, lib):
    from pfs_neural_net_b200 import gnn as pg
    from pfs_neural_net_b200.train_step import TrainStep
    batch = to_batch(tensors, dev)
    class_info = tensors[2].to(dev)
    res = {"graphs": G}
    for mode in ("eager", "graph"):
        torch.manual_seed(0)
        model = pg.GNN(B=B, Fdim=F, T=T, F_s=1, F_t=2).to(dev).train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
        step = TrainStep(model, batch, class_info, opt, use_graph=(mode == "graph"))
        if mode == "eager":
            step(0.5)
            torch.cuda.synchronize(dev)
            n0 = lib.pfs_launch_count()
            step(0.5)
            torch.cuda.synchronize(dev)
            res["launches_per_step"] = int(lib.pfs_launch_count() - n0)
            continue
        for _ in range(warmup):
            step(0.5)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            loss, util = step(0.5 + 0.5 * i / steps)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / steps
        res.update(ms_per_step=ms, graph_steps_per_s=G * 1e3 / ms, edge_layers_per_s=G * S * T * B * 1e3 / ms,
                   loss=float(loss), finite=bool(torch.isfinite(util).all()))
        del step, model, opt
    torch.cuda.empty_cache()
    return res


def time_loss(G, steps, warmup, dev, lib):
    from pfs_neural_net_b200 import loss as pl
    gen = torch.Generator(device=dev).manual_seed(2)
    time_d = (2 * 42.0 / T) * torch.rand(G, S * T, generator=gen, device=dev)
    noise = torch.rand(G, S * T, generator=gen, device=dev)
    class_info = make_batch(G)[2].to(dev)

    def batched():
        t = time_d.detach().requires_grad_(True)
        pl.loss_from_times(t, class_info, S, T, noise=noise)[0].sum().backward()

    def loop():
        for g in range(G):
            t = time_d[g].detach().requires_grad_(True)
            pl.loss_from_times(t, class_info[g], S, T, noise=noise[g])[0].backward()

    out = {"graphs": G}
    for name, fn in (("batched", batched), ("loop", loop)):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize(dev)
        n0 = lib.pfs_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        out[name + "_ms"] = e0.elapsed_time(e1) / steps
        out[name + "_launches"] = (lib.pfs_launch_count() - n0) // steps
    out["loop_over_batched"] = out["loop_ms"] / out["batched_ms"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graphs", default="1,8,64,256", help="comma-separated batch sizes G")
    ap.add_argument("--loss-graphs", type=int, default=256)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()
    sizes = [int(x) for x in args.graphs.split(",")]
    make_batch(min(sizes))                                    # inputs are built the same way with or without a GPU
    if not torch.cuda.is_available():
        sys.exit("batched_train_bench.py needs a CUDA device: it measures the step on the GPU (there is no CPU fallback)")
    from pfs_neural_net_b200 import _abi
    dev = torch.device("cuda", 0)
    lib = _abi.load_library()
    rec = {"card": card(), "workload": "reference training step (%d x %d complete graph, Fdim %d, %d Blocks, loss_function, "
                                        "Adam capturable, one CUDA-graph replay per step) on a batch of G graphs" % (S, T, F, B),
           "steps": args.steps, "warmup": args.warmup, "train": [], "loss": None}
    for G in sizes:
        r = time_step(G, make_batch(G), args.steps, args.warmup, dev, lib)
        rec["train"].append(r)
        print("G=%4d  %8.3f ms/step  %10.1f graph-steps/s  %.3e edge-layers/s  %d launches/step"
              % (G, r["ms_per_step"], r["graph_steps_per_s"], r["edge_layers_per_s"], r["launches_per_step"]), file=sys.stderr)
    rec["loss"] = time_loss(args.loss_graphs, args.steps, args.warmup, dev, lib)
    lr = rec["loss"]
    print("loss fwd+bwd, %d graphs: batched %.3f ms (%d launches), loop of single-graph calls %.3f ms (%d launches): %.1fx"
          % (lr["graphs"], lr["batched_ms"], lr["batched_launches"], lr["loop_ms"], lr["loop_launches"], lr["loop_over_batched"]),
          file=sys.stderr)
    print("card: %s" % rec["card"], file=sys.stderr)
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
