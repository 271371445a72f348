"""Time the training step of one graph whose fibres are sharded over the GPUs (shard.fibre_sharded(), DESIGN.md section 7).

One process per GPU, NCCL; with one GPU a one-rank group.  --graph c4 (the default): rank r holds the C4 slab,
--fibres-per-rank fibres x 512 classes, a canonical complete local graph.  --graph c5: the C5b edge list of bench.py
(100 000 x 512, 10 % Bernoulli, seed 7, shuffled), split by shard.partition_fibres; each rank trains its part with the
partition's edge_ids (the sharded edge-list loss).  x_s = global fibre index, x_t = the class table [T, 2], random bf16
edge features.  The model is GNN(B=--blocks, Fdim=128, F_s=1, F_t=2) in bf16, trained by loss_function and Adam in eager
steps (collectives are not captured into a CUDA graph).  Reports, with the card's name and power limit read in the same
run:
  ms per training step (CUDA events over --steps steps after --warmup, the maximum over the ranks) and edge-layers/s;
  the loss alone (sharded loss_from_times forward + backward with given noise) and the full-graph noise draw of the
  default noise (one torch.rand over all fibres x classes; for c5 over all edges, plus the gather of the rank's edges),
  each as ms and as a share of the step;
  collectives and bytes per step (shard.traffic()); peak memory per rank.
Writes one JSON line to stdout (and to --out if given).

  python tools/sharded_train_bench.py --steps 10 --warmup 3
  python tools/sharded_train_bench.py --graph c5 --steps 10 --warmup 3
"""
import argparse
import json
import os
import socket
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T, F = 512, 128                    # BASELINE configs C4 / C5: 512 classes, Fdim 128
S_C5 = 100000                      # C5b: fibres of the sparse graph


def card(index):
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in out.split(",")]
    except Exception as e:           # the numbers still stand; the card's settings are then unknown
        info["power_limit"] = "unknown (%s)" % str(e)[:60]
    return info


def class_table():
    g = torch.Generator().manual_seed(1)
    return torch.stack([0.5 + 3 * torch.rand(T, generator=g), 50 + 400 * torch.rand(T, generator=g)], 1)


def c5_edge_index():
    """the C5b edge list of bench.wide_graph: 10 % Bernoulli over S_C5 x T, seed 7, shuffled ([2, E] int64, CPU)"""
    g = torch.Generator().manual_seed(7)
    e = torch.nonzero(torch.rand(S_C5 * T, generator=g) < 0.1).flatten()
    e = e[torch.randperm(e.numel(), generator=g)]
    return torch.stack([e // T, e % T]).contiguous()


def _events(fn, n, dev):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / n


def _rank(rank, world, port, args, out):
    import torch.distributed as dist
    from bench import shutdown_process_group
    from pfs_neural_net_b200 import gnn as pg, loss as pl, shard
    from oracle import block_oracle as bo
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    ci = class_table().to(dev)
    graph = pg.BipartiteData.__new__(pg.BipartiteData)
    if args.graph == "c5":                                # this rank's fibres of the C5b edge list and their edge ids
        local, sl, edge_ids = shard.partition_fibres(c5_edge_index(), S_C5, world, rank)
        graph.edge_index, edge_ids = local.to(dev), edge_ids.to(dev)
        f0, S = sl.start, sl.stop - sl.start
    else:
        S = args.fibres_per_rank
        f0, edge_ids = rank * S, None
        graph.edge_index = bo.complete_bipartite(S, T).to(dev)
    E = graph.edge_index.shape[1]
    graph.x_s = torch.arange(f0, f0 + S, dtype=torch.float32, device=dev).reshape(S, 1).bfloat16()
    graph.x_t = ci.bfloat16()
    graph.x_e = torch.randn(E, F, generator=gen, device=dev, dtype=torch.bfloat16)
    graph.x_u = torch.zeros(1, F, dtype=torch.bfloat16, device=dev)
    graph.num_nodes = T
    torch.manual_seed(0)                                  # the same initial model on every rank
    model = pg.GNN(B=args.blocks, Fdim=F, T=T, F_s=1, F_t=2).to(torch.bfloat16).to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    rec = {}
    with shard.fibre_sharded():
        S_total = shard.total_count(S)
        E_total = shard.total_count(E, kind="edges")

        def step():
            opt.zero_grad(set_to_none=True)
            loss, _ = pl.loss_function(model, model(graph), ci, sharpness=0.5, edge_ids=edge_ids)
            loss.backward()
            opt.step()
            return loss

        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        shard.reset_traffic()
        rec["step_ms"] = _events(step, args.steps, dev)
        calls, nbytes = shard.traffic()
        rec["collectives_per_step"], rec["bytes_per_step"] = calls / args.steps, nbytes / args.steps
        rec["peak_mem_gb"] = torch.cuda.max_memory_allocated(dev) / 1e9
        with torch.no_grad():
            time = model.edge_prediction(model(graph).x_e, scale=42 / T).squeeze(-1).float()
        noise = torch.rand(E, generator=gen, device=dev)
        ei = graph.edge_index if edge_ids is not None else None

        def loss_alone():
            t = time.detach().requires_grad_(True)
            pl.loss_from_times(t, ci, S, T, sharpness=0.5, noise=noise, edge_index=ei, edge_ids=edge_ids)[0].backward()

        for _ in range(args.warmup):
            loss_alone()
        torch.cuda.synchronize(dev)
        rec["loss_ms"] = _events(loss_alone, args.steps, dev)
        if edge_ids is None:
            draw = lambda: torch.rand(S_total * T, device=dev)  # noqa: E731  (the default noise's full-graph draw)
        else:
            draw = lambda: torch.rand(E_total, device=dev)[edge_ids]  # noqa: E731  (the full edge list's, gathered)
        draw()
        rec["noise_draw_ms"] = _events(draw, args.steps, dev)
        rec["final_loss"] = float(step())
        rec["fibres"], rec["edges"], rec["edges_total"] = S, E, E_total
    if rank == 0:
        rec["card"] = card(dev.index)
    out[rank] = rec
    del model, opt, graph, time, noise, edge_ids
    torch.cuda.synchronize(dev)
    shutdown_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=0, help="ranks, one GPU each (0: every visible GPU)")
    ap.add_argument("--graph", choices=("c4", "c5"), default="c4",
                    help="c4: a complete slab per rank; c5: the C5b edge list split by fibre ranges")
    ap.add_argument("--blocks", type=int, default=3)
    ap.add_argument("--fibres-per-rank", type=int, default=12500, help="c4 only")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    class_table()                                         # inputs are built the same way with or without a GPU
    if not torch.cuda.is_available():
        sys.exit("sharded_train_bench.py needs a CUDA device: it measures the sharded step on the GPU (there is no CPU "
                 "fallback)")
    world = args.gpus or torch.cuda.device_count()
    if world > torch.cuda.device_count():
        sys.exit("sharded_train_bench.py: --gpus %d but %d visible GPUs (one rank per GPU)" % (world, torch.cuda.device_count()))
    import torch.multiprocessing as mp
    with mp.Manager() as mgr:
        res = mgr.dict()
        mp.spawn(_rank, args=(world, _free_port(), args, res), nprocs=world, join=True)
        res = dict(res)
    step_ms = max(res[r]["step_ms"] for r in range(world))
    loss_ms = max(res[r]["loss_ms"] for r in range(world))
    draw_ms = max(res[r]["noise_draw_ms"] for r in range(world))
    edges = res[0]["edges_total"]
    if args.graph == "c5":
        workload = ("fibre-sharded training step of an edge list: C5b, 10 %% Bernoulli %d x %d (%d edges), shuffled, split "
                    "by shard.partition_fibres (edges per rank %s), Fdim %d, bf16, GNN with %d Blocks, loss_function with "
                    "edge_ids, Adam, eager" % (S_C5, T, edges, [res[r]["edges"] for r in range(world)], F, args.blocks))
    else:
        workload = ("fibre-sharded training step: complete %d x %d graph (%d fibres per rank), Fdim %d, bf16, GNN with %d "
                    "Blocks, loss_function, Adam, eager" % (world * args.fibres_per_rank, T, args.fibres_per_rank, F,
                                                            args.blocks))
    rec = {"card": res[0]["card"], "ranks": world,
           "workload": workload,
           "steps": args.steps, "warmup": args.warmup, "edges": edges,
           "ms_per_step": step_ms, "edge_layers_per_s": edges * args.blocks * 1e3 / step_ms,
           "loss_ms": loss_ms, "loss_share": loss_ms / step_ms, "noise_draw_ms": draw_ms, "noise_draw_share": draw_ms / step_ms,
           "collectives_per_step": res[0]["collectives_per_step"], "bytes_per_step": res[0]["bytes_per_step"],
           "peak_mem_gb_per_rank": [res[r]["peak_mem_gb"] for r in range(world)],
           "final_loss": [res[r]["final_loss"] for r in range(world)]}
    print("%d rank(s), %d edges: %.2f ms/step, %.3e edge-layers/s; loss %.3f ms (%.1f %%), noise draw %.3f ms (%.1f %%); "
          "%.0f collectives / %.0f bytes per step; peak %.1f GB per rank; card %s"
          % (world, edges, step_ms, rec["edge_layers_per_s"], loss_ms, 100 * rec["loss_share"], draw_ms,
             100 * rec["noise_draw_share"], rec["collectives_per_step"], rec["bytes_per_step"],
             max(rec["peak_mem_gb_per_rank"]), rec["card"]), file=sys.stderr)
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
