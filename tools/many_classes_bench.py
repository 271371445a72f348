"""Time the fp32 path on graphs whose classes do not fit the one-CTA TModel tail: the class-tiled tail.

Workloads (one process, one GPU):
  * c5a_F16: the C5a edge list of bench.py (100 000 x 512, each pair an edge with probability 0.1, seed 7, shuffled)
    at Fdim 16, where the TModel tail runs class-tiled (T > 399 at Fdim 16);
  * complete_2000x1024_F10: the complete 2 000 x 1 024 graph at Fdim 10 (class-tiled: T > 639 at Fdim 10);
  * c5a_F10: the C5a edge list at Fdim 10, for comparison: there the one-CTA tail still runs.
For each: one fp32 Block forward + backward, and the training step of GNN(B=3) + loss + capturable Adam as a captured
TrainStep.  Reported: ms (CUDA events over --steps calls / graph replays after --warmup), library launches per call or
step (pfs_launch_count; a step's are counted on an eager step), and the time of the TModel tail kernels
(k_target_tail_*) with pfs_profile on an eager call or step, over the profiled library kernel time and over the
replayed step time, and the time of the EdgeModel backward kernel (k_edge_bwd, or k_edge_bwd2 where its staged tiles
do not fit: Fdim 16 edge lists of 72 fibres or more) of the Block call.  The card's name and power limit are read in the same run.
Writes one JSON line to stdout (and to --out if given).

  python tools/many_classes_bench.py --steps 10 --warmup 3 --out profiles/r03_many_classes_bench.json
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from sparse_train_bench import c5a_edge_index, card  # noqa: E402

B = 3
WORKLOADS = {
    "c5a_F16": dict(graph="c5a", F=16),
    "complete_2000x1024_F10": dict(graph="complete", S=2000, T=1024, F=10),
    "c5a_F10": dict(graph="c5a", F=10),
}
TAIL_PREFIX = "k_target_tail"


def tail_ms(report):
    tail = sum(ms for name, (n, ms) in report.items() if name.startswith(TAIL_PREFIX))
    total = sum(ms for n, ms in report.values())
    return tail, total, sorted(name for name in report if name.startswith(TAIL_PREFIX))


def profiled(lib, fn):
    from pfs_neural_net_b200 import _abi
    torch.cuda.synchronize()
    lib.pfs_profile_enable(1)
    n0 = lib.pfs_launch_count()
    fn()
    torch.cuda.synchronize()
    launches = int(lib.pfs_launch_count() - n0)
    report = _abi.profile_report()
    lib.pfs_profile_enable(0)
    return launches, report


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def time_block(ei, S, T, F, steps, warmup, dev, lib):
    from oracle import block_oracle as bo
    from pfs_neural_net_b200 import gnn
    E = ei.shape[1]
    blk = gnn.Block(F)
    blk.load_state_dict(bo.random_block_state(F, seed=0), strict=True)
    blk = blk.to(dev).train()
    gen = torch.Generator(device=dev).manual_seed(1)
    ins = [torch.randn(n, F, generator=gen, device=dev) for n in (S, T, E, 1)]
    ups = [torch.randn(n, F, generator=gen, device=dev) for n in (S, T, E, 1)]

    def call():
        x = [t.detach().requires_grad_(True) for t in ins]
        _, o_s, o_t, o_e, o_u = blk((ei, *x))
        torch.autograd.backward([o_s, o_t, o_e, o_u], ups)

    ms = timed(call, steps, warmup)
    launches, report = profiled(lib, call)
    t_ms, lib_ms, names = tail_ms(report)
    edge_bwd = {n: v[1] for n, v in report.items() if n in ("k_edge_bwd", "k_edge_bwd2")}    # which one ran, its ms
    return dict(ms=ms, launches=launches, tail_ms=t_ms, library_kernel_ms=lib_ms, tail_kernels=names,
                tail_share_of_kernels=t_ms / lib_ms, tail_share_of_call=t_ms / ms, edge_bwd_kernel_ms=edge_bwd)


def time_step(ei, S, T, F, steps, warmup, dev, lib):
    from pfs_neural_net_b200 import gnn as pg
    from pfs_neural_net_b200.train_step import TrainStep
    E = ei.shape[1]
    g = torch.Generator().manual_seed(3)
    graph = pg.BipartiteData(ei, (torch.arange(S, dtype=torch.float32).reshape(-1, 1) / S).to(dev),
                             torch.stack([0.5 + 3 * torch.rand(T, generator=g), 50 + 400 * torch.rand(T, generator=g)],
                                         -1).to(dev),
                             (2 + 8 * torch.rand(E, F, generator=g)).to(dev), torch.zeros(1, F, device=dev))
    class_info = graph.x_t.clone()
    res = {}
    for mode in ("eager", "graph"):
        torch.manual_seed(0)
        model = pg.GNN(B=B, Fdim=F, T=T, F_s=1, F_t=2).to(dev).train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
        step = TrainStep(model, graph, class_info, opt, use_graph=(mode == "graph"))
        if mode == "eager":
            for _ in range(warmup):
                step(0.5)
            launches, report = profiled(lib, lambda: step(0.5))
            t_ms, lib_ms, names = tail_ms(report)
            res.update(launches_per_step=launches, tail_ms_per_step=t_ms, library_kernel_ms_per_step=lib_ms,
                       tail_kernels=names, tail_share_of_kernels=t_ms / lib_ms)
        out = {}

        def call():
            out["loss"] = step(0.5)[0]

        res["ms_per_step_" + mode] = timed(call, steps, warmup)
        res["loss_" + mode] = float(out["loss"].detach())
        res["finite_" + mode] = bool(torch.isfinite(out["loss"].detach()))
        del step, model, opt
    res["tail_share_of_replayed_step"] = res["tail_ms_per_step"] / res["ms_per_step_graph"]
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="timed calls / steps per measurement")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out")
    args = ap.parse_args()
    names = args.workloads.split(",")
    for n in names:
        if n not in WORKLOADS:
            ap.error("unknown workload %s (known: %s)" % (n, ", ".join(WORKLOADS)))
    if not torch.cuda.is_available():
        sys.exit("many_classes_bench.py needs a CUDA device: it measures the fp32 kernels on the GPU "
                 "(there is no CPU fallback)")
    from pfs_neural_net_b200 import _abi
    dev = torch.device("cuda", 0)
    lib = _abi.load_library()
    rec = {"card": card(), "steps": args.steps, "warmup": args.warmup, "gnn_blocks": B, "workloads": {}}
    c5a = None
    for n in names:
        w = WORKLOADS[n]
        if w["graph"] == "c5a":
            if c5a is None:
                c5a = c5a_edge_index().to(dev)
            ei, S, T = c5a, 100000, 512
            desc = "C5a: 100000 x 512, 10 % Bernoulli, seed 7, shuffled"
        else:
            from oracle import block_oracle as bo
            S, T = w["S"], w["T"]
            ei = bo.complete_bipartite(S, T).to(dev)
            desc = "complete %d x %d, canonical order" % (S, T)
        F = w["F"]
        r = {"graph": desc, "S": S, "T": T, "E": int(ei.shape[1]), "Fdim": F,
             "tail": "class-tiled" if 4 * (T * 8 * F + 6 * F) > 200 * 1024 else "one CTA per graph"}
        r["block"] = time_block(ei, S, T, F, args.steps, args.warmup, dev, lib)
        torch.cuda.empty_cache()
        r["train_step"] = time_step(ei, S, T, F, args.steps, args.warmup, dev, lib)
        rec["workloads"][n] = r
        b, s = r["block"], r["train_step"]
        print("%-24s %s tail: Block fwd+bwd %8.3f ms, %d launches, tail %.3f ms (%.1f %% of kernel time); "
              "step %8.3f ms replayed, %8.3f ms eager, %d launches, tail %.1f %% of the replayed step"
              % (n, r["tail"], b["ms"], b["launches"], b["tail_ms"], 100 * b["tail_share_of_kernels"],
                 s["ms_per_step_graph"], s["ms_per_step_eager"], s["launches_per_step"],
                 100 * s["tail_share_of_replayed_step"]), file=sys.stderr)
    print("card: %s" % rec["card"], file=sys.stderr)
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
