"""Time one fp32 Block forward + backward at Fdim 10 on graphs whose fibres have more than 256 edges (split tiles),
with the c5a edge list (no fibre above 256 edges, whole-fibre tiles) for comparison.

Workloads, all in one call:
  complete512  the complete 12 500 x 512 graph (6.4 M edges, every fibre split in two), canonical order
  heavytail    100 000 fibres with heavy-tailed degrees up to ~3000 over 512 classes, shuffled
  c5a          the c5a edge list of bench.py (10 % of 100 000 x 512, shuffled, 5.12 M edges)

Per workload: ms per step by CUDA events over replays of the step captured as a CUDA graph (after warm-up), edges/s,
launches per step (pfs_launch_count on an eager step), per-kernel times from pfs_profile_* on eager steps and the share
of the step spent in the split-tile merge launches (k_split_moments, k_split_sums).  The card name and power limit are
printed with the numbers.  Writes one JSON line to stdout (and to --out if given).

  python tools/high_degree_bench.py --steps 20 --warmup 5
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

MERGE_KERNELS = ("k_split_moments", "k_split_sums")


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in out.split(",")]
    except Exception as e:           # the numbers still stand; the card's settings are then unknown
        info["power_limit"] = "unknown (%s)" % str(e)[:60]
    return info


def graph(name, dev):
    if name == "complete512":
        S, T = 12500, 512
        return S, T, torch.cartesian_prod(torch.arange(S), torch.arange(T)).T.contiguous().to(dev)
    if name == "heavytail":
        # 512 classes (the TModel tail holds T * 8F floats in one CTA); a fibre of more edges than classes revisits them
        S, T = 100000, 512
        g = torch.Generator().manual_seed(11)
        deg = (20 + torch.rand(S, generator=g) ** 12 * 3000).long()    # mean ~250 edges, a few fibres near 3000
        src = torch.repeat_interleave(torch.arange(S), deg)
        # a random first class and a stride coprime to T: the first T edges of a fibre go to T distinct classes
        start = torch.randint(0, T, (S,), generator=g)
        pos = torch.arange(int(deg.sum())) - torch.repeat_interleave(torch.cumsum(deg, 0) - deg, deg)
        tgt = (torch.repeat_interleave(start, deg) + 131 * pos) % T
        perm = torch.randperm(src.numel(), generator=g)
        return S, T, torch.stack([src[perm], tgt[perm]]).contiguous().to(dev)
    if name == "c5a":
        S, T = 100000, 512
        g = torch.Generator().manual_seed(7)
        e = torch.nonzero(torch.rand(S * T, generator=g) < 0.1).flatten()
        e = e[torch.randperm(e.numel(), generator=g)]
        return S, T, torch.stack([e // T, e % T]).contiguous().to(dev)
    raise ValueError(name)


def build_block(F, dev):
    from pfs_neural_net_b200 import gnn
    torch.manual_seed(0)
    blk = gnn.Block(F)
    g = torch.Generator().manual_seed(1)
    for m in blk.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.weight.data = 0.5 + torch.rand(m.weight.shape, generator=g)
            m.bias.data = 2 * torch.rand(m.bias.shape, generator=g) - 1
    return blk.to(dev).train()


def run(name, F, steps, warmup, dev):
    from pfs_neural_net_b200 import _abi
    from pfs_neural_net_b200.topology import get_topology
    lib = _abi.load_library()
    S, T, ei = graph(name, dev)
    E = ei.shape[1]
    gen = torch.Generator(device=dev).manual_seed(1234)
    ins = [torch.randn(n, F, generator=gen, device=dev) for n in (S, T, E, 1)]
    ups = [torch.linspace(0.5, 1.5, t.numel(), device=dev).reshape(t.shape) for t in ins]
    blk = build_block(F, dev)
    topo = get_topology(ei, S, T)
    t = topo.struct(1, F)
    layout = {"max_degree": int(topo.max_degree), "ntiles": int(t.ntiles), "split_fibres": int(t.nsplit),
              "split_tiles": int(t.nslots), "layout": "dense" if topo.dense else "csr"}

    def step():
        for p in blk.parameters():
            p.grad = None
        xs = [x.detach().requires_grad_(True) for x in ins]
        _, o_s, o_t, o_e, o_u = blk((ei, *xs))
        torch.autograd.backward([o_s, o_t, o_e, o_u], ups)

    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(max(warmup, 3)):
            step()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    n0 = lib.pfs_launch_count()
    step()
    torch.cuda.synchronize(dev)
    launches = int(lib.pfs_launch_count() - n0)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    for _ in range(warmup):
        g.replay()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        g.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    # per-kernel times on eager steps (a run of its own: the events slow the host)
    lib.pfs_profile_enable(1)
    for _ in range(steps):
        step()
    torch.cuda.synchronize(dev)
    rep = _abi.profile_report()
    lib.pfs_profile_enable(0)
    tot = sum(v[1] for v in rep.values())
    kernels = {k: {"launches_per_step": v[0] / steps, "ms_per_step": v[1] / steps}
               for k, v in sorted(rep.items(), key=lambda kv: -kv[1][1])}
    merge_ms = sum(rep[k][1] for k in MERGE_KERNELS if k in rep) / steps
    del g
    return {"workload": name, "S": S, "T": T, "E": E, "F": F, **layout, "ms_per_step": ms, "edges_per_s": E / (ms * 1e-3),
            "launches_per_step": launches, "merge_ms_per_step": merge_ms,
            "merge_share_of_kernel_time": merge_ms / (tot / steps) if tot else None, "kernels": kernels}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--fdim", type=int, default=10)
    ap.add_argument("--workloads", default="complete512,heavytail,c5a")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("high_degree_bench.py needs a CUDA device (the fp32 kernels have no CPU fallback)")
    dev = torch.device("cuda:0")
    res = {"card": card(), "results": []}
    for name in args.workloads.split(","):
        res["results"].append(run(name, args.fdim, args.steps, args.warmup, dev))
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    for r in res["results"]:
        print("%-12s %-24s E=%9d  %8.3f ms/step  %.3e edges/s  %3d launches  merge %.1f %% (%s, %s)" % (
            r["workload"], "ntiles=%d split=%d" % (r["ntiles"], r["split_fibres"]), r["E"], r["ms_per_step"],
            r["edges_per_s"], r["launches_per_step"], 100 * (r["merge_share_of_kernel_time"] or 0.0),
            res["card"]["name"], res["card"].get("power_limit")), file=sys.stderr)


if __name__ == "__main__":
    main()
