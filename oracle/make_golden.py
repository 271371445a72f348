"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.pt from the UNMODIFIED reference.

Run in the build container (needs /root/reference):

    python oracle/make_golden.py

Every case runs the reference's own `Block` / `GNN` classes (imported through
`oracle/ref_loader.py`, nothing restated) in fp64 -- and fp32 for the outputs, so tests can show
err(ours) next to err(reference fp32) -- on seeded inputs, and stores inputs, weights, outputs,
input gradients, parameter gradients and the updated BatchNorm buffers.  The loss used for the
gradients is sum_i <out_i, linspace(0.5, 1.5)> over the four Block outputs (SURVEY.md section 8d).
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import block_oracle as bo  # noqa: E402
from oracle.ref_loader import load_reference_gnn  # noqa: E402

OUT_DIR = os.path.join(os.path.dirname(HERE), "tests", "golden")


def upstream(t):
    return torch.linspace(0.5, 1.5, t.numel(), dtype=t.dtype).reshape(t.shape)


def make_edge_index(kind, S, T, gen):
    dense = bo.complete_bipartite(S, T)
    if kind == "dense":
        return dense
    if kind == "fibre_major_permuted":          # like graphs/graph-0.pt (SURVEY.md section 0.10)
        cols = torch.stack([torch.randperm(T, generator=gen) for _ in range(S)]).reshape(-1)
        return torch.stack([dense[0], cols])
    if kind == "class_major":                   # reference src/graph.py:40-44 before the sort
        return torch.stack([torch.arange(S).repeat(T), torch.arange(T).repeat_interleave(S)])
    if kind == "shuffled":
        return dense[:, torch.randperm(S * T, generator=gen)]
    if kind == "sparse":                        # ~30 % density, shuffled, some empty fibres/classes
        keep = torch.rand(S * T, generator=gen) < 0.3
        keep &= dense[0] != 3                   # fibre 3 has no edges at all
        keep &= dense[1] != 1                   # class 1 has no edges at all
        e = dense[:, keep]
        return e[:, torch.randperm(e.shape[1], generator=gen)]
    if kind == "duplicates":
        e = dense[:, torch.randint(0, S * T, (S * T,), generator=gen)]
        return e
    raise ValueError(kind)


def run_block_case(ref, F, S, T, kind, seed, training, u_zero=False, normed=True):
    gen = torch.Generator().manual_seed(seed)
    sd32 = bo.random_block_state(F, seed=seed)
    if not training:
        # eval uses the running buffers: make them non-trivial
        for k in sd32:
            if k.endswith("running_mean"):
                sd32[k] = torch.randn(sd32[k].shape, generator=gen) * 0.3
            if k.endswith("running_var"):
                sd32[k] = 0.5 + torch.rand(sd32[k].shape, generator=gen)
    edge_index = make_edge_index(kind, S, T, gen)
    E = edge_index.shape[1]
    x_s = torch.randn(S, F, generator=gen, dtype=torch.float64)
    x_t = torch.randn(T, F, generator=gen, dtype=torch.float64)
    x_e = torch.randn(E, F, generator=gen, dtype=torch.float64)
    u = torch.zeros(1, F, dtype=torch.float64) if u_zero else torch.randn(1, F, generator=gen, dtype=torch.float64)

    out = {"F": F, "S": S, "T": T, "kind": kind, "training": training, "normed": normed,
           "edge_index": edge_index, "x_s": x_s, "x_t": x_t, "x_e": x_e, "u": u,
           "state": {k: v.clone() for k, v in sd32.items() if normed or ".norm." not in k}}
    for dtype, tag in ((torch.float64, "f64"), (torch.float32, "f32")):
        blk = ref.Block(F, normed=normed).to(dtype)
        state = bo.cast_state(sd32, dtype)
        blk.load_state_dict({k: v for k, v in state.items() if k in blk.state_dict()}, strict=True)
        blk.train(training)
        ins = [t.to(dtype).clone().requires_grad_(True) for t in (x_s, x_t, x_e, u)]
        _, o_s, o_t, o_e, o_u = blk((edge_index, ins[0], ins[1], ins[2], ins[3]))
        loss = sum((o * upstream(o)).sum() for o in (o_s, o_t, o_e, o_u))
        loss.backward()
        out["out_" + tag] = {"x_s": o_s.detach(), "x_t": o_t.detach(), "x_e": o_e.detach(), "u": o_u.detach()}
        out["gin_" + tag] = {n: t.grad.detach() for n, t in zip(("x_s", "x_t", "x_e", "u"), ins)}
        if dtype == torch.float64:   # fp32 parameter gradients are not stored (fixture size)
            out["gparam_" + tag] = {k: p.grad.detach() for k, p in blk.named_parameters() if p.grad is not None}
        out["buffers_" + tag] = {k: v.detach().clone() for k, v in blk.named_buffers()}
    return out


def run_gnn_case(ref, S, seed):
    """Shipped weights + train.py-style inputs (reference src/train.py:88-104), scaled down to S
    fibres; stores block outputs and the time head (src/gnn.py:307-312) with scale 42/12."""
    ck = torch.load(os.path.join(os.environ.get("PFS_REFERENCE_ROOT", "/root/reference"), "params",
                                 "model_gnn_0.pth"), map_location="cpu", weights_only=False)
    sd = ck["model_state"]
    gen = torch.Generator().manual_seed(seed)
    T, F = 12, 10
    class_info = torch.tensor([[2, 68200], [2, 69300], [2, 96300], [3, 7400], [6, 4500], [6, 8300], [6, 22000],
                               [6, 22000], [8, 9700], [12, 2800], [12, 14000], [12, 144008]], dtype=torch.float64)
    x_s = torch.arange(S, dtype=torch.float64).reshape(-1, 1)
    x_t = class_info
    edge_index = bo.complete_bipartite(S, T)
    x_e = 2.0 + 8.0 * torch.rand(S * T, F, generator=gen, dtype=torch.float64)
    u = torch.zeros(1, F, dtype=torch.float64)
    out = {"S": S, "T": T, "F": F, "edge_index": edge_index, "x_s": x_s, "x_t": x_t, "x_e": x_e, "u": u,
           "class_info": class_info,
           "state": {k: v.clone() for k, v in sd.items()}}      # shipped params/model_gnn_0.pth weights
    for training in (True, False):
        for dtype, tag in ((torch.float64, "f64"), (torch.float32, "f32")):
            model = ref.GNN(Fdim=F, B=3, F_s=1, F_t=2, T=T).to(dtype)
            model.load_state_dict(bo.cast_state(sd, dtype), strict=True)
            model.train(training)
            graph = ref.BipartiteData(edge_index, x_s.to(dtype), x_t.to(dtype), x_e.to(dtype), u.to(dtype))
            g2 = model(graph)
            time = model.edge_prediction(g2.x_e, scale=42 / 12)
            key = ("train_" if training else "eval_") + tag
            out[key] = {"x_s": g2.x_s.detach(), "x_t": g2.x_t.detach(), "x_e": g2.x_e.detach(), "u": g2.x_u.detach(),
                        "time": time.detach()}
            if training and dtype == torch.float64:
                time.sum().backward()
                out["gparam_train_f64"] = {k: p.grad.detach() for k, p in model.named_parameters()
                                           if p.grad is not None}
    return out


def main():
    ref = load_reference_gnn()
    os.makedirs(OUT_DIR, exist_ok=True)
    spec = [
        # name,                F,  S,  T, kind,                   seed, training, extra
        ("dense_train",        10, 40, 12, "dense",                11, True, {}),
        ("dense_eval",         10, 40, 12, "dense",                12, False, {}),
        ("dense_train_u0",     10, 23, 12, "dense",                13, True, {"u_zero": True}),
        ("dense_train_T5",     10, 50, 5, "dense",                 14, True, {}),
        ("dense_train_F16",    16, 21, 7, "dense",                 15, True, {}),
        ("dense_train_F4",     4, 33, 3, "dense",                  16, True, {}),
        ("dense_unnormed",     10, 17, 12, "dense",                17, True, {"normed": False}),
        ("permuted_train",     10, 40, 12, "fibre_major_permuted", 21, True, {}),
        ("class_major_train",  10, 31, 12, "class_major",          22, True, {}),
        ("shuffled_train",     10, 29, 12, "shuffled",             23, True, {}),
        ("sparse_train",       10, 45, 12, "sparse",               24, True, {}),
        ("sparse_eval",        10, 45, 12, "sparse",               25, False, {}),
        ("duplicates_train",   10, 25, 6, "duplicates",            26, True, {}),
    ]
    os.makedirs(os.path.join(OUT_DIR, "block_cases"), exist_ok=True)
    for name, F, S, T, kind, seed, training, extra in spec:
        case = run_block_case(ref, F, S, T, kind, seed, training, **extra)
        # one file per case keeps every golden file under 1 MB
        torch.save(case, os.path.join(OUT_DIR, "block_cases", name + ".pt"))
        print("block case", name, "E =", case["edge_index"].shape[1])
    gnn_case = run_gnn_case(ref, S=64, seed=31)
    torch.save(gnn_case, os.path.join(OUT_DIR, "gnn_shipped_weights.pt"))
    for f in os.listdir(OUT_DIR):
        print(f, os.path.getsize(os.path.join(OUT_DIR, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
