"""Shared helpers for the parity tests (norm-wise error metric of SURVEY.md section 4.3)."""
import os

import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_loss_cases():
    """The reference's training loss on four cases in fp64, then the same four in fp32 (oracle/make_golden_loss.py)."""
    return [c for tag in ("f64", "f32") for c in torch.load(os.path.join(GOLDEN, "loss_cases_%s.pt" % tag))]


def upstream(t):
    return torch.linspace(0.5, 1.5, t.numel(), dtype=t.dtype, device=t.device).reshape(t.shape)


def nerr(a, b):
    """norm-wise error max|a-b| / max|b| (0 when both are all-zero)."""
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    assert a.shape == b.shape, (a.shape, b.shape)
    if b.numel() == 0:
        return 0.0
    scale = b.abs().max().item()
    diff = (a - b).abs().max().item()
    if scale == 0.0:
        return diff
    return diff / scale


def run_oracle_block(bo, case, dtype, training=None):
    """Run oracle/block_oracle.block on a golden case; returns outs, input grads, param grads, buffers."""
    training = case["training"] if training is None else training
    sd = bo.cast_state(case["state"], dtype)
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()
              if v.is_floating_point() and "running" not in k}
    full = dict(sd)
    full.update(params)
    ins = {n: case[n].to(dtype).clone().requires_grad_(True) for n in ("x_s", "x_t", "x_e", "u")}
    buffers = {}
    o_s, o_t, o_e, o_u = bo.block(full, "", case["edge_index"], ins["x_s"], ins["x_t"], ins["x_e"], ins["u"],
                                  training=training, normed=case.get("normed", True), buffers=buffers)
    loss = sum((o * upstream(o)).sum() for o in (o_s, o_t, o_e, o_u))
    loss.backward()
    outs = {"x_s": o_s.detach(), "x_t": o_t.detach(), "x_e": o_e.detach(), "u": o_u.detach()}
    gin = {n: t.grad for n, t in ins.items()}
    gparam = {k: p.grad for k, p in params.items() if p.grad is not None}
    return outs, gin, gparam, buffers
