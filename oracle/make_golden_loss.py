"""TEST INFRASTRUCTURE ONLY -- golden vectors of the reference training loss (run in the build container):

    python oracle/make_golden_loss.py

Calls the UNMODIFIED `train.loss_function` (/root/reference/src/train.py:29-80) with a stand-in for the module-global
`gnn` whose `edge_prediction` returns preset edge times (the loss reads the model only through that call,
src/train.py:42) and with the config globals NFIBERS / NCLASSES overridden for small cases.  The noise the reference
draws inside `softfloor` (torch.rand_like, src/train.py:22) is reproduced by seeding the default generator identically
and recorded next to the outputs.  Writes tests/golden/loss_cases_f64.pt and loss_cases_f32.pt (one file per
dtype keeps each under 1 MB).
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import block_oracle as bo  # noqa: E402
from oracle.ref_loader import load_reference_train  # noqa: E402

OUT_DIR = os.path.join(os.path.dirname(HERE), "tests", "golden")


class _Stub:
    def __init__(self, time):
        self.time = time

    def edge_prediction(self, x_e, scale=1):
        return self.time.unsqueeze(-1)


class _Graph:
    pass


def run_case(train, S, T, seed, dtype, spread):
    g = torch.Generator().manual_seed(seed)
    hours = (0.5 + 3 * torch.rand(T, generator=g)).to(dtype)
    counts = (50 + 400 * torch.rand(T, generator=g)).to(dtype)           # N_i * NFIELDS
    class_info = torch.stack([hours, counts], 1)
    time = (spread * torch.rand(S * T, generator=g)).to(dtype).requires_grad_(True)
    ei = bo.complete_bipartite(S, T)
    graph = _Graph()
    graph.edge_index, graph.x_e = ei, torch.zeros(S * T, 1, dtype=dtype)
    train.gnn = _Stub(time)
    train.NFIBERS, train.NCLASSES = S, T
    torch.manual_seed(seed)
    noise = torch.rand_like(time.detach())                               # what softfloor will draw
    torch.manual_seed(seed)
    loss, utils, comp, n_prime, fibers, time2, variance = train.loss_function(graph, class_info, finaloutput=True)
    loss.backward()
    return dict(S=S, T=T, seed=seed, class_info=class_info, time=time.detach(), noise=noise, loss=loss.detach(),
                totutils=utils.detach(), completeness=torch.as_tensor(comp), n_prime=n_prime.detach(),
                fiber_time=torch.as_tensor(fibers), time2=time2.detach(), variance=variance.detach(),
                g_time=time.grad.clone(), nfields=train.NFIELDS, total_time=train.TOTAL_TIME, wutils=train.wutils,
                wvar=train.wvar)


def main():
    train = load_reference_train()
    for dtype, tag in ((torch.float64, "f64"), (torch.float32, "f32")):
        cases = [run_case(train, S, T, seed, dtype, spread)
                 for S, T, seed, spread in ((50, 12, 1, 6.0), (2000, 12, 2, 7.0), (64, 16, 3, 40.0), (37, 4, 4, 3.0))]
        out = os.path.join(OUT_DIR, "loss_cases_%s.pt" % tag)
        torch.save(cases, out)
        print("wrote %d cases to %s (%.1f KB)" % (len(cases), out, os.path.getsize(out) / 1e3))


if __name__ == "__main__":
    main()
