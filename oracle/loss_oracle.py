"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference training loss (SURVEY.md section 8f, row N1).

Restates `softfloor` (/root/reference/src/train.py:21-27) and `loss_function` (src/train.py:29-80) as
pure functions of the edge times (the output of `GNN.edge_prediction`, src/train.py:42), the uniform
noise the reference draws with `torch.rand_like` (src/train.py:22) and the class table; the constants
of src/config.py:16-28 are arguments.  Any floating dtype; gradients by autograd, like the reference.
Only tests/ may import it.  PARITY PIN: tests/golden/loss_cases_f64.pt / loss_cases_f32.pt, produced by oracle/make_golden_loss.py
from the UNMODIFIED reference functions (tests/test_oracle_golden.py::test_loss_oracle_matches_reference).
"""
import math

import torch

from .block_oracle import segment_sum

NOISELEVEL = 0.3      # softfloor default, reference src/train.py:21


def softfloor(x, noise, sharpness=20, noiselevel=NOISELEVEL):
    """reference src/train.py:21-27 with the uniform draw `noise` in [0, 1) made explicit."""
    x = x + noiselevel * (noise - 0.5)
    r = 0.0 if sharpness == 0 else math.exp(-1.0 / sharpness)
    two_pi_x = 2 * math.pi * x
    return x + 1 / math.pi * (torch.arctan(r * torch.sin(two_pi_x) / (1 - r * torch.cos(two_pi_x)))
                              - math.atan(r / (1.0 - r)))


def loss_terms(time, noise, class_info, edge_index, nfibers, nclasses, nfields=10, total_time=42, wutils=2000.0,
               wvar=1.0, pclass=0.1, pfiber=1.0, sharpness=0.5):
    """reference src/train.py:29-80 from `time = gnn.edge_prediction(...).squeeze(-1)` on; returns a dict with the
    loss, the utility and the diagnostics of `finaloutput=True`."""
    src, tgt = edge_index[0], edge_index[1]
    T_i = class_info[:, 0].unsqueeze(0).expand(nfibers, -1).reshape(-1)
    N_i = class_info[:, 1] / nfields
    visited = time / T_i
    galaxies = softfloor(visited, noise, sharpness)
    galaxies = torch.maximum(torch.zeros_like(galaxies), galaxies)
    n_prime = segment_sum(galaxies, tgt, nclasses)
    time2 = galaxies * T_i
    completeness = n_prime / N_i
    totutils = torch.min(completeness)
    class_over = torch.relu(n_prime - N_i)
    class_penalty = pclass * torch.sum(class_over ** 2)
    fiber_time = segment_sum(time2, src, nfibers)
    overtime = fiber_time - total_time
    fiber_penalty = pfiber * torch.sum(torch.nn.functional.leaky_relu(overtime, 0.1) ** 2)
    variance = torch.sum(torch.var(time2.reshape(nfibers, nclasses), dim=0))
    loss = -wutils * totutils + fiber_penalty + class_penalty - wvar * variance
    return dict(loss=loss, totutils=totutils, completeness=completeness, n_prime=n_prime, fiber_time=fiber_time,
                time=time2, variance=variance, class_penalty=class_penalty, fiber_penalty=fiber_penalty)
