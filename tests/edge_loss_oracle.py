"""TEST INFRASTRUCTURE ONLY -- fp64 statement of the training loss on a general edge list (DESIGN.md section 8b).

Built from the reference restatement in oracle/loss_oracle.py (its `softfloor`, and `segment_sum` of
oracle/block_oracle.py); `loss_terms` there stays pinned to the unmodified reference, and
tests/test_edge_list_loss_oracle.py checks that `loss_terms_edges` equals it on the complete graph in any order.
"""
import torch

from oracle.block_oracle import segment_sum
from oracle.loss_oracle import softfloor


def loss_terms_edges(time, noise, class_info, edge_index, nfibers, nclasses, nfields=10, total_time=42, wutils=2000.0,
                     wvar=1.0, pclass=0.1, pfiber=1.0, sharpness=0.5):
    """The loss on any edge list: `time` and `noise` [E] in the order of `edge_index` [2, E], edge e = (fibre src[e],
    class tgt[e]), duplicates and fibres or classes without edges allowed.  As oracle.loss_oracle.loss_terms, with
    T_i = hours[tgt[e]], and the variance over the fibre x class matrix of cells c_ki = sum of time2 over the edges
    (k, i), 0 where there is none: the reference's var(time2.reshape(S, T), dim=0) of the matrix the edge list
    describes.  On the canonical complete graph this is `loss_terms`; on a permutation of it, `loss_terms` of the
    un-permuted graph.  Returns the keys of `loss_terms` ("time" is time2 in edge order) and "cells" [S, T]."""
    src, tgt = edge_index[0], edge_index[1]
    T_i = class_info[:, 0][tgt]
    N_i = class_info[:, 1] / nfields
    galaxies = softfloor(time / T_i, noise, sharpness)
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
    cells = segment_sum(time2, src * nclasses + tgt, nfibers * nclasses).reshape(nfibers, nclasses)
    variance = torch.sum(torch.var(cells, dim=0))
    loss = -wutils * totutils + fiber_penalty + class_penalty - wvar * variance
    return dict(loss=loss, totutils=totutils, completeness=completeness, n_prime=n_prime, fiber_time=fiber_time,
                time=time2, variance=variance, class_penalty=class_penalty, fiber_penalty=fiber_penalty, cells=cells)
