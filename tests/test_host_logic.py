"""Host-side bookkeeping of the Block-level fusions (functional.XeGradBus), on CPU tensors: no library call involved."""
import torch

from pfs_neural_net_b200 import functional as pf


def test_grad_bus_fuses_each_part_once_in_any_order():
    like = torch.zeros(2, 6, 4)
    bus = pf.XeGradBus()
    assert bus.addend_for_target(like) is None and bus.addend_for_source(like) is None      # nothing there yet
    bus.g_o = torch.ones(2, 6, 4)
    a = bus.addend_for_target(like)                      # TModel runs after the output tap: takes the output gradient
    assert a is not None and torch.equal(a, bus.g_o) and bus.o_used
    assert bus.addend_for_target(like) is None           # ... once
    bus.g_t = torch.full((2, 6, 4), 2.0)
    b = bus.addend_for_source(like)                      # SModel takes what TModel stored (which already holds g_o)
    assert b is bus.g_t and bus.t_used
    # SModel before TModel (TModel's output unused): it takes the output gradient itself
    bus.clear()
    bus.g_o = torch.ones(2, 6, 4)
    c = bus.addend_for_source(like)
    assert c is not None and bus.o_used and not bus.t_used
    # a gradient of another shape / dtype is left to autograd
    bus.clear()
    bus.g_o = torch.ones(2, 6, 4, dtype=torch.float64)
    assert bus.addend_for_target(like) is None and not bus.o_used


def test_fanout_adds_only_what_the_kernels_did_not_fuse():
    x = torch.randn(2, 3, 4, requires_grad=True)
    bus = pf.XeGradBus()
    a, b, c = pf.XeFanout.apply(x, bus)
    ga, gb, gc = torch.ones_like(x), 2 * torch.ones_like(x), 4 * torch.ones_like(x)
    bus.t_used = True                                    # the TModel part was fused into the SModel store (= ga here)
    torch.autograd.backward([a, b, c], [ga, gb, gc])
    assert torch.equal(x.grad, ga + gc)                  # gb not added again, gc (not fused) added
    assert not bus.t_used and not bus.o_used             # cleared for the next step
