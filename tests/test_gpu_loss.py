"""GPU parity of the training-loss kernels (reference src/train.py:21-80; SURVEY.md 8f row N1) against the golden
vectors of the unmodified reference and against the fp64 oracle: loss terms to rtol 1e-4 (fp32), gradient w.r.t. the
edge times norm-wise 1e-4, bit-reproducible run to run."""
import pytest
import torch

from oracle import block_oracle as bo
from oracle import loss_oracle as lo
from tests.util import golden_loss_cases

pytestmark = pytest.mark.gpu


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _cases():
    return [c for c in golden_loss_cases() if c["time"].dtype == torch.float64]


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


@pytest.mark.parametrize("idx", range(4))
def test_loss_matches_reference_golden(idx):
    from pfs_neural_net_b200 import loss as pl
    dev = _dev()
    c = _cases()[idx]
    S, T = c["S"], c["T"]
    time = c["time"].float().to(dev).requires_grad_(True)
    out = pl.loss_from_times(time, c["class_info"].float().to(dev), S, T, nfields=c["nfields"], total_time=c["total_time"],
                             wutils=c["wutils"], wvar=c["wvar"], noise=c["noise"].float().to(dev))
    loss, sc, n_prime, fibre_time, time2 = out
    loss.backward()
    torch.cuda.synchronize()
    # the same fp32-rounded inputs through the fp64 oracle (the golden file pins the oracle to the reference)
    t64 = c["time"].float().double().requires_grad_(True)
    r = lo.loss_terms(t64, c["noise"].float().double(), c["class_info"].float().double(), bo.complete_bipartite(S, T), S, T,
                      nfields=c["nfields"], total_time=c["total_time"], wutils=c["wutils"], wvar=c["wvar"])
    r["loss"].backward()
    assert _rel(sc[1], r["totutils"]) < 1e-4
    assert _rel(n_prime, r["n_prime"]) < 1e-4
    assert _rel(fibre_time, r["fiber_time"]) < 1e-4
    assert _rel(time2, r["time"]) < 1e-4
    assert _rel(sc[4], r["variance"]) < 1e-4
    assert _rel(sc[2], r["class_penalty"]) < 1e-4 or r["class_penalty"].abs().item() < 1e-6
    assert _rel(sc[3], r["fiber_penalty"]) < 1e-4
    # the loss is a difference of large terms: judge it on the scale of its largest term
    scale = max(abs(r["loss"].item()), c["wutils"] * abs(r["totutils"].item()), r["fiber_penalty"].item(), r["variance"].item())
    assert abs(loss.item() - r["loss"].item()) < 1e-4 * scale
    assert _rel(time.grad, t64.grad) < 1e-4
    # and directly against the reference's own fp64 numbers
    assert abs(loss.item() - c["loss"].item()) < 2e-4 * scale
    assert _rel(time.grad, c["g_time"]) < 2e-4
    # deterministic
    t2 = c["time"].float().to(dev).requires_grad_(True)
    l2 = pl.loss_from_times(t2, c["class_info"].float().to(dev), S, T, nfields=c["nfields"], total_time=c["total_time"],
                            wutils=c["wutils"], wvar=c["wvar"], noise=c["noise"].float().to(dev))[0]
    l2.backward()
    assert torch.equal(l2, loss) and torch.equal(t2.grad, time.grad)


def test_loss_function_drop_in_through_the_model():
    """`loss_function(gnn, graph, class_info)` end to end (GNN forward, time head, loss, backward into the weights),
    with the noise drawn like the reference draws it."""
    from pfs_neural_net_b200 import gnn as pg, loss as pl
    dev = _dev()
    S, T, F = 64, 12, 10
    torch.manual_seed(0)
    model = pg.GNN(B=1, Fdim=F, T=T, F_s=1, F_t=2).to(dev).train()
    g = torch.Generator().manual_seed(1)
    class_info = torch.stack([0.5 + 3 * torch.rand(T, generator=g), 50 + 400 * torch.rand(T, generator=g)], 1).to(dev)
    ei = bo.complete_bipartite(S, T).to(dev)
    graph = pg.BipartiteData(ei, torch.arange(S, dtype=torch.float32).reshape(-1, 1), class_info.cpu(),
                             2 + 8 * torch.rand(S * T, F, generator=g), torch.zeros(1, F))
    out = model(graph)
    torch.manual_seed(5)
    loss, utils = pl.loss_function(model, out, class_info)
    torch.manual_seed(5)
    noise = torch.rand(S * T, device=dev)
    loss2, _ = pl.loss_function(model, out, class_info, noise=noise)
    assert torch.equal(loss, loss2)                      # the generator is consumed exactly like rand_like(time)
    loss.backward()
    assert model.decoder_e[0].weight.grad is not None and torch.isfinite(model.decoder_e[0].weight.grad).all()
    assert model.mpb[0].edge_model[0].weight.grad.abs().max().item() > 0
    full = pl.loss_function(model, model(graph), class_info, finaloutput=True)
    assert len(full) == 7 and full[2].shape == (T,) and full[4].shape == (S,)
    with pytest.raises(Exception):
        pl.loss_from_times(torch.zeros(S * T), class_info.cpu(), S, T)      # CPU tensors: no fallback
