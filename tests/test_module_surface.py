"""The drop-in boundary (SURVEY.md section 8b): same module tree, state_dict keys, shapes and registration
order as the reference's src/gnn.py, checked against the shipped checkpoint's weights (golden fixture)."""
import pytest
import torch

from oracle import block_oracle as bo
from pfs_neural_net_b200 import gnn


def test_shipped_checkpoint_loads_strict(golden_gnn_case):
    model = gnn.GNN(Fdim=10, B=3, F_s=1, F_t=2, T=12)
    state = golden_gnn_case["state"]
    assert model.load_state_dict(state, strict=True).missing_keys == []
    assert list(model.state_dict().keys()) == list(state.keys())          # same order: Adam state is index-keyed
    assert len(list(model.parameters())) == 109
    assert sum(p.numel() for p in model.parameters()) == 55233
    for k, v in model.state_dict().items():
        assert v.shape == state[k].shape and v.dtype == state[k].dtype, k


def test_block_state_dict_matches_reference_layout():
    blk = gnn.Block(10)
    expect = bo.block_param_shapes(10)
    assert [k for k, _ in expect] == list(blk.state_dict().keys())
    for k, shape in expect:
        assert tuple(blk.state_dict()[k].shape) == tuple(shape), k


def test_unnormed_block_has_no_norm_entries():
    blk = gnn.Block(10, normed=False)
    assert not any("norm" in k for k in blk.state_dict())
    assert gnn.Block(10, s_model=False, u_model=False).state_dict().keys() == {
        k for k in gnn.Block(10).state_dict() if k.startswith(("edge_model", "t_model"))}


def test_no_cpu_fallback():
    blk = gnn.Block(10)
    ei = bo.complete_bipartite(5, 3)
    with pytest.raises(RuntimeError, match="CUDA"):
        blk((ei, torch.randn(5, 10), torch.randn(3, 10), torch.randn(15, 10), torch.randn(1, 10)))
    model = gnn.GNN(Fdim=10, B=1)
    with pytest.raises(RuntimeError, match="CUDA"):
        model.edge_prediction(torch.randn(15, 10))


def test_round_is_the_identity_like_the_reference():
    model = gnn.GNN(Fdim=10, B=1)
    x = torch.tensor([0.4, 1.6])
    assert torch.equal(model.eval().round(x), x) and torch.equal(model.train().round(x), x)


def test_bipartite_data_bag():
    g = gnn.BipartiteData(bo.complete_bipartite(4, 3), torch.zeros(4, 2), torch.zeros(3, 2), torch.zeros(12, 2),
                          torch.zeros(1, 2))
    assert g.num_nodes == 3
    inc = g.__inc__("edge_index", g.edge_index)
    assert inc.flatten().tolist() == [4, 3]
    assert g.__inc__("x_s", g.x_s) == 0
