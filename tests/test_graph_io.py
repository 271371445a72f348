"""On-disk graph formats (SURVEY.md section 8f row N3): the generator emits the canonical dense order, graph files
round-trip, the host-side CSR/CSC arrays are consistent, a crafted graph file runs no code."""
import torch

from pfs_neural_net_b200 import graph_io as gio


def test_generator_is_canonical_and_round_trips(tmp_path):
    info = torch.tensor([[1.5, 100.0], [2.0, 250.0], [0.5, 40.0]])
    g = gio.make_graph(info, nfibers=7, fdim=4)
    assert gio.is_canonical(g.edge_index, 3)
    assert g.x_t.shape == (3, 4) and g.x_s.shape == (7, 4) and g.x_e.shape == (21, 4) and g.x_u.shape == (1, 4)
    p = gio.save_graph(str(tmp_path / "g.pt"), g)
    h = gio.load_graph(p)
    for k in ("edge_index", "x_s", "x_t", "x_e", "x_u"):
        assert torch.equal(getattr(g, k), getattr(h, k)), k


def test_host_csr_csc_arrays(tmp_path):
    gen = torch.Generator().manual_seed(0)
    S, T = 9, 5
    keep = torch.rand(S * T, generator=gen) < 0.5
    e = torch.nonzero(keep).flatten()
    e = e[torch.randperm(e.numel(), generator=gen)]
    ei = torch.stack([e // T, e % T])
    a = gio.csr_arrays(ei, S, T)
    E = ei.shape[1]
    # CSR: positions of fibre k are rowptr[k]..rowptr[k+1], in original edge order (stable)
    for k in range(S):
        seg = a["csr_eid"][a["csr_rowptr"][k]:a["csr_rowptr"][k + 1]].long()
        assert (ei[0][seg] == k).all() and (seg[1:] > seg[:-1]).all()
    assert torch.equal(a["csr_src"].long(), ei[0][a["csr_eid"].long()]) and torch.equal(a["csr_tgt"].long(), ei[1][a["csr_eid"].long()])
    # CSC: class-sorted CSR positions
    for c in range(T):
        q = a["csc_q"][a["csc_colptr"][c]:a["csc_colptr"][c + 1]].long()
        assert (a["csr_tgt"][q] == c).all()
    assert int(a["csr_rowptr"][-1]) == E and int(a["csc_colptr"][-1]) == E
    g = gio.make_graph(torch.rand(T, 2), S, 4)
    g.edge_index, g.x_e = ei, torch.zeros(E, 4)
    d = torch.load(gio.save_graph(str(tmp_path / "s.pt"), g))
    assert not bool(d["canonical"]) and "csr_rowptr" in d and d["format"] == gio.FORMAT


def test_crafted_graph_file_executes_nothing(tmp_path):
    """A pickle may name any importable callable; the loader maps everything outside its allow-list (tensor rebuild
    helpers, plain containers) to an inert attribute bag, so a crafted graph file runs no code (ADVICE round 1)."""
    marker = tmp_path / "pwned"

    class Evil:
        def __reduce__(self):
            import os as _os
            return (_os.system, ("touch %s" % marker,))

    g = gio.make_graph(torch.rand(3, 2), 4, 4)
    payload = {"edge_index": g.edge_index, "x_s": g.x_s, "x_t": g.x_t, "x_e": g.x_e, "x_u": g.x_u, "extra": Evil()}
    p = str(tmp_path / "evil.pt")
    torch.save(payload, p)
    h = gio.load_graph(p)                       # loads the tensors ...
    assert torch.equal(h.edge_index, g.edge_index)
    assert not marker.exists()                  # ... and never called os.system
