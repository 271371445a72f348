"""Topology cache: turns the reference's `edge_index` [2, E] int64 (src/gnn.py:98,135,187) into what
the kernels consume.

  * canonical dense order (reference src/train.py:94, e = k*T + i) is DETECTED on the device, never
    assumed -- `graphs/graph-0.pt` is fibre-major but class-permuted (SURVEY.md section 0.10);
  * anything else gets int32 CSR (fibre-sorted) and CSC (class-sorted) arrays plus a tile table
    from `pfs_build_topology`, built once per `edge_index` and cached here;
  * when a fibre has more than PFS_TILE_EDGES edges, the fp32 kernels take the split tile table of
    `pfs_build_split_tiles` instead (built on first use by `struct()`; the bf16 wide path never asks).
"""
import collections
import ctypes as ct

import torch

from . import _abi


class Topology:
    def __init__(self, edge_index, num_src, num_tgt):
        if not edge_index.is_cuda:
            raise _abi.PfsError("pfs_b200 needs CUDA tensors: edge_index is on %s (no CPU fallback)" % edge_index.device)
        if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.shape[0] != 2:
            raise ValueError("edge_index must be an int64 tensor of shape [2, E]")
        lib = _abi.load_library()
        self.edge_index = edge_index.contiguous()
        self.device = edge_index.device
        self.S, self.T, self.E = int(num_src), int(num_tgt), int(edge_index.shape[1])
        if self.E == 0:
            raise ValueError("graph has no edges")
        stream = torch.cuda.current_stream(self.device).cuda_stream
        flag = torch.zeros(1, dtype=torch.int32, device=self.device)
        _abi.check(lib.pfs_detect_dense(self.edge_index.data_ptr(), self.E, self.S, self.T, flag.data_ptr(), stream),
                   "pfs_detect_dense")
        self.canonical = bool(flag.item())            # e = k*T + i (reference src/train.py:94)
        self.dense = self.canonical and self.T <= _abi.PFS_TILE_EDGES   # what the narrow fp32 kernels call dense
        self.arrays = None
        self.ntiles = 0
        self.max_degree = self.T if self.canonical else None
        self._wide = None
        self._split = None
        self._workspaces = {}

    def csr(self):
        """int32 CSR / CSC arrays of pfs_build_topology, built on first use and cached."""
        if self.arrays is None:
            lib = _abi.load_library()
            self._build_csr(lib, torch.cuda.current_stream(self.device).cuda_stream)
        return self.arrays

    def wide(self):
        """Segments / index arrays for the wide (bf16, tensor-core) path."""
        if self._wide is None:
            from .wide import WideTopology
            self._wide = WideTopology(self)
        return self._wide

    def _build_csr(self, lib, stream):
        lo = int(self.edge_index.min().item())
        hi_s = int(self.edge_index[0].max().item())
        hi_t = int(self.edge_index[1].max().item())
        if lo < 0 or hi_s >= self.S or hi_t >= self.T:
            raise IndexError("edge_index out of range for %d fibres x %d classes" % (self.S, self.T))
        i32 = dict(dtype=torch.int32, device=self.device)
        a = {
            "csr_rowptr": torch.empty(self.S + 1, **i32), "csr_eid": torch.empty(self.E, **i32),
            "csr_src": torch.empty(self.E, **i32), "csr_tgt": torch.empty(self.E, **i32),
            "csc_colptr": torch.empty(self.T + 1, **i32), "csc_q": torch.empty(self.E, **i32),
            "tile_fibre": torch.empty(self.S + 2, **i32),
        }
        scalars = torch.zeros(2, **i32)
        tmp_bytes = lib.pfs_build_topology_temp_bytes(self.E, self.S, self.T)
        tmp = torch.empty(tmp_bytes, dtype=torch.uint8, device=self.device)
        _abi.check(lib.pfs_build_topology(
            self.edge_index.data_ptr(), self.E, self.S, self.T, a["csr_rowptr"].data_ptr(), a["csr_eid"].data_ptr(),
            a["csr_src"].data_ptr(), a["csr_tgt"].data_ptr(), a["csc_colptr"].data_ptr(), a["csc_q"].data_ptr(),
            a["tile_fibre"].data_ptr(), scalars[0:1].data_ptr(), scalars[1:2].data_ptr(), tmp.data_ptr(), tmp_bytes,
            stream), "pfs_build_topology")
        self.ntiles, self.max_degree = (int(v) for v in scalars.tolist())
        self.arrays = a

    def split_tiles(self):
        """Tile table of pfs_build_split_tiles (fibres of more than PFS_TILE_EDGES edges cut into chunks), built
        on first use and cached: {"tile_fibre", "tile_q", "tile_slot", "split_fibre", "split_ptr"} (int32,
        trimmed to their lengths) and the counts "ntiles", "nsplit", "nslots"."""
        if self._split is None:
            a = self.csr()
            lib = _abi.load_library()
            cap = self.S + self.E // _abi.PFS_TILE_EDGES + 2
            i32 = dict(dtype=torch.int32, device=self.device)
            b = {"tile_fibre": torch.empty(cap, **i32), "tile_q": torch.empty(cap, **i32),
                 "tile_slot": torch.empty(cap, **i32), "split_fibre": torch.empty(self.S, **i32),
                 "split_ptr": torch.empty(self.S + 1, **i32)}
            counts = torch.zeros(3, **i32)
            _abi.check(lib.pfs_build_split_tiles(
                a["csr_rowptr"].data_ptr(), self.S, b["tile_fibre"].data_ptr(), b["tile_q"].data_ptr(),
                b["tile_slot"].data_ptr(), b["split_fibre"].data_ptr(), b["split_ptr"].data_ptr(), counts.data_ptr(),
                torch.cuda.current_stream(self.device).cuda_stream), "pfs_build_split_tiles")
            nt, ns, nslots = (int(v) for v in counts.tolist())
            for k, n in (("tile_fibre", nt + 1), ("tile_q", nt + 1), ("tile_slot", nt), ("split_fibre", ns),
                         ("split_ptr", ns + 1)):
                b[k] = b[k][:n]
            b.update(ntiles=nt, nsplit=ns, nslots=nslots)
            self._split = b
        return self._split

    def struct(self, G, F):
        t = _abi.TopologyStruct()
        t.layout = _abi.PFS_LAYOUT_DENSE if self.dense else _abi.PFS_LAYOUT_CSR
        t.G, t.F, t.S, t.T, t.E = int(G), int(F), self.S, self.T, self.E
        if not self.dense:
            a = self.csr()
            t.csr_rowptr, t.csr_eid = a["csr_rowptr"].data_ptr(), a["csr_eid"].data_ptr()
            t.csr_src, t.csr_tgt = a["csr_src"].data_ptr(), a["csr_tgt"].data_ptr()
            t.tile_fibre, t.ntiles = a["tile_fibre"].data_ptr(), self.ntiles
            t.csc_colptr, t.csc_q = a["csc_colptr"].data_ptr(), a["csc_q"].data_ptr()
            if self.max_degree > _abi.PFS_TILE_EDGES:
                b = self.split_tiles()
                t.tile_fibre, t.ntiles = b["tile_fibre"].data_ptr(), b["ntiles"]
                t.tile_q, t.tile_slot = b["tile_q"].data_ptr(), b["tile_slot"].data_ptr()
                t.split_fibre, t.split_ptr = b["split_fibre"].data_ptr(), b["split_ptr"].data_ptr()
                t.nsplit, t.nslots = b["nsplit"], b["nslots"]
        return t

    def workspace(self, G, F):
        """One scratch buffer per (G, F), shared by every module call on this topology (calls are
        stream-ordered, so the forward/backward kernels never overlap on it)."""
        key = (int(G), int(F))
        ws = self._workspaces.get(key)
        if ws is None:
            t = self.struct(G, F)
            nbytes = _abi.load_library().pfs_workspace_bytes(ct.byref(t))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            self._workspaces[key] = ws
        return ws


_CACHE = collections.OrderedDict()
_CACHE_MAX = 16


def get_topology(edge_index, num_src, num_tgt):
    """Cached Topology for this `edge_index` tensor (keyed on storage, version counter and sizes; the
    entry keeps the tensor alive so the address cannot be recycled under a stale key)."""
    key = (edge_index.data_ptr(), edge_index._version, tuple(edge_index.shape), int(num_src), int(num_tgt),
           str(edge_index.device))
    topo = _CACHE.get(key)
    if topo is None:
        topo = Topology(edge_index, num_src, num_tgt)
        topo._key_tensor = edge_index
        _CACHE[key] = topo
        while len(_CACHE) > _CACHE_MAX:
            _CACHE.popitem(last=False)
    else:
        _CACHE.move_to_end(key)
    return topo


def clear_cache():
    _CACHE.clear()
