"""Graph store: V/E loader + device-resident CSR with a degree-binned row schedule.

Drop-in for ``clane.graph`` of the reference (/root/reference/clane/graph.py): same
constructor, attributes and methods (``Graph(data_root, embedding_dim)``, ``.d .vertex_ids
.X .V .E .dispense_pair``, ``len(g)``, ``g[idx]``, ``.A``, ``.get_nbrs``, ``.build_P``,
``.Z``, ``.set_Z``), but the adjacency is coalesced ONCE into a CSR (graph.py:104-110 does it
on every access) and everything the iterative update touches lives in HBM:

    rowptr int32[N+1] | col int32[E] | erow int32[E] | w fp32[E]
    X fp32[N, ld] | Z fp32[3][N, ld]   (ld = d rounded up to 4 floats: 16-byte aligned rows; three rotating buffers)
    (float64 features: w, X and Z are fp64 with ld = d rounded up to 2, and the update runs in double, DESIGN.md 7b)
    clane_plan: the degree-sorted row-block schedule (hub groups / row groups, sinks dropped)

All arithmetic is done by libclane_b200.so through the C-ABI (clane_b200/_lib.py); torch
only owns the device memory.  There is no CPU fallback: ``build_P`` and the Embedder raise
without a CUDA device.
"""
from __future__ import annotations

import ctypes
import os
import random
from pathlib import Path

import numpy as np
import torch
from torch.utils.data import Dataset

from . import _lib
from .similarity import AsymmertricSimilarity

HUB_THRESHOLD = 0      # 0 = library default: rows longer than (edges of the plan / 4096), clamped to [256, 16384]


class Vertex(object):
    """Per-node record (graph.py:9-21).  ``x`` / ``z`` are row views resolved on access."""

    def __init__(self, graph: "Graph", idx: int) -> None:
        self._graph = graph
        self.idx = idx
        self.id_ = graph.vertex_ids[idx]

    @property
    def x(self) -> torch.Tensor:
        return self._graph.X[self.idx]

    @property
    def z(self) -> torch.Tensor:
        return self._graph._row_of_Z(self.idx)

    @z.setter
    def z(self, value) -> None:
        # the reference assigns rows in place (`v.z = ...`, embedder.py:92, graph.py:138)
        self._graph._set_row_of_Z(self.idx, value)

    @property
    def outgoing_indices(self):
        g = self._graph
        return g._raw_dst[g._raw_src == self.idx].tolist()

    @property
    def incoming_indices(self):
        g = self._graph
        return g._raw_src[g._raw_dst == self.idx].tolist()


class Edge(object):
    """(src, dst) pair of Vertex records (graph.py:24-30)."""

    def __init__(self, src: Vertex, dst: Vertex) -> None:
        self.src, self.dst = src, dst


class _LazySeq(object):
    """Sequence that materialises its items on access (N + E_raw Python objects are not
    affordable at 62M edges; the reference builds them eagerly, graph.py:61-89)."""

    def __init__(self, n, make):
        self._n, self._make = n, make

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self._make(j) for j in range(*i.indices(self._n))]
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError(i)
        return self._make(i)

    def __iter__(self):
        return (self._make(i) for i in range(self._n))


def _parse_vertex_ids(path: Path):
    # graph.py:44-45 -- FileNotFoundError propagates
    with open(path, "r") as io:
        return io.read().strip().split("\n")


def _parse_edges(path: Path, vertex_ids):
    """graph.py:73-81: lines ``src_id<TAB>dst_id``; ids map to their FIRST position in V;
    a line without exactly one tab or with an unknown id raises ValueError.  Parsed natively
    (clane_edges_open: hash map over V, one file piece per host thread) -- the reference's
    ``vertex_ids.index`` loop is O(E*N)."""
    open(path, "r").close()                     # FileNotFoundError etc. exactly as the reference raises them
    L = _lib.lib()
    joined = "\n".join(vertex_ids).encode("utf-8")
    handle, e_raw, err_line = ctypes.c_void_p(), ctypes.c_int64(), ctypes.c_int64(-1)
    err = ctypes.create_string_buffer(512)
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    rc = L.clane_edges_open(joined, len(joined), len(vertex_ids), str(path).encode(), threads, ctypes.byref(handle),
                            ctypes.byref(e_raw), ctypes.byref(err_line), err, len(err))
    if rc == -6:                                # CLANE_EPARSE: the reference's tuple-unpacking error
        raise ValueError(err.value.decode("utf-8", "replace"))
    if rc == -7:                                # CLANE_EUNKNOWNID: list.index's error
        raise ValueError(f"{err.value.decode('utf-8', 'replace')!r} is not in list")
    _lib.check(rc, "clane_edges_open")
    try:
        src = np.empty(e_raw.value, np.int64)
        dst = np.empty(e_raw.value, np.int64)
        _lib.check(L.clane_edges_read(handle, src.ctypes.data, dst.ctypes.data), "clane_edges_read")
    finally:
        L.clane_edges_close(handle)
    return src, dst


class Graph(Dataset):
    def __init__(self, data_root: Path, embedding_dim: int = 128) -> None:
        super(Graph, self).__init__()
        self.d = embedding_dim
        data_root = Path(data_root)
        self.vertex_ids = _parse_vertex_ids(data_root.joinpath("V"))

        # content embeddings C (graph.py:49-59): C.npy (dtype preserved), C.pt, else N(0,1)
        # drawn from the global CPU generator with the reference's exact call.
        try:
            self.X = torch.from_numpy(np.load(data_root.joinpath("C.npy")))
        except FileNotFoundError:
            try:
                self.X = torch.load(data_root.joinpath("C.pt"))
            except FileNotFoundError:
                self.X = torch.normal(0, 1, [len(self.vertex_ids), self.d])

        src, dst = _parse_edges(data_root.joinpath("E"), self.vertex_ids)
        self._init_from_arrays(src, dst)

    # -- construction -----------------------------------------------------------------------
    @classmethod
    def from_arrays(cls, n: int, src, dst, X, vertex_ids=None) -> "Graph":
        """Build from index arrays (synthetic benchmarks; skips the text files)."""
        g = cls.__new__(cls)
        Dataset.__init__(g)
        g.vertex_ids = vertex_ids if vertex_ids is not None else _LazySeq(n, str)
        g.X = torch.as_tensor(X)
        g.d = int(g.X.shape[1])
        g._init_from_arrays(np.ascontiguousarray(src, np.int64), np.ascontiguousarray(dst, np.int64))
        return g

    def _init_from_arrays(self, src: np.ndarray, dst: np.ndarray) -> None:
        n = len(self.vertex_ids)
        if self.X.dim() != 2 or self.X.shape[0] != n:
            raise ValueError(f"content embeddings have shape {tuple(self.X.shape)}, expected [{n}, d]")
        self._n = n
        self._raw_src, self._raw_dst = src, dst
        self.V = _LazySeq(n, lambda i: Vertex(self, i))
        self.E = _LazySeq(len(src), lambda k: Edge(Vertex(self, int(src[k])), Vertex(self, int(dst[k]))))
        self.dispense_pair = False

        # coalesced CSR, once (replaces the per-access rebuild of graph.py:104-110)
        L = _lib.lib()
        rowptr = np.zeros(n + 1, np.int32)
        col = np.zeros(max(len(src), 1), np.int32)
        e = L.clane_csr_from_edges(src.ctypes.data, dst.ctypes.data, len(src), n, rowptr.ctypes.data, col.ctypes.data)
        if e < 0:
            _lib.check(int(e), "clane_csr_from_edges")
        self._rowptr, self._col = rowptr, col[:e].copy()
        self._nnz = int(e)
        self._Z_host = self.X      # z aliases x until the first update (graph.py:18-19)
        self._dev = None

    # -- Dataset protocol (graph.py:93-102) -------------------------------------------------
    def __len__(self):
        return self._n

    def __getitem__(self, idx):
        if self.dispense_pair:
            randomly_chosen_idx = random.randint(0, len(self) - 1)
            a, b = self._rowptr[idx], self._rowptr[idx + 1]
            is_neighbor = bool(np.any(self._col[a:b] == randomly_chosen_idx))
            return (idx, random.randint(0, len(self) - 1), is_neighbor)
        return idx

    # -- adjacency --------------------------------------------------------------------------
    def _coo_indices(self) -> torch.Tensor:
        rows = np.repeat(np.arange(self._n, dtype=np.int64), np.diff(self._rowptr))
        return torch.from_numpy(np.stack([rows, self._col.astype(np.int64)]))

    @property
    def A(self) -> torch.Tensor:
        """Coalesced COO adjacency (graph.py:104-110); values count merged duplicates."""
        vals = torch.ones(len(self._raw_src))
        idx = torch.from_numpy(np.stack([self._raw_src, self._raw_dst])) if len(self._raw_src) else \
            torch.zeros([2, 0], dtype=torch.long)
        return torch.sparse_coo_tensor(indices=idx, values=vals, size=(self._n, self._n)).coalesce()

    def get_nbrs(self, idx: int) -> torch.LongTensor:
        """Out-neighbour positions of vertex idx, ascending, 1-D int64 (graph.py:112-116)."""
        a, b = self._rowptr[idx], self._rowptr[idx + 1]
        return torch.from_numpy(self._col[a:b].astype(np.int64))

    # -- device residency -------------------------------------------------------------------
    def _device_state(self):
        if self._dev is None:
            dev = _lib.require_cuda()
            if self.X.dtype not in (torch.float32, torch.float64):
                raise NotImplementedError(
                    f"clane_b200 computes in fp32 or fp64; content embeddings are {self.X.dtype} "
                    "(the reference would run its whole update in that dtype, graph.py:51)")
            L = _lib.lib()
            n, e, d = self._n, self._nnz, int(self.X.shape[1])
            S = type("DeviceState", (), {})()
            S.dtype = self.X.dtype
            f64 = S.dtype == torch.float64
            ld = int(L.clane_padded_ld_f64(d) if f64 else L.clane_padded_ld(d))
            S.device, S.n, S.e, S.d, S.ld = dev, n, e, d, ld
            S.rowptr = torch.from_numpy(self._rowptr).to(dev)
            S.col = torch.from_numpy(self._col if e else np.zeros(1, np.int32)).to(dev)
            S.erow = torch.zeros(max(e, 1), dtype=torch.int32, device=dev)
            # fp64 runs without a plan: its kernels take plain sizes and the reduction scratch S.work
            S.plan = None if f64 else _lib.Plan(n, e, d, self._rowptr, 0, n, HUB_THRESHOLD)   # module attribute: tests lower it
            S.X = torch.zeros([max(n, 1), ld], dtype=S.dtype, device=dev)
            S.X[:n, :d] = self.X.to(dev)
            S.Z = [torch.zeros_like(S.X) for _ in range(3)]     # rotating: sweep t reads Z[(cur + t) % 3], writes the next
            S.Zptrs = (ctypes.c_void_p * 3)(*[z.data_ptr() for z in S.Z])
            S.cur = 0
            S.w = torch.zeros(max(e, 1), dtype=S.dtype, device=dev)
            S.norms2 = torch.zeros(2, dtype=S.dtype, device=dev)
            S.amount = torch.zeros(1, dtype=S.dtype, device=dev)
            if f64:
                S.state = torch.zeros(ctypes.sizeof(_lib.Patience64), dtype=torch.uint8, device=dev)
                S.state_host = torch.zeros(ctypes.sizeof(_lib.Patience64), dtype=torch.uint8).pin_memory()
                S.work = torch.zeros(int(L.clane_work_f64(max(n * d, e * d))), dtype=torch.float64, device=dev)
            else:
                S.state = torch.zeros(8, dtype=torch.int32, device=dev)          # struct clane_patience
                S.state_host = torch.zeros(8, dtype=torch.int32).pin_memory()
            S.log_cap = 1 << 16
            S.log = torch.zeros(S.log_cap, dtype=S.dtype, device=dev)
            S.stream = torch.cuda.Stream(device=dev)   # sweeps run here (a capturable stream: CUDA-graph replay)
            _lib.check(L.clane_edge_rows(S.rowptr.data_ptr(), n, e, S.erow.data_ptr(), _lib.stream_handle()),
                       "clane_edge_rows")
            self._dev = S
            self._upload_Z(self._Z_host)
        return self._dev

    def _upload_Z(self, Z: torch.Tensor) -> None:
        S = self._dev
        if tuple(Z.shape) != (S.n, S.d):
            raise ValueError(f"Z has shape {tuple(Z.shape)}, expected {(S.n, S.d)}")
        S.Z[0].zero_()
        S.Z[0][:S.n, :S.d] = Z.to(device=S.device, dtype=S.dtype)
        S.Z[1].copy_(S.Z[0])
        S.Z[2].copy_(S.Z[0])
        S.cur = 0

    @property
    def Z_device(self) -> torch.Tensor:
        """Current embeddings as a [N, d] view of the device buffer (no copy)."""
        S = self._device_state()
        return S.Z[S.cur][:S.n, :S.d]

    # -- embeddings -------------------------------------------------------------------------
    @property
    def Z(self) -> torch.Tensor:
        """Current embeddings [N, d] on the host (graph.py:130-134), materialised on demand."""
        if self._dev is None:
            return self._Z_host if self._Z_host is not self.X else self.X.clone()
        return self.Z_device.cpu()

    def _row_of_Z(self, idx: int) -> torch.Tensor:
        """One row of the current embeddings on the host (a 4*d-byte copy, not the whole matrix)."""
        if self._dev is None:
            return self._Z_host[idx].clone() if self._Z_host is self.X else self._Z_host[idx]
        S = self._dev
        return S.Z[S.cur][idx, :S.d].cpu()

    def _set_row_of_Z(self, idx: int, value) -> None:
        value = torch.as_tensor(value)
        if self._dev is None:
            if self._Z_host is self.X:          # z stops aliasing x at the first write (graph.py:18-19)
                self._Z_host = self.X.clone()
            self._Z_host[idx] = value.to(self._Z_host.dtype)
        else:
            S = self._dev
            row = value.to(device=S.device, dtype=S.dtype).reshape(S.d)
            for z in S.Z:                       # every buffer: rows without out-neighbours are never rewritten by a sweep
                z[idx, :S.d] = row

    def set_Z(self, Z: torch.Tensor) -> None:
        """Replace the embeddings (graph.py:136-138)."""
        Z = torch.as_tensor(Z)
        if self._dev is None:
            self._Z_host = Z.detach().cpu().clone()
        else:
            self._upload_Z(Z)

    # -- P ----------------------------------------------------------------------------------
    def _build_P_device(self, similarity) -> torch.Tensor:
        """Row-stochastic weights w[E] of the coalesced edges, on the device (graph.py:118-128)."""
        S = self._device_state()
        L = _lib.lib()
        Zc = S.Z[S.cur]
        stream = _lib.stream_handle()
        if S.dtype == torch.float64:
            return self._build_P_device_f64(similarity, S, L, Zc, stream)
        if getattr(similarity, "_clane_kernel", None) == "cosine":
            _lib.check(L.clane_build_p_cosine(S.plan.handle, Zc.data_ptr(), S.rowptr.data_ptr(), S.erow.data_ptr(),
                                              S.col.data_ptr(), S.w.data_ptr(), S.norms2.data_ptr(), stream),
                       "clane_build_p_cosine")
        elif (getattr(similarity, "_clane_kernel", None) == "asym" and S.e > 0
              and type(similarity).forward is AsymmertricSimilarity.forward):
            # trainable bilinear scorer: every node projected once on the tensor cores, then per-edge dots + row softmax.
            # A subclass that overrides forward is scored by its own forward (the generic path below).
            if getattr(S, "asym_work", None) is None:
                # P_src | P_dst, then the split of the stacked weights (the fp32 kernel's scratch)
                S.asym_work = torch.zeros(2 * S.n * S.ld + 4 * S.d * S.ld, dtype=torch.float32, device=S.device)
                S.asym_error = torch.zeros(1, dtype=torch.int32, device=S.device)
            S.asym_error.zero_()
            if L.clane_asym_supported(S.d):
                # d in {32, 64, 96, 128}: the TF32 kernel
                name = "clane_build_p_asym"
                W = similarity.stacked_weights(S.device)
                rc = L.clane_build_p_asym(S.plan.handle, Zc.data_ptr(), W.data_ptr(), S.rowptr.data_ptr(), S.erow.data_ptr(),
                                          S.col.data_ptr(), S.w.data_ptr(), S.asym_work.data_ptr(), S.asym_error.data_ptr(),
                                          stream)
            else:
                # every other width: the fp32-faithful 3xTF32 kernel, W padded to rows of ld floats
                name = "clane_build_p_asym_fp32"
                W = torch.zeros([2 * S.d, S.ld], dtype=torch.float32, device=S.device)
                W[:, :S.d] = similarity.stacked_weights(S.device)
                rc = L.clane_build_p_asym_fp32(S.plan.handle, Zc.data_ptr(), W.data_ptr(), S.ld, S.rowptr.data_ptr(),
                                               S.erow.data_ptr(), S.col.data_ptr(), S.w.data_ptr(), S.asym_work.data_ptr(),
                                               S.asym_error.data_ptr(), stream)
            _lib.check(rc, name)
            if int(S.asym_error.item()):          # synchronises: W must outlive the launch anyway
                raise _lib.ClaneError(f"{name}: the projection kernel timed out waiting for its TMA copies")
        else:
            # user plugin: honour its scores, still on the device; the softmax stays fused
            Zv = Zc[:S.n, :S.d]
            src_Z, dst_Z = Zv[S.erow[:S.e].long()], Zv[S.col[:S.e].long()]
            scores = similarity(src_Z, dst_Z).detach().to(device=S.device, dtype=torch.float32).reshape(-1).contiguous()
            if scores.numel() != S.e:
                raise ValueError(f"similarity returned {scores.numel()} scores for {S.e} edges")
            _lib.check(L.clane_row_softmax(scores.data_ptr(), 0, 0, S.n, S.rowptr.data_ptr(), S.w.data_ptr(), stream),
                       "clane_row_softmax")
        return S.w[:S.e]

    def _build_P_device_f64(self, similarity, S, L, Zc, stream) -> torch.Tensor:
        """build_P in double: cosine on the fused fp64 kernels; any other scorer (the trainable asymmetric one
        included, whose fp32 weights then raise torch's dtype error as upstream) scores in double as a plugin."""
        if getattr(similarity, "_clane_kernel", None) == "cosine":
            _lib.check(L.clane_build_p_cosine_f64(S.n, S.e, S.d, Zc.data_ptr(), S.rowptr.data_ptr(), S.erow.data_ptr(),
                                                  S.col.data_ptr(), S.w.data_ptr(), S.norms2.data_ptr(),
                                                  S.work.data_ptr(), stream), "clane_build_p_cosine_f64")
        else:
            Zv = Zc[:S.n, :S.d]
            src_Z, dst_Z = Zv[S.erow[:S.e].long()], Zv[S.col[:S.e].long()]
            scores = similarity(src_Z, dst_Z).detach().to(device=S.device, dtype=torch.float64).reshape(-1).contiguous()
            if scores.numel() != S.e:
                raise ValueError(f"similarity returned {scores.numel()} scores for {S.e} edges")
            _lib.check(L.clane_row_softmax_f64(scores.data_ptr(), None, 0, S.n, S.rowptr.data_ptr(), S.w.data_ptr(),
                                               stream), "clane_row_softmax_f64")
        return S.w[:S.e]

    def build_P(self, similarity) -> torch.Tensor:
        """Coalesced sparse COO N x N with the per-source softmax weights (graph.py:118-128)."""
        w = self._build_P_device(similarity)
        return torch.sparse_coo_tensor(indices=self._coo_indices(), values=w.cpu(), size=(self._n, self._n)).coalesce()
