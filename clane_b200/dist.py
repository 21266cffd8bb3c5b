"""Row-partitioned multi-GPU sweep (SURVEY.md section 8e): one process per GPU of one NVLink domain.

Nodes are partitioned by contiguous id range; every rank keeps the full CSR and a full replica
of Z (out-neighbours span all ranks) and sweeps its own rows.  The exchange is fused into the
sweep: the Z buffers (three, rotating; slices of one peer-mapped symmetric allocation) are known
to the sweep kernel on every rank (clane_plan_set_peers / _third), which stores a span's finished
rows of Znext to ALL ranks' buffers -- one bulk store per destination, issued from inside the
kernel, overlapping the gathers, no collective on the data path.  ShardedSweeper.sweeps() pipelines
the rest: a token all-reduce orders the ranks between sweeps on the main stream, the exact L1 of
sweep t runs on a tail stream and a second process group beside sweep t + 1.  Where symmetric
memory is unavailable the slices are exchanged with one NCCL all-gather per sweep instead.  The
three global scalars stay bit-identical on every rank:

  * L1 change per sweep (embedder.py:94): the ATen cascade's level-1 nodes are independent, so
    each rank reduces the nodes of its OWN rows right after its sweep, from local data only (the
    row ranges are cut at multiples of lcm(node, d) / d rows so that no node straddles two
    ranks); the ranks all-reduce(SUM) the node slots -- every slot is written by exactly one rank
    and is +0 elsewhere, so the sum is exact -- together with the <= 31 trailing element values,
    and each rank finishes levels 2-3 and the patience state machine itself
    (clane_l1_finish_values).  In the synchronous form (sweep()) that all-reduce is also the only
    inter-rank ordering a sweep needs: once it completes on a rank, every rank has finished
    reading Zcur and its peer stores of Znext have landed.  Patience is replicated, never broadcast.  When the shape
    cannot be cut that way (d odd, tiny n) the ranks first synchronise, then reduce balanced
    node ranges of the full array.
  * the two Frobenius norms of build_P (similarity.py:37) are cascade sums over the flattened [E*d] gathered
    arrays: each rank reduces a balanced, contiguous range of the cascade's level-1 nodes (it holds the full Z and
    CSR, so any node range is local work), the ranks all-reduce the node slots exactly as for the L1 change, and every
    rank finishes the fixed-order combine itself; dots and softmax only for the rank's own rows.

The helpers at the top are pure host logic (tested under gloo on CPU); ShardedSweeper needs CUDA.
"""
from __future__ import annotations

import ctypes
import math
import os

import numpy as np
import torch
import torch.distributed as dist

from . import _lib

ROW_ALIGN = 8   # slices are cut at multiples of the sweep's row-group size


def node_align_rows(n: int, d: int) -> int:
    """Rows per alignment unit such that a cut at a multiple of it never splits a level-1 node of
    the ATen cascade over the flattened [n*d] array: lcm(node elements, d) / d."""
    ni = (n * d) // 32
    p = max(4, ((ni - 1).bit_length() if ni > 1 else 0) // 4)
    node_elems = 32 * (1 << p) * (1 << p)
    return node_elems // math.gcd(node_elems, d)


def rows_per_rank(n: int, world: int, align: int = ROW_ALIGN) -> int:
    """Equal slice length (a multiple of `align`) such that world * length >= n."""
    per = -(-n // world)
    return -(-per // align) * align


def aligned_rows_per_rank(n: int, d: int, world: int):
    """Slice length cut at level-1 node boundaries, or None when the nodes are too coarse for this
    shape (fewer than 4 alignment units per rank: the cut would unbalance the ranks)."""
    a = node_align_rows(n, d)
    if a % ROW_ALIGN or a * 4 * world > n:
        return None
    return rows_per_rank(n, world, a)


def row_range(n: int, world: int, rank: int, per: int | None = None) -> tuple[int, int]:
    """Rows [lo, hi) owned by `rank`; trailing ranks may own fewer (or no) rows."""
    per = rows_per_rank(n, world) if per is None else per
    lo = min(rank * per, n)
    return lo, min(lo + per, n)


def own_node_range(n: int, d: int, n_nodes: int, lo: int, hi: int) -> tuple[int, int]:
    """Level-1 nodes covered by rows [lo, hi) of a node-aligned cut (the last rank takes the
    trailing partial node)."""
    ni = (n * d) // 32
    p = max(4, ((ni - 1).bit_length() if ni > 1 else 0) // 4)
    node_elems = 32 * (1 << p) * (1 << p)
    if lo >= hi:
        return n_nodes if lo >= n else 0, n_nodes if lo >= n else 0
    nlo = (lo * d) // node_elems
    nhi = n_nodes if hi >= n else (hi * d) // node_elems
    return min(nlo, n_nodes), min(nhi, n_nodes)


def node_range(n_nodes: int, world: int, rank: int) -> tuple[int, int]:
    """Level-1 cascade nodes [lo, hi) reduced by `rank` (contiguous, balanced)."""
    base, rem = divmod(n_nodes, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


_TAIL_GROUP = None


def tail_group():
    """A second process group (its own communicator and stream) for the all-reduce of the L1 slots, so that it can
    run beside the ordering all-reduce of the next sweep.  Created once per process, by every rank, at the first
    ShardedSweeper."""
    global _TAIL_GROUP
    if _TAIL_GROUP is None:
        _TAIL_GROUP = dist.new_group()
    return _TAIL_GROUP


def gather_rows(local: torch.Tensor, full: torch.Tensor, group=None) -> None:
    """all-gather equal-length row slices into `full` ([world * per, ld], contiguous)."""
    dist.all_gather_into_tensor(full, local.contiguous(), group=group)


class ShardedSweeper:
    """Sweeps of one propagate() call over this rank's rows, with the per-sweep exchange."""

    def __init__(self, graph, similarity, gamma: float, tol: int = 10, max_sweeps: int = 0, exchange: str = "auto"):
        if graph.X.dtype != torch.float32:
            raise NotImplementedError(f"sharded sweeps run in fp32 only; content embeddings are {graph.X.dtype} "
                                      "(use Embedder on one GPU for fp64)")
        n_ld = graph._n * int(_lib.lib().clane_padded_ld(int(graph.X.shape[1])))
        if n_ld >= 2 ** 31:
            # the sharded exchange and its kernels are verified only below 2^31 elements per [N, ld] matrix
            raise NotImplementedError(f"sharded sweeps need N*ld < 2^31; this graph has N*ld = {n_ld} "
                                      "(use Embedder on one GPU for wider graphs)")
        self.g, self.sim, self.gamma = graph, similarity, float(np.float32(gamma))
        self.world, self.rank = dist.get_world_size(), dist.get_rank()
        self.dev = _lib.require_cuda()
        L = _lib.lib()
        n, e, d = graph._n, graph._nnz, int(graph.X.shape[1])
        ld = int(L.clane_padded_ld(d))
        self.n, self.e, self.d, self.ld = n, e, d, ld
        aligned = aligned_rows_per_rank(n, d, self.world)
        self.aligned = aligned is not None
        self.per = aligned if self.aligned else rows_per_rank(n, self.world)
        self.lo, self.hi = row_range(n, self.world, self.rank, self.per)
        npad = self.per * self.world
        dev = self.dev
        self.rowptr = torch.from_numpy(graph._rowptr).to(dev)
        self.col = torch.from_numpy(graph._col if e else np.zeros(1, np.int32)).to(dev)
        self.erow = torch.zeros(max(e, 1), dtype=torch.int32, device=dev)
        # X: only this rank's rows travel host -> device (a sweep reads x_v of its own rows only); the initial Z = X of
        # the other ranks' rows arrives over NVLink (one all-gather of the slices) instead of 8 x the PCIe upload
        self.X = torch.zeros([npad, ld], dtype=torch.float32, device=dev)
        if self.hi > self.lo:
            self.X[self.lo:self.hi, :d] = graph.X[self.lo:self.hi].to(dev, non_blocking=True)
        if self.world > 1:
            lo_pad = self.rank * self.per
            gather_rows(self.X[lo_pad:lo_pad + self.per].clone(), self.X)
        self.plan = _lib.Plan(n, e, d, graph._rowptr, self.lo, self.hi, 0)
        self.chunks = []          # exchange "ce": (plan, row_lo, row_hi) per chunk of this rank's rows
        self.exchange = self._alloc_z(npad, ld, exchange)
        self.cur = 0
        self.w = torch.zeros(max(e, 1), dtype=torch.float32, device=dev)
        self.norms2 = torch.zeros(2, dtype=torch.float32, device=dev)
        self.amount = torch.zeros(1, dtype=torch.float32, device=dev)
        self.state = torch.zeros(8, dtype=torch.int32, device=dev)
        self.state_host = torch.zeros(8, dtype=torch.int32).pin_memory()
        self.log_cap = 1 << 16
        self.log = torch.zeros(self.log_cap, dtype=torch.float32, device=dev)
        nodes = ctypes.c_int64()
        _lib.check(L.clane_cascade_shape(n * d, ctypes.byref(nodes), None))
        self.n1 = int(nodes.value)
        if self.aligned:
            self.nlo, self.nhi = own_node_range(n, d, self.n1, self.lo, self.hi)
        else:
            self.nlo, self.nhi = node_range(self.n1, self.world, self.rank)
        # level-1 slots [n1 + 2][32] + the trailing element values [32]: one all-reduce
        self.p1 = torch.zeros((self.n1 + 3) * 32, dtype=torch.float32, device=dev)
        # the norms of build_P: level-1 nodes of the cascade over [E*d], two quantities per node
        _lib.check(L.clane_cascade_shape(e * d, ctypes.byref(nodes), None))
        self.nn = int(nodes.value)
        self.nn_lo, self.nn_hi = node_range(self.nn, self.world, self.rank)
        self.pn = torch.zeros((self.nn + 2) * 64, dtype=torch.float32, device=dev)
        self.sync_token = torch.zeros(1, dtype=torch.float32, device=dev)
        s = _lib.stream_handle()
        _lib.check(L.clane_edge_rows(self.rowptr.data_ptr(), n, e, self.erow.data_ptr(), s))
        self.tol, self.max_sweeps = tol, max_sweeps
        # pipelined sweeps (three buffers): the exact-L1 pass of sweep t on its own stream / process group, beside sweep t + 1
        self.pipelined = len(self.Z) == 3 and self.aligned and self.exchange == "p2p" and self.world > 1
        if self.pipelined:
            self.tail_stream = torch.cuda.Stream(device=dev)
            self.tail_pg = tail_group()
            self.ring = 16
            self.amounts_dev = torch.zeros(self.ring, dtype=torch.float32, device=dev)
            self.amounts_host = torch.zeros(self.ring, dtype=torch.float32).pin_memory()
        self.launches_last_sweep = 0
        self.timing, self.phase_ms = False, {}     # measurement aid: CUDA-event brackets around the phases of a sweep
        self.build_p()
        _lib.check(L.clane_patience_reset(self.state.data_ptr(), tol, max_sweeps, s))

    def _alloc_z(self, npad: int, ld: int, exchange: str) -> str:
        """The Z buffers (three for the pipelined fused exchange, else two): peer-mapped symmetric memory (exchange fused into the sweep kernel) when
        available, plain device memory + NCCL all-gather otherwise."""
        L = _lib.lib()
        self.symm = None
        if exchange in ("auto", "p2p", "multicast", "ce") and self.world > 1:
            try:
                import torch.distributed._symmetric_memory as symm_mem
                # "auto" / "p2p": three rotating buffers, so that the L1 reduction of a sweep can run beside the next sweep
                nbuf = 3 if exchange in ("auto", "p2p") and os.environ.get("CLANE_DIST_PIPELINE", "1") != "0" else 2
                # one allocation, one rendezvous (the expensive part of the setup): the buffers are slices of it
                whole = symm_mem.empty((nbuf * npad, ld), dtype=torch.float32, device=self.dev)
                hdl = symm_mem.rendezvous(whole, dist.group.WORLD)
                bufs = [whole[i * npad:(i + 1) * npad] for i in range(nbuf)]
                step = npad * ld * 4
                ptrs = [(ctypes.c_uint64 * self.world)(*[int(p) + i * step for p in hdl.buffer_ptrs]) for i in range(nbuf)]
                for b in bufs:
                    b.copy_(self.X)
                torch.cuda.synchronize()
                dist.barrier()
                self.Z, self.symm, self._symm_whole = bufs, hdl, whole
                if exchange == "ce":
                    # Copy-engine exchange (opt-in): the rank's rows are swept in a few chunks; each finished chunk goes
                    # to every peer's Znext with one peer-to-peer cudaMemcpyAsync per peer on copy streams while the next
                    # chunk is swept.  Measured at products shape: SLOWER than the stores from inside the sweep kernel --
                    # 3.21 vs 2.90 ms per sweep on 2 GPUs, 2.84 vs 1.85 ms on 8 (28 copies of 30 MB per sweep reach
                    # ~390 GB/s per rank; the in-kernel stores ~500 GB/s) -- so "auto" keeps the fused exchange.
                    self._setup_copy_engine_exchange(npad, ld)
                    return "ce"
                _lib.check(L.clane_plan_set_peers(self.plan.handle, self.world, self.rank, ptrs[0], ptrs[1]),
                           "clane_plan_set_peers")
                if nbuf == 3:
                    _lib.check(L.clane_plan_set_peers_third(self.plan.handle, ptrs[2]), "clane_plan_set_peers_third")
                mc0 = int(getattr(hdl, "multicast_ptr", 0) or 0)
                mc = [mc0 + i * step if mc0 else 0 for i in range(2)]
                # opt-in: measured at products shape on 4 GPUs, one multimem.st per row piece (1.82 ms row kernel) is
                # slower than three unicast stores (1.60 ms) -- every rank ingests the same bytes either way
                if exchange == "multicast" and all(mc):
                    _lib.check(L.clane_plan_set_multicast(self.plan.handle, mc[0], mc[1]), "clane_plan_set_multicast")
                    return "multicast"
                return "p2p"
            except Exception as exc:       # no VMM / fabric handles on this box: fall back to NCCL
                if exchange in ("p2p", "ce"):
                    raise
                self.symm_error = repr(exc)
                self.chunks = []
        self.Z = [self.X.clone(), self.X.clone()]
        return "nccl" if self.world > 1 else "none"

    def _setup_copy_engine_exchange(self, npad: int, ld: int, n_chunks: int = 0) -> None:
        n_chunks = n_chunks or int(os.environ.get("CLANE_CE_CHUNKS", "4"))
        rows = self.hi - self.lo
        step = max(ROW_ALIGN, -(-rows // n_chunks) // ROW_ALIGN * ROW_ALIGN)
        if step * n_chunks < rows:
            step += ROW_ALIGN
        lo = self.lo
        while lo < self.hi:
            hi = min(lo + step, self.hi)
            self.chunks.append((_lib.Plan(self.n, self.e, self.d, self.g._rowptr, lo, hi, 0), lo, hi))
            lo = hi
        # views of every peer's Z buffers (peer-mapped symmetric memory) and a few copy streams
        nbuf = len(self.Z)
        whole = [self.symm.get_buffer(r, (nbuf * npad, ld), torch.float32) for r in range(self.world)]
        self.peer_Z = [[w[i * npad:(i + 1) * npad] for w in whole] for i in range(nbuf)]
        self.copy_streams = [torch.cuda.Stream(device=self.dev) for _ in range(min(self.world - 1, 4))]

    def _sweep_chunks(self, zc: torch.Tensor, zn: torch.Tensor, which: int) -> int:
        """The rank's rows chunk by chunk; chunk k travels to the peers while chunk k + 1 is swept."""
        L = _lib.lib()
        cur = torch.cuda.current_stream()
        s = cur.cuda_stream
        launches = 0
        for plan, lo, hi in self.chunks:
            _lib.check(L.clane_sweep(plan.handle, self.X.data_ptr(), zc.data_ptr(), zn.data_ptr(), self.rowptr.data_ptr(),
                                     self.col.data_ptr(), self.w.data_ptr(), ctypes.c_float(self.gamma), 0, 0, 0, 0, s),
                       "clane_sweep")
            launches += plan.launches_per_sweep - 2
            ev = torch.cuda.Event()
            ev.record(cur)
            j = 0
            for r in range(self.world):
                if r == self.rank:
                    continue
                cs = self.copy_streams[j % len(self.copy_streams)]
                j += 1
                cs.wait_event(ev)
                with torch.cuda.stream(cs):
                    self.peer_Z[which][r][lo:hi].copy_(zn[lo:hi], non_blocking=True)
        for cs in self.copy_streams:     # the sweep is over when its rows have been handed to every peer's copy engine queue
            cur.wait_stream(cs)
        return launches

    def build_p(self) -> None:
        """Graph.build_P for this rank's rows: dots of the own edges, the two global norms reduced by level-1 node
        range (each rank its share of the nodes of the cascade over [E*d], one all-reduce of the slots -- every slot is
        written by exactly one rank, so the sum is exact and identical everywhere), softmax of the own rows."""
        L = _lib.lib()
        s = _lib.stream_handle()
        z = self.Z[self.cur].data_ptr()
        if self.e == 0:
            return
        if self.world == 1:
            _lib.check(L.clane_build_p_cosine(self.plan.handle, z, self.rowptr.data_ptr(), self.erow.data_ptr(),
                                              self.col.data_ptr(), self.w.data_ptr(), self.norms2.data_ptr(), s),
                       "clane_build_p_cosine")
            return
        elo, ehi = int(self.g._rowptr[self.lo]), int(self.g._rowptr[self.hi])
        _lib.check(L.clane_scores_cosine(self.plan.handle, z, self.erow.data_ptr(), self.col.data_ptr(), elo, ehi,
                                         self.w.data_ptr(), 0, s), "clane_scores_cosine")
        self.pn.zero_()
        _lib.check(L.clane_norms_partial(self.plan.handle, z, self.erow.data_ptr(), self.col.data_ptr(), self.nn_lo,
                                         self.nn_hi, self.pn.data_ptr(), s), "clane_norms_partial")
        dist.all_reduce(self.pn, op=dist.ReduceOp.SUM)
        _lib.check(L.clane_norms_finish(self.plan.handle, z, self.erow.data_ptr(), self.col.data_ptr(), self.pn.data_ptr(),
                                        self.norms2.data_ptr(), s), "clane_norms_finish")
        _lib.check(L.clane_plan_softmax(self.plan.handle, self.w.data_ptr(), self.norms2.data_ptr(), self.rowptr.data_ptr(),
                                        self.w.data_ptr(), s), "clane_plan_softmax")

    def sweep(self, with_l1: bool = True) -> int:
        """One sweep: own rows (stored to every rank's Znext when the exchange is fused), exact L1 +
        patience.  Returns the number of kernels this rank launched."""
        L = _lib.lib()
        s = _lib.stream_handle()
        nxt = (self.cur + 1) % len(self.Z)
        zc, zn = self.Z[self.cur], self.Z[nxt]
        marks = [] if self.timing else None

        def mark(name):
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                marks.append((name, ev))

        mark("start")
        if self.chunks:
            launches = self._sweep_chunks(zc, zn, nxt)
        else:
            _lib.check(L.clane_sweep(self.plan.handle, self.X.data_ptr(), zc.data_ptr(), zn.data_ptr(), self.rowptr.data_ptr(),
                                     self.col.data_ptr(), self.w.data_ptr(), ctypes.c_float(self.gamma), 0, 0, 0, 0, s),
                       "clane_sweep")
            launches = self.plan.launches_per_sweep - 2  # a rank's plan is never fused: no fix-up kernel; L1 counted below
        mark("sweep")
        if self.exchange == "nccl":
            lo = self.rank * self.per
            gather_rows(zn[lo:lo + self.per], zn)
            mark("all_gather")
        vals = self.p1[(self.n1 + 2) * 32:]
        if with_l1:
            if self.exchange in ("p2p", "multicast", "ce") and not self.aligned:
                dist.all_reduce(self.sync_token)       # every rank's rows have landed before the full-array pass
            self.p1.zero_()
            _lib.check(L.clane_l1_partial(self.plan.handle, zn.data_ptr(), zc.data_ptr(), self.nlo, self.nhi,
                                          self.p1.data_ptr(), s), "clane_l1_partial")
            if self.hi == self.n and self.lo < self.hi or (self.n == 0 and self.rank == 0):
                _lib.check(L.clane_l1_tail_values(self.plan.handle, zn.data_ptr(), zc.data_ptr(), vals.data_ptr(), s),
                           "clane_l1_tail_values")
                launches += 1
            mark("l1_partial")
            dist.all_reduce(self.p1, op=dist.ReduceOp.SUM)
            mark("all_reduce")
            _lib.check(L.clane_l1_finish_values(self.plan.handle, self.p1.data_ptr(), vals.data_ptr(),
                                                self.amount.data_ptr(), 0, 0, 0, s), "clane_l1_finish_values")
            mark("finish")
            launches += 3
        elif self.exchange in ("p2p", "multicast", "ce"):
            dist.all_reduce(self.sync_token)           # order the ranks between sweeps
        self.cur = nxt
        if marks is not None:
            marks[-1][1].synchronize()
            for (_, a), (name, b) in zip(marks, marks[1:]):
                self.phase_ms[name] = self.phase_ms.get(name, 0.0) + a.elapsed_time(b)
            self.phase_ms["sweeps"] = self.phase_ms.get("sweeps", 0) + 1
        return launches

    def last_amount(self) -> float:
        return float(self.amount.cpu()[0])

    def sweeps(self, max_sweeps: int = 0, until_stop: bool = False) -> list:
        """Up to `max_sweeps` sweeps (0: unbounded, with `until_stop`), optionally ended by the strict-minimum patience
        counter of embedder.py:94-108.  Returns the per-sweep L1 amounts (fp32).

        Pipelined over three rotating buffers when the exchange is fused and the slices are node-aligned: sweep t + 1
        (main stream) needs only the rows of sweep t on every rank -- one all-reduce of a token orders the ranks -- so
        the exact L1 of sweep t (own level-1 nodes, all-reduce of the slots on a second process group, finish, amount
        into a pinned ring) runs beside it on the tail stream, and the host reads amount t while sweep t + 1 runs.
        A sweep overwrites the buffer the L1 pass of two sweeps earlier read: the ordering all-reduce before it is
        issued only after that pass.  At most ONE speculative sweep runs after the stop, into a buffer that is not the
        result (the same contract as clane_sweeps on one GPU).  Otherwise: a loop over sweep()."""
        if not (max_sweeps or until_stop):
            raise ValueError("sweeps(): give max_sweeps or until_stop")
        minimum, patience, amounts = np.float32(np.inf), self.tol, []
        if not self.pipelined or self.timing:
            while True:
                self.sweep(True)
                amount = np.float32(self.amount.cpu().numpy()[0])
                amounts.append(amount)
                if until_stop:
                    if minimum > amount:
                        patience, minimum = self.tol, amount
                    else:
                        patience -= 1
                    if patience == 0:
                        return amounts
                if max_sweeps and len(amounts) >= max_sweeps:
                    return amounts
        L = _lib.lib()
        main, tail = torch.cuda.current_stream(), self.tail_stream
        s_main, s_tail = main.cuda_stream, tail.cuda_stream
        start, ring = self.cur, self.ring
        l1_read, done = {}, {}
        with_tail_values = (self.hi == self.n and self.lo < self.hi) or (self.n == 0 and self.rank == 0)
        vals = self.p1[(self.n1 + 2) * 32:]

        def issue(t: int) -> None:
            c = (start + t) % 3
            zc, zn = self.Z[c], self.Z[(c + 1) % 3]
            if t >= 2:
                main.wait_event(l1_read.pop(t - 2))    # this rank's L1 pass has read the buffer sweep t overwrites everywhere
            dist.all_reduce(self.sync_token)           # every rank's previous sweep has landed
            _lib.check(L.clane_sweep(self.plan.handle, self.X.data_ptr(), zc.data_ptr(), zn.data_ptr(), self.rowptr.data_ptr(),
                                     self.col.data_ptr(), self.w.data_ptr(), ctypes.c_float(self.gamma), 0, 0, 0, 0, s_main),
                       "clane_sweep")
            swept = torch.cuda.Event()
            swept.record(main)
            with torch.cuda.stream(tail):
                tail.wait_event(swept)
                self.p1.zero_()
                _lib.check(L.clane_l1_partial(self.plan.handle, zn.data_ptr(), zc.data_ptr(), self.nlo, self.nhi,
                                              self.p1.data_ptr(), s_tail), "clane_l1_partial")
                if with_tail_values:
                    _lib.check(L.clane_l1_tail_values(self.plan.handle, zn.data_ptr(), zc.data_ptr(), vals.data_ptr(), s_tail),
                               "clane_l1_tail_values")
                ev = torch.cuda.Event()
                ev.record(tail)
                l1_read[t] = ev
                dist.all_reduce(self.p1, op=dist.ReduceOp.SUM, group=self.tail_pg)
                slot = self.amounts_dev[t % ring:t % ring + 1]
                _lib.check(L.clane_l1_finish_values(self.plan.handle, self.p1.data_ptr(), vals.data_ptr(), slot.data_ptr(),
                                                    0, 0, 0, s_tail), "clane_l1_finish_values")
                self.amounts_host[t % ring:t % ring + 1].copy_(slot, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(tail)
                done[t] = ev

        limit = max_sweeps if max_sweeps else 1 << 62
        issue(0)
        issued = 1
        while True:
            if issued < limit:
                issue(issued)                          # one sweep ahead of the amount the host looks at
                issued += 1
            t = len(amounts)
            done.pop(t).synchronize()
            amount = np.float32(self.amounts_host[t % ring].item())
            amounts.append(amount)
            if until_stop:
                if minimum > amount:
                    patience, minimum = self.tol, amount
                else:
                    patience -= 1
                if patience == 0:
                    break
            if len(amounts) >= limit:
                break
        main.wait_stream(tail)                         # whatever follows on the main stream sees the tails finished
        k = len(amounts)
        self.cur = (start + k) % 3
        self.amount.copy_(self.amounts_dev[(k - 1) % ring:(k - 1) % ring + 1])
        self.launches_last_sweep = self.plan.launches_per_sweep - 2 + 3 + (1 if with_tail_values else 0)
        return amounts

    # -- the reference's loops, replicated on every rank (never broadcast: the amounts are bit-identical) ----
    def propagate(self, max_sweeps: int = 0) -> list:
        """One Embedder.propagate() call (/root/reference/clane/embedder.py:71-108): build_P once, then sweeps
        until the strict-minimum patience counter reaches 0.  Returns the per-sweep L1 amounts.  The counter
        runs on the host here (one scalar read per sweep: microseconds against a multi-millisecond sharded
        sweep), on fp32 values, exactly as the reference compares them."""
        self.build_p()
        return self.sweeps(max_sweeps, until_stop=True)

    def iterate(self, max_outer: int = 0):
        """Embedder.iterate() (embedder.py:56-69).  Returns (sweeps per propagate() call, outer amounts)."""
        L = _lib.lib()
        minimum, patience = np.float32(np.inf), self.tol
        sweeps_per_call, outer_amounts = [], []
        prev = torch.empty_like(self.Z[0])
        outer = torch.zeros(1, dtype=torch.float32, device=self.dev)
        while True:
            prev.copy_(self.Z[self.cur])
            sweeps_per_call.append(len(self.propagate()))
            # every rank holds the full Z after the sweep's all-reduce: the outer L1 needs no exchange
            _lib.check(L.clane_l1_diff(self.plan.handle, self.Z[self.cur].data_ptr(), prev.data_ptr(), outer.data_ptr(),
                                       _lib.stream_handle()), "clane_l1_diff")
            amount = np.float32(outer.cpu().numpy()[0])
            outer_amounts.append(amount)
            if minimum > amount:
                patience, minimum = self.tol, amount
            else:
                patience -= 1
            if patience == 0 or (max_outer and len(sweeps_per_call) >= max_outer):
                return sweeps_per_call, outer_amounts

    def Z_host(self) -> torch.Tensor:
        return self.Z[self.cur][:self.n, :self.d].cpu()

    def Z_host_slice(self) -> torch.Tensor:
        """This rank's rows of the current embeddings on the host (the ranks' slices together are Z)."""
        return self.Z[self.cur][self.lo:self.hi, :self.d].cpu()
