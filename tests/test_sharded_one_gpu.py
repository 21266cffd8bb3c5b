"""The row-partitioned multi-GPU sweep (clane_b200/dist.py and the kernel code that exists only for it), run on ONE
device against the CPU oracle, bit-exact.

A peer store is an ordinary global store, so "rank q's Z buffer" can be any allocation on the same GPU, and the
kernels have no device-side waits across CTAs or launches, so several emulated ranks on one device cannot deadlock.

Layer 1 drives W ranks' plans in sequence through the C-ABI, doing in one thread what ShardedSweeper.sweep() does on
each rank: per-rank build_P (dots over the rank's own edges, the norms reduced by node range, the plan's softmax),
sweeps whose rows every rank stores into every rank's replica (bulk stores to up to 15 peers, lane stores, hub-chain
peer stores), and the exact L1 change reduced by node range.  Every destination is checked separately: after one
rank's sweep alone, every replica holds the oracle's values in that rank's rows and NaN everywhere else.

Layer 2 runs ShardedSweeper itself, one thread per rank in one process, with torch.distributed and its symmetric
memory replaced by host-side fakes: every collective meets the other ranks at a barrier of its group and checks that
they all called the same collective with the same shape (a mismatch is a deadlock under NCCL).

Every case first asserts the regime it was built for (row cuts, bulk or lane stores, hub chains, exchange mode), so
that a change to the planner or to dist.py fails here instead of moving the case to an easier path.
"""
import collections
import ctypes
import threading
import types

import numpy as np
import pytest
import torch

import clane_b200.dist as cdist
from clane_b200 import _lib, similarity
from clane_b200.graph import Graph
from oracle import oracle as O
from tests.test_host import group_schedule, sweep_program
from tests.test_sweep_regimes import exact_edges

pytestmark = pytest.mark.gpu

GAMMA = 0.76
HUB = 256                # explicit hub threshold of the layer-1 plans: rows of > 256 neighbours take segments + chains
HEAVY = 20003            # neighbours of the heavy hub row: 2500 8-blocks >= kLongBlocks, the heavy chain kernel
LONG_BLOCKS = 2048       # kLongBlocks (program.cuh)
MAX_PEERS = 15           # kMaxPeers (program.cuh): remote destinations of one sweep
TOL = 2                  # patience of every run to the stop
BARRIER_TIMEOUT = 300.0  # seconds: a rank that never arrives fails the case instead of hanging it


def oracle_csr(deg, d, seed):
    rng = np.random.default_rng(seed)
    n = len(deg)
    src, dst = exact_edges(deg, rng)
    X = rng.standard_normal((n, d), dtype=np.float32)
    O.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, n)
    assert np.array_equal(np.diff(rowptr), deg)                   # exact degrees: the regimes below rest on them
    return src, dst, X, rowptr, col


def cuts(n, d, world):
    """dist.py's row cut: node-aligned when the shape allows it, else equal multiples of 8 rows."""
    aligned = cdist.aligned_rows_per_rank(n, d, world)
    per = aligned if aligned is not None else cdist.rows_per_rank(n, world)
    return aligned is not None, per, [cdist.row_range(n, world, r, per) for r in range(world)]


def cascade_nodes(elems):
    nodes = ctypes.c_int64()
    _lib.check(_lib.lib().clane_cascade_shape(elems, ctypes.byref(nodes), None))
    return int(nodes.value)


def rows_equal(got, want):
    """Bit-exact row comparison on the device; NaN in `want` means "must be NaN" (never written)."""
    both_nan = torch.isnan(want) & torch.isnan(got)
    return ((got == want) | both_nan).all(1)


def assert_buffer(got, want, what):
    ok = rows_equal(got, want)
    if not bool(ok.all()):
        bad = torch.nonzero(~ok).flatten()[:8].tolist()
        raise AssertionError(f"{what}: {int((~ok).sum())} rows differ, first {bad} (NaN: never written)")


# =====================================================================================================================
# Layer 1: W ranks' plans on one device, driven in sequence through the C-ABI
# =====================================================================================================================
# (d, W, aligned cut): d = 128 / 100 / 33 / 7 store a span's rows in bulk (one 128-column slab), d = 500 lane by lane
# over 4 slabs; 16 ranks = 15 remote destinations, the last lane of flush_rows.  d = 7 runs on n = 13.
L1_CASES = [(128, 2, True), (128, 8, True), (128, 16, True), (100, 2, True), (100, 3, True), (100, 8, False),
            (500, 4, False), (33, 3, False), (7, 4, False)]
# d -> (ld, slabs of 128 columns, tail float4s past the 16-column blocks)
assert max(w for _, w, _ in L1_CASES) == MAX_PEERS + 1       # the widest case stores through every peer slot
WIDTHS = {128: (128, 1, 0), 100: (100, 1, 1), 500: (500, 4, 1), 33: (36, 1, 1), 7: (8, 1, 2)}


def layer1_degrees(n, world, ranges, rng):
    """1-4 neighbours per row; the heavy hub as the first row of rank 1, light hubs at the last row of rank 0, inside
    the last rank and at row n - 1 (the rows the L1 tail reads), a sink as the first row of a rank, and a whole rank of
    sinks from W = 4 on.  n = 13: small rows only, a sink as the first row of rank 1."""
    deg = rng.integers(1, 5, n)
    if n < 1000:
        deg[ranges[1][0]] = 0
        return deg
    deg[ranges[1][0]] = HEAVY
    deg[ranges[0][1] - 1] = 300
    lo, hi = ranges[world - 1]
    deg[(lo + hi) // 2] = 333
    deg[n - 1] = 317
    deg[ranges[world - 1][0] if world >= 3 else 0] = 0
    if world >= 4:
        deg[ranges[world - 2][0]:ranges[world - 2][1]] = 0
    return deg


def patience(state):
    return _lib.Patience.from_buffer_copy(state.cpu().numpy().tobytes())


@pytest.mark.parametrize("d,world,aligned", L1_CASES)
def test_rank_plans_in_sequence_against_oracle(d, world, aligned):
    L = _lib.lib()
    n = 13 if d == 7 else 40000
    ld = int(L.clane_padded_ld(d))
    al, _, ranges = cuts(n, d, world)
    deg = layer1_degrees(n, world, ranges, np.random.default_rng(d * 100 + world))
    _, _, X, rowptr, col = oracle_csr(deg, d, d * 1000 + world)
    rp32 = rowptr.astype(np.int32)

    # ---- the regime ----
    assert al == aligned
    limit = d // 16 * 16
    assert (ld, (ld + 127) // 128, (ld - limit) // 4) == WIDTHS[d]
    if d == 7:
        assert [hi - lo for lo, hi in ranges] == [8, 5, 0, 0] and n * d < 32 * 16 * 16 and cascade_nodes(n * d) == 1
    else:
        assert all(hi > lo for lo, hi in ranges)
        assert deg[ranges[1][0]] == HEAVY and deg[ranges[0][1] - 1] > HUB and deg[n - 1] > HUB
        tasks = sweep_program(rp32, n, d, *ranges[1], HUB)
        seg = tasks[(tasks[:, 3] & 512) != 0]
        blocks = {int(f) >> 10: int(b) for f, b in zip(seg[:, 3], seg[:, 6])}
        assert blocks[0] == HEAVY // 8 >= LONG_BLOCKS                   # rank 1's first row: the heavy chain
        if world >= 4:
            assert not np.any(deg[slice(*ranges[world - 2])])
    sweep_rank_plans(X, rowptr, col, deg, ranges, aligned)


def sweep_rank_plans(X, rowptr, col, deg, ranges, aligned):
    """What ShardedSweeper does on every rank, one rank after the other: build_P, then sweeps to the oracle's patience
    stop with every rank's rows stored into every rank's replica, and the exact L1 change reduced by node range."""
    L = _lib.lib()
    n, d = X.shape
    world = len(ranges)
    ld = int(L.clane_padded_ld(d))
    e = len(col)
    rp32 = rowptr.astype(np.int32)
    n1, nn = cascade_nodes(n * d), cascade_nodes(e * d)
    plans = [_lib.Plan(n, e, d, rp32, lo, hi, HUB) for lo, hi in ranges]
    for (lo, hi), plan in zip(ranges, plans):
        assert (plan.group_rows, plan.fused_l1) == (8, False)          # a rank's plan is never fused: G = 8
        hubs = [v for v in range(lo, hi) if deg[v] > HUB]
        hr = group_schedule(rp32, n, d, lo, hi, HUB)[3]
        assert sorted(hr.tolist()) == hubs and plan.n_hub_rows == len(hubs)
        if not np.any(deg[lo:hi]):                                     # no rows, or a whole rank of sinks
            assert plan.n_spans == 0 and plan.n_hub_rows == 0

    dev = torch.device("cuda")
    s = _lib.stream_handle()
    Xd = torch.zeros((n, ld), device=dev)
    Xd[:, :d] = torch.from_numpy(X).to(dev)
    rowptr_d = torch.from_numpy(rp32).to(dev)
    col_d = torch.from_numpy(col if e else np.zeros(1, np.int32)).to(dev)
    erow = torch.zeros(max(e, 1), dtype=torch.int32, device=dev)
    _lib.check(L.clane_edge_rows(rowptr_d.data_ptr(), n, e, erow.data_ptr(), s))
    Z = [[Xd.clone() for _ in range(3)] for _ in range(world)]          # rank r's replica i, all X to begin with
    ptrs = [(ctypes.c_uint64 * world)(*[Z[q][i].data_ptr() for q in range(world)]) for i in range(3)]
    for r, plan in enumerate(plans):
        _lib.check(L.clane_plan_set_peers(plan.handle, world, r, ptrs[0], ptrs[1]))
        _lib.check(L.clane_plan_set_peers_third(plan.handle, ptrs[2]))

    # ---- build_P per rank: own dots, norms by node range, one "all-reduce" of the slots, finish + own softmax ----
    w = [torch.full((max(e, 1),), float("nan"), device=dev) for _ in range(world)]   # foreign weights: NaN
    pn = []
    for r, ((lo, hi), plan) in enumerate(zip(ranges, plans)):
        z0 = Z[r][0].data_ptr()
        _lib.check(L.clane_scores_cosine(plan.handle, z0, erow.data_ptr(), col_d.data_ptr(), int(rowptr[lo]),
                                         int(rowptr[hi]), w[r].data_ptr(), 0, s))
        p = torch.zeros((nn + 2) * 64, device=dev)
        _lib.check(L.clane_norms_partial(plan.handle, z0, erow.data_ptr(), col_d.data_ptr(), *cdist.node_range(nn, world, r),
                                         p.data_ptr(), s))
        pn.append(p)
    pn_sum = torch.stack(pn).sum(0)            # every slot written by exactly one rank: the sum is exact
    norms = []
    for r, plan in enumerate(plans):
        mine = pn_sum.clone()
        nr = torch.zeros(2, device=dev)
        _lib.check(L.clane_norms_finish(plan.handle, Z[r][0].data_ptr(), erow.data_ptr(), col_d.data_ptr(), mine.data_ptr(),
                                        nr.data_ptr(), s))
        _lib.check(L.clane_plan_softmax(plan.handle, w[r].data_ptr(), nr.data_ptr(), rowptr_d.data_ptr(), w[r].data_ptr(), s))
        norms.append(nr)
    torch.cuda.synchronize()
    wo = O.build_p(X, rowptr, col)
    _, s1, s2 = O.scores_raw(X, rowptr, col)
    w_all = np.full(e, np.nan, np.float32)
    for r, (lo, hi) in enumerate(ranges):
        w_all[rowptr[lo]:rowptr[hi]] = w[r][rowptr[lo]:rowptr[hi]].cpu().numpy()
        assert norms[r].cpu().numpy().tolist() == [s1, s2], f"rank {r}: norms"
    assert np.array_equal(w_all, wo)

    # ---- sweeps to the oracle's patience stop ----
    Zo, amounts, _ = O.propagate(X, X, rowptr, col, GAMMA, TOL)
    T = len(amounts)
    assert 4 <= T <= 200, T
    sink = torch.from_numpy(np.flatnonzero(deg == 0)).to(dev)
    states, logs, amount, diff = [], [], [], []
    for r in range(world):
        st = torch.zeros(8, dtype=torch.int32, device=dev)
        _lib.check(L.clane_patience_reset(st.data_ptr(), TOL, 0, s))
        states.append(st)
        logs.append(torch.zeros(256, device=dev))
        amount.append(torch.zeros(1, device=dev))
        diff.append(torch.zeros(1, device=dev))
    p1 = [torch.zeros((n1 + 3) * 32, device=dev) for _ in range(world)]
    node_ranges = [cdist.own_node_range(n, d, n1, lo, hi) if aligned else cdist.node_range(n1, world, r)
                   for r, (lo, hi) in enumerate(ranges)]
    tail_rank = [r for r, (lo, hi) in enumerate(ranges) if hi == n and lo < hi]
    assert len(tail_rank) == 1
    nan_rows = torch.full((n, d), float("nan"), device=dev)
    z_host = X
    expect = [Xd[:, :d].clone() for _ in range(3)]             # what every replica's buffer i holds
    for t in range(T):
        c, nx = t % 3, (t + 1) % 3
        want_h = O.sweep(X, z_host, rowptr, col, wo, GAMMA)
        want = torch.from_numpy(want_h).to(dev)

        def sweep(r):
            _lib.check(L.clane_sweep(plans[r].handle, Xd.data_ptr(), Z[r][c].data_ptr(), Z[r][nx].data_ptr(),
                                     rowptr_d.data_ptr(), col_d.data_ptr(), w[r].data_ptr(), ctypes.c_float(GAMMA),
                                     0, 0, 0, 0, s), f"clane_sweep rank {r}")

        if t < 3:
            # placement: each rank alone, into targets that hold NaN outside the sink rows -- every replica must hold the
            # oracle's values in exactly that rank's swept rows; the two other buffers of every replica stay untouched
            for r, (lo, hi) in enumerate(ranges):
                for q in range(world):
                    Z[q][nx].fill_(float("nan"))
                    Z[q][nx][sink] = Xd[sink]
                sweep(r)
                placed = nan_rows.clone()
                placed[lo:hi] = want[lo:hi]
                placed[sink] = Xd[sink, :d]
                for q in range(world):
                    assert_buffer(Z[q][nx][:, :d], placed, f"sweep {t}: rank {r}'s rows in replica {q}, buffer {nx}")
                    for i in (c, (t + 2) % 3):
                        assert_buffer(Z[q][i][:, :d], expect[i], f"sweep {t}: rank {r} touched replica {q}, buffer {i}")
        for r in range(world):
            sweep(r)
        for q in range(world):
            assert_buffer(Z[q][nx][:, :d], want, f"sweep {t}: replica {q}")
        expect[nx] = want

        # exact L1 change: own (aligned) or balanced (unaligned) node ranges, the tail values, one sum, finish per rank
        for r, plan in enumerate(plans):
            p1[r].zero_()
            zn, zc = Z[r][nx].data_ptr(), Z[r][c].data_ptr()
            _lib.check(L.clane_l1_partial(plan.handle, zn, zc, *node_ranges[r], p1[r].data_ptr(), s))
            if r in tail_rank:
                _lib.check(L.clane_l1_tail_values(plan.handle, zn, zc, p1[r][(n1 + 2) * 32:].data_ptr(), s))
        p1_sum = torch.stack(p1).sum(0)
        for r, plan in enumerate(plans):
            mine = p1_sum.clone()
            _lib.check(L.clane_l1_finish_values(plan.handle, mine.data_ptr(), mine[(n1 + 2) * 32:].data_ptr(),
                                                amount[r].data_ptr(), states[r].data_ptr(), logs[r].data_ptr(), 256, s))
            _lib.check(L.clane_l1_diff(plan.handle, Z[r][nx].data_ptr(), Z[r][c].data_ptr(), diff[r].data_ptr(), s))
        torch.cuda.synchronize()
        for r in range(world):
            got = np.float32(amount[r].item())
            assert got == amounts[t], f"sweep {t}, rank {r}: L1 {got} != oracle {amounts[t]}"
            assert np.float32(diff[r].item()) == got, f"sweep {t}, rank {r}: value finish != clane_l1_diff"
            st = patience(states[r])
            assert (st.sweeps, st.stop) == (t + 1, int(t == T - 1)), f"sweep {t}, rank {r}: patience {st.sweeps} {st.stop}"
        z_host = want_h
    assert np.array_equal(z_host, Zo)
    for r in range(world):
        assert np.array_equal(logs[r][:T].cpu().numpy(), amounts)


def test_peer_stores_and_value_finish_two_ranks():
    """Two ranks, one peer each: a light hub row (700 neighbours: hub segments + a light chain) in rank 0, at a
    node-aligned cut (d = 128) and an unaligned one (d = 100).  Then the argument checks of clane_plan_set_peers: more
    than 1 + kMaxPeers ranks, a rank outside the world and missing addresses are refused; the third buffer needs a peer
    set first; n_peers = 0 turns the exchange off."""
    for n, d, aligned in [(6000, 128, True), (3001, 100, False)]:
        al, _, ranges = cuts(n, d, 2)
        deg = np.random.default_rng(n + d).integers(1, 5, n)
        deg[17] = 700
        _, _, X, rowptr, col = oracle_csr(deg, d, 3 * n + d)
        assert al == aligned and ranges[0][0] <= 17 < ranges[0][1] and (700 // 8) < LONG_BLOCKS
        sweep_rank_plans(X, rowptr, col, deg, ranges, aligned)

    L = _lib.lib()
    rowptr = np.arange(0, 3 * 65, 3, dtype=np.int32)
    plan = _lib.Plan(64, int(rowptr[-1]), 8, rowptr, 0, 32, HUB)
    a = (ctypes.c_uint64 * 17)(*range(4096, 4096 + 17 * 256, 256))
    b = (ctypes.c_uint64 * 17)(*range(8192, 8192 + 17 * 256, 256))
    assert L.clane_plan_set_peers_third(plan.handle, a) == -1
    assert L.clane_plan_set_peers(plan.handle, MAX_PEERS + 2, 0, a, b) == -1
    assert L.clane_plan_set_peers(plan.handle, 2, 2, a, b) == -1
    assert L.clane_plan_set_peers(plan.handle, 2, -1, a, b) == -1
    assert L.clane_plan_set_peers(plan.handle, -1, 0, a, b) == -1
    assert L.clane_plan_set_peers(plan.handle, 2, 0, None, b) == -1
    assert L.clane_plan_set_peers(plan.handle, 2, 0, a, None) == -1
    assert L.clane_plan_set_peers(plan.handle, MAX_PEERS + 1, MAX_PEERS, a, b) == 0
    assert L.clane_plan_set_peers_third(plan.handle, None) == -1
    assert L.clane_plan_set_peers_third(plan.handle, a) == 0
    assert L.clane_plan_set_peers(plan.handle, 0, 0, None, None) == 0
    assert L.clane_plan_set_peers_third(plan.handle, a) == -1


# =====================================================================================================================
# Layer 2: ShardedSweeper itself, one thread per rank, with fake collectives and fake symmetric memory
# =====================================================================================================================
class _Group:
    def __init__(self, world, name):
        self.name = name
        self.barrier = threading.Barrier(world, timeout=BARRIER_TIMEOUT)
        self.slots = [None] * world


class FakeDist:
    """The part of torch.distributed that dist.py uses, for `world` threads of one process on one device.  A collective
    synchronises the calling thread's current stream, meets the other ranks at the group's barrier, checks that they all
    called the same collective with the same shape, combines on the host's order, synchronises and meets them again.
    Nothing here waits on the device."""

    class ReduceOp:
        SUM = "sum"

    def __init__(self, world):
        self.world = world
        self._local = threading.local()
        self._lock = threading.Lock()
        self.WORLD = _Group(world, "WORLD")
        self.group = types.SimpleNamespace(WORLD=self.WORLD)
        self._made = []                       # new_group() groups, by call index (the same on every rank)
        self.calls = collections.Counter()    # (group, collective) -> calls by rank 0

    def bind(self, rank):
        self._local.rank, self._local.n_new = rank, 0

    def abort(self):
        for g in [self.WORLD, *self._made]:
            g.barrier.abort()

    def get_world_size(self, group=None):
        return self.world

    def get_rank(self, group=None):
        return self._local.rank

    def new_group(self, *args, **kwargs):
        i = self._local.n_new
        self._local.n_new += 1
        with self._lock:
            while len(self._made) <= i:
                self._made.append(_Group(self.world, f"group{len(self._made) + 1}"))
            return self._made[i]

    def meet(self, group, kind, shape, payload):
        """Returns every rank's payload, in rank order."""
        group = group or self.WORLD
        r = self._local.rank
        torch.cuda.current_stream().synchronize()
        group.slots[r] = (kind, shape, payload)
        if r == 0:
            self.calls[(group.name, kind)] += 1
        group.barrier.wait()
        calls = [(k, s) for k, s, _ in group.slots]
        if len(set(calls)) != 1:
            raise AssertionError(f"ranks disagree on the collective of {group.name}: {calls}")
        return [p for _, _, p in group.slots]

    def leave(self, group):
        torch.cuda.current_stream().synchronize()
        (group or self.WORLD).barrier.wait()

    def all_reduce(self, tensor, op=ReduceOp.SUM, group=None, async_op=False):
        assert op == self.ReduceOp.SUM and not async_op
        parts = self.meet(group, "all_reduce", tuple(tensor.shape), tensor.clone())
        total = parts[0].clone()
        for p in parts[1:]:
            total += p
        tensor.copy_(total)
        self.leave(group)

    def all_gather_into_tensor(self, output, input, group=None, async_op=False):
        assert not async_op
        parts = self.meet(group, "all_gather", tuple(input.shape), input.clone())    # the input may alias the output
        output.copy_(torch.cat(parts).view_as(output))
        self.leave(group)

    def barrier(self, group=None, **kwargs):
        self.meet(group, "barrier", None, None)
        self.leave(group)


class FakeSymmetricMemory:
    """torch.distributed._symmetric_memory for ranks that share one device: a buffer is plain device memory, and the
    rendezvous hands every rank every rank's base pointer (no multicast object)."""

    def __init__(self, fake_dist, fail=False):
        self.dist, self.fail = fake_dist, fail

    def empty(self, shape, dtype, device):
        if self.fail:
            raise RuntimeError("symmetric memory is not available")
        return torch.empty(shape, dtype=dtype, device=device)

    def rendezvous(self, tensor, group):
        bufs = self.dist.meet(group, "rendezvous", (tuple(tensor.shape), tensor.dtype), tensor)
        self.dist.leave(group)

        def get_buffer(rank, shape, dtype):
            assert tuple(shape) == tuple(bufs[rank].shape) and dtype == bufs[rank].dtype
            return bufs[rank]
        return types.SimpleNamespace(buffer_ptrs=[b.data_ptr() for b in bufs], multicast_ptr=0, get_buffer=get_buffer)


def run_ranks(world, fake, fn):
    """fn(rank) on `world` threads (each on the default stream, as a torchrun rank); a failure on any rank breaks every
    barrier, so the others fail too instead of waiting.  Returns the ranks' results."""
    results, errors = [None] * world, []

    def body(r):
        fake.bind(r)
        try:
            results[r] = fn(r)
        except BaseException as exc:          # noqa: BLE001 -- re-raised on the main thread
            errors.append((r, exc))
            fake.abort()

    threads = [threading.Thread(target=body, args=(r,), name=f"rank{r}") for r in range(world)]
    try:
        for t in threads:
            t.start()
    finally:
        for t in threads:
            t.join()
    if errors:
        first = [e for e in errors if not isinstance(e[1], threading.BrokenBarrierError)] or errors
        r, exc = first[0]
        raise AssertionError(f"rank {r} failed: {exc!r}") from exc
    return results


def layer2_graph(n, d, world, seed):
    """1-4 neighbours per row, and hub rows in rank 1 and the last rank: > 256 neighbours, a hub under the per-rank
    automatic threshold (edges / 4096, at least 256)."""
    rng = np.random.default_rng(seed)
    _, _, ranges = cuts(n, d, world)
    deg = rng.integers(1, 5, n)
    deg[ranges[min(1, world - 1)][0] + 5] = 700
    deg[n - 2] = 300
    deg[n // 3] = 0
    src, dst, X, rowptr, col = oracle_csr(deg, d, seed + 1)
    return Graph.from_arrays(n, src, dst, X), X, rowptr, col, deg


# case -> (W, exchange, CLANE_DIST_PIPELINE, symmetric memory fails, n, d), (exchange, pipelined, Z buffers, aligned).
# n * d % 32 != 0 at d = 100 and 33: the last rank reduces trailing element values (clane_l1_tail_values).
L2_CASES = {
    "w1": ((1, "auto", "1", False, 70001, 100), ("none", False, 2, True)),
    "w2": ((2, "auto", "1", False, 70001, 100), ("p2p", True, 3, True)),
    "w4": ((4, "auto", "1", False, 70001, 100), ("p2p", True, 3, True)),
    "w8": ((8, "auto", "1", False, 70001, 100), ("p2p", True, 3, True)),
    "w3-two-buffers": ((3, "auto", "0", False, 70001, 100), ("p2p", False, 2, True)),
    "w2-nccl": ((2, "auto", "1", True, 20000, 128), ("nccl", False, 2, True)),
    "w4-ce": ((4, "ce", "1", False, 20000, 128), ("ce", False, 2, True)),
    "w4-odd-d": ((4, "auto", "1", False, 20003, 33), ("p2p", False, 3, False)),
}
N_SMALL = 3001           # iterate() runs on a small graph: d = 128 (node-aligned up to 8 ranks), or the case's odd d


@pytest.mark.parametrize("case", list(L2_CASES))
def test_sharded_sweeper_threads_against_oracle(case, monkeypatch):
    (world, exchange, pipeline, symm_fails, n, d), want_flags = L2_CASES[case]
    import torch.distributed._symmetric_memory  # noqa: F401 -- imported now, so that the patched attribute stays
    fake = FakeDist(world)
    symm = FakeSymmetricMemory(fake, fail=symm_fails)
    monkeypatch.setattr(cdist, "dist", fake)
    monkeypatch.setattr(torch.distributed, "_symmetric_memory", symm)
    monkeypatch.setattr(cdist, "_TAIL_GROUP", None)
    monkeypatch.setenv("CLANE_DIST_PIPELINE", pipeline)
    monkeypatch.delenv("CLANE_CE_CHUNKS", raising=False)
    _lib.Plan(1, 0, 1)                          # the library's one-time kernel setup, before the threads start

    g, X, rowptr, col, deg = layer2_graph(n, d, world, 7 * world + d)
    ds = d if d % 2 else 128
    gs, Xs, rowptr_s, col_s, _ = layer2_graph(N_SMALL, ds, world, 11 * world + d)
    sim = similarity.CosineSimilarity()
    wo = O.build_p(X, rowptr, col)
    Zo, amounts, _ = O.propagate(X, X, rowptr, col, GAMMA, TOL)
    Z4, amounts4, _ = O.propagate(X, X, rowptr, col, GAMMA, 1 << 30, max_sweeps=4)
    Zi, spc, outer = O.iterate(Xs, rowptr_s, col_s, GAMMA, TOL)
    assert len(amounts) >= 4 and len(spc) >= 2

    def rank(r):
        keep, out = [], {}
        sw = cdist.ShardedSweeper(g, sim, GAMMA, tol=TOL, exchange=exchange)
        keep.append(sw)
        out["flags"] = (sw.exchange, sw.pipelined, len(sw.Z), sw.aligned)
        out["range"] = (sw.lo, sw.hi, sw.plan.n_hub_rows)
        out["chunks"] = [(lo, hi) for _, lo, hi in sw.chunks]
        out["peer_Z"] = len(sw.peer_Z[0]) if sw.chunks else 0
        out["symm_error"] = getattr(sw, "symm_error", None)
        out["X"] = sw.X[:n, :d].cpu().numpy()
        elo, ehi = int(rowptr[sw.lo]), int(rowptr[sw.hi])
        out["w"] = sw.w[elo:ehi].cpu().numpy()
        out["amounts"] = np.float32(sw.propagate())
        out["Z"] = sw.Z_host().numpy()
        out["slice"] = sw.Z_host_slice().numpy()
        # a fresh sweeper: the pipelined call twice, the first one stopping with a speculative sweep in flight
        sw2 = cdist.ShardedSweeper(g, sim, GAMMA, tol=TOL, exchange=exchange)
        keep.append(sw2)
        out["amounts4"] = np.float32(sw2.sweeps(3) + sw2.sweeps(1))
        out["Z4"] = sw2.Z_host().numpy()
        sw3 = cdist.ShardedSweeper(gs, sim, GAMMA, tol=TOL, exchange=exchange)
        keep.append(sw3)
        out["iterate"] = sw3.iterate()
        out["Zi"] = sw3.Z_host().numpy()
        out["small_flags"] = (sw3.exchange, sw3.pipelined)
        torch.cuda.synchronize()
        cdist.dist.barrier()                    # no rank frees its buffers while another may still store into them
        return out

    res = run_ranks(world, fake, rank)

    # ---- the flags and the cut ----
    al, _, ranges = cuts(n, d, world)
    for r, o in enumerate(res):
        assert o["flags"] == want_flags, (r, o["flags"])
        assert o["range"][:2] == ranges[r]
    assert al == want_flags[3]
    for o in res:                               # the small graph takes the same exchange (and pipeline, at d = 128)
        assert o["small_flags"] == want_flags[:2]
    hub_ranks = [r for r, (lo, hi) in enumerate(ranges) if np.any(deg[lo:hi] > 256)]
    assert all(res[r]["range"][2] >= 1 for r in hub_ranks) and (world == 1 or hub_ranks[0] > 0)
    if want_flags[0] == "nccl":
        assert res[0]["symm_error"] and fake.calls[("WORLD", "all_gather")] > 1
    else:
        assert fake.calls[("WORLD", "all_gather")] == (3 if world > 1 else 0)      # X, once per sweeper
    if want_flags[0] == "ce":
        for r, o in enumerate(res):
            lo, hi = ranges[r]
            assert len(o["chunks"]) >= 2 and o["chunks"][0][0] == lo and o["chunks"][-1][1] == hi and o["peer_Z"] == world
    if want_flags[1]:
        assert any(name != "WORLD" for name, _ in fake.calls)                    # the tail all-reduce's own group

    # ---- every rank against the oracle ----
    for r, o in enumerate(res):
        lo, hi = ranges[r]
        assert np.array_equal(o["X"], X), f"rank {r}: gathered X"
        assert np.array_equal(o["w"], wo[rowptr[lo]:rowptr[hi]]), f"rank {r}: own rows of P"
        assert np.array_equal(o["amounts"], amounts), f"rank {r}: propagate() amounts"
        assert np.array_equal(o["Z"], Zo), f"rank {r}: Z after propagate()"
        assert np.array_equal(o["amounts4"], amounts4), f"rank {r}: sweeps(3) + sweeps(1)"
        assert np.array_equal(o["Z4"], Z4), f"rank {r}: Z after sweeps(3) + sweeps(1)"
        got_spc, got_outer = o["iterate"]
        assert got_spc == spc.tolist() and np.array_equal(np.float32(got_outer), outer), f"rank {r}: iterate()"
        assert np.array_equal(o["Zi"], Zi), f"rank {r}: Z after iterate()"
    assert np.array_equal(np.concatenate([o["slice"] for o in res]), Zo)
