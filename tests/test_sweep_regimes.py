"""The sweep kernel in every schedule regime the planner produces, against the CPU oracle, bit-exact.

The row kernel's control flow depends on the schedule clane_group_schedule derives from (n, d) and the degrees: the
fused-L1 group size G (4 / 8 / 16 / 32 rows = one level-0 chunk of the L1 cascade, or no fusion), direct spans (one
warp per whole group, which writes the group's L1 partial itself), fix groups (partial recomputed from memory), light
and heavy hub chains, and the columns of the sequential regime.  Every case below first asserts that its graph
reached the regime it was built for -- a change to the planner then fails here instead of moving the case to an
easier path -- and then compares P, every L1 amount and Z with the oracle, through Embedder.propagate, through one
clane_sweep into a NaN-filled Znext (a row the kernel never writes shows up as NaN, not as a stale value) and
through the conditional-WHILE launch of clane_sweeps.
"""
import ctypes

import numpy as np
import pytest
import torch

import clane_b200.graph as graph_module
from clane_b200 import _lib, similarity
from clane_b200.embedder import Embedder
from clane_b200.graph import Graph
from oracle import oracle as O
from tests.test_gpu_parity import while_launch_required
from tests.test_host import group_schedule, sweep_program

pytestmark = pytest.mark.gpu

GAMMA = 0.76
TOL = 10                 # patience never runs out within the few sweeps of a case: max_sweeps ends every run
HUB = 256                # hub threshold of every plan here: rows of > 256 neighbours take the segment + chain path
SPAN_EDGES = 128         # span budget of clane_plan_create
LONG_BLOCKS = 2048       # kLongBlocks (program.cuh): hub rows of >= 2048 8-blocks take the heavy chain kernel


def exact_edges(deg, rng):
    """Edges giving row v exactly deg[v] distinct out-neighbours: dst = (v + shift_v + j * stride_v) % n for j < deg[v]
    with (deg[v] - 1) * stride_v < n, so nothing is merged when the CSR is coalesced."""
    n = len(deg)
    src = np.repeat(np.arange(n, dtype=np.int64), deg)
    j = np.arange(len(src)) - np.repeat(np.cumsum(deg) - deg, deg)
    stride = rng.integers(1, np.maximum(1, (n - 1) // np.maximum(deg, 1)) + 1)
    shift = rng.integers(0, n, n)
    return src, (src + shift[src] + j * stride[src]) % n


def make_case(deg, d, seed, monkeypatch):
    monkeypatch.setattr(graph_module, "HUB_THRESHOLD", HUB)
    rng = np.random.default_rng(seed)
    n = len(deg)
    src, dst = exact_edges(deg, rng)
    X = rng.standard_normal((n, d), dtype=np.float32)
    g = Graph.from_arrays(n, src, dst, X)
    O.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, n)
    assert np.array_equal(np.diff(rowptr), deg)                   # exact degrees: the regimes below rest on them
    assert np.array_equal(g._rowptr, rowptr) and np.array_equal(g._col, col)
    return g, X, rowptr, col


def assert_rows_equal(got, want, what):
    bad = np.flatnonzero(~(got == want).all(1))
    assert len(bad) == 0, f"{what}: {len(bad)} rows differ, first {bad[:8].tolist()} (NaN: never written)"


def check_against_oracle(g, X, rowptr, col, sweeps):
    n, d = X.shape
    L = _lib.lib()
    Zo, amounts, w = O.propagate(X, X, rowptr, col, GAMMA, TOL, max_sweeps=sweeps)
    assert len(amounts) == sweeps

    # 1. Embedder.propagate: P, every L1 amount and Z
    emb = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=GAMMA, tolerence=TOL)
    emb.verbose = False
    emb.propagate(max_sweeps=sweeps)
    S = g._device_state()
    assert np.array_equal(S.w[:S.e].cpu().numpy(), w)
    assert_rows_equal(g.Z.numpy(), Zo, "propagate")
    assert np.array_equal(emb.amounts_per_call[0], amounts)

    # 2. one clane_sweep from Zcur != X into a Znext whose swept rows hold NaN; sink rows are never written
    Z1 = O.sweep(X, X, rowptr, col, w, GAMMA)
    Zc_h = O.sweep(X, Z1, rowptr, col, w, GAMMA)
    want = O.sweep(X, Zc_h, rowptr, col, w, GAMMA)
    sink = np.diff(rowptr) == 0
    Zc = torch.zeros_like(S.X)
    Zc[:n, :d] = torch.from_numpy(Zc_h).cuda()
    Zn = torch.full_like(S.X, float("nan"))
    Zn[torch.from_numpy(np.flatnonzero(sink)).cuda()] = Zc[torch.from_numpy(np.flatnonzero(sink)).cuda()]
    amount = torch.full((1,), float("nan"), device="cuda")
    _lib.check(L.clane_sweep(S.plan.handle, S.X.data_ptr(), Zc.data_ptr(), Zn.data_ptr(), S.rowptr.data_ptr(),
                             S.col.data_ptr(), S.w.data_ptr(), ctypes.c_float(float(np.float32(GAMMA))),
                             amount.data_ptr(), 0, 0, 0, _lib.stream_handle()))
    torch.cuda.synchronize()
    assert_rows_equal(Zn[:n, :d].cpu().numpy(), want, "clane_sweep")
    assert np.float32(amount.item()) == O.l1_diff(want, Zc_h)

    # 3. the conditional-WHILE launch (one graph launch for the whole propagate()), from Z = X again
    g.set_Z(torch.from_numpy(X))
    sh = S.stream.cuda_stream
    S.stream.wait_stream(torch.cuda.current_stream())
    _lib.check(L.clane_patience_reset(S.state.data_ptr(), TOL, sweeps, sh))
    rc = L.clane_sweeps(S.plan.handle, S.X.data_ptr(), S.Zptrs, 0, S.rowptr.data_ptr(), S.col.data_ptr(), S.w.data_ptr(),
                        ctypes.c_float(float(np.float32(GAMMA))), 0, 1, S.state.data_ptr(), S.log.data_ptr(), S.log_cap, sh)
    if rc == _lib.CLANE_EUNSUPPORTED and not while_launch_required():
        return
    assert rc == 0, rc
    S.stream.synchronize()
    st = _lib.Patience.from_buffer_copy(S.state.cpu().numpy().tobytes())
    assert st.stop == 1 and st.sweeps == sweeps
    assert_rows_equal(S.Z[sweeps % 3][:n, :d].cpu().numpy(), Zo, "clane_sweeps WHILE")
    assert np.array_equal(S.log[:sweeps].cpu().numpy(), amounts)


# ---- fused group sizes ---------------------------------------------------------------------------------------------
# (d, n, G): every (d, G) the planner fuses (n * d <= 2^24: 512-element chunks, above: 1024), plus an unfused control.
# n % G != 0 throughout, so the last group is ragged.
GROUP_CASES = [(128, 5003, 4), (128, 140003, 8), (64, 5003, 8), (64, 300005, 16), (32, 5003, 16), (32, 600005, 32),
               (100, 5003, None)]

FULL, MIXED, ALL_SINK, WINDOW, SPLIT, HUB0 = 1, 2, 3, 4, 5, 6     # group indices of the special groups
HUB_DEGREES = [264 + i for i in range(8)]                          # 0..7 mod 8: every count of 8-block leftovers


def group_degrees(n, G, last_sink, rng):
    """1-4 neighbours per row (a group of <= 32 such rows stays within the span budget: a direct span of G rows),
    then the special groups at known indices."""
    deg = rng.integers(1, 5, n)
    r = lambda grp: grp * G                                         # noqa: E731
    mids = sorted({G // 3, 2 * G // 3} - {0, G - 1})
    if len(mids) + 2 >= G:
        mids = mids[:1]
    deg[r(MIXED) + np.array([0, G - 1] + mids)] = 0                 # sinks at the first, the last and middle rows
    deg[r(ALL_SINK):r(ALL_SINK) + G] = 0                           # never updated, partial +0
    deg[r(WINDOW):r(WINDOW) + G - 1] = 0                           # one row of 200 > 128: the window is restaged,
    deg[r(WINDOW) + G - 1] = 200                                   # and the span is still the whole group
    deg[r(SPLIT):r(SPLIT) + G] = -(-192 // G)                       # > 128 edges: several spans, a fix group
    for i, k in enumerate(HUB_DEGREES):                             # light hub rows, at every position of a group
        deg[r(HUB0 + i) + i % G] = k
    deg[n - 1] = 0 if last_sink else 3
    return deg


@pytest.mark.parametrize("last_sink", [False, True], ids=["last-row-swept", "last-row-sink"])
@pytest.mark.parametrize("d,n,G", GROUP_CASES)
def test_every_fused_group_size_against_oracle(d, n, G, last_sink, monkeypatch):
    fused = G is not None
    G = G or 8
    assert n % G > 1
    deg = group_degrees(n, G, last_sink, np.random.default_rng(n + d))
    g, X, rowptr, col = make_case(deg, d, n * 3 + d + last_sink, monkeypatch)

    # the regime: group size, fusion, which groups are direct spans of all their rows, which are fix groups
    sr, sm, fx, hr, G_, fused_ = group_schedule(g._rowptr, n, d, 0, n, HUB, SPAN_EDGES)
    assert (G_, fused_) == (G, fused)
    n_groups = -(-n // G)
    hub_groups = list(range(HUB0, HUB0 + len(HUB_DEGREES)))
    assert sorted(hr.tolist()) == [grp * G + i % G for i, grp in enumerate(hub_groups)]
    assert deg[hr].tolist() == sorted(HUB_DEGREES, reverse=True)
    nrows, direct = sm & 0xff, (sm >> 8) & 1
    want_direct = sorted(set(range(n_groups)) - {ALL_SINK, SPLIT, *hub_groups})
    assert sorted((sr[direct == 1] // G).tolist()) == want_direct
    assert np.all(sr[direct == 1] % G == 0)
    assert np.all(nrows[direct == 1] == np.minimum(G, n - sr[direct == 1]))
    assert ((sr >= SPLIT * G) & (sr < SPLIT * G + G)).sum() >= 2
    assert fx.tolist() == (sorted([SPLIT, *hub_groups]) if fused else [])
    # what the kernel receives: direct spans of G rows (32 rows: lane 31 sweeps the group's last row)
    tasks = sweep_program(g._rowptr, n, d, 0, n, HUB, SPAN_EDGES)
    spans = tasks[(tasks[:, 3] & 512) == 0]
    direct_tasks = spans[(spans[:, 3] & 256) != 0]
    assert len(direct_tasks) == (len(want_direct) if fused else 0)
    if fused:
        assert ((direct_tasks[:, 3] & 0xff) == G).sum() == len(want_direct) - 1
    S = g._device_state()
    assert (S.plan.group_rows, S.plan.fused_l1) == (G, fused)
    assert S.plan.n_hub_rows == len(HUB_DEGREES) and S.plan.n_fix_groups == len(fx) and S.plan.n_spans == len(sr)

    check_against_oracle(g, X, rowptr, col, sweeps=4)


# ---- heavy and light hub chains ------------------------------------------------------------------------------------
# three long rows: light with 7 leftovers (2047 blocks), heavy at exactly kLongBlocks, heavy with 3 leftovers
CHAIN_ROWS = {1001: 16383, 2050: 16384, 30007: 20003}


@pytest.mark.parametrize("d", [15, 32, 100, 111, 128, 500])
def test_hub_chain_widths_against_oracle(d, monkeypatch):
    """d = 15: sequential regime only (no 32-column slab); 32: fused G = 16 beside a heavy row; 100: one tail float4;
    111: ld = 112, a 16-column tail; 128: no tail warp; 500: several 128-column slabs."""
    n = 40000
    rng = np.random.default_rng(d)
    deg = rng.integers(1, 5, n)
    for r, k in CHAIN_ROWS.items():
        deg[r] = k
    g, X, rowptr, col = make_case(deg, d, 7 * d, monkeypatch)

    L = _lib.lib()
    ld = L.clane_padded_ld(d)
    limit = d // 16 * 16                                   # columns below it use the 8-block order
    assert (ld, limit, (ld - limit) // 4) == {15: (16, 0, 4), 32: (32, 32, 0), 100: (100, 96, 1), 111: (112, 96, 4),
                                              128: (128, 128, 0), 500: (500, 496, 1)}[d]
    sr, sm, fx, hr, G, fused = group_schedule(g._rowptr, n, d, 0, n, HUB, SPAN_EDGES)
    assert hr.tolist() == sorted(CHAIN_ROWS, key=CHAIN_ROWS.get, reverse=True)
    assert (G, fused) == {32: (16, True), 128: (4, True)}.get(d, (8, False))
    # the program's segments: blocks per hub row, hence which rows take the heavy chain kernel
    tasks = sweep_program(g._rowptr, n, d, 0, n, HUB, SPAN_EDGES)
    seg = tasks[(tasks[:, 3] & 512) != 0]
    blocks = {int(f) >> 10: int(b) for f, b in zip(seg[:, 3], seg[:, 6])}
    assert [blocks[h] for h in range(3)] == [k // 8 for k in sorted(CHAIN_ROWS.values(), reverse=True)]
    assert sum(b >= LONG_BLOCKS for b in blocks.values()) == 2 and min(blocks.values()) == LONG_BLOCKS - 1
    S = g._device_state()
    assert S.plan.n_hub_rows == 3 and (S.plan.group_rows, S.plan.fused_l1) == (G, fused)

    check_against_oracle(g, X, rowptr, col, sweeps=3)
