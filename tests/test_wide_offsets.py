"""Graphs whose [N, ld] matrices hold 2^31 or more elements, on one GPU, against the CPU oracles.

The fp32 kernels address the rows of an [N, ld] matrix by 32-bit unsigned float4 indices: they cover N * ld <= 2^34
(CLANE_MAX_MATRIX_FLOATS, refused beyond with CLANE_ERANGE); the fp64 kernels use 64-bit offsets.  Every graph here
is relabelled so that the longest rows and the most-gathered columns get the highest ids: the hub rows, many spans and
many gathered neighbours lie past element 2^31 of every matrix.  Each case needs tens of GB of device and host memory
and skips, stating the amounts, where either is short.

At these sizes the L1 change is never fused into the sweep: a level-0 chunk of the cascade over N * d >= 2^31
elements is 64 or more cascade rows, more than one warp stages (fusion needs N * d <= 2^28).
"""
import ctypes
import gc
import types

import numpy as np
import pytest
import torch

from clane_b200 import _lib, similarity, synth
from clane_b200.embedder import Embedder
from clane_b200.graph import Graph
from oracle import oracle as O
from oracle_f64 import oracle_f64 as O64

GAMMA, TOL = 0.76, 10
WIDE = 2 ** 31
LONG_ROW = 16384        # hub rows of at least this many neighbours take the heavy chain kernel (kLongBlocks * 8)


def _host_available() -> int:
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    return 0


def _require(device_gb: float, host_gb: float) -> None:
    gc.collect()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    host = _host_available()
    if free < device_gb * 1e9 or host < host_gb * 1e9:
        pytest.skip(f"needs {device_gb} GB of free device memory and {host_gb} GB of host memory; "
                    f"{free / 1e9:.1f} GB and {host / 1e9:.1f} GB are available")


def _release(g: Graph) -> None:
    g._dev = None
    gc.collect()
    torch.cuda.empty_cache()


def _wide_graph(n: int, e: int, d: int, seed: int, features: str, dtype=np.float32):
    """Power-law edges relabelled by degree, ascending (hubs and the most-gathered columns last); X in chunks."""
    rng = np.random.default_rng(seed)
    src, dst = synth.make_edges(n, e, "powerlaw", rng)
    deg = np.bincount(src, minlength=n) + np.bincount(dst, minlength=n)
    new = np.empty(n, np.int64)
    new[np.argsort(deg, kind="stable")] = np.arange(n)
    src, dst = new[src], new[dst]
    del deg, new
    X = np.empty((n, d), dtype)
    for a in range(0, n, 1 << 20):
        b = min(n, a + (1 << 20))
        if features == "bow":      # ~18 words per document, 0/1
            X[a:b] = rng.random((b - a, d), dtype=np.float32) < 18.0 / d
        else:                      # scaled so that the asymmetric scores are of order one
            X[a:b] = rng.standard_normal((b - a, d)) * 0.5
    return src, dst, X


def _first_wide_row(ld: int) -> int:
    return -(-WIDE // ld)


def _check_layout(rowptr: np.ndarray, col: np.ndarray, ld: int) -> None:
    """The longest row, many rows and many gathers lie past element 2^31 of an [N, ld] matrix."""
    first = _first_wide_row(ld)
    deg = np.diff(rowptr)
    assert len(deg) * ld > WIDE
    assert int(np.argmax(deg)) >= first
    assert np.count_nonzero(deg[first:]) >= 10_000
    assert np.count_nonzero(col >= first) >= 100_000


def _asym_truth(X: np.ndarray, W: np.ndarray, rowptr: np.ndarray, col: np.ndarray, rows: np.ndarray):
    """(edge indices, P there) for whole source rows, in fp64: project, per-edge dots, row softmax."""
    d = X.shape[1]
    W64 = W.astype(np.float64)
    rowptr = rowptr.astype(np.int64)
    deg = rowptr[rows + 1] - rowptr[rows]
    rows, deg = rows[deg > 0], deg[deg > 0]
    edges = np.repeat(rowptr[rows], deg) + (np.arange(deg.sum()) - np.repeat(np.cumsum(deg) - deg, deg))
    psrc = X[rows].astype(np.float64) @ W64[:d].T
    cols, inv = np.unique(col[edges], return_inverse=True)
    pdst = X[cols].astype(np.float64) @ W64[d:].T
    s = np.einsum("ij,ij->i", np.repeat(psrc, deg, axis=0), pdst[inv])
    starts = np.cumsum(deg) - deg
    m = np.maximum.reduceat(s, starts)
    ex = np.exp(s - np.repeat(m, deg))
    return edges, ex / np.repeat(np.add.reduceat(ex, starts), deg)


def _check_asym(g: Graph, X: np.ndarray, tol: float, seed: int) -> None:
    """Graph.build_P with AsymmertricSimilarity (Z = X): P of 2000 random source rows past element 2^31 and of the
    longest row, against fp64 truth."""
    torch.manual_seed(seed)
    sim = similarity.AsymmertricSimilarity(n_dim=g.d)
    S = g._device_state()
    first = _first_wide_row(S.ld)
    rows = np.unique(np.concatenate([np.random.default_rng(seed).choice(np.arange(first, g._n), 2000, replace=False),
                                     [int(np.argmax(np.diff(g._rowptr)))]]))
    got = g._build_P_device(sim)
    W = sim.stacked_weights("cpu").numpy()
    edges, want = _asym_truth(X, W, g._rowptr, g._col, rows)
    assert np.count_nonzero(np.diff(g._rowptr)[rows]) >= 1000
    assert np.abs(got[torch.from_numpy(edges).to(got.device)].cpu().numpy() - want).max() <= tol
    S.asym_work = None                         # its 2 * N * ld floats are not needed by the sweeps
    gc.collect()
    torch.cuda.empty_cache()


def _propagate_against_oracle(g: Graph, src, dst, X):
    """Cosine P, two sweeps (amounts) and Z, bit-exact against the oracle; returns (Embedder Z, amounts)."""
    O.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, g._n)
    assert np.array_equal(g._rowptr, rowptr) and np.array_equal(g._col, col)
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=GAMMA, tolerence=TOL)
    e.verbose = False
    e.propagate(max_sweeps=2)
    S = g._device_state()
    w_dev = S.w[:S.e].cpu().numpy()
    Zo, amounts, w = O.propagate(X, X, rowptr, col, GAMMA, TOL, max_sweeps=2)
    assert np.array_equal(w_dev, w)
    assert len(amounts) == 2 and np.array_equal(e.amounts_per_call[0], amounts)
    Z = g.Z.numpy()
    assert np.array_equal(Z, Zo)
    return Z, amounts


@pytest.mark.gpu
def test_d128_hub_chains_asym_and_session_past_2_31():
    """d = 128, N = 18 M, E = 36 M (N * ld = 2.3e9): span tasks, heavy and light hub chains and the unfused cascade
    past element 2^31; the TF32 asymmetric scorer; the session C-ABI on the same graph."""
    _require(60, 45)
    n, d = 18_000_000, 128
    src, dst, X = _wide_graph(n, 2 * n, d, seed=11, features="normal")
    g = Graph.from_arrays(n, src, dst, X)
    _check_layout(g._rowptr, g._col, 128)
    deg = np.diff(g._rowptr)
    plan = g._device_state().plan
    n_long = int(np.count_nonzero(deg >= LONG_ROW))
    assert n_long >= 1 and plan.n_hub_rows > n_long and not plan.fused_l1
    assert plan.launches_per_sweep == 6          # spans, hub segments, heavy chains, light chains, cascade level 0/1, finish
    _check_asym(g, X, 2e-3, seed=1)              # the TF32 kernel's bound (test_gpu_parity)
    Z, amounts = _propagate_against_oracle(g, src, dst, X)
    del src, dst
    _release(g)
    h = ctypes.c_void_p()
    L = _lib.lib()
    _lib.check(L.clane_session_create(ctypes.byref(h), n, g._nnz, d, g._rowptr.ctypes.data, g._col.ctypes.data,
                                      X.ctypes.data, 0), "clane_session_create")
    try:
        am = np.zeros(8, np.float32)
        k = ctypes.c_int32()
        _lib.check(L.clane_session_propagate(h, ctypes.c_float(GAMMA), TOL, 2, am.ctypes.data, 8, ctypes.byref(k)),
                   "clane_session_propagate")
        assert k.value == 2 and np.array_equal(am[:2], amounts)
        Zs = np.empty((n, d), np.float32)
        _lib.check(L.clane_session_get_z(h, Zs.ctypes.data), "clane_session_get_z")
        assert np.array_equal(Zs, Z)
    finally:
        L.clane_session_destroy(h)


@pytest.mark.gpu
def test_d1433_multi_slab_rows_and_asym_fp32_past_2_31():
    """d = 1433 bag of words, N = 1.6 M, E = 3.2 M (N * ld = 2.3e9): 12 column slabs per row, the fma dot order,
    hub chains with sequential-regime columns, the unfused cascade; the 3xTF32 asymmetric scorer."""
    _require(60, 45)
    n, d = 1_600_000, 1433
    src, dst, X = _wide_graph(n, 2 * n, d, seed=12, features="bow")
    g = Graph.from_arrays(n, src, dst, X)
    _check_layout(g._rowptr, g._col, 1436)
    plan = g._device_state().plan
    assert plan.n_hub_rows >= 1 and not plan.fused_l1
    _check_asym(g, X, 1e-5, seed=2)
    _propagate_against_oracle(g, src, dst, X)
    _release(g)


@pytest.mark.gpu
def test_fp64_d64_past_2_31():
    """float64, d = 64, N = 34 M, E = 68 M (N * ld = 2.18e9): P, two sweeps' amounts and Z bit-exact against the fp64
    oracle."""
    _require(100, 75)
    n, d = 34_000_000, 64
    src, dst, X = _wide_graph(n, 2 * n, d, seed=13, features="normal", dtype=np.float64)
    g = Graph.from_arrays(n, src, dst, torch.from_numpy(X))
    _check_layout(g._rowptr, g._col, 64)
    O.set_threads(O.max_threads())
    O64.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, n)
    del src, dst
    assert np.array_equal(g._rowptr, rowptr) and np.array_equal(g._col, col)
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=GAMMA, tolerence=TOL)
    e.verbose = False
    e.propagate(max_sweeps=2)
    w_dev = g._dev.w[:g._nnz].cpu().numpy()
    Zo, amounts, w = O64.propagate(X, X, rowptr, col, GAMMA, TOL, max_sweeps=2)
    assert np.array_equal(w_dev, w)
    assert len(amounts) == 2 and np.array_equal(e.amounts_per_call[0], amounts)
    assert np.array_equal(g.Z.numpy(), Zo)
    _release(g)


@pytest.mark.gpu
def test_cosine_pairs_past_2_33():
    """CosineSimilarity._raw over E = 9 M pairs at d = 500: its helper matrix [2E, 500] holds 9e9 floats, so the second
    operand of the last pairs lies past float 2^33 (float4 index 2^31).  Per-pair dots are independent of the batch:
    they must equal the dots of the same pairs computed in slices of 3 M pairs."""
    _require(80, 4)
    e, d = 9_000_000, 500
    assert (2 * e - 1) * d >= 2 ** 33
    gen = torch.Generator(device="cuda")
    gen.manual_seed(14)
    v1 = torch.randn((e, d), generator=gen, device="cuda")
    v2 = torch.randn((e, d), generator=gen, device="cuda")
    dots, _ = similarity.CosineSimilarity._raw(v1, v2)
    dots = dots[:e].cpu()
    for a in range(0, e, 3_000_000):
        b = min(e, a + 3_000_000)
        part, _ = similarity.CosineSimilarity._raw(v1[a:b], v2[a:b])
        assert torch.equal(part[:b - a].cpu(), dots[a:b])
    del v1, v2
    gc.collect()
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_plan_refuses_matrices_past_2_34_floats():
    """Scores-only plans included: N * ld = 2^34 is accepted, one float4 more per row is CLANE_ERANGE."""
    _lib.Plan(2 ** 30, 0, 16)
    with pytest.raises(_lib.ClaneError, match="out of range"):
        _lib.Plan(2 ** 30, 0, 17)


def test_sharded_sweeper_refuses_wide_graphs():
    """Sharded sweeps are verified only below 2^31 elements per matrix: wider graphs are refused before any device
    or process-group work."""
    from clane_b200.dist import ShardedSweeper
    g = types.SimpleNamespace(_n=WIDE // 128, X=torch.empty((0, 128)))
    with pytest.raises(NotImplementedError, match="2\\^31"):
        ShardedSweeper(g, similarity.CosineSimilarity(), GAMMA)
