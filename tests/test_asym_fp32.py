"""AsymmertricSimilarity at fp32 accuracy for every width: the 3xTF32 projection (clane_asym_project_fp32), the whole
build_P on it (clane_build_p_asym_fp32), the dispatch of Graph.build_P and one propagate() on top of it.

Truth is the exact product computed in fp64 from the same fp32 inputs.  The projection bound is the one the kernel
states: |p - p_exact| <= (4 + 3d) 2^-23 sum_k |z_k w_k|.
"""
import ctypes

import numpy as np
import pytest
import torch

from clane_b200 import _lib, similarity, synth
from clane_b200.embedder import Embedder
from clane_b200.graph import Graph
from oracle import oracle as O

CLANE_EINVAL = -1

WIDTHS = [1, 2, 3, 16, 31, 33, 100, 127, 129, 160, 255, 256, 257, 500, 1433]
ROWS = [0, 1, 127, 128, 129, 1000]
SENTINEL = -7.25


def _stacked(d: int, seed: int) -> np.ndarray:
    torch.manual_seed(seed)
    return similarity.AsymmertricSimilarity(n_dim=d).stacked_weights("cpu").numpy()


def _padded(a: np.ndarray, ld: int, rows: int | None = None) -> torch.Tensor:
    rows = a.shape[0] if rows is None else rows
    t = torch.zeros([max(rows, 1), ld], dtype=torch.float32)
    t[:a.shape[0], :a.shape[1]] = torch.from_numpy(a)
    return t.cuda()


def _project_fp32(Z: np.ndarray, W: np.ndarray, extra_rows: int = 0):
    """(P [2, n + extra_rows, ld] as written by clane_asym_project_fp32 over sentinel-filled buffers, error flag)."""
    L = _lib.lib()
    n, d = Z.shape
    ld = L.clane_padded_ld(d)
    Zd, Wd = _padded(Z, ld), _padded(W, ld)
    P = torch.full([2, n + extra_rows, ld], SENTINEL, device="cuda")
    work = torch.zeros(4 * d * ld, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    _lib.check(L.clane_asym_project_fp32(Zd.data_ptr(), n, d, ld, Wd.data_ptr(), ld, P[0].data_ptr(), P[1].data_ptr(),
                                         work.data_ptr(), err.data_ptr(), _lib.stream_handle()), "clane_asym_project_fp32")
    return P.cpu().numpy(), int(err.item())


def _exact(Z: np.ndarray, W: np.ndarray):
    """(exact [n, 2d] in fp64, sum_k |z_k w_k| [n, 2d])."""
    Z64, W64 = Z.astype(np.float64), W.astype(np.float64)
    return Z64 @ W64.T, np.abs(Z64) @ np.abs(W64).T


def _stacked_view(P: np.ndarray, n: int, d: int) -> np.ndarray:
    return np.concatenate([P[0, :n, :d], P[1, :n, :d]], axis=1)


# ---- 1. the projection -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("d", WIDTHS)
def test_projection_within_fp32_bound(d):
    L = _lib.lib()
    ld = L.clane_padded_ld(d)
    W = _stacked(d, d)
    rng = np.random.default_rng(d)
    for n in ROWS:
        Z = rng.standard_normal((n, d), dtype=np.float32)
        P, err = _project_fp32(Z, W, extra_rows=3)
        assert err == 0
        # nothing beyond column d - 1 of a row, nor past row n - 1
        assert np.all(P[:, :, d:ld] == SENTINEL) and np.all(P[:, n:, :] == SENTINEL)
        if n == 0:
            continue
        exact, mag = _exact(Z, W)
        got = _stacked_view(P, n, d).astype(np.float64)
        bound = (4 + 3 * d) * 2.0 ** -23 * mag
        assert np.all(np.abs(got - exact) <= bound), (n, float(np.max(np.abs(got - exact) / np.maximum(mag, 1e-300))))


@pytest.mark.gpu
def test_bound_separates_tf32_from_fp32():
    """Control: at d = 128 the TF32 kernel's error, measured the same way, is at least 10x the fp32 kernel's."""
    L = _lib.lib()
    n, d = 1000, 128
    W = _stacked(d, 5)
    Z = np.random.default_rng(5).standard_normal((n, d), dtype=np.float32)
    exact, mag = _exact(Z, W)
    P32, err = _project_fp32(Z, W)
    assert err == 0
    Zd, Wd = _padded(Z, d), torch.from_numpy(W).cuda()
    out = torch.zeros([2, n, d], device="cuda")
    e = torch.zeros(1, dtype=torch.int32, device="cuda")
    _lib.check(L.clane_asym_project(Zd.data_ptr(), n, d, d, Wd.data_ptr(), out[0].data_ptr(), out[1].data_ptr(),
                                    e.data_ptr(), _lib.stream_handle()))
    assert int(e.item()) == 0
    rel32 = np.abs(_stacked_view(P32, n, d) - exact) / mag
    relt = np.abs(_stacked_view(out.cpu().numpy(), n, d) - exact) / mag
    assert relt.max() >= 10 * rel32.max()


# ---- 2./3. build_P against fp64 truth ----------------------------------------------------------------------------
def _truth_p(X: np.ndarray, W: np.ndarray, rowptr: np.ndarray, col: np.ndarray, rows=None):
    """P in fp64 (project every node, per-edge dots, softmax per row); for `rows` only: (edge indices, P there)."""
    d = X.shape[1]
    W64 = W.astype(np.float64)
    n = len(rowptr) - 1
    rows = np.arange(n) if rows is None else np.asarray(rows)
    rowptr = rowptr.astype(np.int64)
    deg = rowptr[rows + 1] - rowptr[rows]
    rows, deg = rows[deg > 0], deg[deg > 0]
    edges = np.repeat(rowptr[rows], deg) + (np.arange(deg.sum()) - np.repeat(np.cumsum(deg) - deg, deg))
    psrc = X[rows].astype(np.float64) @ W64[:d].T
    pdst = X.astype(np.float64) @ W64[d:].T
    s = np.einsum("ij,ij->i", np.repeat(psrc, deg, axis=0), pdst[col[edges]])
    starts = np.cumsum(deg) - deg
    m = np.maximum.reduceat(s, starts)
    e = np.exp(s - np.repeat(m, deg))
    p = e / np.repeat(np.add.reduceat(e, starts), deg)
    return edges, p


def _hub_graph(n: int, d: int, rng, scale: float):
    src, dst = synth.make_edges(n, n * 6, "powerlaw", rng)
    for hub, k in ((3, 70), (11, 300)):                   # rows of >= 64 neighbours: k_row_softmax_long
        extra = rng.permutation(n)[:k]
        extra = extra[extra != hub]
        src, dst = np.concatenate([src, np.full(len(extra), hub)]), np.concatenate([dst, extra])
    X = (rng.standard_normal((n, d)) * scale).astype(np.float32)
    return Graph.from_arrays(n, src, dst, X), X


@pytest.mark.gpu
@pytest.mark.parametrize("d", [2, 100, 200, 500, 1433])
def test_build_p_against_fp64_and_module(d):
    rng = np.random.default_rng(100 + d)
    n = 1500
    g, X = _hub_graph(n, d, rng, d ** -0.25)          # scores of order one
    assert np.any(np.diff(g._rowptr) == 0) and np.diff(g._rowptr).max() >= 64    # sinks and long rows
    torch.manual_seed(d)
    sim = similarity.AsymmertricSimilarity(n_dim=d)
    W = sim.stacked_weights("cpu").numpy()
    got = g.build_P(sim).values().numpy()
    edges, want = _truth_p(X, W, g._rowptr, g._col)
    assert len(edges) == len(got) and np.array_equal(edges, np.arange(len(got)))
    assert np.abs(got - want).max() <= 1e-5
    # the reference's build_P: the fp32 module on gathered rows, then the row softmax
    rows, cols = g._coo_indices()
    Xt = torch.from_numpy(X)
    with torch.no_grad():
        scores = sim(Xt[rows], Xt[cols]).numpy().astype(np.float32)
    module = O.softmax_rows(scores, g._rowptr.astype(np.int64))
    assert np.abs(got - module).max() <= 1e-5
    sums = np.add.reduceat(got.astype(np.float64), g._rowptr[:-1][np.diff(g._rowptr) > 0])
    assert np.abs(sums - 1).max() <= 1e-5
    dense = torch.sparse_coo_tensor(torch.from_numpy(np.stack([rows.numpy(), cols.numpy()])), torch.from_numpy(got),
                                    (n, n)).to_dense().sum(1).numpy()
    assert np.all(dense[np.diff(g._rowptr) == 0] == 0)


def _build_p_fp32_direct(g: Graph, W: np.ndarray) -> np.ndarray:
    """clane_build_p_asym_fp32 on the graph's device state (any width, d = 128 included)."""
    L = _lib.lib()
    S = g._device_state()
    Wd = _padded(W, S.ld)
    work = torch.zeros(2 * S.n * S.ld + 4 * S.d * S.ld, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    _lib.check(L.clane_build_p_asym_fp32(S.plan.handle, S.Z[S.cur].data_ptr(), Wd.data_ptr(), S.ld, S.rowptr.data_ptr(),
                                         S.erow.data_ptr(), S.col.data_ptr(), S.w.data_ptr(), work.data_ptr(),
                                         err.data_ptr(), _lib.stream_handle()), "clane_build_p_asym_fp32")
    assert int(err.item()) == 0
    return S.w[:S.e].cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["cora", "pubmed", "arxiv"])
def test_benchmark_shapes_every_edge(shape):
    n, src, dst, X = synth.make_graph(shape, seed=0)
    g = Graph.from_arrays(n, src, dst, X)
    W = _stacked(X.shape[1], 0)
    got = _build_p_fp32_direct(g, W)
    edges, want = _truth_p(X, W, g._rowptr, g._col)
    assert np.array_equal(edges, np.arange(len(got)))
    assert np.abs(got - want).max() <= 1e-5


@pytest.mark.gpu
def test_products_shape_sampled_rows():
    """Every node projected on the GPU; P checked on a seeded sample of 200,000 whole source rows."""
    n, src, dst, X = synth.make_graph("products", seed=0)
    g = Graph.from_arrays(n, src, dst, X)
    W = _stacked(X.shape[1], 0)
    del src, dst
    got = _build_p_fp32_direct(g, W)
    rows = np.sort(np.random.default_rng(7).choice(n, 200_000, replace=False))
    edges, want = _truth_p(X, W, g._rowptr, g._col, rows)
    assert len(edges) > 1_000_000
    assert np.abs(got[edges] - want).max() <= 1e-5


# ---- 4. dispatch --------------------------------------------------------------------------------------------------
def _small_graph(d: int, seed: int):
    rng = np.random.default_rng(seed)
    n = 600
    src, dst = synth.make_edges(n, n * 5, "powerlaw", rng)
    X = (rng.standard_normal((n, d)) * d ** -0.25).astype(np.float32)
    return Graph.from_arrays(n, src, dst, X), X


@pytest.mark.gpu
def test_build_p_fuses_d100_without_calling_forward():
    g, X = _small_graph(100, 1)
    torch.manual_seed(1)
    sim = similarity.AsymmertricSimilarity(n_dim=100)

    def boom(*args, **kwargs):
        raise AssertionError("the fused path must not call the plugin")

    sim.forward = boom
    got = g.build_P(sim).values().numpy()
    assert np.array_equal(got, _build_p_fp32_direct(g, sim.stacked_weights("cpu").numpy()))


class _Scaled(similarity.AsymmertricSimilarity):
    calls = 0

    def forward(self, z_src, z_dst):
        type(self).calls += 1
        return 0.5 * super().forward(z_src, z_dst)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [100, 128])
def test_subclass_overriding_forward_is_honoured(d):
    g, X = _small_graph(d, 2)
    torch.manual_seed(2)
    sim = _Scaled(n_dim=d).cuda()          # the generic path calls the plugin on device tensors
    _Scaled.calls = 0
    got = g.build_P(sim).values().numpy()
    assert _Scaled.calls == 1
    rows, cols = g._coo_indices()
    Xt = torch.from_numpy(X).cuda()
    with torch.no_grad():
        scores = sim(Xt[rows.cuda()], Xt[cols.cuda()]).cpu().numpy().astype(np.float32)
    want = O.softmax_rows(scores, g._rowptr.astype(np.int64))
    assert np.abs(got - want).max() <= 1e-5
    # the unmodified plugin with the same weights scores twice as sharply: a different P
    plain = similarity.AsymmertricSimilarity(n_dim=d)
    plain.load_state_dict(sim.state_dict())
    assert np.abs(g.build_P(plain).values().numpy() - got).max() > 1e-4


@pytest.mark.gpu
def test_d128_default_stays_on_tf32_kernel():
    L = _lib.lib()
    g, X = _small_graph(128, 3)
    torch.manual_seed(3)
    sim = similarity.AsymmertricSimilarity(n_dim=128)
    got = g.build_P(sim).values().numpy()
    S = g._device_state()
    W = sim.stacked_weights(S.device)
    S.w.zero_()
    work = torch.zeros(2 * S.n * S.ld, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    _lib.check(L.clane_build_p_asym(S.plan.handle, S.Z[S.cur].data_ptr(), W.data_ptr(), S.rowptr.data_ptr(),
                                    S.erow.data_ptr(), S.col.data_ptr(), S.w.data_ptr(), work.data_ptr(), err.data_ptr(),
                                    _lib.stream_handle()))
    assert int(err.item()) == 0
    assert np.array_equal(got, S.w[:S.e].cpu().numpy())


# ---- 5. end to end ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_propagate_d100_bit_exact_against_oracle_with_gpu_p():
    d, gamma, tol = 100, 0.76, 3
    g, X = _hub_graph(1200, d, np.random.default_rng(9), d ** -0.25)
    torch.manual_seed(9)
    e = Embedder(g, similarity.AsymmertricSimilarity(n_dim=d), device=torch.device("cuda"), gamma=gamma, tolerence=tol)
    e.verbose = False
    e.propagate()
    w = g._dev.w[:g._nnz].cpu().numpy()
    rowptr = g._rowptr.astype(np.int64)
    # the reference's propagate loop with that P: sweep, L1 change, patience on a strict new minimum
    Z, amounts, minimum, patience = X.copy(), [], np.inf, tol
    while patience > 0 and len(amounts) < 100_000:
        Zn = O.sweep(X, Z, rowptr, g._col, w, gamma)
        a = O.l1_diff(Zn, Z)
        amounts.append(a)
        Z = Zn
        if minimum > a:
            minimum, patience = a, tol
        else:
            patience -= 1
    assert e.sweeps_per_call == [len(amounts)]
    assert np.array_equal(e.amounts_per_call[0], np.array(amounts, np.float32))
    assert np.array_equal(g.Z.numpy(), Z)


# ---- 6. C-ABI argument checks (host-side: no device needed) ---------------------------------------------------------
def test_fp32_entry_points_reject_bad_arguments():
    L = _lib.lib()
    p = ctypes.c_void_p(4096)            # never dereferenced: every call below fails its argument check first
    s = None

    def project(Z=p, n=10, d=5, ld=8, W=p, ldw=8, Ps=p, Pd=p, work=p, err=p):
        return L.clane_asym_project_fp32(Z, n, d, ld, W, ldw, Ps, Pd, work, err, s)

    for bad in ({"Z": None}, {"W": None}, {"Ps": None}, {"Pd": None}, {"work": None}, {"err": None},
                {"d": 0}, {"d": -3}, {"ld": 4}, {"ldw": 4}, {"n": -1}):
        assert project(**bad) == CLANE_EINVAL, bad
    assert L.clane_build_p_asym_fp32(None, p, p, 8, p, p, p, p, p, p, s) == CLANE_EINVAL


@pytest.mark.gpu
def test_build_p_fp32_rejects_bad_arguments():
    L = _lib.lib()
    g, X = _small_graph(100, 4)
    S = g._device_state()
    buf = torch.zeros(2 * S.n * S.ld + 4 * S.d * S.ld, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    ok = dict(Z=S.Z[0].data_ptr(), W=buf.data_ptr(), ldw=S.ld, rowptr=S.rowptr.data_ptr(), erow=S.erow.data_ptr(),
              col=S.col.data_ptr(), w=S.w.data_ptr(), work=buf.data_ptr(), err=err.data_ptr())

    def call(**kw):
        a = {**ok, **kw}
        return L.clane_build_p_asym_fp32(S.plan.handle, a["Z"], a["W"], a["ldw"], a["rowptr"], a["erow"], a["col"], a["w"],
                                         a["work"], a["err"], _lib.stream_handle())

    for bad in ({"Z": None}, {"W": None}, {"rowptr": None}, {"erow": None}, {"col": None}, {"w": None}, {"work": None},
                {"err": None}, {"ldw": 96}):
        assert call(**bad) == CLANE_EINVAL, bad
    torch.cuda.synchronize()
    assert int(err.item()) == 0
