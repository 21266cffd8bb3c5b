"""GPU parity tests proper: the CUDA path, called through the C-ABI (ctypes), against the CPU
oracle and the golden vectors of the real reference.

Bars (BASELINE.json north_star): CSR / neighbour indexing bit-exact; identical iteration
counts; final embeddings within max-abs 1e-5 / rel 1e-4 in fp32.  Because the kernels
reproduce the reference's rounding sequence, every comparison below is also asserted
BIT-EXACT (np.array_equal), which implies the stated tolerance.
"""
import ctypes
from pathlib import Path

import numpy as np
import pytest
import torch

from clane_b200 import _lib, similarity, synth
from clane_b200.embedder import Embedder
from clane_b200.graph import Graph
from oracle import oracle as O

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
GOLD = ROOT / "tests" / "golden"
REF_CASES = sorted(p.stem for p in GOLD.glob("ref_*.npz"))
ATOL, RTOL = 1e-5, 1e-4      # north_star tolerance for final embeddings


def within_tolerance(a, b):
    return bool(np.all(np.abs(a - b) <= ATOL + RTOL * np.abs(b)))


def gpu_l1(a: np.ndarray, b: np.ndarray) -> np.float32:
    """clane_l1_diff on two [n, d] host arrays."""
    L = _lib.lib()
    n, d = a.shape
    ld = L.clane_padded_ld(d)
    A = torch.zeros([n, ld], device="cuda"); A[:, :d] = torch.from_numpy(a).cuda()
    B = torch.zeros([n, ld], device="cuda"); B[:, :d] = torch.from_numpy(b).cuda()
    out = torch.zeros(1, device="cuda")
    plan = _lib.Plan(n, 0, d)
    _lib.check(L.clane_l1_diff(plan.handle, A.data_ptr(), B.data_ptr(), out.data_ptr(), _lib.stream_handle()))
    return np.float32(out.cpu().numpy()[0])


# ---- cascade sum (embedder.py:60,94) -------------------------------------------------------------
@pytest.mark.parametrize("n,d", [(1, 1), (1, 3), (1, 7), (2, 4), (3, 5), (17, 2), (34, 2), (100, 8), (64, 128),
                                 (257, 100), (40, 1433), (3000, 500), (8192, 128), (8193, 128), (70001, 31),
                                 (169343, 128)])
def test_l1_cascade_bit_exact(n, d):
    rng = np.random.default_rng(n * 31 + d)
    a = rng.standard_normal((n, d)).astype(np.float32)
    b = rng.standard_normal((n, d)).astype(np.float32)
    assert gpu_l1(a, b) == O.l1_diff(a, b)
    assert gpu_l1(a, a) == np.float32(0)


def test_l1_cascade_matches_torch_sum_live():
    torch.set_num_threads(1)
    if torch.backends.cpu.get_cpu_capability() != "AVX512":
        pytest.skip("torch.sum order was characterised on the AVX-512 host")
    rng = np.random.default_rng(5)
    a = rng.standard_normal((5000, 128)).astype(np.float32)
    b = rng.standard_normal((5000, 128)).astype(np.float32)
    assert gpu_l1(a, b) == (torch.from_numpy(a) - torch.from_numpy(b)).abs().sum().item()


# ---- build_P: scores + norms + softmax (graph.py:118-128, similarity.py:26-37) ----------------------
@pytest.mark.parametrize("case", REF_CASES)
def test_build_p_bit_exact_with_reference(case):
    G = np.load(GOLD / f"{case}.npz")
    g = Graph.from_arrays(int(G["n"]), G["raw_src"], G["raw_dst"], G["X"])
    P = g.build_P(similarity.CosineSimilarity())
    assert np.array_equal(P.indices().numpy(), G["P0_indices"])
    assert np.array_equal(P.values().numpy(), G["P0_values"])
    rs = P.to_dense().sum(1)
    assert abs(rs.max().item() - 1) < 1e-3 and abs(rs.min().item()) < 1e-3 or int(G["n"]) == len(set(G["A_indices"][0]))


def test_row_softmax_generic_plugin_and_long_rows():
    rng = np.random.default_rng(11)
    ks = [1, 2, 7, 15, 16, 17, 31, 32, 33, 48, 100, 255, 1000, 8234, 0, 5]
    rowptr = np.concatenate([[0], np.cumsum(ks)]).astype(np.int32)
    for scale in (0.01, 1.0, 30.0):
        s = (rng.standard_normal(rowptr[-1]) * scale).astype(np.float32)
        want = O.softmax_rows(s, rowptr.astype(np.int64))
        L = _lib.lib()
        sd, rp = torch.from_numpy(s).cuda(), torch.from_numpy(rowptr).cuda()
        w = torch.zeros_like(sd)
        _lib.check(L.clane_row_softmax(sd.data_ptr(), 0, 0, len(ks), rp.data_ptr(), w.data_ptr(), _lib.stream_handle()))
        assert np.array_equal(w.cpu().numpy(), want)
        _lib.check(L.clane_row_softmax(sd.data_ptr(), 0, 0, len(ks), rp.data_ptr(), sd.data_ptr(), _lib.stream_handle()))
        assert np.array_equal(sd.cpu().numpy(), want)      # in place


def test_user_plugin_is_honoured():
    G = np.load(GOLD / "ref_hub60_d20.npz")
    g = Graph.from_arrays(int(G["n"]), G["raw_src"], G["raw_dst"], G["X"])

    class Dot:
        def __call__(self, a, b):
            assert a.is_cuda and a.shape == b.shape
            return (a * b).sum(1)

    P = g.build_P(Dot())
    rows, cols = G["A_indices"]
    s = (torch.from_numpy(G["X"]).cuda()[rows] * torch.from_numpy(G["X"]).cuda()[cols]).sum(1).cpu().numpy()
    want = O.softmax_rows(s, G["nbr_ptr"])
    assert np.array_equal(P.values().numpy(), want)


# ---- similarity plugin KATs (reference tests/test_similarity.py) -----------------------------------
def test_cosine_plugin_known_answers():
    cos = similarity.CosineSimilarity()
    v = torch.Tensor([1, 2, 3])
    assert abs(cos(v, v.clone()).item() - 1) < 1e-4
    assert abs(cos(torch.Tensor([0, 1]), torch.Tensor([1, 0])).item()) < 1e-4
    assert abs(cos(v, v.neg()).item() + 1) < 1e-4
    a, b = torch.rand(10), torch.rand(10)
    assert torch.equal(cos(a, b), cos(b, a))
    assert cos(torch.rand(4, 16), torch.rand(4, 16)).size() == torch.Size([4])


@pytest.mark.parametrize("e,d", [(1, 3), (64, 2), (64, 128), (50, 399), (50, 400), (30, 1433)])
def test_cosine_plugin_batched_quirk_bit_exact(e, d):
    rng = np.random.default_rng(e * 7 + d)
    a = rng.standard_normal((e, d)).astype(np.float32)
    b = rng.standard_normal((e, d)).astype(np.float32)
    rowptr = np.concatenate([np.arange(e + 1), np.full(e, e)]).astype(np.int64)
    dots, s1, s2 = O.scores_raw(np.concatenate([a, b]), rowptr, np.arange(e, 2 * e, dtype=np.int32))
    want = (dots / np.float32(np.sqrt(s1, dtype=np.float32) * np.sqrt(s2, dtype=np.float32))).astype(np.float32)
    got = similarity.CosineSimilarity()(torch.from_numpy(a), torch.from_numpy(b))
    assert not got.is_cuda and np.array_equal(got.numpy(), want)


def test_cosine_plugin_single_row_against_batch_matches_reference():
    """[1, d] against [E, d] (the reference's matmul broadcasts, similarity.py:35-37): golden values of the real
    reference, both argument orders."""
    G = np.load(GOLD / "prim_cosine_broadcast.npz")
    cos = similarity.CosineSimilarity()
    for i, (e, d) in enumerate(G["cases"]):
        rng = np.random.default_rng(5000 + i)
        a = torch.from_numpy(rng.standard_normal((1, d)).astype(np.float32))
        b = torch.from_numpy(rng.standard_normal((e, d)).astype(np.float32))
        assert np.array_equal(cos(a, b).numpy(), G[f"ab_{e}_{d}"])
        assert np.array_equal(cos(b, a).numpy(), G[f"ba_{e}_{d}"])
        assert np.array_equal(cos(a[0], b).numpy(), G[f"ab_{e}_{d}"])          # 1-D input is unsqueezed first
    with pytest.raises(RuntimeError):
        cos(torch.rand(3, 8), torch.rand(4, 8))


def test_vertex_z_assignment_writes_through():
    """`v.z = ...` is how the reference updates a row (embedder.py:92, graph.py:138)."""
    G = np.load(GOLD / "ref_cyclic100_d8.npz")
    g = Graph.from_arrays(int(G["n"]), G["raw_src"], G["raw_dst"], G["X"])
    g.V[3].z = torch.full([8], 2.5)                         # before the device state exists
    assert torch.equal(g.Z[3], torch.full([8], 2.5)) and torch.equal(g.X[3], torch.from_numpy(G["X"][3]))
    g._device_state()
    g.V[5].z = torch.arange(8.0)
    assert torch.equal(g.V[5].z, torch.arange(8.0)) and torch.equal(g.Z[3], torch.full([8], 2.5))
    Z = g.Z
    Z[3], Z[5] = g.X[3], g.X[5]
    assert torch.equal(Z, g.X)


# ---- sweep (embedder.py:84-94) ---------------------------------------------------------------------
@pytest.mark.parametrize("case", REF_CASES)
def test_first_sweep_bit_exact_with_reference(case):
    G = np.load(GOLD / f"{case}.npz")
    g = Graph.from_arrays(int(G["n"]), G["raw_src"], G["raw_dst"], G["X"])
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=float(G["gamma"]),
                 tolerence=int(G["tol"]))
    e.verbose = False
    e.propagate(max_sweeps=1)
    assert np.array_equal(g.Z.numpy(), G["Z_after_first_sweep"])
    assert e.amounts_per_call[0][0] == G["amounts"][0]


# ---- full iterate: counts + embeddings ---------------------------------------------------------------
@pytest.mark.parametrize("case", REF_CASES)
def test_iterate_matches_reference(case, capsys):
    G = np.load(GOLD / f"{case}.npz")
    g = Graph.from_arrays(int(G["n"]), G["raw_src"], G["raw_dst"], G["X"])
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=float(G["gamma"]),
                 tolerence=int(G["tol"]), save_history=(case == "ref_toy_d2"))
    e.iterate()
    assert e.sweeps_per_call == G["sweeps_per_call"].tolist()            # identical iteration counts
    assert np.array_equal(np.concatenate(e.amounts_per_call), G["amounts"])
    Z = g.Z.numpy()
    assert within_tolerance(Z, G["Z_final"])                             # the stated bar
    assert np.array_equal(Z, G["Z_final"])                               # and in fact bit-exact
    lines = capsys.readouterr().out.strip().split("\n")
    assert len(lines) == len(G["amounts"])
    assert [int(l.split()[-1]) for l in lines] == G["counters"].tolist() # the printed patience counters
    if e.save_history:
        assert [len(h) for h in e.history["Z"]] == G["sweeps_per_call"].tolist()
        assert np.array_equal(e.history["Z"][0][0].numpy(), G["Z_after_first_sweep"])
        assert np.array_equal(e.history["Z"][0][-1].numpy(), G["Z_after_first_call"])


def test_session_api_host_buffers():
    """The pure-C host-buffer API (what bench.py's e2e leg and a C consumer call)."""
    G = np.load(GOLD / "ref_n120_d128.npz")
    n, d = int(G["n"]), int(G["d"])
    L = _lib.lib()
    g = Graph.from_arrays(n, G["raw_src"], G["raw_dst"], G["X"])
    X = np.ascontiguousarray(G["X"])
    h = ctypes.c_void_p()
    _lib.check(L.clane_session_create(ctypes.byref(h), n, g._nnz, d, g._rowptr.ctypes.data, g._col.ctypes.data,
                                      X.ctypes.data, 0))
    try:
        w = np.zeros(g._nnz, np.float32)
        _lib.check(L.clane_session_build_p(h, w.ctypes.data))
        assert np.array_equal(w, G["P0_values"])
        spc = np.zeros(64, np.int32)
        outer = ctypes.c_int32()
        mn = ctypes.c_float(float("inf"))
        _lib.check(L.clane_session_iterate(h, ctypes.c_float(float(G["gamma"])), int(G["tol"]), 0, ctypes.byref(mn),
                                           spc.ctypes.data, 64, ctypes.byref(outer)))
        assert spc[:outer.value].tolist() == G["sweeps_per_call"].tolist()
        Z = np.zeros((n, d), np.float32)
        _lib.check(L.clane_session_get_z(h, Z.ctypes.data))
        assert np.array_equal(Z, G["Z_final"])
        assert mn.value == G["outer_amounts"].min()
        # set_Z + bounded propagate
        _lib.check(L.clane_session_set_z(h, X.ctypes.data))
        am = np.zeros(8, np.float32)
        k = ctypes.c_int32()
        _lib.check(L.clane_session_propagate(h, ctypes.c_float(float(G["gamma"])), int(G["tol"]), 5, am.ctypes.data, 8,
                                             ctypes.byref(k)))
        assert k.value == 5 and np.array_equal(am[:5], G["amounts"][:5])
    finally:
        L.clane_session_destroy(h)


# ---- the reference's own tests, restated against the new package -------------------------------------
def test_reference_test_graph_build_p(data_root):
    g = Graph(data_root=data_root, embedding_dim=16)
    P = g.build_P(similarity.CosineSimilarity()).to_dense()
    assert P.shape == (34, 34)
    assert abs(P.sum(1).max().item() - 1) < 1e-3 and abs(P.sum(1).min().item()) < 1e-3


def test_reference_test_embedder(data_root):
    g = Graph(data_root=data_root, embedding_dim=16)
    e = Embedder(graph=g, similarity_measure=similarity.CosineSimilarity(), gamma=0.74, device=torch.device("cpu"))
    e.verbose = False
    e.iterate()
    assert (g.Z - g.X).abs().sum() != 0


def test_reference_test_cli(tmp_path, data_root, monkeypatch):
    from clane_b200.__main__ import embedding, get_parser
    G = np.load(GOLD / "ref_toy_d2.npz")
    torch.manual_seed(int(G["seed"]))
    out = tmp_path / "test_output"
    args = get_parser().parse_args(["--data_root", str(data_root), "--output_root", str(out), "--config_file",
                                    str(ROOT / "tests" / "config.yaml"), "--save_history"])
    embedding(args)
    Z0 = np.load(out / "0" / "Z_0.npy")
    Z = np.load(out / "Z.npy")
    assert Z0.shape == (34, 2) and Z.shape == (34, 2) and Z.dtype == np.float32
    assert np.array_equal(Z0, G["Z_after_first_sweep"]) and np.array_equal(Z, G["Z_final"])   # config 1, end to end
    assert sorted(p.name for p in out.iterdir() if p.is_dir()) == sorted(str(i) for i in range(len(G["sweeps_per_call"])))


# ---- BASELINE shapes: oracle comparison at sizes it finishes in seconds, properties at full size ------
@pytest.mark.parametrize("shape,scale", [("cora", 1.0), ("pubmed", 1.0), ("arxiv", 1.0)])
def test_baseline_shapes_against_oracle(shape, scale):
    n, src, dst, X = synth.make_graph(shape, seed=0, scale=scale)
    g = Graph.from_arrays(n, src, dst, X)
    O.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, n)
    assert np.array_equal(g._rowptr, rowptr) and np.array_equal(g._col, col)
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=0.76, tolerence=10)
    e.verbose = False
    e.propagate(max_sweeps=3)
    Zo, amounts, w = O.propagate(X, X, rowptr.astype(np.int64), col, 0.76, 10, max_sweeps=3)
    S = g._device_state()
    assert np.array_equal(S.w[:S.e].cpu().numpy(), w)                    # P bit-exact
    assert np.array_equal(e.amounts_per_call[0], amounts)                # L1 amounts bit-exact
    Z = g.Z.numpy()
    assert within_tolerance(Z, Zo) and np.array_equal(Z, Zo)
    sinks = np.diff(rowptr) == 0
    assert np.array_equal(Z[sinks], X[sinks])                            # embedder.py:88-89


@pytest.mark.parametrize("n,d,hub_deg,tol", [(3000, 128, 900, 2), (3000, 64, 400, 2), (5000, 32, 300, 2), (3000, 100, 700, 2),
                                             (700, 500, 600, 1), (300, 1433, 290, 1), (140003, 128, 9000, 1)])
def test_hub_rows_and_fused_l1_against_oracle(n, d, hub_deg, tol, monkeypatch):
    """Power-law graphs with hub rows (shared-memory ring path), every d regime: fused L1
    (d = 32/64/128, level step 16 and 32), padded / multi-slab rows (100, 500, 1433)."""
    import clane_b200.graph as graph_module
    monkeypatch.setattr(graph_module, "HUB_THRESHOLD", 128)     # default is 1024: force the hub kernel on these sizes
    rng = np.random.default_rng(n + d)
    e = n * 6
    src, dst = synth.make_edges(n, e, "powerlaw", rng)
    hubs = rng.permutation(n)[:3]
    extra_src = np.repeat(hubs, [hub_deg, hub_deg // 2 + 3, 257])
    extra_dst = np.concatenate([rng.permutation(n)[:k] for k in (hub_deg, hub_deg // 2 + 3, 257)])
    src, dst = np.concatenate([src, extra_src]), np.concatenate([dst, extra_dst])
    X = rng.standard_normal((n, d), dtype=np.float32)
    g = Graph.from_arrays(n, src, dst, X)
    emb = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=0.76, tolerence=tol)
    emb.verbose = False
    emb.propagate(max_sweeps=4)
    S = g._device_state()
    assert S.plan.n_hub_rows >= 3 and S.plan.fused_l1 == (d in (32, 64, 128))
    assert (S.plan.n_fix_groups >= 3) == S.plan.fused_l1
    O.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, n)
    Zo, amounts, w = O.propagate(X, X, rowptr, col, 0.76, tol, max_sweeps=4)
    assert np.array_equal(S.w[:S.e].cpu().numpy(), w)
    assert np.array_equal(emb.amounts_per_call[0], amounts)
    assert np.array_equal(g.Z.numpy(), Zo)


def test_default_hub_threshold_long_rows_in_row_kernel():
    """Rows up to the default threshold (256 neighbours on a small graph) stay whole in the row kernel; longer
    rows take the segment + chain path.  Both against the oracle."""
    rng = np.random.default_rng(77)
    n, d = 6000, 128
    src, dst = synth.make_edges(n, n * 5, "powerlaw", rng)
    extra = [(5, 1500), (6, 1030), (900, 250), (901, 200), (902, 255), (4001, 129)]
    src = np.concatenate([src] + [np.full(k, r) for r, k in extra])
    dst = np.concatenate([dst] + [rng.permutation(n)[:k] for _, k in extra])
    X = rng.standard_normal((n, d), dtype=np.float32)
    g = Graph.from_arrays(n, src, dst, X)
    emb = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=0.76, tolerence=2)
    emb.verbose = False
    emb.propagate(max_sweeps=3)
    S = g._device_state()
    assert 2 <= S.plan.n_hub_rows <= 6 and S.plan.fused_l1
    O.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, n)
    Zo, amounts, w = O.propagate(X, X, rowptr, col, 0.76, 2, max_sweeps=3)
    assert np.array_equal(emb.amounts_per_call[0], amounts)
    assert np.array_equal(g.Z.numpy(), Zo)


def test_split_l1_reduction_matches_whole():
    """clane_l1_partial over disjoint node ranges + clane_l1_finish == clane_l1_diff (multi-GPU path)."""
    L = _lib.lib()
    rng = np.random.default_rng(9)
    for n, d in [(50000, 100), (169343, 128), (3000, 500), (10, 3)]:
        a = rng.standard_normal((n, d)).astype(np.float32)
        b = rng.standard_normal((n, d)).astype(np.float32)
        ld = L.clane_padded_ld(d)
        A = torch.zeros([n, ld], device="cuda"); A[:, :d] = torch.from_numpy(a).cuda()
        B = torch.zeros([n, ld], device="cuda"); B[:, :d] = torch.from_numpy(b).cuda()
        plan = _lib.Plan(n, 0, d)
        nodes = ctypes.c_int64()
        _lib.check(L.clane_cascade_shape(n * d, ctypes.byref(nodes), None))
        k = nodes.value
        parts = []
        cuts = [0, k // 3, k // 3, (2 * k) // 3 + (1 if k else 0), k]     # includes an empty range
        cuts = sorted(min(c, k) for c in cuts)
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            p1 = torch.zeros((k + 2) * 32, device="cuda")
            _lib.check(L.clane_l1_partial(plan.handle, A.data_ptr(), B.data_ptr(), lo, hi, p1.data_ptr(), _lib.stream_handle()))
            parts.append(p1)
        total = torch.stack(parts).sum(0)              # what an all-reduce(SUM) of disjoint slots gives
        out = torch.zeros(1, device="cuda")
        _lib.check(L.clane_l1_finish(plan.handle, A.data_ptr(), B.data_ptr(), total.data_ptr(), out.data_ptr(), 0, 0, 0,
                                     _lib.stream_handle()))
        assert np.float32(out.cpu().numpy()[0]) == O.l1_diff(a, b)


def test_full_convergence_cora_shape_counts_match_oracle():
    n, src, dst, X = synth.make_graph("cora", seed=0)
    g = Graph.from_arrays(n, src, dst, X)
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=0.76, tolerence=10)
    e.verbose = False
    e.iterate()
    O.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, n)
    Zo, spc, _ = O.iterate(X, rowptr, col, 0.76, 10)
    assert e.sweeps_per_call == spc.tolist()
    assert np.array_equal(g.Z.numpy(), Zo)


@pytest.mark.parametrize("shape", ["pubmed", "arxiv"])
def test_full_convergence_counts_match_oracle_at_baseline_shapes(shape):
    """Embedder.iterate() to convergence at BASELINE configs 3 and 4: per-call sweep counts, outer amounts and the
    final embeddings against the oracle (the CPU port needs ~10-60 s for these)."""
    n, src, dst, X = synth.make_graph(shape, seed=0)
    g = Graph.from_arrays(n, src, dst, X)
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=0.76, tolerence=10)
    e.verbose = False
    e.iterate()
    O.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, n)
    Zo, spc, oam = O.iterate(X, rowptr, col, 0.76, 10)
    assert e.sweeps_per_call == spc.tolist()
    assert e.minimum_amount_updated_Z == oam.min()
    Z = g.Z.numpy()
    assert within_tolerance(Z, Zo) and np.array_equal(Z, Zo)


def test_products_shape_full_size_against_oracle():
    """BASELINE config 5 at full size on one GPU (2.45 M nodes / 61.9 M edges / d = 100): CSR, P, the L1 amounts of
    two sweeps and Z, bit-exact against the oracle."""
    n, src, dst, X = synth.make_graph("products", seed=0)
    g = Graph.from_arrays(n, src, dst, X)
    O.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, n)
    assert g._nnz == 61859140 and np.array_equal(g._rowptr, rowptr) and np.array_equal(g._col, col)
    del src, dst
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=0.76, tolerence=10)
    e.verbose = False
    e.propagate(max_sweeps=2)
    S = g._device_state()
    assert S.plan.n_hub_rows >= 1 and not S.plan.fused_l1
    Zo, amounts, w = O.propagate(X, X, rowptr, col, 0.76, 10, max_sweeps=2)
    assert np.array_equal(S.w[:S.e].cpu().numpy(), w)
    assert np.array_equal(e.amounts_per_call[0], amounts)
    Z = g.Z.numpy()
    assert within_tolerance(Z, Zo) and np.array_equal(Z, Zo)


def test_adjacent_hub_rows_across_build_p_calls(monkeypatch):
    """Several short hub rows with consecutive ids (their chain scratch regions are neighbours), whole iterate():
    every propagate() call rebuilds P, so weights parked for one call must never leak into the next."""
    import clane_b200.graph as graph_module
    monkeypatch.setattr(graph_module, "HUB_THRESHOLD", 16)
    rng = np.random.default_rng(123)
    n, d = 400, 64
    src, dst = synth.make_edges(n, n * 3, "uniform", rng)
    ks = [17, 18, 19, 25, 33, 41, 23, 17]
    hub_src = np.concatenate([np.full(k, 100 + i) for i, k in enumerate(ks)])
    hub_dst = np.concatenate([rng.permutation(n)[:k] for k in ks])
    src, dst = np.concatenate([src, hub_src]), np.concatenate([dst, hub_dst])
    X = rng.standard_normal((n, d), dtype=np.float32)
    g = Graph.from_arrays(n, src, dst, X)
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=0.76, tolerence=2)
    e.verbose = False
    e.iterate()
    assert g._device_state().plan.n_hub_rows >= len(ks)
    rowptr, col = O.csr_from_edges(src, dst, n)
    Zo, spc, _ = O.iterate(X, rowptr, col, 0.76, 2)
    assert e.sweeps_per_call == spc.tolist() and len(spc) >= 3
    assert np.array_equal(g.Z.numpy(), Zo)


def while_launch_required() -> bool:
    """clane_sweeps(until_stop=1) must take the conditional-WHILE graph on a B200."""
    return torch.cuda.get_device_capability()[0] == 10


def test_sweeps_batches_equal_single_sweeps():
    """clane_sweeps (three rotating buffers, L1 tail of a sweep beside the next sweep's rows, at most one speculative sweep
    after the stop) against one clane_sweep call per sweep: same amounts, same count, same Z -- for a run that stops in
    the middle of a batch, for a bounded run, and through the conditional-WHILE launch."""
    L = _lib.lib()
    rng = np.random.default_rng(31)
    for n, d, tol in [(4000, 128, 2), (3000, 100, 1), (900, 500, 2)]:
        src, dst = synth.make_edges(n, n * 5, "powerlaw", rng)
        src = np.concatenate([src, np.full(400, 11)])           # one hub row
        dst = np.concatenate([dst, rng.permutation(n)[:400]])
        X = rng.standard_normal((n, d), dtype=np.float32)
        rowptr, col = O.csr_from_edges(src, dst, n)
        Zo, amounts, _ = O.propagate(X, X, rowptr, col, 0.76, tol)
        for mode in ("while", "batches", "bounded"):
            g = Graph.from_arrays(n, src, dst, X)
            S = g._device_state()
            g._build_P_device(similarity.CosineSimilarity())
            sh = S.stream.cuda_stream
            S.stream.wait_stream(torch.cuda.current_stream())
            cap = 5 if mode == "bounded" else 0
            _lib.check(L.clane_patience_reset(S.state.data_ptr(), tol, cap, sh))
            args = (S.plan.handle, S.X.data_ptr(), S.Zptrs, 1, S.rowptr.data_ptr(), S.col.data_ptr(), S.w.data_ptr(),
                    ctypes.c_float(float(np.float32(0.76))))
            S.Z[1].copy_(S.Z[0])
            if mode == "while":
                rc = L.clane_sweeps(*args, 0, 1, S.state.data_ptr(), S.log.data_ptr(), S.log_cap, sh)
                if rc == _lib.CLANE_EUNSUPPORTED and not while_launch_required():
                    continue
                assert rc == 0, rc
            else:
                for _ in range(-(-(len(amounts) + 2) // 7)):    # batches of 7: the rotation does not close, stops mid-batch
                    start = (1 + 7 * _) % 3
                    a2 = args[:3] + (start,) + args[4:]
                    _lib.check(L.clane_sweeps(*a2, 7, 0, S.state.data_ptr(), S.log.data_ptr(), S.log_cap, sh))
            S.stream.synchronize()
            st = _lib.Patience.from_buffer_copy(S.state.cpu().numpy().tobytes())
            want = 5 if mode == "bounded" else len(amounts)
            assert st.stop == 1 and st.sweeps == want, (mode, st.sweeps, want)
            assert np.array_equal(S.log[:want].cpu().numpy(), amounts[:want])
            if mode != "bounded":
                assert np.array_equal(S.Z[(1 + want) % 3][:n, :d].cpu().numpy(), Zo)


def test_norms_reduced_by_node_range_equal_whole():
    """clane_norms_partial over disjoint node ranges + a sum of the slots + clane_norms_finish == the norms of
    clane_scores_cosine (the multi-GPU build_P), and the plan's softmax == the row-range softmax."""
    L = _lib.lib()
    rng = np.random.default_rng(41)
    for n, d in [(5000, 128), (3000, 100), (200, 1433), (50, 3)]:
        src, dst = synth.make_edges(n, n * (6 if n >= 1000 else 2), "powerlaw" if n >= 1000 else "uniform", rng)
        X = rng.standard_normal((n, d), dtype=np.float32)
        g = Graph.from_arrays(n, src, dst, X)
        S = g._device_state()
        s = _lib.stream_handle()
        z = S.Z[0].data_ptr()
        dots = torch.zeros(S.e, device="cuda")
        norms = torch.zeros(2, device="cuda")
        _lib.check(L.clane_scores_cosine(S.plan.handle, z, S.erow.data_ptr(), S.col.data_ptr(), 0, S.e, dots.data_ptr(),
                                         norms.data_ptr(), s))
        nodes = ctypes.c_int64()
        _lib.check(L.clane_cascade_shape(S.e * d, ctypes.byref(nodes), None))
        k = nodes.value
        parts = []
        for lo, hi in [(0, k // 3), (k // 3, k // 3), (k // 3, k)]:
            p1 = torch.zeros((k + 2) * 64, device="cuda")
            _lib.check(L.clane_norms_partial(S.plan.handle, z, S.erow.data_ptr(), S.col.data_ptr(), lo, hi, p1.data_ptr(), s))
            parts.append(p1)
        total = torch.stack(parts).sum(0)
        norms2 = torch.zeros(2, device="cuda")
        _lib.check(L.clane_norms_finish(S.plan.handle, z, S.erow.data_ptr(), S.col.data_ptr(), total.data_ptr(),
                                        norms2.data_ptr(), s))
        assert np.array_equal(norms2.cpu().numpy(), norms.cpu().numpy())
        rowptr, col = O.csr_from_edges(src, dst, n)
        od, s1, s2 = O.scores_raw(X, rowptr, col)
        assert np.array_equal(dots.cpu().numpy(), od) and norms.cpu().numpy().tolist() == [s1, s2]
        w1, w2 = torch.zeros_like(dots), torch.zeros_like(dots)
        _lib.check(L.clane_plan_softmax(S.plan.handle, dots.data_ptr(), norms.data_ptr(), S.rowptr.data_ptr(), w1.data_ptr(), s))
        _lib.check(L.clane_row_softmax(dots.data_ptr(), norms.data_ptr(), 0, n, S.rowptr.data_ptr(), w2.data_ptr(), s))
        assert np.array_equal(w1.cpu().numpy(), w2.cpu().numpy())
        assert np.array_equal(w1.cpu().numpy(), O.build_p(X, rowptr, col))


@pytest.mark.parametrize("n,e,d", [(50, 3, 128), (50, 33, 128), (900, 4001, 128), (40000, 270003, 128), (700, 3001, 64),
                                   (30000, 530001, 64), (900, 5003, 32), (60000, 1050007, 32)])
def test_scores_cosine_every_norm_chunk_size(n, e, d):
    """clane_scores_cosine (the dots on a side stream beside the norm cascade) against the oracle at every level-0
    chunk size of the norm cascade (4 / 8 / 16 / 32 edges per chunk at d = 128 / 64 / 32), with partial last chunks
    and partial tiles of 32 edges."""
    L = _lib.lib()
    rng = np.random.default_rng(n + e + d)
    src, dst = synth.make_edges(n, e, "powerlaw" if n >= 900 else "uniform", rng)
    X = rng.standard_normal((n, d), dtype=np.float32)
    g = Graph.from_arrays(n, src, dst, X)
    S = g._device_state()
    assert S.e == e
    s = _lib.stream_handle()
    dots = torch.zeros(S.e, device="cuda")
    norms = torch.zeros(2, device="cuda")
    _lib.check(L.clane_scores_cosine(S.plan.handle, S.Z[0].data_ptr(), S.erow.data_ptr(), S.col.data_ptr(), 0, S.e,
                                     dots.data_ptr(), norms.data_ptr(), s))
    O.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, n)
    od, s1, s2 = O.scores_raw(X, rowptr, col)
    assert np.array_equal(dots.cpu().numpy(), od)
    assert norms.cpu().numpy().tolist() == [s1, s2]


@pytest.mark.parametrize("n,d", [(1000, 128), (300, 64), (4097, 32), (777, 96)])
def test_asymmetric_scorer_fused_build_p(n, d):
    """AsymmertricSimilarity through Graph.build_P: the tcgen05 projection + per-edge dots + row softmax against the
    fp32 torch module on gathered rows (what the reference's build_P would do with this plugin, graph.py:120-123).
    Tolerance: the tensor cores read TF32 inputs (10-bit mantissa) and accumulate in fp32 -- projected values within
    2e-3 of the row scale, scores within 1e-2 * |z|^2-scale, weights of P within 2e-3 absolute."""
    L = _lib.lib()
    torch.manual_seed(d)
    rng = np.random.default_rng(n + d)
    src, dst = synth.make_edges(n, n * 5, "powerlaw", rng)
    X = (rng.standard_normal((n, d)) * 0.5).astype(np.float32)
    g = Graph.from_arrays(n, src, dst, X)
    sim = similarity.AsymmertricSimilarity(n_dim=d)
    assert sim.is_trainable() and hasattr(sim, "parameters")
    # the projection alone, against fp32 matmul
    S = g._device_state()
    W = sim.stacked_weights(S.device)
    work = torch.zeros(2 * n * S.ld, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    _lib.check(L.clane_asym_project(S.Z[0].data_ptr(), n, d, S.ld, W.data_ptr(), work.data_ptr(), work[n * S.ld:].data_ptr(),
                                    err.data_ptr(), _lib.stream_handle()))
    assert int(err.item()) == 0
    P = work.view(2, n, S.ld)[:, :, :d].cpu().numpy()
    Xt = torch.from_numpy(X)
    want_src = (Xt @ sim.Phi_src.weight.detach().T).numpy()
    want_dst = (Xt @ sim.Phi_dst.weight.detach().T).numpy()
    scale = np.abs(want_src).max()
    assert np.abs(P[0] - want_src).max() <= 2e-3 * scale and np.abs(P[1] - want_dst).max() <= 2e-3 * scale
    # the whole build_P
    Pm = g.build_P(sim)
    rows, cols = g._coo_indices()
    with torch.no_grad():
        scores = sim(Xt[rows], Xt[cols]).numpy().astype(np.float32)
    want = O.softmax_rows(scores, g._rowptr.astype(np.int64))
    got = Pm.values().numpy()
    assert np.abs(got - want).max() <= 2e-3
    rs = Pm.to_dense().sum(1)
    assert abs(rs.max().item() - 1) < 1e-3
    # other widths fall back to the generic plugin path (scores by the module itself, softmax in CUDA)
    assert L.clane_asym_supported(100) == 0 and L.clane_asym_supported(128) == 1


@pytest.mark.parametrize("n,d", [(7, 1), (5, 3), (33, 5), (1000, 7)])
def test_value_finish_small_and_ragged(n, d):
    """n*d < 8 (ATen's scalar path), and ragged tails: the values the finish needs come from the 32-float buffer."""
    L = _lib.lib()
    rng = np.random.default_rng(n * 31 + d)
    a = rng.standard_normal((n, d)).astype(np.float32)
    b = rng.standard_normal((n, d)).astype(np.float32)
    ld = L.clane_padded_ld(d)
    A = torch.zeros([n, ld], device="cuda"); A[:, :d] = torch.from_numpy(a).cuda()
    B = torch.zeros([n, ld], device="cuda"); B[:, :d] = torch.from_numpy(b).cuda()
    plan = _lib.Plan(n, 0, d)
    nodes = ctypes.c_int64()
    _lib.check(L.clane_cascade_shape(n * d, ctypes.byref(nodes), None))
    k = nodes.value
    p1 = torch.zeros((k + 3) * 32, device="cuda")
    vals = p1[(k + 2) * 32:]
    s = _lib.stream_handle()
    _lib.check(L.clane_l1_partial(plan.handle, A.data_ptr(), B.data_ptr(), 0, k, p1.data_ptr(), s))
    _lib.check(L.clane_l1_tail_values(plan.handle, A.data_ptr(), B.data_ptr(), vals.data_ptr(), s))
    out = torch.zeros(1, device="cuda")
    _lib.check(L.clane_l1_finish_values(plan.handle, p1.data_ptr(), vals.data_ptr(), out.data_ptr(), 0, 0, 0, s))
    assert np.float32(out.cpu().numpy()[0]) == O.l1_diff(a, b)


@pytest.mark.parametrize("shape", ["cora", "arxiv"])
def test_bench_dump_outputs_are_the_timed_sweeps(shape, tmp_path):
    """bench.py --dump-outputs: the warm-up and timed sweeps are one sequence from Z = X, so Z after the last timed
    sweep and the L1 change of each timed sweep equal the oracle's propagate() of warmup + steps sweeps, bit-exact;
    arxiv's Z is larger than the dump's budget and is sampled."""
    import json
    import subprocess
    import sys
    steps = 7
    cmd = [sys.executable, str(ROOT / "bench.py"), "--workload", shape, "--steps", str(steps), "--warmup", "2",
           "--no-cpu-baseline", "--no-converge", "--dump-outputs", str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.split("\n") if ln.startswith("{")][-1])
    assert line["steps"] == steps and line["warmup"] >= 2
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    n, src, dst, X = synth.make_graph(shape, seed=0)
    O.set_threads(O.max_threads())
    rowptr, col = O.csr_from_edges(src, dst, n)
    Zo, amounts, _ = O.propagate(X, X, rowptr, col, 0.76, 1 << 30, max_sweeps=line["warmup"] + steps)
    amounts = amounts[-steps:]
    rows = np.load(tmp_path / "Z_rows.npy")
    assert rows.dtype == np.float64 and np.all(np.diff(rows) > 0)
    assert len(rows) == (n if shape == "cora" else 65536)
    Z = np.load(tmp_path / "Z.npy")
    assert Z.dtype == np.float32 and np.array_equal(Z, Zo[rows.astype(np.int64)])
    assert np.array_equal(np.load(tmp_path / "amounts.npy"), amounts) and len(amounts) == steps


def test_sharded_run_equals_single_gpu_when_two_gpus_are_present():
    """tools/check_dist.py under torchrun (2 ranks, fused peer-store exchange): bit-identical to the single-GPU
    run at four shapes.  Skipped on a one-GPU box."""
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", str(ROOT / "tools" / "check_dist.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("sharded == single-GPU: True") == 5
