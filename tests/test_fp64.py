"""float64 content embeddings on the GPU: the whole update in double, bit-exact with the fixtures of
tests/golden/make_golden_f64.py (the reference's hot path restated in torch) and with the fp64 oracle."""
import ctypes
from pathlib import Path

import numpy as np
import pytest
import torch

from clane_b200 import _lib, similarity, synth
from clane_b200.embedder import Embedder
from clane_b200.graph import Graph
from oracle_f64 import oracle_f64 as O
from tests.test_f64_host import _scratch_needed

F64 = Path(__file__).resolve().parent / "golden" / "f64"
CASES = sorted(p.stem for p in F64.glob("ref_*.npz"))

pytestmark = pytest.mark.gpu


def _write_root(root: Path, G) -> Path:
    ids = [str(x) for x in G["ids"]]
    root.mkdir(parents=True, exist_ok=True)
    (root / "V").write_text("\n".join(ids))
    (root / "E").write_text("\n".join(f"{ids[a]}\t{ids[b]}" for a, b in zip(G["raw_src"], G["raw_dst"])))
    np.save(root / "C.npy", G["X"])
    return root


def _csr(src, dst, n):
    idx = np.unique(np.stack([src, dst]).astype(np.int64), axis=1)
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(idx[0], minlength=n))]).astype(np.int64)
    return rowptr, idx[1].astype(np.int32)


@pytest.mark.parametrize("case", CASES)
def test_fixture_through_graph_and_embedder(case, tmp_path):
    G = np.load(F64 / f"{case}.npz")
    g = Graph(_write_root(tmp_path / "data", G), embedding_dim=int(G["d"]))
    assert g.X.dtype == torch.float64
    rows = np.repeat(np.arange(len(g)), np.diff(g._rowptr))
    assert np.array_equal(rows, G["A_indices"][0]) and np.array_equal(g._col, G["A_indices"][1])
    P = g.build_P(similarity.CosineSimilarity())
    assert P.values().dtype == torch.float64 and np.array_equal(P.values().numpy(), G["P0_values"])
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=float(G["gamma"]),
                 tolerence=int(G["tol"]))
    e.verbose = False
    e.iterate()
    assert e.sweeps_per_call == G["sweeps_per_call"].tolist()
    amounts = np.concatenate(e.amounts_per_call)
    assert amounts.dtype == np.float64 and np.array_equal(amounts, G["amounts"])
    assert e.minimum_amount_updated_Z == G["outer_amounts"].min()
    Z = g.Z
    assert Z.dtype == torch.float64 and np.array_equal(Z.numpy(), G["Z_final"])
    assert g.V[5].z.dtype == torch.float64 and np.array_equal(g.V[5].z.numpy(), G["Z_final"][5])


def test_amounts_print_as_float64(capsys):
    G = np.load(F64 / "ref_toy_d16.npz")
    g = Graph.from_arrays(int(G["n"]), G["raw_src"], G["raw_dst"], torch.from_numpy(G["X"]))
    Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=float(G["gamma"]),
             tolerence=int(G["tol"])).propagate()
    first = capsys.readouterr().out.strip().split("\n")[0]
    want = torch.tensor(G["amounts"][0])
    assert want.dtype == torch.float64 and first == f"{str(want)} {int(G['tol'])}"


@pytest.mark.parametrize("shape", ["cora", "pubmed", "arxiv"])
def test_shapes_against_oracle(shape):
    n, src, dst, X = synth.make_graph(shape, seed=3)
    X = X.astype(np.float64)
    g = Graph.from_arrays(n, src, dst, torch.from_numpy(X))
    rowptr, col = _csr(src, dst, n)
    assert np.array_equal(g._rowptr, rowptr) and np.array_equal(g._col, col)
    O.set_threads(8)
    Zo, amounts, w = O.propagate(X, X, rowptr, col, 0.76, 3, max_sweeps=3)
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=0.76, tolerence=3)
    e.verbose = False
    e.propagate(max_sweeps=3)
    assert np.array_equal(g._dev.w[:g._nnz].cpu().numpy(), w)
    assert np.array_equal(e.amounts_per_call[0], amounts)
    assert np.array_equal(g.Z.numpy(), Zo)
    # a whole propagate() from X stops on the same sweep
    g.set_Z(torch.from_numpy(X))
    e.propagate()
    _, amounts_full, _ = O.propagate(X, X, rowptr, col, 0.76, 3)
    assert e.sweeps_per_call[1] == len(amounts_full)
    assert np.array_equal(e.amounts_per_call[1], amounts_full)


@pytest.mark.parametrize("d", [1, 15, 100, 128, 500])
def test_long_rows(d):
    """Rows of 150,000, 20,003 and 16,383 neighbours are single serial chains per column."""
    n = 150_010
    rng = np.random.default_rng(d)
    src = [np.zeros(150_000, np.int64), np.ones(20_003, np.int64), np.full(16_383, 2, np.int64)]
    dst = [rng.permutation(n)[:150_000], rng.permutation(n)[:20_003], rng.permutation(n)[:16_383]]
    small = rng.integers(3, n, 3000)
    src.append(small)
    dst.append(rng.integers(0, n, 3000))
    src, dst = np.concatenate(src), np.concatenate(dst)
    X = rng.standard_normal((n, d))
    g = Graph.from_arrays(n, src, dst, torch.from_numpy(X))
    rowptr, col = _csr(src, dst, n)
    O.set_threads(8)
    Zo, amounts, w = O.propagate(X, X, rowptr, col, 0.76, 3, max_sweeps=2)
    e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=0.76, tolerence=3)
    e.verbose = False
    e.propagate(max_sweeps=2)
    assert np.array_equal(g._dev.w[:g._nnz].cpu().numpy(), w)
    assert np.array_equal(e.amounts_per_call[0], amounts)
    assert np.array_equal(g.Z.numpy(), Zo)


@pytest.mark.parametrize("n,e,d", [(65_536, 70_000, 128), (100_000, 80_000, 100)])
def test_scratch_at_shapes_straddling_a_cascade_step(n, e, d):
    """n*d and e*d on opposite sides of a cascade step change (2^19 rows of 16): the smaller reduction needs the
    larger scratch.  The sweeps' L1 (first case) or build_P's norms (second) must still use an adequate buffer."""
    rng = np.random.default_rng(n)
    src, dst = rng.integers(0, n, e + e // 50), rng.integers(0, n, e + e // 50)
    key = np.unique(src * n + dst)[:e]
    src, dst = key // n, key % n
    X = rng.standard_normal((n, d))
    g = Graph.from_arrays(n, src, dst, torch.from_numpy(X))
    rowptr, col = _csr(src, dst, n)
    assert g._nnz == e
    O.set_threads(8)
    Zo, amounts, w = O.propagate(X, X, rowptr, col, 0.76, 3, max_sweeps=3)
    e_ = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=0.76, tolerence=3)
    e_.verbose = False
    e_.propagate(max_sweeps=3)
    assert g._dev.work.numel() >= max(_scratch_needed(n * d), _scratch_needed(e * d))
    assert np.array_equal(g._dev.w[:g._nnz].cpu().numpy(), w)
    assert np.array_equal(e_.amounts_per_call[0], amounts)
    assert np.array_equal(g.Z.numpy(), Zo)


def test_batched_sweeps_equal_single_sweeps():
    """clane_sweeps_f64 (batches, no-ops after the stop) against one clane_sweep_f64 per call."""
    n, src, dst, X = synth.make_graph("cora", seed=5, scale=0.5)
    X = X.astype(np.float64)
    runs = []
    for history in (False, True):
        g = Graph.from_arrays(n, src, dst, torch.from_numpy(X))
        e = Embedder(g, similarity.CosineSimilarity(), device=torch.device("cuda"), gamma=0.76, tolerence=3,
                     save_history=history)
        e.verbose = False
        e.propagate()
        runs.append((e.sweeps_per_call[0], e.amounts_per_call[0], g.Z.numpy()))
        if history:
            assert len(e.history["Z"][0]) == e.sweeps_per_call[0]
            assert e.history["Z"][0][-1].dtype == torch.float64
            assert np.array_equal(e.history["Z"][0][-1].numpy(), runs[-1][2])
    assert runs[0][0] == runs[1][0]
    assert np.array_equal(runs[0][1], runs[1][1]) and np.array_equal(runs[0][2], runs[1][2])
    # the raw C-ABI: a batch longer than the call leaves the sweep count and the result buffer at the stop
    g = Graph.from_arrays(n, src, dst, torch.from_numpy(X))
    g.build_P(similarity.CosineSimilarity())
    S, L = g._dev, _lib.lib()
    s = _lib.stream_handle()
    _lib.check(L.clane_patience_reset_f64(S.state.data_ptr(), 3, 0, s))
    _lib.check(L.clane_sweeps_f64(S.n, S.d, S.rowptr.data_ptr(), S.col.data_ptr(), S.w.data_ptr(), S.X.data_ptr(),
                                  S.Zptrs, 0, ctypes.c_double(0.76), runs[0][0] + 7, S.state.data_ptr(),
                                  S.log.data_ptr(), S.log_cap, S.work.data_ptr(), s))
    st = _lib.Patience64.from_buffer_copy(S.state.cpu().numpy().tobytes())
    assert st.stop == 1 and st.sweeps == runs[0][0] and st.last_amount == runs[0][1][-1]
    assert np.array_equal(S.Z[st.sweeps % 3][:S.n, :S.d].cpu().numpy(), runs[0][2])


class DotPlugin(similarity.Similarity):
    """A user scorer: plain per-pair dot products."""

    def __call__(self, v1, v2):
        return (v1 * v2).sum(-1)


def test_user_plugin_scores_in_double():
    n, src, dst, X = synth.make_graph("pubmed", seed=2, scale=0.3)
    X = X.astype(np.float64)
    g = Graph.from_arrays(n, src, dst, torch.from_numpy(X))
    sim = DotPlugin()
    P = g.build_P(sim)
    S = g._dev
    Z = S.Z[S.cur][:S.n, :S.d]
    scores = sim(Z[S.erow[:S.e].long()], Z[S.col[:S.e].long()])
    assert scores.dtype == torch.float64
    assert np.array_equal(P.values().numpy(), O.softmax_rows(scores.cpu().numpy(), g._rowptr.astype(np.int64)))


def test_asymmetric_scorer_raises_torch_dtype_error():
    G = np.load(F64 / "ref_toy_d16.npz")
    g = Graph.from_arrays(int(G["n"]), G["raw_src"], G["raw_dst"], torch.from_numpy(G["X"]))
    with pytest.raises(RuntimeError, match="dtype"):
        g.build_P(similarity.AsymmertricSimilarity(int(G["d"])).cuda())


def test_fp16_still_raises():
    g = Graph.from_arrays(3, [0, 1], [1, 2], torch.zeros(3, 4, dtype=torch.float16))
    with pytest.raises(NotImplementedError):
        g.Z_device


def test_cli_writes_float64_Z(tmp_path):
    from clane_b200.__main__ import main
    G = np.load(F64 / "ref_hub60_d20.npz")
    root = _write_root(tmp_path / "data", G)
    cfg = tmp_path / "config.yaml"
    cfg.write_text(f'graph:\n  embedding_dim: {int(G["d"])}\n\nsimilarity:\n  method: "CosineSimilarity"\n  kwargs: {{}}\n\n'
                   f'embedder:\n  gamma: {float(G["gamma"])}\n  tolerence: {int(G["tol"])}\n')
    main(["--data_root", str(root), "--output_root", str(tmp_path / "out"), "--config_file", str(cfg)])
    Z = np.load(tmp_path / "out" / "Z.npy")
    assert Z.dtype == np.float64 and np.array_equal(Z, G["Z_final"])
