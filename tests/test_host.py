"""Host-side logic (no GPU): loader semantics of graph.py, CSR build, row schedule, the C-ABI
surface, CLI parser and plugin registry.  Known answers come from the reference's own tests
(tests/test_graph.py) and from the golden files."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from clane_b200 import _lib, similarity
from clane_b200.__main__ import get_parser
from clane_b200.graph import Graph
from oracle import oracle as O

ROOT = Path(__file__).resolve().parent.parent
GOLD = ROOT / "tests" / "golden"


def write_graph(root, ids, edges, X=None):
    root.mkdir(parents=True, exist_ok=True)
    (root / "V").write_text("\n".join(ids))
    (root / "E").write_text("\n".join(f"{a}\t{b}" for a, b in edges))
    if X is not None:
        np.save(root / "C.npy", X)


# ---- reference tests/test_graph.py restated ---------------------------------------------------
def test_load_zachary(data_root):
    g = Graph(data_root=data_root, embedding_dim=16)
    assert len(g.vertex_ids) == 34 and len(g.V) == 34 and len(g.E) == 78 and len(g) == 34
    for v in g.V:
        assert isinstance(v.x, torch.Tensor) and v.x.shape[-1] == 16


def test_build_A_and_neighbour_kat(data_root):
    g = Graph(data_root=data_root, embedding_dim=16)
    assert g.A.shape[0] == 34 and g.A.shape[1] == 34
    assert g.get_nbrs(33).tolist() == [8, 9, 13, 14, 15, 18, 19, 20, 22, 23, 26, 27, 28, 29, 30, 31, 32]
    for v in g.V:
        nb = g.get_nbrs(v.idx)
        assert nb.dim() == 1 and nb.dtype == torch.int64


def test_same_random_features_as_reference(data_root):
    G = np.load(GOLD / "ref_toy_d2.npz")
    torch.manual_seed(int(G["seed"]))
    g = Graph(data_root=data_root, embedding_dim=2)
    assert np.array_equal(g.X.numpy(), G["X"])          # graph.py:56: identical torch.normal call
    assert np.array_equal(g.A.indices().numpy(), G["A_indices"])


# ---- loader semantics (graph.py:44-45, :73-81) ---------------------------------------------------
def test_first_occurrence_wins_and_coalesce(tmp_path):
    ids = ["a", "b", "a", "c"]                            # duplicate id: index() finds position 0
    write_graph(tmp_path, ids, [("a", "b"), ("c", "a"), ("a", "b"), ("b", "b"), ("c", "c")],
                np.zeros((4, 3), np.float32))
    g = Graph(tmp_path, 3)
    assert len(g) == 4 and len(g.E) == 5                 # raw count keeps duplicates and self-loops
    assert g.A._nnz() == 4                               # (0,1) merged; self-loops kept
    assert g.A.values().tolist() == [2.0, 1.0, 1.0, 1.0]
    assert g.get_nbrs(0).tolist() == [1] and g.get_nbrs(1).tolist() == [1]
    assert g.get_nbrs(2).tolist() == [] and g.get_nbrs(3).tolist() == [0, 3]
    assert g.V[0].outgoing_indices == [1, 1] and g.V[1].incoming_indices == [0, 0, 1]
    assert g.E[1].src.idx == 3 and g.E[1].dst.idx == 0


def test_loader_errors(tmp_path):
    with pytest.raises(FileNotFoundError):
        Graph(tmp_path / "missing", 4)
    write_graph(tmp_path / "noE", ["a", "b"], [("a", "b")])
    (tmp_path / "noE" / "E").unlink()
    with pytest.raises(FileNotFoundError):
        Graph(tmp_path / "noE", 4)
    write_graph(tmp_path / "bad", ["a", "b"], [("a", "b")])
    (tmp_path / "bad" / "E").write_text("a b")           # no tab
    with pytest.raises(ValueError):
        Graph(tmp_path / "bad", 4)
    (tmp_path / "bad" / "E").write_text("a\tb\tc")       # two tabs
    with pytest.raises(ValueError):
        Graph(tmp_path / "bad", 4)
    (tmp_path / "bad" / "E").write_text("a\tzzz")        # unknown id
    with pytest.raises(ValueError):
        Graph(tmp_path / "bad", 4)
    (tmp_path / "bad" / "E").write_text("")              # empty file: the reference fails to unpack
    with pytest.raises(ValueError):
        Graph(tmp_path / "bad", 4)


def test_feature_file_precedence(tmp_path):
    X = np.arange(6, dtype=np.float32).reshape(2, 3)
    write_graph(tmp_path, ["a", "b"], [("a", "b")], X)
    g = Graph(tmp_path, 99)                              # C.npy wins over embedding_dim (graph.py:51)
    assert np.array_equal(g.X.numpy(), X) and g.V[1].x.tolist() == [3.0, 4.0, 5.0]
    (tmp_path / "C.npy").unlink()
    torch.save(torch.from_numpy(X) + 1, tmp_path / "C.pt")
    assert np.array_equal(Graph(tmp_path, 99).X.numpy(), X + 1)


def test_vertex_z_assignment_on_the_host(data_root):
    """`v.z = ...` (embedder.py:92, graph.py:138) before any device state exists: z stops aliasing x."""
    g = Graph(data_root=data_root, embedding_dim=4)
    x3 = g.X[3].clone()
    g.V[3].z = torch.full([4], 7.0)
    assert torch.equal(g.V[3].z, torch.full([4], 7.0)) and torch.equal(g.V[3].x, x3)
    assert torch.equal(g.Z[3], torch.full([4], 7.0)) and torch.equal(g.Z[4], g.X[4])


def test_dataset_protocol(data_root):
    g = Graph(data_root=data_root, embedding_dim=4)
    assert g[5] == 5
    g.dispense_pair = True
    idx, other, is_nbr = g[33]
    assert idx == 33 and 0 <= other < 34 and isinstance(is_nbr, bool)


# ---- CSR build and schedule (C-ABI host functions) vs the oracle / golden --------------------------
@pytest.mark.parametrize("case", sorted(p.stem for p in GOLD.glob("ref_*.npz")))
def test_csr_bit_exact_with_reference(case):
    G = np.load(GOLD / f"{case}.npz")
    n = int(G["n"])
    g = Graph.from_arrays(n, G["raw_src"], G["raw_dst"], G["X"])
    rows = np.repeat(np.arange(n), np.diff(g._rowptr))
    assert np.array_equal(rows, G["A_indices"][0]) and np.array_equal(g._col, G["A_indices"][1])
    assert g._rowptr.dtype == np.int32 and g._col.dtype == np.int32
    for v in (0, n // 2, n - 1):
        a, b = G["nbr_ptr"][v], G["nbr_ptr"][v + 1]
        assert g.get_nbrs(v).tolist() == G["nbr_idx"][a:b].tolist()


def test_csr_random_multigraph_vs_oracle():
    rng = np.random.default_rng(7)
    n, e = 500, 20000
    src, dst = rng.integers(0, n, e), rng.integers(0, n, e)
    g = Graph.from_arrays(n, src, dst, np.zeros((n, 4), np.float32))
    rowptr, col = O.csr_from_edges(src, dst, n)
    assert np.array_equal(g._rowptr, rowptr) and np.array_equal(g._col, col)
    assert g._nnz == len(np.unique(src * n + dst))


def test_csr_rejects_out_of_range():
    L = _lib.lib()
    src, dst = np.array([0, 5], np.int64), np.array([1, 1], np.int64)
    rowptr, col = np.zeros(4, np.int32), np.zeros(2, np.int32)
    assert L.clane_csr_from_edges(src.ctypes.data, dst.ctypes.data, 2, 3, rowptr.ctypes.data, col.ctypes.data) == -2
    with pytest.raises(_lib.ClaneError):
        Graph.from_arrays(3, src, dst, np.zeros((3, 2), np.float32))


def group_schedule(rowptr, n, d, lo, hi, hub=128, span_edges=128):
    L = _lib.lib()
    cap = hi - lo + 1
    sr, sm, fx, hr = (np.zeros(cap, np.int32) for _ in range(4))
    ns, nf, nhr, G, fu = (ctypes.c_int32() for _ in range(5))
    _lib.check(L.clane_group_schedule(rowptr.ctypes.data, n, d, lo, hi, hub, span_edges, sr.ctypes.data, sm.ctypes.data,
                                      ctypes.byref(ns), fx.ctypes.data, ctypes.byref(nf), hr.ctypes.data,
                                      ctypes.byref(nhr), ctypes.byref(G), ctypes.byref(fu)))
    return sr[:ns.value], sm[:ns.value], fx[:nf.value], hr[:nhr.value], G.value, bool(fu.value)


def test_group_schedule_degree_sorted_row_blocks():
    rng = np.random.default_rng(3)
    n = 2003
    deg = np.minimum((rng.pareto(1.0, n) * 3).astype(np.int64), n - 1)
    deg[:5] = [0, 1, 33, 257, 1500]
    deg[64:80] = 0                                    # two whole groups of sinks
    deg[96:104] = [0, 0, 0, 300, 0, 0, 0, 0]          # a group whose only non-sink row is a hub
    deg[200:208] = [100, 100, 20, 5, 90, 90, 0, 120]  # a group that must be cut into several spans
    src = np.repeat(np.arange(n), deg)
    dst = np.concatenate([rng.permutation(n)[:k] for k in deg])
    g = Graph.from_arrays(n, src, dst, np.zeros((n, 4), np.float32))
    k = np.diff(g._rowptr)
    hub, budget = 128, 128
    for d, lo, hi in [(100, 0, n), (128, 0, n), (128, 500, 1700), (1433, 0, n)]:
        sr, sm, fx, hr, G, fused = group_schedule(g._rowptr, n, d, lo, hi, hub, budget)
        assert fused == (d == 128 and lo == 0 and hi == n)
        assert G == (4 if fused else 8)               # n*d < 2^24: level step 16 -> 512-element chunks
        nrows, direct = sm & 0xff, sm >> 8
        kk = np.where(k > hub, 0, k)                  # hub rows are not part of a span's work
        work = np.array([kk[r:r + m].sum() for r, m in zip(sr, nrows)])
        assert np.all(work > 0) and np.all(np.diff(work) <= 0)                        # longest first, no empty span
        assert np.all(np.diff(sr)[np.diff(work) == 0] > 0)                            # equal spans stay in row order (stable)
        covered = np.zeros(n, bool)
        for r, m, w_, dr in zip(sr, nrows, work, direct):
            assert (r - lo) // G == (r + m - 1 - lo) // G                              # a span stays inside one group
            assert not covered[r:r + m].any()
            covered[r:r + m] = True
            assert w_ <= budget or (kk[r:r + m] > 0).sum() == 1 or kk[r:r + m - 1].sum() + 0 <= budget
            if dr:                                                                      # whole group, no hub row
                g0 = lo + (r - lo) // G * G
                assert r == g0 and m == min(G, hi - g0) and k[r:r + m].max() <= hub
        ordinary = (k > 0) & (k <= hub)
        ordinary[:lo] = False
        ordinary[hi:] = False
        assert np.all(covered[ordinary])                                                # every ordinary row is swept
        want_hr = [v for v in range(lo, hi) if k[v] > hub]
        assert sorted(hr.tolist()) == want_hr and np.all(np.diff(k[hr]) <= 0)
        if fused:
            ng = (hi - lo + G - 1) // G
            nd = np.zeros(ng, int)
            for r, dr in zip(sr, direct):
                nd[(r - lo) // G] += 1
            has_hub = np.array([k[lo + i * G: min(lo + (i + 1) * G, hi)].max() > hub for i in range(ng)])
            is_direct = np.zeros(ng, bool)
            is_direct[[(r - lo) // G for r, dr in zip(sr, direct) if dr]] = True
            assert fx.tolist() == np.nonzero(((nd > 0) | has_hub) & ~is_direct)[0].tolist()
        else:
            assert len(fx) == 0
    sr, sm, fx, hr, G, fused = group_schedule(g._rowptr, n, 100, 0, n, hub, budget)
    rows200 = sorted((int(r), int(m & 0xff)) for r, m in zip(sr, sm) if 200 <= r < 208)
    assert rows200 == [(200, 1), (201, 3), (204, 1), (205, 2), (207, 1)]
    # a graph large enough for level step 32: 1024-element chunks = 8 rows of 128
    rp = np.zeros(140001, np.int32)
    assert group_schedule(rp, 140000, 128, 0, 140000)[4:] == (8, True)
    assert group_schedule(rp, 140000, 64, 0, 140000)[4:] == (8, True)      # 8.96M elements: step 16, 512 / 64
    assert group_schedule(rp, 140000, 100, 0, 140000)[4:] == (8, False)


@pytest.mark.parametrize("d", [32, 64, 128])
def test_group_schedule_fused_group_size_at_the_level_step_boundaries(d):
    """A fused group is one level-0 chunk of the L1 cascade over n*d (32 * level step elements): the step goes from
    16 to 32 above n*d = 2^24 and from 32 to 64 above 2^28, where the chunk outgrows a warp's 1024 floats and fusion
    turns off."""
    for elems, G, fused in [(1 << 24, 512 // d, True), ((1 << 24) + d, 1024 // d, True),
                            (1 << 28, 1024 // d, True), ((1 << 28) + d, 8, False)]:
        n = elems // d
        assert group_schedule(np.zeros(n + 1, np.int32), n, d, 0, n)[4:] == (G, fused), (n, d)


def test_group_schedule_direct_32_row_spans():
    """d = 32 above 2^24 elements: 32-row groups, and a low-degree graph sweeps every group as one direct span --
    lane 31 of the warp holds a row of its own."""
    rng = np.random.default_rng(17)
    n, d = 600000, 32
    rowptr = np.concatenate([[0], np.cumsum(rng.integers(1, 5, n))]).astype(np.int32)
    sr, sm, fx, hr, G, fused = group_schedule(rowptr, n, d, 0, n, 256)
    assert (G, fused) == (32, True) and len(fx) == 0 and len(hr) == 0
    assert np.array_equal(np.sort(sr), np.arange(0, n, 32)) and np.all(sm == 32 | (1 << 8))
    tasks = sweep_program(rowptr, n, d, 0, n, 256)
    assert len(tasks) == n // 32 and np.all(tasks[:, 3] == 32 | (1 << 8))
    for t in tasks[::997]:
        _, direct, out = emulate_task(t, rowptr)
        assert direct and [r for r, _ in out] == list(range(t[2], t[2] + 32))
        assert out[31][1] == list(range(rowptr[t[2] + 31], rowptr[t[2] + 32]))


def test_cascade_shape():
    L = _lib.lib()
    nodes, per = ctypes.c_int64(), ctypes.c_int64()
    _lib.check(L.clane_cascade_shape(169343 * 128, ctypes.byref(nodes), ctypes.byref(per)))
    assert (nodes.value, per.value) == (662, 32768)
    _lib.check(L.clane_cascade_shape(2708 * 1433, ctypes.byref(nodes), ctypes.byref(per)))
    assert (nodes.value, per.value) == (474, 8192)


# ---- C-ABI surface -------------------------------------------------------------------------------
def test_library_exports_every_declared_symbol():
    header = (ROOT / "include" / "clane_b200.h").read_text()
    declared = set(re.findall(r"\b(clane_[a-z0-9_]+)\s*\(", header))
    declared -= {"clane_patience", "clane_plan", "clane_session"}
    assert len(declared) >= 20
    L = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in declared:
        assert hasattr(L, name), f"{name} declared in clane_b200.h but not exported"
    assert declared == set(_lib.SIGNATURES), "ctypes binding out of sync with the header"
    assert ctypes.sizeof(_lib.Patience) == 32
    assert _lib.lib().clane_version() >= 100
    assert _lib.lib().clane_padded_ld(1433) == 1436 and _lib.lib().clane_padded_ld(128) == 128
    assert b"invalid argument" in _lib.lib().clane_error_string(-1)


def test_kernel_entry_points_reject_bad_arguments_without_a_device():
    L = _lib.lib()
    assert L.clane_sweep(0, 0, 0, 0, 0, 0, 0, 0.5, 0, 0, 0, 0, 0) == -1
    assert L.clane_row_softmax(0, 0, 0, 1, 0, 0, 0) == -1
    assert L.clane_scores_cosine(0, 0, 0, 0, 0, 1, 0, 0, 0) == -1
    assert L.clane_l1_diff(0, 0, 0, 0, 0) == -1 and L.clane_plan_info(0, None, None, None, None, None, None) == -1
    assert L.clane_plan_destroy(0) == 0
    assert L.clane_group_schedule(0, 1, 1, 0, 1, 128, 128, 0, 0, None, 0, None, 0, None, None, None) == -1


def test_no_cpu_fallback_without_cuda(data_root):
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    g = Graph(data_root=data_root, embedding_dim=4)
    with pytest.raises(_lib.ClaneError):
        g.build_P(similarity.CosineSimilarity())
    with pytest.raises(_lib.ClaneError):
        similarity.CosineSimilarity()(torch.ones(3), torch.ones(3))


def test_product_never_imports_the_oracle():
    for py in (ROOT / "clane_b200").rglob("*.py"):
        text = py.read_text()
        assert "import oracle" not in text and "from oracle" not in text, py
    for src in (ROOT / "clane_b200" / "csrc").iterdir():
        assert "oracle" not in src.read_text().lower(), src


# ---- CLI / registry ------------------------------------------------------------------------------
def test_cli_flags_match_reference():
    args = get_parser().parse_args(["--data_root", "a", "--output_root", "b", "--config_file", "c.yaml",
                                    "--save_history", "--num_workers", "3", "--gpu"])
    assert args.data_root == Path("a") and args.output_root == Path("b") and args.config_file == Path("c.yaml")
    assert args.save_history and args.gpu and args.num_workers == 3
    d = get_parser().parse_args([])
    assert d.num_workers == 0 and not d.save_history and not d.gpu


def test_plugin_registry():
    assert hasattr(similarity, "CosineSimilarity") and hasattr(similarity, "AsymmertricSimilarity")
    sim = similarity.CosineSimilarity(foo="bar")        # kwargs swallowed (tests/config.yaml:6-7)
    assert not sim.is_trainable() and not hasattr(sim, "parameters")
    assert similarity.AsymmertricSimilarity(n_dim=2).is_trainable()
    from clane.graph import Graph as AliasGraph         # the drop-in alias package
    from clane.embedder import Embedder, IterativeEmbedder  # noqa: F401
    from clane.__main__ import embedding, get_parser as gp  # noqa: F401
    assert AliasGraph is Graph


def test_cli_missing_config_and_unknown_method(tmp_path, data_root):
    from clane_b200.__main__ import embedding
    args = get_parser().parse_args(["--data_root", str(data_root), "--output_root", str(tmp_path / "o"),
                                    "--config_file", str(tmp_path / "nope.yaml")])
    with pytest.raises(FileNotFoundError):
        embedding(args)
    cfg = tmp_path / "c.yaml"
    cfg.write_text('graph:\n  embedding_dim: 2\nsimilarity:\n  method: "Nope"\n  kwargs: {}\nembedder: {}\n')
    args = get_parser().parse_args(["--data_root", str(data_root), "--output_root", str(tmp_path / "o"),
                                    "--config_file", str(cfg)])
    with pytest.raises(AttributeError, match="Given similarity method Nope not found."):
        embedding(args)


# ---------------------------------------------------------------------------------------------
# the sweep kernel's task list: a host emulation of k_sweep_rows' control flow (run_span / run_segment in sweep.cuh)
# ---------------------------------------------------------------------------------------------
def sweep_program(rowptr, n, d, lo, hi, hub, span_edges=128):
    L = _lib.lib()
    nt = ctypes.c_int64()
    _lib.check(L.clane_sweep_program(rowptr.ctypes.data, n, d, lo, hi, hub, span_edges, 0, 0, ctypes.byref(nt)))
    tasks = np.zeros((max(nt.value, 1), 8), np.int32)
    _lib.check(L.clane_sweep_program(rowptr.ctypes.data, n, d, lo, hi, hub, span_edges, tasks.ctypes.data, nt.value,
                                     ctypes.byref(nt)))
    assert L.clane_sweep_program(rowptr.ctypes.data, n, d, lo, hi, hub, span_edges, tasks.ctypes.data, nt.value - 1,
                                 ctypes.byref(nt)) == (-3 if nt.value else 0)
    return tasks[:nt.value]


def emulate_task(task, rowptr):
    """Walk one task exactly as a warp of k_sweep_rows does, with edge ids instead of data.  Returns
    (segment, direct, [(row or scratch block, [edge ids in reduction order])])."""
    e_first, e_total, r0, flags, nb, blk_base, nblk_row, _ = (int(x) for x in task)
    segment, direct, nrows = bool(flags & 512), bool(flags & 256), flags & 0xff
    if segment:        # whole (offset, w) stream in the window, batches of 8 in order
        assert e_total <= 128 and e_total == 8 * nb and r0 + nb <= nblk_row
        return True, False, [(blk_base + r0 + b, list(range(e_first + 8 * b, e_first + 8 * b + 8))) for b in range(nb)]
    # span: lane l takes the degree of row r0 + l from rowptr[r0 + min(l, nrows)] and rowptr[r0 + min(l + 1, nrows)]
    # (lanes past the span: 0), a 128-entry window of the edge stream, restaged when a batch starts at its end (only a
    # single row longer than the window gets there)
    assert 1 <= nrows <= 32 and e_first == rowptr[r0] and e_total == rowptr[r0 + nrows] - e_first
    lane_deg = [int(rowptr[r0 + min(lane + 1, nrows)] - rowptr[r0 + min(lane, nrows)]) for lane in range(32)]
    nonsink = sum(1 for r in range(nrows) if rowptr[r0 + r + 1] > rowptr[r0 + r])
    assert e_total <= 128 or nonsink == 1          # a row longer than the window is the only row with edges in its span
    state = [e_first, e_total]
    window = list(range(e_first, e_first + min(e_total, 128)))
    mpos, out = 0, []

    def batch(m):
        nonlocal mpos, window
        if mpos == 128:
            state[0] += 128
            state[1] -= 128
            assert state[1] > 0
            window = list(range(state[0], state[0] + min(state[1], 128)))
            mpos = 0
        assert mpos + m <= len(window), "batch runs past the staged window"
        got = window[mpos:mpos + m]
        mpos += m
        return got

    for r in range(nrows):
        k = lane_deg[r]
        if k == 0:
            continue
        cur = []
        while k >= 8:
            cur += batch(8)
            k -= 8
        if k:
            cur += batch(k)
        out.append((r0 + r, cur))
    return False, direct, out


@pytest.mark.parametrize("d,lo,hi,hub", [(128, 0, 2003, 128), (100, 0, 2003, 64), (128, 500, 1700, 128), (7, 0, 2003, 1 << 20)])
def test_sweep_program_covers_every_edge_in_order(d, lo, hi, hub):
    rng = np.random.default_rng(5)
    n = 2003
    deg = np.minimum((rng.pareto(1.0, n) * 3).astype(np.int64), n - 1)
    deg[:6] = [0, 1, 33, 257, 1500, 2002]
    deg[64:80] = 0
    deg[96:104] = [0, 0, 0, 300, 0, 0, 0, 0]
    deg[200:208] = [100, 100, 20, 5, 90, 90, 0, 120]
    deg[300:308] = [7, 8, 9, 15, 16, 17, 1, 2]
    src = np.repeat(np.arange(n), deg)
    dst = np.concatenate([rng.permutation(n)[:k] for k in deg])
    g = Graph.from_arrays(n, src, dst, np.zeros((n, 4), np.float32))
    rowptr = g._rowptr
    k = np.diff(rowptr)
    tasks = sweep_program(rowptr, n, d, lo, hi, hub)
    sr, sm, fx, hr, G, fused = group_schedule(rowptr, n, d, lo, hi, hub, 128)
    seen_rows, seen_blocks, n_seg = {}, {}, 0
    work = []
    for t in tasks:
        segment, direct, out = emulate_task(t, rowptr)
        work.append((not segment, -int(t[1])))
        if segment:
            n_seg += 1
            for blk, edges in out:
                assert blk not in seen_blocks
                seen_blocks[blk] = edges
        else:
            assert direct == (fused and any(int(r) == int(t[2]) and (m >> 8) for r, m in zip(sr, sm)))
            for row, edges in out:
                assert row not in seen_rows
                seen_rows[row] = edges
    spans_only = [w_ for w_ in work if w_[0]]
    assert work[len(work) - len(spans_only):] == spans_only == sorted(spans_only)   # segments first, spans by edge count
    for v in range(lo, hi):
        if 0 < k[v] <= hub:
            assert seen_rows[v] == list(range(rowptr[v], rowptr[v + 1]))
        else:
            assert v not in seen_rows
    # hub rows: their full 8-blocks, rows in degree-descending order, every row's scratch starting at an even block
    blk, nblocks = 0, 0
    for v in hr:
        for b in range(k[v] // 8):
            assert seen_blocks[blk + b] == list(range(rowptr[v] + 8 * b, rowptr[v] + 8 * b + 8))
        nblocks += k[v] // 8
        blk += (k[v] // 8 + 1) & ~1
    assert nblocks == len(seen_blocks)
    assert n_seg == sum(-(-(k[v] // 8) // 16) for v in hr)


# ---------------------------------------------------------------------------------------------
# native edge-file ingest (clane_edges_open) against the reference's own parsing expression
# ---------------------------------------------------------------------------------------------
def reference_parse(data_root):
    """graph.py:44-45 and :73-81 of the reference, verbatim semantics (list.index replaced by a first-position
    dict, which returns the same positions)."""
    with open(data_root / "V", "r") as io:
        vertex_ids = io.read().strip().split("\n")
    with open(data_root / "E", "r") as io:
        lines = io.read().strip().split("\n")
    first = {}
    for i, vid in enumerate(vertex_ids):
        first.setdefault(vid, i)
    src, dst = [], []
    for line in lines:
        src_id, dst_id = line.split("\t")
        for k, out in ((src_id, src), (dst_id, dst)):
            if k not in first:
                raise ValueError(f"{k!r} is not in list")
            out.append(first[k])
    return vertex_ids, np.array(src, np.int64), np.array(dst, np.int64)


def _write(tmp_path, v_bytes, e_bytes):
    (tmp_path / "V").write_bytes(v_bytes)
    (tmp_path / "E").write_bytes(e_bytes)
    np.save(tmp_path / "C.npy", np.zeros((len(v_bytes.decode().strip().split("\n")), 4), np.float32))
    return tmp_path


@pytest.mark.parametrize("v,e", [
    (b"a\nb\nc\n", b"a\tb\nb\tc\nc\ta\n"),
    (b"a\nb\nc", b"\n\n  a\tb\r\nb\tc\rc\ta\r\n\r\n"),                  # CRLF, lone CR, surrounding whitespace
    (b"x y\n\nz\nx y\n", b"x y\tz\n\tz\nz\t\nz\tx y\n"),                          # ids with spaces, the empty id, a repeated id
    ("é\n日本\nq\n".encode(), "日本\té\nq\t日本".encode()),                 # non-ASCII ids
    (b"0\n1\n2\n3\n", b"0\t1\n0\t1\n2\t2\n3\t0"),                         # duplicates and a self-loop are kept
])
def test_native_edge_ingest_matches_reference_expression(tmp_path, v, e):
    root = _write(tmp_path, v, e)
    ids, src, dst = reference_parse(root)
    g = Graph(root, 4)
    assert g.vertex_ids == ids and len(g.E) == len(src)
    assert np.array_equal(g._raw_src, src) and np.array_equal(g._raw_dst, dst)


@pytest.mark.parametrize("e,msg", [
    (b"a\tb\nab\nb\tc", "not enough values to unpack (expected 2, got 1)"),
    (b"a\tb\tc\nzz\tq", "too many values to unpack (expected 2)"),       # the FIRST bad line wins
    (b"a\tb\n\nb\tc", "not enough values to unpack (expected 2, got 1)"),  # a blank line in the middle
    (b"", "not enough values to unpack (expected 2, got 1)"),              # an empty E file, as upstream
    (b"a\tb\nb\tzz\nyy\ta", "'zz' is not in list"),
    (b"qq\tzz", "'qq' is not in list"),                                   # src is looked up before dst
])
def test_native_edge_ingest_errors_like_the_reference(tmp_path, e, msg):
    root = _write(tmp_path, b"a\nb\nc\n", e)
    with pytest.raises(ValueError) as ref:
        reference_parse(root)
    assert str(ref.value) == msg
    with pytest.raises(ValueError) as ours:
        Graph(root, 4)
    assert str(ours.value) == msg


def test_native_edge_ingest_large_file_many_pieces(tmp_path):
    """~3 MB of edges: cut into one piece per host thread; mixed line terminators across the cuts."""
    rng = np.random.default_rng(11)
    n, e = 5000, 200000
    ids = [f"node-{i * 7919 % 100003}" for i in range(n)]
    src, dst = rng.integers(0, n, e), rng.integers(0, n, e)
    term = np.array(["\n", "\r\n", "\r"])[rng.integers(0, 3, e)]
    body = "".join(f"{ids[a]}\t{ids[b]}{t}" for a, b, t in zip(src, dst, term))
    root = _write(tmp_path, ("\n".join(ids) + "\n").encode(), body.encode())
    _, rs, rd = reference_parse(root)
    g = Graph(root, 4)
    assert np.array_equal(g._raw_src, rs) and np.array_equal(g._raw_dst, rd) and np.array_equal(rs, src)
    # an unknown id deep inside the file: same error, whichever thread finds it
    bad = body.replace(f"{ids[src[150000]]}\t{ids[dst[150000]]}", f"{ids[src[150000]]}\tnope", 1)
    (tmp_path / "E").write_bytes(bad.encode())
    with pytest.raises(ValueError, match="'nope' is not in list"):
        Graph(root, 4)


def test_native_edge_ingest_missing_file(tmp_path):
    (tmp_path / "V").write_bytes(b"a\nb\n")
    np.save(tmp_path / "C.npy", np.zeros((2, 4), np.float32))
    with pytest.raises(FileNotFoundError):
        Graph(tmp_path, 4)
    L = _lib.lib()
    h, n, line = ctypes.c_void_p(), ctypes.c_int64(), ctypes.c_int64()
    err = ctypes.create_string_buffer(256)
    assert L.clane_edges_open(b"a\nb", 3, 2, str(tmp_path / "E").encode(), 0, ctypes.byref(h), ctypes.byref(n),
                              ctypes.byref(line), err, 256) == -5
    assert err.value.decode().endswith("/E")


def test_csr_build_is_thread_count_independent():
    """The two-level counting sort gives torch.coalesce()'s order whatever the number of host threads, on a skewed
    multigraph with duplicates, self-loops, empty rows and more buckets than rows per bucket."""
    import os
    L = _lib.lib()
    rng = np.random.default_rng(8)
    n, e = 70001, 400000
    src = (n * rng.random(e) ** 3).astype(np.int64)           # heavy head
    dst = rng.integers(0, n, e)
    src[:5000], dst[:5000] = src[5000:10000], dst[5000:10000]  # duplicates
    dst[10000:10100] = src[10000:10100]                        # self-loops
    key = np.unique(src * n + dst)
    want_rp = np.searchsorted(key // n, np.arange(n + 1)).astype(np.int32)
    want_col = (key % n).astype(np.int32)
    have = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    try:
        for k in (1, 2, 3, len(have) if have else 1):
            if have:
                os.sched_setaffinity(0, set(sorted(have)[:k]))
            rp, col = np.zeros(n + 1, np.int32), np.zeros(e, np.int32)
            E = L.clane_csr_from_edges(src.ctypes.data, dst.ctypes.data, e, n, rp.ctypes.data, col.ctypes.data)
            assert E == len(key) and np.array_equal(rp, want_rp) and np.array_equal(col[:E], want_col)
    finally:
        if have:
            os.sched_setaffinity(0, have)


def test_bench_reference_arm_line_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): one JSON line with the contract's
    keys, same metric / unit / config object as the GPU arm; ranks other than 0 print nothing and exit 0."""
    import json
    import subprocess
    import sys
    root = Path(__file__).resolve().parent.parent
    cmd = [sys.executable, str(root / "bench.py"), "--impl", "reference", "--workload", "cora", "--steps", "2", "--warmup", "1"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.strip().split("\n") if ln.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "edges_per_sec_per_sweep" and j["unit"] == "edges/s"
    assert j["higher_is_better"] is True and j["steps"] == 2 and j["warmup"] == 1 and j["value"] > 0
    assert j["config"]["workload"].startswith("cora") and j["config"]["nodes"] == 2708
    assert j["cpu_baseline"]["kind"] in ("port", "reference") and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"] == {"value": j["value"], "unit": j["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=root, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
