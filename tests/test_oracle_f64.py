"""The fp64 oracle (oracle_f64/) against the float64 fixtures of tests/golden/make_golden_f64.py, and the torch
restatement behind those fixtures against the fixtures the real reference wrote.  Bit-exact everywhere."""
import importlib.util
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle_f64 import oracle_f64 as O

GOLD = Path(__file__).resolve().parent / "golden"
F64 = GOLD / "f64"
F64_CASES = sorted(p.stem for p in F64.glob("ref_*.npz"))


def _make_golden_f64():
    spec = importlib.util.spec_from_file_location("make_golden_f64", GOLD / "make_golden_f64.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def prim():
    return np.load(F64 / "prim_torch_f64.npz")


def test_f64_fixtures_present():
    assert F64_CASES == ["ref_cyclic100_d8", "ref_hub60_d20", "ref_tfidf30_d500", "ref_toy_d16"]


@pytest.mark.parametrize("case", ["ref_toy_d16", "ref_hub60_d20", "ref_cyclic100_d8"])
def test_restatement_in_fp32_reproduces_reference(case):
    """The torch restatement that wrote the float64 fixtures, run in float32, equals the real reference."""
    mg = _make_golden_f64()
    G = np.load(GOLD / f"{case}.npz")
    n = int(G["n"])
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        idx = mg.coalesced_indices(n, G["raw_src"], G["raw_dst"])
        assert np.array_equal(idx.numpy(), G["A_indices"])
        out = mg.restated_iterate(torch.from_numpy(G["X"]), idx, float(G["gamma"]), int(G["tol"]))
    finally:
        torch.set_num_threads(threads)
    assert np.array_equal(out["scores0"], G["scores0"])
    assert np.array_equal(out["P0_values"], G["P0_values"])
    assert out["sweeps_per_call"].tolist() == G["sweeps_per_call"].tolist()
    assert np.array_equal(out["amounts"], G["amounts"])
    assert np.array_equal(out["outer_amounts"], G["outer_amounts"])
    assert np.array_equal(out["Z_after_first_sweep"], G["Z_after_first_sweep"])
    assert np.array_equal(out["Z_final"], G["Z_final"])


@pytest.mark.parametrize("threads", [1, 4])
def test_cascade_sum_matches_torch_sum(prim, threads):
    O.set_threads(threads)
    for i, n in enumerate(prim["sum_n"]):
        x = np.abs(np.random.default_rng(1000 + i).standard_normal(int(n)))
        assert O.aten_sum(x) == prim["sum_out"][i], f"n={n}"


def test_softmax_rows_match_torch(prim):
    for i, k in enumerate(prim["softmax_k"]):
        for j, scale in enumerate((0.01, 1.0, 30.0, 300.0)):
            s = np.random.default_rng(2000 + 10 * i + j).standard_normal(int(k)) * scale
            w = O.softmax_rows(s, np.array([0, k]))
            assert np.array_equal(w, prim[f"softmax_{k}_{j}"]), f"k={k} scale={scale}"


def test_row_update_matches_torch_mm(prim):
    for i, (k, d) in enumerate(prim["mm_cases"]):
        rng = np.random.default_rng(3000 + i)
        w = rng.random(k)
        w /= w.sum()
        Z = rng.standard_normal((k, d))
        Zc = np.concatenate([np.zeros((1, d)), Z])       # node 0 -> nodes 1..k, x = 0, gamma = 1
        rowptr = np.zeros(k + 2, np.int64)
        rowptr[1:] = k
        Zn = O.sweep(np.zeros_like(Zc), Zc, rowptr, np.arange(1, k + 1, dtype=np.int32), w, 1.0)
        assert np.array_equal(Zn[0], prim[f"mm_{k}_{d}"]), f"k={k} d={d}"
        assert np.array_equal(Zn[1:], Zc[1:])


def test_batched_dot_matches_torch(prim):
    for i, d in enumerate(prim["dot_d"]):
        rng = np.random.default_rng(4000 + i)
        a, b = rng.standard_normal((64, d)), rng.standard_normal((64, d))
        rowptr = np.concatenate([np.arange(65), np.full(64, 64)]).astype(np.int64)
        dots, _, _ = O.scores_raw(np.concatenate([a, b]), rowptr, np.arange(64, 128, dtype=np.int32))
        assert np.array_equal(dots, prim[f"dot_{d}"]), f"d={d}"


def test_exp_edges():
    """Sleef expd u10 as restated: exact at 0, flushed below -1000, and monotone on a fine grid."""
    x = np.array([0.0, -1e-300, -745.2, -1000.0, -1000.5, -2000.0])
    e = O.exp(x)
    assert e[0] == 1.0 and e[1] == 1.0 and e[4] == 0.0 and e[5] == 0.0
    g = O.exp(np.linspace(-30, 0, 100001))
    assert np.all(np.diff(g) >= 0)


@pytest.mark.parametrize("case", F64_CASES)
def test_oracle_f64_reproduces_fixture(case):
    G = np.load(F64 / f"{case}.npz")
    n = int(G["n"])
    O.set_threads(2)
    rows, col = G["A_indices"][0], G["A_indices"][1].astype(np.int32)
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))]).astype(np.int64)
    dots, s1, s2 = O.scores_raw(G["X"], rowptr, col)
    assert np.array_equal(dots / (np.sqrt(s1) * np.sqrt(s2)), G["scores0"])
    w = O.build_p(G["X"], rowptr, col)
    assert np.array_equal(w, G["P0_values"])
    gamma, tol = float(G["gamma"]), int(G["tol"])
    assert np.array_equal(O.sweep(G["X"], G["X"], rowptr, col, w, gamma), G["Z_after_first_sweep"])
    Z1, amounts, _ = O.propagate(G["X"], G["X"], rowptr, col, gamma, tol)
    k0 = int(G["sweeps_per_call"][0])
    assert len(amounts) == k0 and np.array_equal(amounts, G["amounts"][:k0])
    assert np.array_equal(Z1, G["Z_after_first_call"])
    Z, spc, oam = O.iterate(G["X"], rowptr, col, gamma, tol)
    assert spc.tolist() == G["sweeps_per_call"].tolist()
    assert np.array_equal(oam, G["outer_amounts"])
    assert np.array_equal(Z, G["Z_final"]) and Z.dtype == np.float64


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour without a CUDA device")
@pytest.mark.parametrize("dtype", [torch.float64, torch.float16])
def test_device_state_without_cuda_raises(dtype):
    from clane_b200 import _lib
    from clane_b200.graph import Graph
    g = Graph.from_arrays(3, [0, 1], [1, 2], torch.zeros(3, 4, dtype=dtype))
    with pytest.raises(_lib.ClaneError):
        g.Z_device
