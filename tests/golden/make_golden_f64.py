"""Generate the float64 golden fixtures under tests/golden/f64/ with torch alone (one CPU thread):

    python tests/golden/make_golden_f64.py

When C.npy holds float64 the reference runs its whole hot path in double (graph.py:51 keeps the dtype).
This script does not need a reference checkout: ``restated_iterate`` is a literal torch restatement of the
reference's hot path -- the per-vertex loop of Embedder.propagate with ``P[idx].values() @ Z[nbrs]``, then
``x + gamma * (.)``, ``torch.sum(torch.abs(.))`` and the strict-``>`` patience of both loops (embedder.py:56-108),
Graph.build_P's per-source ``softmax(0)`` of CosineSimilarity's scores (graph.py:118-128, similarity.py:26-37).
Run in float32 it reproduces the fixtures the real reference wrote (ref_toy_d16, ref_hub60_d20, ref_cyclic100_d8)
bit for bit; tests/test_oracle_f64.py checks that, which is what makes its float64 output the reference's.

Two kinds of fixtures:
* ``prim_torch_f64.npz`` -- torch.sum, softmax(0), mm and bmm in double on the grids of prim_torch.npz
  (inputs are regenerated from the same seeds by the tests);
* ``ref_<case>.npz`` -- inputs and every output of ``restated_iterate`` in double.
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
OUT = HERE / "f64"


def coalesced_indices(n: int, raw_src, raw_dst) -> torch.Tensor:
    """Graph.A (graph.py:104-110): the coalesced COO index set."""
    idx = torch.from_numpy(np.stack([np.asarray(raw_src, np.int64), np.asarray(raw_dst, np.int64)]))
    return torch.sparse_coo_tensor(indices=idx, values=torch.ones(idx.shape[1]), size=(n, n)).coalesce().indices()


def cosine(v1: torch.Tensor, v2: torch.Tensor) -> torch.Tensor:
    """CosineSimilarity.__call__ (similarity.py:35-37): batched dots over the two global norms."""
    dots = v1.unsqueeze(1).matmul(v2.unsqueeze(-1)).view(-1)
    return dots / (torch.sqrt(torch.sum(v1 * v1)) * torch.sqrt(torch.sum(v2 * v2)))


def build_P(Z: torch.Tensor, idx: torch.Tensor):
    """Graph.build_P (graph.py:118-128): per-source softmax(0) of the scores.  Returns (scores, w)."""
    scores = cosine(Z[idx[0]], Z[idx[1]])
    w = scores.clone()
    for u in idx[0].unique():
        mask = idx[0] == u
        w[mask] = scores[mask].softmax(0)
    return scores, w


def restated_iterate(X: torch.Tensor, idx: torch.Tensor, gamma: float, tol: int):
    """Embedder.iterate (embedder.py:56-69) over propagate (embedder.py:71-108), in X's dtype."""
    n = X.shape[0]
    rowptr = np.zeros(n + 1, np.int64)
    np.add.at(rowptr, idx[0].numpy() + 1, 1)
    rowptr = np.cumsum(rowptr)
    col = idx[1]
    Z = X.clone()
    out = dict(amounts=[], sweeps_per_call=[], outer_amounts=[])
    g_min, g_tol = float("inf"), tol
    first_call = True
    while True:
        prev = Z.clone()
        scores, w = build_P(Z, idx)
        if first_call:
            out["scores0"], out["P0_values"] = scores.numpy().copy(), w.numpy().copy()
        p_min, p_tol, sweeps = float("inf"), tol, 0
        while True:
            current_Z = Z.clone()
            Zn = Z.clone()
            for v in range(n):
                a, b = int(rowptr[v]), int(rowptr[v + 1])
                if b == a:                      # embedder.py:88-89
                    continue
                Zn[v] = X[v] + gamma * (w[a:b].view(1, -1) @ current_Z[col[a:b]]).view(-1)
            amount = torch.sum(torch.abs(Zn - current_Z))
            Z = Zn
            sweeps += 1
            out["amounts"].append(amount.item())
            if first_call and sweeps == 1:
                out["Z_after_first_sweep"] = Z.numpy().copy()
            if p_min > amount:
                p_tol, p_min = tol, amount
            else:
                p_tol -= 1
            if p_tol == 0:
                break
        if first_call:
            out["Z_after_first_call"] = Z.numpy().copy()
        first_call = False
        out["sweeps_per_call"].append(sweeps)
        amount = torch.sum(torch.abs(Z - prev))
        out["outer_amounts"].append(amount.item())
        if g_min > amount:
            g_tol, g_min = tol, amount
        else:
            g_tol -= 1
        if g_tol == 0:
            break
    out["Z_final"] = Z.numpy().copy()
    dt = np.float64 if X.dtype == torch.float64 else np.float32
    out["amounts"] = np.array(out["amounts"], dt)
    out["outer_amounts"] = np.array(out["outer_amounts"], dt)
    out["sweeps_per_call"] = np.array(out["sweeps_per_call"], np.int64)
    return out


def case(name, n, e_raw, d, gamma, tol, seed, features="normal", hub=None, dups=0, loops=0, weird_ids=False):
    rng = np.random.default_rng(seed)
    src = rng.integers(0, n, e_raw)
    dst = rng.integers(0, n, e_raw)
    if hub is not None:
        src = np.concatenate([src, np.full(hub, 3)])
        dst = np.concatenate([dst, rng.permutation(n)[:hub]])
    if dups:
        sel = rng.integers(0, len(src), dups)
        src, dst = np.concatenate([src, src[sel]]), np.concatenate([dst, dst[sel]])
    if loops:
        lp = rng.integers(0, n, loops)
        src, dst = np.concatenate([src, lp]), np.concatenate([dst, lp])
    order = rng.permutation(len(src))
    src, dst = src[order], dst[order]
    if features == "normal":
        X = rng.standard_normal((n, d))
    else:                                   # tf-idf-like: sparse, non-negative
        X = (rng.random((n, d)) < 0.1) * rng.random((n, d)) * 0.2
    ids = [f"v{(7 * i + 3) % n:03d}x" if weird_ids else str(i) for i in range(n)]
    idx = coalesced_indices(n, src, dst)
    out = restated_iterate(torch.from_numpy(X), idx, gamma, tol)
    out.update(X=X, n=np.int64(n), d=np.int64(d), gamma=np.float64(gamma), tol=np.int64(tol), raw_src=src,
               raw_dst=dst, A_indices=idx.numpy(), ids=np.array(ids))
    np.savez_compressed(OUT / f"ref_{name}.npz", **out)
    print(name, "sweeps/call", out["sweeps_per_call"].tolist(), "E", idx.shape[1])


def case_toy(name, d, gamma, tol, seed):
    """The karate-club graph of tests/data_root with float64 N(0, 1) features from a seeded generator."""
    root = HERE.parent / "data_root"
    ids = (root / "V").read_text().strip().split("\n")
    pos = {v: i for i, v in reversed(list(enumerate(ids)))}
    pairs = [line.split("\t") for line in (root / "E").read_text().strip().split("\n")]
    src = np.array([pos[a] for a, _ in pairs], np.int64)
    dst = np.array([pos[b] for _, b in pairs], np.int64)
    X = np.random.default_rng(seed).standard_normal((len(ids), d))
    idx = coalesced_indices(len(ids), src, dst)
    out = restated_iterate(torch.from_numpy(X), idx, gamma, tol)
    out.update(X=X, n=np.int64(len(ids)), d=np.int64(d), gamma=np.float64(gamma), tol=np.int64(tol), raw_src=src,
               raw_dst=dst, A_indices=idx.numpy(), ids=np.array(ids))
    np.savez_compressed(OUT / f"ref_{name}.npz", **out)
    print(name, "sweeps/call", out["sweeps_per_call"].tolist(), "E", idx.shape[1])


def prim_fixtures():
    """torch's double primitives on the grids of prim_torch.npz (same seeds, float64 inputs)."""
    out = {}
    sum_n = [1, 2, 3, 5, 7, 8, 31, 32, 33, 100, 511, 512, 513, 4096, 16384, 16385, 65536, 100000, 524288,
             524289 + 77, 1 << 20, (1 << 21) + 12345, 5_000_011, 21_675_904, 40_000_003]
    res = []
    for i, n in enumerate(sum_n):
        x = np.abs(np.random.default_rng(1000 + i).standard_normal(n))
        res.append(torch.from_numpy(x).sum().item())
    out["sum_n"], out["sum_out"] = np.array(sum_n, np.int64), np.array(res, np.float64)
    sm_k = [1, 2, 3, 7, 8, 9, 15, 16, 17, 31, 32, 33, 48, 100, 255, 1000, 8234]
    for i, k in enumerate(sm_k):
        for j, scale in enumerate((0.01, 1.0, 30.0, 300.0)):
            s = np.random.default_rng(2000 + 10 * i + j).standard_normal(k) * scale
            out[f"softmax_{k}_{j}"] = torch.from_numpy(s).softmax(0).numpy()
    out["softmax_k"] = np.array(sm_k, np.int64)
    mm_cases = [(1, 2), (3, 8), (7, 16), (8, 16), (9, 17), (8, 2), (16, 20), (23, 24), (33, 3), (40, 100), (8, 128),
                (15, 128), (64, 128), (200, 130), (300, 128), (1000, 64), (2000, 128), (20000, 128), (5, 500),
                (33, 500), (12, 1433), (9, 15), (50, 31), (50, 33)]
    for i, (k, d) in enumerate(mm_cases):
        rng = np.random.default_rng(3000 + i)
        w = rng.random(k)
        w /= w.sum()
        Z = rng.standard_normal((k, d))
        out[f"mm_{k}_{d}"] = torch.from_numpy(w).view(1, -1).mm(torch.from_numpy(Z)).numpy()[0]
    out["mm_cases"] = np.array(mm_cases, np.int64)
    dot_d = [2, 5, 8, 64, 100, 128, 399, 400, 500, 1433]
    for i, d in enumerate(dot_d):
        rng = np.random.default_rng(4000 + i)
        a, b = rng.standard_normal((64, d)), rng.standard_normal((64, d))
        out[f"dot_{d}"] = torch.from_numpy(a).unsqueeze(1).matmul(torch.from_numpy(b).unsqueeze(-1)).view(-1).numpy()
    out["dot_d"] = np.array(dot_d, np.int64)
    np.savez_compressed(OUT / "prim_torch_f64.npz", **out)
    print("prim fixtures written")


def main():
    torch.set_num_threads(1)
    OUT.mkdir(exist_ok=True)
    prim_fixtures()
    case_toy("toy_d16", 16, 0.74, 10, seed=0)
    case("cyclic100_d8", 100, 390, 8, 0.76, 3, seed=0, dups=4)
    case("hub60_d20", 60, 500, 20, 0.76, 3, seed=1, hub=51, dups=20, loops=6, weird_ids=True)
    case("tfidf30_d500", 30, 200, 500, 0.76, 2, seed=3, features="tfidf", hub=24)


if __name__ == "__main__":
    sys.exit(main())
