"""Time the fp32 path on graphs whose [N, ld] matrices hold more than 2^31 floats (one GPU).

    python tools/bench_wide.py [--out DIR] [--sweeps 20] [--warmup 3]

Two shapes, power-law edges (E = 2N) relabelled by degree so that hub rows and the most-gathered columns get the
highest ids, as in tests/test_wide_offsets.py:
  * d = 128, N = 18 M (N * ld = 2.30e9): normal features, heavy and light hub chains;
  * d = 1433, N = 1.6 M (N * ld = 2.30e9): Cora-style bag of words, 12 column slabs per row.
For each: ms per sweep (CUDA events around --sweeps sweeps of one clane_sweeps batch, exact L1 included, patience stop
disabled), G edges/s, the sweep's algorithmic bytes (bench.py's model: 12*d*N + 8*E + 4*(N+1)) over time as a share of
the 7.7 TB/s data-sheet HBM bandwidth, and build_P ms (cosine; CUDA events, mean of 3 after one warm-up call).  The
working sets (tens of GB) do not fit the 126 MB L2.  One JSON line per shape on stdout and in DIR/bench_wide.json,
with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from clane_b200 import _lib, similarity, synth  # noqa: E402
from clane_b200.graph import Graph  # noqa: E402

HBM_TBS = 7.7
GAMMA = 0.76
SHAPES = {"d128": (18_000_000, 128, "normal", 11), "d1433": (1_600_000, 1433, "bow", 12)}


def wide_graph(n: int, d: int, features: str, seed: int):
    rng = np.random.default_rng(seed)
    src, dst = synth.make_edges(n, 2 * n, "powerlaw", rng)
    deg = np.bincount(src, minlength=n) + np.bincount(dst, minlength=n)
    new = np.empty(n, np.int64)
    new[np.argsort(deg, kind="stable")] = np.arange(n)
    src, dst = new[src], new[dst]
    X = np.empty((n, d), np.float32)
    for a in range(0, n, 1 << 20):
        b = min(n, a + (1 << 20))
        if features == "bow":
            X[a:b] = rng.random((b - a, d), dtype=np.float32) < 18.0 / d
        else:
            X[a:b] = rng.standard_normal((b - a, d)) * 0.5
    return src, dst, X


def measure(name: str, sweeps: int, warmup: int) -> dict:
    n, d, features, seed = SHAPES[name]
    src, dst, X = wide_graph(n, d, features, seed)
    g = Graph.from_arrays(n, src, dst, X)
    del src, dst
    L, S = _lib.lib(), g._device_state()
    sim = similarity.CosineSimilarity()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g._build_P_device(sim)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(3):
        g._build_P_device(sim)
    ev1.record()
    torch.cuda.synchronize()
    build_p_ms = ev0.elapsed_time(ev1) / 3
    gamma = ctypes.c_float(float(np.float32(GAMMA)))
    sh = S.stream.cuda_stream

    def run(k):
        _lib.check(L.clane_patience_reset(S.state.data_ptr(), 1 << 30, 0, sh))
        _lib.check(L.clane_sweeps(S.plan.handle, S.X.data_ptr(), S.Zptrs, S.cur, S.rowptr.data_ptr(), S.col.data_ptr(),
                                  S.w.data_ptr(), gamma, k, 0, S.state.data_ptr(), S.log.data_ptr(), S.log_cap, sh))
        S.cur = (S.cur + k) % 3

    run(warmup)
    run(sweeps)         # untimed: the batch graphs the timed call replays exist before the clock starts
    torch.cuda.synchronize()
    ev0.record(S.stream)
    run(sweeps)
    ev1.record(S.stream)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / sweeps
    e = g._nnz
    nbytes = 12 * d * n + 8 * e + 4 * (n + 1)
    gbs = nbytes / (ms * 1e-3) / 1e9
    deg = np.diff(g._rowptr)
    line = {"shape": name, "n": n, "e": e, "d": d, "n_ld": n * S.ld, "max_degree": int(deg.max()),
            "n_hub_rows": S.plan.n_hub_rows, "n_long_hub_rows": int(np.count_nonzero(deg >= 16384)),
            "sweeps": sweeps, "ms_per_sweep": round(ms, 3), "G_edges_per_s": round(e / (ms * 1e-3) / 1e9, 3),
            "bytes_per_sweep": nbytes, "GBps": round(gbs, 1), "share_of_hbm": round(gbs / (HBM_TBS * 1e3), 3),
            "build_p_ms": round(build_p_ms, 3)}
    g._dev = None
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".")
    ap.add_argument("--sweeps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="d128,d1433")
    a = ap.parse_args()
    _lib.require_cuda()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().split("\n")[0]
    lines = []
    for name in a.shapes.split(","):
        line = measure(name, a.sweeps, a.warmup)
        line["gpu"] = gpu
        print(json.dumps(line), flush=True)
        lines.append(line)
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "bench_wide.json").write_text(json.dumps(lines, indent=1) + "\n")


if __name__ == "__main__":
    main()
