"""Time the float64 path at arXiv shape (169,343 nodes, 1,166,243 edges, d = 128) with fp64 features.

    python tools/bench_f64.py [--sweeps 1000] [--warmup 20]

Prints one JSON line: ms per sweep (CUDA events around --sweeps sweeps of one clane_sweeps_f64 batch with the
patience stop disabled), build_P ms, the sweep's algorithmic bytes -- 24*d*N (read X and Z, write Znext) + 12*E
(col, w) + 4*(N+1) (rowptr), plus 16*d*N for the unfused L1 pass (read Znext and Zcur) -- over time, that rate
as a share of the 7.7 TB/s data-sheet HBM bandwidth, and the card's name and power limit read in the same run.
A working set of ~0.5 GB does not fit the 126 MB L2.

--drop-rows-over K removes the out-edges of every row of more than K neighbours before timing (a diagnostic: it
shows how much of the sweep the longest rows, each one serial chain per column, account for).
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sweeps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--drop-rows-over", type=int, default=0, metavar="K")
    a = ap.parse_args()
    _lib.require_cuda()
    n, src, dst, X = synth.make_graph("arxiv", seed=0)
    if a.drop_rows_over > 0:
        keep = np.bincount(src, minlength=n)[src] <= a.drop_rows_over
        src, dst = src[keep], dst[keep]
    g = Graph.from_arrays(n, src, dst, torch.from_numpy(X.astype(np.float64)))
    sim = similarity.CosineSimilarity()
    g._build_P_device(sim)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(5):
        g._build_P_device(sim)
    t1.record()
    torch.cuda.synchronize()
    build_p_ms = t0.elapsed_time(t1) / 5
    S, L = g._dev, _lib.lib()
    s = _lib.stream_handle()

    def run(k):
        # max_sweeps = 0 and a patience larger than the run: every sweep does its full work, L1 and patience step
        _lib.check(L.clane_patience_reset_f64(S.state.data_ptr(), 1 << 30, 0, s))
        _lib.check(L.clane_sweeps_f64(S.n, S.d, S.rowptr.data_ptr(), S.col.data_ptr(), S.w.data_ptr(), S.X.data_ptr(),
                                      S.Zptrs, 0, ctypes.c_double(0.76), k, S.state.data_ptr(), S.log.data_ptr(),
                                      S.log_cap, S.work.data_ptr(), s))

    run(a.warmup)
    torch.cuda.synchronize()
    t0.record()
    run(a.sweeps)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / a.sweeps
    st = _lib.Patience64.from_buffer_copy(S.state.cpu().numpy().tobytes())
    assert st.sweeps == a.sweeps and not st.stop
    d, e = g.d, g._nnz
    sweep_bytes = 24 * d * n + 12 * e + 4 * (n + 1)
    l1_bytes = 16 * d * n
    gbs = (sweep_bytes + l1_bytes) / (ms * 1e-3) / 1e9
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")[0]
    print(json.dumps({"shape": "arxiv", "dtype": "float64", "drop_rows_over": a.drop_rows_over,
                      "max_degree": int(np.diff(g._rowptr).max()), "n": n, "e": e, "d": d, "sweeps": a.sweeps,
                      "ms_per_sweep": round(ms, 4), "build_p_ms": round(build_p_ms, 3),
                      "bytes_per_sweep": sweep_bytes + l1_bytes, "GBps": round(gbs, 1),
                      "share_of_hbm": round(gbs / (HBM_TBS * 1e3), 3), "gpu": q}))


if __name__ == "__main__":
    main()
