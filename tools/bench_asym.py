"""Time the AsymmertricSimilarity scorer at the benchmark shapes and write one JSON file.

    python tools/bench_asym.py OUT_DIR [--shapes arxiv,products,pubmed,cora] [--reps 50]

For each synthetic shape (clane_b200.synth) it reports, from CUDA events over `reps` launches after warm-up:
  * fp32_project: clane_asym_project_fp32 (3xTF32, any width);
  * fp32_build_p: clane_build_p_asym_fp32 (projection + per-edge dots + row softmax);
  * at d in {32, 64, 96, 128} also tf32_project / tf32_build_p (clane_asym_project / clane_build_p_asym);
  * generic_build_p: Graph.build_P with a subclass that overrides forward (the module scores gathered [E, d] rows),
    or "did not fit" when the device runs out of memory.
Each projection carries its algorithmic bytes (4 n d read + 8 n d written + 8 d^2 of W) against 7.7 TB/s and its
FLOPs (4 n d^2 useful; x3 executed for 3xTF32) against 1,125 TFLOP/s dense TF32 (HGX B200 data sheet, one GPU, a card
allowed 1,000 W), and which of the two bounds it.  The device name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from clane_b200 import _lib, similarity, synth  # noqa: E402
from clane_b200.graph import Graph  # noqa: E402

PEAK_BYTES = 7.7e12
PEAK_TF32 = 1.125e15


class _Generic(similarity.AsymmertricSimilarity):
    """The same scorer through the generic plugin path (Graph.build_P fuses only the unmodified class)."""

    def forward(self, z_src, z_dst):
        return super().forward(z_src, z_dst)


def _device():
    q = "--query-gpu=name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", q, "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return {"name": torch.cuda.get_device_name(), "nvidia_smi": out or "unavailable"}


def _time(fn, reps: int, warmup: int = 3) -> float:
    """Mean milliseconds per call from CUDA events around `reps` back-to-back calls."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def _roofline(ms: float, n: int, d: int, passes: int) -> dict:
    nbytes = 4 * n * d + 8 * n * d + 8 * d * d
    flops = 4 * n * d * d
    t_bytes, t_flops = nbytes / PEAK_BYTES, passes * flops / PEAK_TF32
    t = ms * 1e-3
    return {"ms": ms, "bytes": nbytes, "flops_useful": flops, "flops_executed": passes * flops,
            "achieved_TBps": nbytes / t / 1e12, "achieved_TFLOPs_executed": passes * flops / t / 1e12,
            "bound": "memory" if t_bytes >= t_flops else "compute",
            "share_of_bound": max(t_bytes, t_flops) / t}


def run_shape(shape: str, reps: int) -> dict:
    L = _lib.lib()
    t0 = time.time()
    n, src, dst, X = synth.make_graph(shape, seed=0)
    g = Graph.from_arrays(n, src, dst, X)
    del src, dst
    d = X.shape[1]
    S = g._device_state()
    torch.manual_seed(0)
    sim = similarity.AsymmertricSimilarity(n_dim=d)
    W = torch.zeros([2 * d, S.ld], device="cuda")
    W[:, :d] = sim.stacked_weights(S.device)
    Wc = sim.stacked_weights(S.device)
    work = torch.zeros(2 * S.n * S.ld + 4 * d * S.ld, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    Z = S.Z[S.cur]
    psrc, pdst, wsplit = work.data_ptr(), work[S.n * S.ld:].data_ptr(), work[2 * S.n * S.ld:].data_ptr()
    st = _lib.stream_handle()
    res = {"shape": shape, "n": n, "e": S.e, "d": d, "setup_s": round(time.time() - t0, 1)}

    def proj32():
        _lib.check(L.clane_asym_project_fp32(Z.data_ptr(), n, d, S.ld, W.data_ptr(), S.ld, psrc, pdst, wsplit,
                                             err.data_ptr(), st))

    def bp32():
        _lib.check(L.clane_build_p_asym_fp32(S.plan.handle, Z.data_ptr(), W.data_ptr(), S.ld, S.rowptr.data_ptr(),
                                             S.erow.data_ptr(), S.col.data_ptr(), S.w.data_ptr(), work.data_ptr(),
                                             err.data_ptr(), st))

    res["fp32_project"] = _roofline(_time(proj32, reps), n, d, 3)
    res["fp32_build_p_ms"] = _time(bp32, reps)
    if L.clane_asym_supported(d):
        def projtf():
            _lib.check(L.clane_asym_project(Z.data_ptr(), n, d, S.ld, Wc.data_ptr(), psrc, pdst, err.data_ptr(), st))

        def bptf():
            _lib.check(L.clane_build_p_asym(S.plan.handle, Z.data_ptr(), Wc.data_ptr(), S.rowptr.data_ptr(),
                                            S.erow.data_ptr(), S.col.data_ptr(), S.w.data_ptr(), work.data_ptr(),
                                            err.data_ptr(), st))

        res["tf32_project"] = _roofline(_time(projtf, reps), n, d, 1)
        res["tf32_build_p_ms"] = _time(bptf, reps)
    torch.cuda.synchronize()
    res["error_flag"] = int(err.item())
    del work
    gen = _Generic(n_dim=d)
    gen.load_state_dict(sim.state_dict())
    gen = gen.cuda()
    torch.cuda.empty_cache()
    try:
        res["generic_build_p_ms"] = _time(lambda: g._build_P_device(gen), max(1, min(reps, 5)), warmup=1)
        res["generic_peak_GB"] = torch.cuda.max_memory_allocated() / 1e9
    except torch.cuda.OutOfMemoryError as exc:
        res["generic_build_p_ms"] = "did not fit"
        res["generic_error"] = str(exc).split("\n")[0][:200]
    torch.cuda.empty_cache()
    return res


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("out_dir")
    ap.add_argument("--shapes", default="arxiv,products,pubmed,cora")
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    _lib.require_cuda()
    out = {"device": _device(), "peaks": {"hbm_TBps": PEAK_BYTES / 1e12, "tf32_dense_TFLOPs": PEAK_TF32 / 1e12},
           "shapes": []}
    for shape in args.shapes.split(","):
        torch.cuda.reset_peak_memory_stats()
        r = run_shape(shape, args.reps)
        print(json.dumps(r), flush=True)
        out["shapes"].append(r)
    Path(args.out_dir).mkdir(parents=True, exist_ok=True)
    (Path(args.out_dir) / "bench_asym.json").write_text(json.dumps(out, indent=1))
    return 0


if __name__ == "__main__":
    sys.exit(main())
