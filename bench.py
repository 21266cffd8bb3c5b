#!/usr/bin/env python
"""bench.py -- edges/sec per sweep of the CLANE embedding update on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload arxiv|products|pubmed|cora]
    python bench.py --impl reference ...      # the CPU arm: oracle port on all host threads
    python bench.py --dump-outputs DIR ...    # also write what the timed sweeps computed (one GPU; see dump_outputs)

A "step" is one Jacobi sweep of Embedder.propagate (/root/reference/clane/embedder.py:84-108)
over the whole graph with P frozen: the fused gather-SpMM + residual kernel(s), the exact
(ATen-cascade-order) L1 change and the device-side patience update.  Inputs are resident in
HBM when the timed region starts; `e2e` is the same metric through the host-buffer C-ABI
(clane_session_*) with every host<->device copy inside the timed region.

One JSON line is printed by rank 0.  See DESIGN.md section "Measurement" for the definitions.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

METRIC = "edges_per_sec_per_sweep"
UNIT = "edges/s"
GAMMA = 0.76


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="clane_b200", choices=["clane_b200", "reference"])
    ap.add_argument("--workload", default=None, help="cora | pubmed | arxiv | products (default: arxiv at 1 GPU, products at >1)")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (debug only; marks the line invalid)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-converge", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (single-GPU arm; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "clane_b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm")
    return args


def workload_name(args) -> str:
    if args.workload:
        return args.workload
    return "arxiv" if args.gpus == 1 else "products"


def workload_config(name, n, e, d, scale):
    """The `config` object: identical in both arms (the driver compares them)."""
    ws = 3 * n * d * 4 + 8 * e
    return {"workload": f"{name}-shape synthetic", "nodes": n, "edges": e, "dim": d, "gamma": GAMMA,
            "similarity": "CosineSimilarity", "scale": scale,
            "l2": f"no flush: working set {ws / 1e6:.0f} MB exceeds the 126 MB L2" if ws > 126e6
                  else "no flush: working set fits L2 (the steady state of the iteration; Cora/Pubmed shapes)"}


def sweep_bytes(n, e, d):
    """Algorithmic bytes of one sweep (SURVEY.md 8d): X, Z_cur read, Z_next written, col, w, rowptr."""
    return 12 * d * n + 8 * e + 4 * (n + 1)


DUMP_Z_BYTES = 32 << 20


def dump_outputs(out_dir, S, steps):
    """What the timed sweeps computed, as a caller of Embedder.propagate receives it, so that two builds can be compared
    output for output.  All sweeps of a run, warm-up (the line's `warmup` counts them) and timed, are one sequence from
    Z = X with P built from X, so the same arguments give the same outputs:

        Z.npy        float32 [rows, d]  embeddings after the last timed sweep: every row, or, when Z is larger than
                                        DUMP_Z_BYTES, a fixed sample of rows (seed 0, ascending)
        Z_rows.npy   float64 [rows]     the row ids of Z.npy
        amounts.npy  float32 [steps]    the exact L1 change of every timed sweep, the last one last"""
    import torch
    n, d = S.n, S.d
    rows = np.arange(n)
    if n * d * 4 > DUMP_Z_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_Z_BYTES // (4 * d), replace=False))
    Z = S.Z[S.cur][torch.from_numpy(rows).to(S.device), :d].cpu().numpy()
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "Z.npy", Z)
    np.save(out / "Z_rows.npy", rows.astype(np.float64))
    np.save(out / "amounts.npy", S.log[:steps].cpu().numpy())


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload: str):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(workload)
        except Exception:
            return None
    return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": float(self.max_mhz) if self.max_mhz else None,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's path on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_sweeps(n, src, dst, X, budget_s: float, min_sweeps: int, max_sweeps: int, step_budget_s: float = 0.0):
    """Time CPU sweeps (row update + exact L1 change) of the oracle on the host threads.

    Returns (edges per timed step, all edges, threads, times, sample description).  When a whole sweep is
    slower than step_budget_s (> 0), each timed step covers a contiguous row range holding about
    that much work -- a bounded sample of the same workload."""
    from oracle import oracle as O
    rowptr, col = O.csr_from_edges(src, dst, n)
    O.set_threads(O.max_threads())
    w = O.build_p(X, rowptr, col)
    Z = np.ascontiguousarray(X)
    Zn = Z.copy()
    # use as many host threads as actually help (shared/virtualised hosts can anti-scale)
    best = None
    for t in sorted({1, max(1, O.max_threads() // 2), O.max_threads()}):
        O.set_threads(t)
        O.sweep_range(X, Z, Zn, 0, n, rowptr, col, w, GAMMA)
        t0 = time.perf_counter()
        O.sweep_range(X, Z, Zn, 0, n, rowptr, col, w, GAMMA)
        O.l1_diff(Zn, Z)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, t)
    t_full, threads = best
    O.set_threads(threads)
    hi = n
    if step_budget_s > 0 and t_full > step_budget_s:
        target = rowptr[n] * step_budget_s / t_full
        hi = max(1, int(np.searchsorted(rowptr, target)))
    edges = int(rowptr[hi])
    what = "whole sweeps" if hi == n else f"sweeps of rows [0, {hi}) = {edges} of {int(rowptr[n])} edges"
    times = []
    t_end = time.perf_counter() + budget_s
    while len(times) < max_sweeps and (len(times) < min_sweeps or time.perf_counter() < t_end):
        t0 = time.perf_counter()
        O.sweep_range(X, Z, Zn, 0, hi, rowptr, col, w, GAMMA)
        O.l1_diff(Zn[:hi], Z[:hi])
        times.append(time.perf_counter() - t0)
        if hi == n:
            Z, Zn = Zn, Z
    return edges, int(rowptr[n]), threads, times, what


def run_reference(args):
    from clane_b200 import synth
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = workload_name(args)
    n, src, dst, X = synth.make_graph(name, seed=0, scale=args.scale)
    d = X.shape[1]
    # each step = one CPU sweep of the same workload (bounded: the whole run ends within minutes)
    total = args.warmup + args.steps
    e, e_all, threads, times, what = cpu_sweeps(n, src, dst, X, budget_s=1e9, min_sweeps=total, max_sweeps=total,
                                         step_budget_s=150.0 / total)
    timed = times[args.warmup:]
    ms = 1e3 * float(np.mean(timed))
    value = e / (ms * 1e-3)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, n, e_all, d, args.scale),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{len(timed)} {what} (row update + exact L1) of the {name}-shape graph, "
                                   f"oracle C port of the reference's path, OpenMP over rows"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference itself is pure Python (O(N*E) per sweep, ~210 edges/s at Cora shape, BASELINE.md) "
                "and cannot run this shape; this arm times its bit-exact C restatement on all host threads",
    }
    print(json.dumps(line))



def single_gpu_steps(torch, L, _lib, g, sim, steps, warmup=3):
    """ms per sweep (exact L1 included) of graph `g` on THIS rank's GPU alone: the strong-scaling reference."""
    S = g._device_state()
    g.set_Z(g.X)
    g._build_P_device(sim)
    gamma = ctypes.c_float(float(np.float32(GAMMA)))
    sh = S.stream.cuda_stream

    def run(k):
        _lib.check(L.clane_patience_reset(S.state.data_ptr(), 1 << 30, 0, sh))
        _lib.check(L.clane_sweeps(S.plan.handle, S.X.data_ptr(), S.Zptrs, S.cur, S.rowptr.data_ptr(), S.col.data_ptr(),
                                  S.w.data_ptr(), gamma, k, 0, S.state.data_ptr(), S.log.data_ptr(), S.log_cap, sh))
        S.cur = (S.cur + k) % 3
    torch.cuda.synchronize()
    run(warmup)
    run(steps)          # untimed: the batch graphs the timed call replays exist before the clock starts
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(S.stream)
    run(steps)
    ev1.record(S.stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / steps


def vectorised_cpu_sweeps(n, src, dst, X, budget_s=6.0):
    """BASELINE.md section 3 item (iii): a best-effort VECTORISED torch-CPU restatement (CSR SpMM + axpy + L1 on all
    host threads) -- timing only: its summation order is torch's, not the reference's, so counts may drift."""
    import torch
    from oracle import oracle as O
    rowptr, col = O.csr_from_edges(src, dst, n)
    w = O.build_p(X, rowptr, col)
    P = torch.sparse_csr_tensor(torch.from_numpy(rowptr), torch.from_numpy(col.astype(np.int64)), torch.from_numpy(w),
                                size=(n, n))
    Xt = torch.from_numpy(np.ascontiguousarray(X))
    has = torch.from_numpy(np.diff(rowptr) > 0).unsqueeze(1)
    Z = Xt.clone()
    times = []
    t_end = time.perf_counter() + budget_s
    while len(times) < 3 or (time.perf_counter() < t_end and len(times) < 50):
        t0 = time.perf_counter()
        Zn = torch.where(has, Xt + GAMMA * (P @ Z), Z)
        amount = (Zn - Z).abs().sum().item()
        times.append(time.perf_counter() - t0)
        Z = Zn
    return int(rowptr[n]), torch.get_num_threads(), times[1:], amount


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from clane_b200 import _lib, similarity, synth
    from clane_b200.embedder import Embedder
    from clane_b200.graph import Graph

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    name = workload_name(args)
    n, src, dst, X = synth.make_graph(name, seed=0, scale=args.scale)
    d = X.shape[1]
    g = Graph.from_arrays(n, src, dst, X)
    e = g._nnz
    L = _lib.lib()
    sim = similarity.CosineSimilarity()
    emb = Embedder(g, sim, device=torch.device("cuda", local_rank), gamma=GAMMA, tolerence=10)
    emb.verbose = False

    if world > 1:
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the outputs of a single-GPU run")
        from clane_b200 import dist as cdist
        runner = cdist.ShardedSweeper(g, sim, GAMMA, exchange=os.environ.get("CLANE_EXCHANGE", "auto"))
        S = None
    else:
        runner = None
        S = g._device_state()
        g._build_P_device(sim)
        if args.dump_outputs and args.steps > S.log_cap:
            raise SystemExit(f"--dump-outputs keeps the L1 change of at most {S.log_cap} timed sweeps")
    stream = S.stream if S is not None else torch.cuda.current_stream()
    torch.cuda.synchronize()
    sh = stream.cuda_stream
    gamma = ctypes.c_float(float(np.float32(GAMMA)))
    launches_per_step = [0]

    def one_step(i, with_l1=True):
        if runner is not None:
            launches_per_step[0] = runner.sweep(with_l1)
            return
        a, b = S.Z[(S.cur + i) % 3], S.Z[(S.cur + i + 1) % 3]
        _lib.check(L.clane_sweep(S.plan.handle, S.X.data_ptr(), a.data_ptr(), b.data_ptr(), S.rowptr.data_ptr(),
                                 S.col.data_ptr(), S.w.data_ptr(), gamma, S.amount.data_ptr() if with_l1 else 0, 0, 0, 0,
                                 sh))
        launches_per_step[0] = S.plan.launches_per_sweep if with_l1 else S.plan.launches_per_sweep - 2 - (
            1 if S.plan.fused_l1 and S.plan.n_fix_groups else 0)

    def many_steps(k):
        """k sweeps the way Embedder.propagate runs them: one clane_sweeps call (replayed graphs of 6 sweeps, the exact
        L1 + patience tail of every sweep beside the rows of the next one); the patience counter is set so that it
        never stops inside the timed region."""
        if runner is not None:
            # the sharded counterpart: ShardedSweeper.sweeps (exact L1 of sweep t beside sweep t + 1, three rotating buffers)
            runner.sweeps(k)
            launches_per_step[0] = runner.launches_last_sweep or launches_per_step[0]
            return
        _lib.check(L.clane_patience_reset(S.state.data_ptr(), 1 << 30, 0, sh))
        _lib.check(L.clane_sweeps(S.plan.handle, S.X.data_ptr(), S.Zptrs, S.cur, S.rowptr.data_ptr(), S.col.data_ptr(),
                                  S.w.data_ptr(), gamma, k, 0, S.state.data_ptr(), S.log.data_ptr(), S.log_cap, sh))
        S.cur = (S.cur + k) % 3
        launches_per_step[0] = S.plan.launches_per_sweep

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_loop(steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record(stream)
        many_steps(steps)
        ev1.record(stream)
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def kernel_loop(steps):
        """The same steps again with the library's event brackets on: average duration of the dominant
        kernel (k_sweep_rows) alone, measured on the stream it is launched on."""
        if runner is not None and runner.chunks:      # copy-engine exchange: several span kernels per sweep, timed as a phase below
            return np.full(4, float("nan"))
        plan = S.plan if runner is None else runner.plan
        _lib.check(L.clane_plan_profile(plan.handle, 1))
        acc = np.zeros(4)
        buf = (ctypes.c_float * 4)()
        for i in range(steps):
            one_step(i, True)
            _lib.check(L.clane_plan_profile_read(plan.handle, buf))
            acc += np.array(buf[:])
        _lib.check(L.clane_plan_profile(plan.handle, 0))
        acc /= steps
        if world > 1:
            t = torch.tensor(acc, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            acc = t.cpu().numpy()
        return acc

    # warm-up: at least W sweeps, rounded up to whole buffer rotations x graph batches, so that the timed region replays
    # graphs that already exist (a graph is keyed by the buffer its first sweep reads)
    warm = -(-max(args.warmup, 3) // 6) * 6 if runner is None else max(args.warmup, 3)
    many_steps(warm)
    if runner is None:
        # ... and three untimed passes of the timed call itself: the batch graphs of every starting buffer and of the
        # remainder (steps mod 6) exist before the clock starts, and the timed pass starts where the first one did
        for _ in range(3):
            many_steps(args.steps)
        warm += 3 * args.steps
    sampler = ClockSampler(local_rank)
    sampler.start()
    total_ms = timed_loop(args.steps)                                  # the metric: whole steps
    if args.dump_outputs:                                              # before kernel_loop overwrites the Z buffers
        dump_outputs(args.dump_outputs, S, args.steps)
    kern = kernel_loop(min(args.steps, 200))                           # per-kernel durations (roofline)
    phases = None
    exch = runner.exchange if runner is not None else "none"
    if runner is not None:                                             # phases of a sharded sweep (events, this rank)
        runner.timing, runner.phase_ms = True, {}
        for i in range(min(args.steps, 20)):
            one_step(i, True)
        runner.timing = False
        k = runner.phase_ms.pop("sweeps")
        phases = {name: ms / k for name, ms in runner.phase_ms.items()}
    clocks = sampler.stop()
    ms_per_step = total_ms / args.steps
    value = e / (ms_per_step * 1e-3)
    if runner is None:
        torch.cuda.synchronize()
        amount = float(_lib.Patience.from_buffer_copy(S.state.cpu().numpy().tobytes()).last_amount)
    else:
        amount = runner.last_amount()

    PLAN = S.plan if runner is None else runner.plan
    peak, peak_src = measured_peak()
    if np.isnan(kern[0]):        # chunked sweep: the whole sweep phase (span kernels of every chunk, exchange beside them)
        t = torch.tensor([phases["sweep"]], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        kern = np.array([float(t.item()), float("nan"), phases.get("l1_partial", 0.0) + phases.get("all_reduce", 0.0) +
                         phases.get("finish", 0.0), 0.0])
    kern_ms = float(kern[0])
    bytes_sweep = sweep_bytes(n, e, d)
    achieved = bytes_sweep / world / (kern_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, n, e, d, args.scale),
        "details": {"parallelism": "single GPU" if world == 1 else
                    f"rows partitioned by contiguous id over {world} GPUs; exchange: " +
                    ("every finished row stored to all ranks' Z (NVLink peer memory) from inside the sweep kernel, "
                     "one all-reduce of the L1 slots per sweep" + (" (multimem.st through the NVSwitch multicast mapping)"
                                                                  if exch == "multicast" else "")
                     if exch in ("p2p", "multicast")
                     else "rows swept in chunks, every finished chunk copied to all ranks' Z by the copy engines (peer-to-peer "
                          "cudaMemcpyAsync over NVLink) while the next chunk is swept; one all-reduce of the L1 slots per sweep"
                     if exch == "ce" else "NCCL all-gather of Z per sweep"),
                     "step": ("span tasks with the hub segments + chains beside them, exact L1 change (fused partials / cascade) "
                             "and device patience of every sweep beside the next sweep's rows (three rotating Z buffers, "
                             "replayed graphs of 6 sweeps); P frozen") if world == 1 else
                            ("span tasks (a span's rows leave as bulk stores to every rank) with the hub segments + chains beside "
                             "them; " + ("exact L1 of sweep t (own level-1 nodes, all-reduce of the slots on a second process "
                                         "group, finish) on a tail stream beside sweep t + 1, three rotating symmetric buffers, "
                                         "one token all-reduce per sweep orders the ranks" if getattr(runner, "pipelined", False)
                                         else "exact L1 (own level-1 nodes, all-reduce of the slots, finish) after every sweep")
                             + "; P frozen"),
                    "plan": {"group_rows": PLAN.group_rows, "spans": PLAN.n_spans, "hub_rows": PLAN.n_hub_rows,
                             "fused_l1": PLAN.fused_l1}},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic(name) if world == 1 else None,
                     "traffic_gbs": (ncu_traffic(name) / (kern_ms * 1e-3) / 1e9) if world == 1 and ncu_traffic(name) else None,
                     "kernel": "k_sweep_rows", "kernel_ms": kern_ms,
                     "sweep_ms_serialized": None if np.isnan(kern[1]) else float(kern[1]), "l1_tail_ms": float(kern[2]), "hub_kernel_ms": float(kern[3]),
                     "algorithmic_bytes_per_launch": bytes_sweep / world, "peak_source": peak_src,
                     "frac_of_nominal_8TBs": achieved / 8000.0,
                     "whole_step_gbs": bytes_sweep / world / (ms_per_step * 1e-3) / 1e9},
        "clocks": clocks,
        "gpu_launches": launches_per_step[0] * args.steps,
        "last_amount": amount,
    }
    if phases is not None:
        line["sharded_phase_ms_rank0"] = phases
        allp = [None] * world
        dist.all_gather_object(allp, phases)
        line["sharded_phase_ms_all_ranks"] = allp

    if world == 1:
        # Graph.build_P (scores + global norms + row softmax), once per propagate() call: its own small roofline
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        g._build_P_device(sim)
        torch.cuda.synchronize()
        evs[0].record()
        for _ in range(10):
            g._build_P_device(sim)
        evs[1].record()
        torch.cuda.synchronize()
        bp_ms = evs[0].elapsed_time(evs[1]) / 10
        bp_bytes = 4 * d * n + 16 * e + 4 * (n + 1)
        line["build_p"] = {"ms": bp_ms, "algorithmic_bytes": bp_bytes, "achieved_gbs": bp_bytes / (bp_ms * 1e-3) / 1e9,
                           "frac": bp_bytes / (bp_ms * 1e-3) / 1e9 / peak,
                           "kernels": "k_dots (warp per 32 edges, tiled) + cascade level 0/1 + finish + row softmax"}
        if rank == 0:
            line["e2e"] = e2e_session(L, g, X, n, e, d, args.steps)
    else:
        # N > 1: the sharded public API from HOST buffers -- every rank uploads the CSR replica and X, builds P,
        # runs `steps` sweeps (exchange fused into the sweep kernel) and downloads the full Z; max over ranks.
        runner = None
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        r2 = cdist.ShardedSweeper(g, sim, GAMMA, exchange=os.environ.get("CLANE_EXCHANGE", "auto"))
        r2.sweeps(args.steps)
        Zh = r2.Z_host_slice()           # every rank downloads its own rows: together they are Z
        amount2 = r2.last_amount()
        dt = torch.tensor([time.perf_counter() - t0], device="cuda")
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        secs = float(dt.item())
        h2d = n * d * 4 + world * (4 * (n + 1) + 4 * e)          # X once (a slice per rank), the CSR on every rank
        d2h = n * d * 4 + 4 * world
        line["e2e"] = {"value": e * args.steps / secs, "unit": UNIT, "h2d_bytes_per_step": h2d / args.steps,
                       "d2h_bytes_per_step": d2h / args.steps, "seconds": secs, "steps": args.steps,
                       "last_amount": amount2,
                       "note": "ShardedSweeper(graph from host arrays) + sweeps(steps) (exact L1 of every sweep) + Z_host_slice() on every rank, "
                               "wall clock, max over ranks; every rank uploads the CSR and its own rows of X (the other rows "
                               "arrive over NVLink) and downloads its own rows of Z; upload, plan build, build_P and the "
                               "download are inside the timed region and amortised over the steps of the call"}
        del r2
        # ---- strong scaling on ONE workload: the same graph on rank 0's GPU alone, in this job ----
        n1 = torch.zeros(1, device="cuda")
        torch.cuda.synchronize()
        dist.barrier()          # every rank has released its sharded buffers (peer unmapping done) before rank 0 measures
        if rank == 0:
            n1[0] = single_gpu_steps(torch, L, _lib, g, sim, min(args.steps, 50))
        dist.broadcast(n1, 0)
        n1_ms = float(n1.item())
        n1_value = e / (n1_ms * 1e-3)
        line["strong_scaling"] = {"workload": f"{name}-shape synthetic", "n1_ms_per_step": n1_ms, "n1_value": n1_value,
                                  "efficiency": value / (world * n1_value),
                                  "how": f"{min(args.steps, 50)} single-GPU sweeps of the same graph on rank 0, same job, CUDA "
                                         "events; efficiency = value / (n_gpus * n1_value)"}
        # ---- parity of the sharded path against the single-GPU path, outside every timed region ----
        K = 3
        rc_ = cdist.ShardedSweeper(g, sim, GAMMA, exchange=os.environ.get("CLANE_EXCHANGE", "auto"))
        am = [float(a) for a in rc_.sweeps(K)]
        Zs = rc_.Z[rc_.cur][:n]
        Zb = torch.empty_like(Zs)
        amb = torch.zeros(K, dtype=torch.float64, device="cuda")
        if rank == 0:
            g.set_Z(g.X)
            emb.sweeps_per_call, emb.amounts_per_call = [], []
            emb.propagate(max_sweeps=K)
            S1 = g._device_state()
            Zb.copy_(S1.Z[S1.cur][:n])
            amb.copy_(torch.from_numpy(np.asarray(emb.amounts_per_call[-1], np.float64)))
        dist.broadcast(Zb, 0)
        dist.broadcast(amb, 0)
        same = torch.tensor([int(torch.equal(Zs, Zb) and am == amb.cpu().tolist())], device="cuda")
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        line["parity_vs_single_gpu"] = bool(same.item())
        line["parity_check"] = f"{K} sweeps from Z = X: every rank's full Z replica and the L1 amounts bit-identical to rank 0's single-GPU run"
        del rc_, Zb
        if not args.no_converge:
            # time-to-converge of the sharded Embedder.iterate() (build_P calls + sweeps + patience on every rank)
            r3 = cdist.ShardedSweeper(g, sim, GAMMA, tol=10, exchange=os.environ.get("CLANE_EXCHANGE", "auto"))
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            spc, _ = r3.iterate()
            torch.cuda.synchronize()
            dt = torch.tensor([time.perf_counter() - t0], device="cuda")
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            line["time_to_converge"] = {"seconds": float(dt.item()), "outer_iterations": len(spc), "sweeps": int(sum(spc)),
                                        "sweeps_per_call": spc, "tolerence": 10}
            del r3
            box = [None]
            if rank == 0:             # the same iterate() on one GPU: counts must agree
                g.set_Z(g.X)
                emb.sweeps_per_call, emb.amounts_per_call = [], []
                emb.minimum_amount_updated_Z = float("inf")
                emb.tolerences["global"].reset()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                emb.iterate()
                torch.cuda.synchronize()
                box[0] = (list(emb.sweeps_per_call), time.perf_counter() - t0)
            dist.broadcast_object_list(box, 0)
            line["time_to_converge"]["single_gpu_sweeps_per_call"] = box[0][0]
            line["time_to_converge"]["single_gpu_seconds"] = box[0][1]
            line["time_to_converge"]["counts_match_single_gpu"] = box[0][0] == list(spc)
            line["parity_vs_single_gpu"] = line["parity_vs_single_gpu"] and box[0][0] == list(spc)

    if not args.no_converge and world == 1:
        g.set_Z(g.X)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        emb.iterate()
        torch.cuda.synchronize()
        line["time_to_converge"] = {"seconds": time.perf_counter() - t0, "outer_iterations": len(emb.sweeps_per_call),
                                    "sweeps": int(sum(emb.sweeps_per_call)), "sweeps_per_call": emb.sweeps_per_call,
                                    "tolerence": 10}

    if world == 1 and name != "products" and args.workload is None and args.scale == 1.0 and not args.no_converge:
        # the strong-scaling reference of the N > 1 lines, taken by the driver's own N = 1 run as well
        n2, s2, d2, X2 = synth.make_graph("products", seed=0)
        g2 = Graph.from_arrays(n2, s2, d2, X2)
        del s2, d2
        ms2 = single_gpu_steps(torch, L, _lib, g2, sim, 30)
        line["products_n1"] = {"workload": "products-shape synthetic", "nodes": n2, "edges": g2._nnz, "dim": int(X2.shape[1]),
                               "ms_per_step": ms2, "value": g2._nnz / (ms2 * 1e-3), "unit": UNIT,
                               "whole_step_gbs": sweep_bytes(n2, g2._nnz, int(X2.shape[1])) / (ms2 * 1e-3) / 1e9,
                               "note": "secondary: the workload of the N > 1 lines on one GPU (30 sweeps, CUDA events); "
                                       "strong-scaling efficiency at N GPUs = value_N / (N * this value)"}
        del g2, X2

    if rank == 0 and not args.no_cpu_baseline and world == 1:
        ve, vthreads, vtimes, _ = vectorised_cpu_sweeps(n, src, dst, X)
        line["cpu_baseline_vectorised"] = {
            "value": ve / float(np.mean(vtimes)), "unit": UNIT, "cores": vthreads, "kind": "port",
            "sample": f"{len(vtimes)} whole sweeps, torch-CPU sparse CSR SpMM + axpy + L1 on all host threads "
                      "(BASELINE.md section 3 item iii; timing only -- torch's summation order, not the reference's)"}
        line["cpu_baseline_reference_python"] = {
            "value": None, "unit": UNIT,
            "sample": "the unmodified reference (pure Python, O(N*E) per sweep; 210 edges/s measured at Cora shape in "
                      "the build container, BASELINE.md) cannot run here: /root/reference does not exist on the GPU box"}
        ce, _, threads, times, what = cpu_sweeps(n, src, dst, X, budget_s=12.0, min_sweeps=3, max_sweeps=200,
                                              step_budget_s=4.0)
        timed = times[1:]
        line["cpu_baseline"] = {"value": ce / float(np.mean(timed)), "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"{len(timed)} {what} of the same {name}-shape graph (after 1 warm-up), "
                                          "oracle C port, OpenMP over rows"}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
        if line.get("parity_vs_single_gpu") is False:
            raise SystemExit("sharded run differs from the single-GPU run")


def e2e_session(L, g, X, n, e, d, steps):
    """Same metric through the host-buffer C-ABI: upload CSR + X from pinned host memory, build P,
    `steps` sweeps with the patience state machine live (its amounts come back), download Z."""
    import torch
    from clane_b200 import _lib
    Xp = torch.from_numpy(np.ascontiguousarray(X)).pin_memory()
    rp = torch.from_numpy(g._rowptr).pin_memory()
    cp = torch.from_numpy(g._col).pin_memory()
    Zout = torch.empty([n, d], dtype=torch.float32).pin_memory()
    amounts = torch.empty(steps, dtype=torch.float32).pin_memory()
    torch.cuda.synchronize()
    best = None
    for _ in range(2):
        t0 = time.perf_counter()
        h = ctypes.c_void_p()
        _lib.check(L.clane_session_create(ctypes.byref(h), n, e, d, rp.data_ptr(), cp.data_ptr(), Xp.data_ptr(), 0))
        k = ctypes.c_int32()
        _lib.check(L.clane_session_propagate(h, ctypes.c_float(float(np.float32(GAMMA))), 1 << 30, steps, amounts.data_ptr(),
                                             steps, ctypes.byref(k)))
        _lib.check(L.clane_session_get_z(h, Zout.data_ptr()))
        dt = time.perf_counter() - t0
        L.clane_session_destroy(h)
        assert k.value == steps
        best = dt if best is None else min(best, dt)
    h2d = n * d * 4 + 4 * (n + 1) + 4 * e
    d2h = n * d * 4 + 4 * steps
    return {"value": e * steps / best, "unit": UNIT, "h2d_bytes_per_step": h2d / steps, "d2h_bytes_per_step": d2h / steps,
            "seconds": best, "steps": steps,
            "note": "clane_session_create + clane_session_propagate(max_sweeps=steps) + clane_session_get_z from pinned "
                    "host buffers; the upload, build_P and the download are inside the timed region and amortised over "
                    "the steps of the call, as in a real propagate()"}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
