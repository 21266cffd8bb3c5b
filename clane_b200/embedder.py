"""Embedder -- drop-in for ``clane.embedder.Embedder`` (/root/reference/clane/embedder.py:12-108).

Same constructor, ``iterate()``, ``propagate()``, ``history`` and ``minimum_amount_updated_Z``;
the per-vertex Python loop of embedder.py:85-92 becomes one ``clane_sweep`` C-ABI call per
sweep (fused gather-SpMM + residual, exact L1 change, device-side patience state machine); a
whole ``propagate()`` is ONE ``clane_sweeps`` call -- a CUDA graph whose conditional WHILE node
repeats batches of sweeps until the device-side patience counter reaches zero.  Work enqueued
after that point is a device-side no-op, so the result is exactly the reference's (same sweep
count, same Z).
"""
from __future__ import annotations

import ctypes
import queue
import threading
from pathlib import Path

import numpy as np
import torch

from . import _lib
from .graph import Graph
from .similarity import Similarity

Inf = float("inf")


class SavedZ(object):
    """History entry that lives on disk (streamed ``--save_history``): quacks like the tensor the reference keeps
    in ``history["Z"]`` as far as its CLI uses it (``.cpu().numpy()``), and loads on demand."""

    def __init__(self, path: Path) -> None:
        self.path = Path(path)

    def cpu(self):
        return self

    def numpy(self) -> np.ndarray:
        return np.load(self.path)

    def __array__(self, dtype=None, copy=None):
        a = np.load(self.path)
        return a if dtype is None else a.astype(dtype)


class HistoryWriter(object):
    """Streams the per-sweep embeddings of ``--save_history`` to ``root/{outer}/Z_{sweep}.npy`` (the layout of
    /root/reference/clane/__main__.py:73-82) while the sweeps run: each sweep's Z goes device -> one of three pinned
    host buffers -> a writer thread, instead of accumulating N*d*4 bytes per sweep in host memory until the end."""

    def __init__(self, root: Path, n: int, d: int, dtype: torch.dtype = torch.float32) -> None:
        self.root = Path(root)
        self.free, self.work = queue.Queue(), queue.Queue()
        for _ in range(3):
            self.free.put(torch.empty([n, d], dtype=dtype).pin_memory())
        self.error = None
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self) -> None:
        while True:
            item = self.work.get()
            if item is None:
                return
            buf, path = item
            try:
                path.parent.mkdir(parents=True, exist_ok=True)
                np.save(path, buf.numpy())
            except Exception as exc:          # surfaced by close()
                self.error = exc
            self.free.put(buf)

    def put(self, z_dev: torch.Tensor, outer: int, sweep: int) -> SavedZ:
        """``z_dev`` [n, d] (a view of the padded device matrix), already final on the current stream's timeline."""
        buf = self.free.get()                 # back-pressure: at most three sweeps in flight
        buf.copy_(z_dev)                      # synchronous device -> pinned copy
        path = self.root.joinpath(f"{outer}", f"Z_{sweep}.npy")
        self.work.put((buf, path))
        return SavedZ(path)

    def close(self) -> None:
        self.work.put(None)
        self.thread.join()
        if self.error is not None:
            raise self.error


class Embedder(object):
    def __init__(
        self,
        graph:              Graph,
        similarity_measure: Similarity,
        device,
        gamma:              float = 0.76,
        tolerence:          int = 10,
        batch_size:         int = 4,
        lr:                 float = 1e-4,
        num_workers:        int = 0,
        save_history:       bool = False,
    ) -> None:
        self.graph = graph
        self.similarity_measure = similarity_measure
        self.device = device
        self.gamma = gamma
        self.tolerences = {
            "global": self.Tolerence(tolerence),
            "propagation": self.Tolerence(tolerence),
            "similarity_model": self.Tolerence(tolerence),
        }
        self.batch_size = batch_size
        self.lr = lr
        self.num_workers = num_workers
        self.save_history = save_history
        if save_history:
            self.history = {"Z": [], "loss_P": []}
        self.minimum_amount_updated_Z = Inf
        self.history_root = None       # set (a directory) to stream history["Z"] to disk while iterating
        self._history_writer = None
        self.verbose = True            # the reference prints `amount counter` per sweep (embedder.py:104)
        self.sweeps_per_call = []      # bookkeeping the parity tests read
        self.amounts_per_call = []

    class Tolerence:
        def __init__(self, initial_value):
            self.initial_value = initial_value
            self.value = initial_value

        def reset(self):
            self.value = self.initial_value

        def endure(self):
            self.value -= 1

    # ---------------------------------------------------------------------------------------
    def iterate(self):
        """Outer loop (embedder.py:56-69): propagate until the outer L1 change stops improving."""
        g = self.graph
        L = _lib.lib()
        S = g._device_state()
        prev = torch.empty_like(S.Z[0])
        if self.save_history and self.history_root is not None:
            self._history_writer = HistoryWriter(self.history_root, S.n, S.d, S.dtype)
        try:
            self._iterate(g, L, S, prev)
        finally:
            if self._history_writer is not None:
                writer, self._history_writer = self._history_writer, None
                writer.close()

    def _iterate(self, g, L, S, prev):
        while True:
            prev.copy_(S.Z[S.cur])
            self.propagate()
            if S.dtype == torch.float64:
                _lib.check(L.clane_l1_diff_f64(S.n, S.d, S.Z[S.cur].data_ptr(), prev.data_ptr(), S.work.data_ptr(),
                                               S.amount.data_ptr(), _lib.stream_handle()), "clane_l1_diff_f64")
            else:
                _lib.check(L.clane_l1_diff(S.plan.handle, S.Z[S.cur].data_ptr(), prev.data_ptr(), S.amount.data_ptr(),
                                           _lib.stream_handle()), "clane_l1_diff")
            amount_updated_Z_current = float(S.amount.cpu()[0])   # synchronises the current stream
            if self.minimum_amount_updated_Z > amount_updated_Z_current:
                self.tolerences['global'].reset()
                self.minimum_amount_updated_Z = amount_updated_Z_current
            else:
                self.tolerences['global'].endure()
            if self.tolerences['global'].value == 0:  # embeddings are no more updated
                break

    # ---------------------------------------------------------------------------------------
    @torch.no_grad()
    def propagate(self, max_sweeps: int = 0):
        """Jacobi sweeps with P frozen until the patience counter reaches 0 (embedder.py:71-108)."""
        g = self.graph
        L = _lib.lib()
        S = g._device_state()
        g._build_P_device(self.similarity_measure)
        tol = self.tolerences['propagation']
        tol.reset()
        # the sweeps run on the graph's own stream (capturable, so whole sweeps replay as CUDA graphs)
        caller = torch.cuda.current_stream()
        S.stream.wait_stream(caller)
        stream = S.stream.cuda_stream
        f64 = S.dtype == torch.float64
        if f64:
            _lib.check(L.clane_patience_reset_f64(S.state.data_ptr(), int(tol.initial_value), int(max_sweeps), stream),
                       "clane_patience_reset_f64")
            gamma = ctypes.c_double(float(self.gamma))     # gamma scales a double tensor: not rounded to fp32
        else:
            _lib.check(L.clane_patience_reset(S.state.data_ptr(), int(tol.initial_value), int(max_sweeps), stream),
                       "clane_patience_reset")
            gamma = ctypes.c_float(float(np.float32(self.gamma)))
        history_Z = [] if self.save_history else None
        start = S.cur

        def read_state():
            with torch.cuda.stream(S.stream):
                S.state_host.copy_(S.state, non_blocking=True)
            S.stream.synchronize()
            return (_lib.Patience64 if f64 else _lib.Patience).from_buffer_copy(S.state_host.numpy().tobytes())

        if f64 and history_Z is None:
            # batches of sweeps enqueued directly, one sync each; sweeps past the stop are device-side no-ops
            st = None
            while st is None or not st.stop:
                _lib.check(L.clane_sweeps_f64(S.n, S.d, S.rowptr.data_ptr(), S.col.data_ptr(), S.w.data_ptr(),
                                              S.X.data_ptr(), S.Zptrs, start, gamma, 12, S.state.data_ptr(),
                                              S.log.data_ptr(), S.log_cap, S.work.data_ptr(), stream), "clane_sweeps_f64")
                st = read_state()    # 12 sweeps = whole rotations: every batch starts at the same buffer
        elif history_Z is None:
            # the whole call is ONE graph launch: a conditional WHILE node repeats batches of sweeps (the L1 / patience
            # tail of every sweep beside the rows of the next one) until the device-side patience counter hits zero
            rc = L.clane_sweeps(S.plan.handle, S.X.data_ptr(), S.Zptrs, start, S.rowptr.data_ptr(), S.col.data_ptr(),
                                S.w.data_ptr(), gamma, 0, 1, S.state.data_ptr(), S.log.data_ptr(), S.log_cap, stream)
            if rc == _lib.CLANE_EUNSUPPORTED:      # long sweeps (enqueued directly) or no conditional nodes: batches, one sync each
                st = None
                while st is None or not st.stop:
                    _lib.check(L.clane_sweeps(S.plan.handle, S.X.data_ptr(), S.Zptrs, start, S.rowptr.data_ptr(),
                                              S.col.data_ptr(), S.w.data_ptr(), gamma, 12, 0, S.state.data_ptr(),
                                              S.log.data_ptr(), S.log_cap, stream), "clane_sweeps")
                    st = read_state()    # 12 sweeps = whole rotations: every batch starts at the same buffer
            else:
                _lib.check(rc, "clane_sweeps")
                st = read_state()
        else:
            # save_history: one sweep per call, its Z copied out before the next one starts
            k = 0
            while True:
                src, dst = S.Z[(start + k) % 3], S.Z[(start + k + 1) % 3]
                if f64:
                    _lib.check(L.clane_sweep_f64(S.n, S.d, S.rowptr.data_ptr(), S.col.data_ptr(), S.w.data_ptr(),
                                                 S.X.data_ptr(), src.data_ptr(), dst.data_ptr(), gamma, None,
                                                 S.state.data_ptr(), S.log.data_ptr(), S.log_cap, S.work.data_ptr(),
                                                 stream), "clane_sweep_f64")
                else:
                    _lib.check(L.clane_sweep(S.plan.handle, S.X.data_ptr(), src.data_ptr(), dst.data_ptr(),
                                             S.rowptr.data_ptr(), S.col.data_ptr(), S.w.data_ptr(), gamma,
                                             0, S.state.data_ptr(), S.log.data_ptr(), S.log_cap, stream), "clane_sweep")
                k += 1
                st = read_state()
                if self._history_writer is not None:
                    history_Z.append(self._history_writer.put(dst[:S.n, :S.d], len(self.history['Z']), len(history_Z)))
                else:
                    history_Z.append(dst[:S.n, :S.d].cpu())
                if st.stop:
                    break
        done = int(st.sweeps)
        caller.wait_stream(S.stream)
        S.cur = (start + done) % 3         # sweep i read Z[(start + i) % 3] and wrote the next buffer
        amounts = S.log[:min(done, S.log_cap)].cpu().numpy()
        self.sweeps_per_call.append(done)
        self.amounts_per_call.append(amounts)

        # replay the counter for the per-sweep line of embedder.py:104 and the final state
        minimum = Inf
        for a in amounts:
            if minimum > a:
                tol.reset()
                minimum = a
            else:
                tol.endure()
            if self.verbose:
                print(torch.tensor(a), tol.value)
        if history_Z is not None:
            self.history['Z'].append(history_Z)
        return


class IterativeEmbedder(Embedder):
    """Named placeholder for the reference's IterativeEmbedder (embedder.py:158-289) -- a spec decision, see DESIGN.md
    section 7.  Upstream the class cannot be constructed (its __init__ omits the required ``device``: TypeError;
    the reference's own asymmetric CLI test errors), reads an undefined ``self.tolerence`` and calls an undefined
    ``self.update_embeddings``: there is no behaviour a parity test could pin, so any working version would be a
    new algorithm.  The name exists so that ``from clane.embedder import IterativeEmbedder`` (reference
    __main__.py:12) keeps importing and the trainable-plugin branch of the CLI fails loudly."""

    def __init__(self, *args, **kwargs):
        raise NotImplementedError(
            "IterativeEmbedder is dead code in the reference (TypeError at construction, undefined attributes past it) "
            "and is deliberately not implemented (DESIGN.md section 7); use Embedder with a non-trainable similarity.")
