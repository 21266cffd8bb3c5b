"""ctypes binding of libclane_b200.so (include/clane_b200.h).

There is no CPU fallback: if the shared library is missing, or a device entry point is
called without a CUDA device, this module raises.  The oracle under ``oracle/`` is never
imported from here.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG = Path(__file__).resolve().parent
import os as _os
LIB_PATH = Path(_os.environ["CLANE_LIB"]) if _os.environ.get("CLANE_LIB") else _PKG / "libclane_b200.so"

c_f32p = C.POINTER(C.c_float)
c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_vp = C.c_void_p


class Patience(C.Structure):
    """Mirror of ``struct clane_patience`` (32 bytes)."""
    _fields_ = [("minimum", C.c_float), ("patience", C.c_int32), ("tol", C.c_int32), ("sweeps", C.c_int32),
                ("max_sweeps", C.c_int32), ("stop", C.c_int32), ("last_amount", C.c_float), ("reserved", C.c_int32)]


class Patience64(C.Structure):
    """Mirror of ``struct clane_patience64`` (40 bytes)."""
    _fields_ = [("minimum", C.c_double), ("last_amount", C.c_double), ("patience", C.c_int32), ("tol", C.c_int32),
                ("sweeps", C.c_int32), ("max_sweeps", C.c_int32), ("stop", C.c_int32), ("reserved", C.c_int32)]


CLANE_EUNSUPPORTED = -9


class ClaneError(RuntimeError):
    pass


# name -> (restype, argtypes); mirrors include/clane_b200.h declaration by declaration
SIGNATURES = {
    "clane_version": (C.c_int, []),
    "clane_error_string": (C.c_char_p, [C.c_int]),
    "clane_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "clane_padded_ld": (C.c_int32, [C.c_int32]),
    "clane_csr_from_edges": (C.c_int64, [c_vp, c_vp, C.c_int64, C.c_int64, c_vp, c_vp]),
    "clane_edges_open": (C.c_int, [C.c_char_p, C.c_int64, C.c_int64, C.c_char_p, C.c_int32, C.POINTER(c_vp), c_i64p, c_i64p,
                                   C.c_char_p, C.c_int32]),
    "clane_edges_read": (C.c_int, [c_vp, c_vp, c_vp]),
    "clane_edges_close": (C.c_int, [c_vp]),
    "clane_group_schedule": (C.c_int, [c_vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_vp, c_vp,
                                       c_i32p, c_vp, c_i32p, c_vp, c_i32p, c_i32p, c_i32p]),
    "clane_sweep_program": (C.c_int, [c_vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_vp, C.c_int64,
                                      c_i64p]),
    "clane_plan_create": (C.c_int, [C.POINTER(c_vp), C.c_int32, C.c_int64, C.c_int32, c_vp, C.c_int32, C.c_int32,
                                    C.c_int32]),
    "clane_plan_destroy": (C.c_int, [c_vp]),
    "clane_plan_info": (C.c_int, [c_vp, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p]),
    "clane_cascade_shape": (C.c_int, [C.c_int64, c_i64p, c_i64p]),
    "clane_edge_rows": (C.c_int, [c_vp, C.c_int32, C.c_int64, c_vp, c_vp]),
    "clane_scores_cosine": (C.c_int, [c_vp, c_vp, c_vp, c_vp, C.c_int64, C.c_int64, c_vp, c_vp, c_vp]),
    "clane_norms_partial": (C.c_int, [c_vp, c_vp, c_vp, c_vp, C.c_int64, C.c_int64, c_vp, c_vp]),
    "clane_norms_finish": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "clane_row_softmax": (C.c_int, [c_vp, c_vp, C.c_int32, C.c_int32, c_vp, c_vp, c_vp]),
    "clane_plan_softmax": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "clane_asym_supported": (C.c_int, [C.c_int32]),
    "clane_asym_project": (C.c_int, [c_vp, C.c_int32, C.c_int32, C.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "clane_build_p_asym": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "clane_asym_project_fp32": (C.c_int, [c_vp, C.c_int32, C.c_int32, C.c_int32, c_vp, C.c_int32, c_vp, c_vp, c_vp, c_vp,
                                          c_vp]),
    "clane_build_p_asym_fp32": (C.c_int, [c_vp, c_vp, c_vp, C.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "clane_cosine_finalize": (C.c_int, [c_vp, c_vp, C.c_int64, c_vp, c_vp]),
    "clane_build_p_cosine": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "clane_sweep": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_float, c_vp, c_vp, c_vp, C.c_int32, c_vp]),
    "clane_sweeps": (C.c_int, [c_vp, c_vp, c_vp, C.c_int32, c_vp, c_vp, c_vp, C.c_float, C.c_int32, C.c_int32, c_vp, c_vp,
                               C.c_int32, c_vp]),
    "clane_l1_diff": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp]),
    "clane_l1_partial": (C.c_int, [c_vp, c_vp, c_vp, C.c_int64, C.c_int64, c_vp, c_vp]),
    "clane_l1_finish": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_int32, c_vp]),
    "clane_l1_tail_values": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp]),
    "clane_l1_finish_values": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_int32, c_vp]),
    "clane_plan_set_peers": (C.c_int, [c_vp, C.c_int32, C.c_int32, c_vp, c_vp]),
    "clane_plan_set_peers_third": (C.c_int, [c_vp, c_vp]),
    "clane_plan_set_multicast": (C.c_int, [c_vp, C.c_uint64, C.c_uint64]),
    "clane_plan_trace": (C.c_int, [c_vp, C.c_int, c_vp]),
    "clane_plan_profile": (C.c_int, [c_vp, C.c_int]),
    "clane_plan_profile_read": (C.c_int, [c_vp, c_f32p]),
    "clane_patience_reset": (C.c_int, [c_vp, C.c_int32, C.c_int32, c_vp]),
    "clane_padded_ld_f64": (C.c_int32, [C.c_int32]),
    "clane_work_f64": (C.c_int64, [C.c_int64]),
    "clane_patience_reset_f64": (C.c_int, [c_vp, C.c_int32, C.c_int32, c_vp]),
    "clane_l1_diff_f64": (C.c_int, [C.c_int32, C.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "clane_row_softmax_f64": (C.c_int, [c_vp, c_vp, C.c_int32, C.c_int32, c_vp, c_vp, c_vp]),
    "clane_build_p_cosine_f64": (C.c_int, [C.c_int32, C.c_int64, C.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                           c_vp]),
    "clane_sweep_f64": (C.c_int, [C.c_int32, C.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_double, c_vp, c_vp, c_vp,
                                  C.c_int32, c_vp, c_vp]),
    "clane_sweeps_f64": (C.c_int, [C.c_int32, C.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp, C.c_int32, C.c_double, C.c_int32,
                                   c_vp, c_vp, C.c_int32, c_vp, c_vp]),
    "clane_session_create": (C.c_int, [C.POINTER(c_vp), C.c_int32, C.c_int64, C.c_int32, c_vp, c_vp, c_vp, C.c_int32]),
    "clane_session_destroy": (C.c_int, [c_vp]),
    "clane_session_set_z": (C.c_int, [c_vp, c_vp]),
    "clane_session_get_z": (C.c_int, [c_vp, c_vp]),
    "clane_session_build_p": (C.c_int, [c_vp, c_vp]),
    "clane_session_propagate": (C.c_int, [c_vp, C.c_float, C.c_int32, C.c_int32, c_vp, C.c_int32, c_i32p]),
    "clane_session_iterate": (C.c_int, [c_vp, C.c_float, C.c_int32, C.c_int32, c_f32p, c_vp, C.c_int32, c_i32p]),
    "clane_session_sweeps": (C.c_int, [c_vp, C.c_float, C.c_int32, c_f32p]),
}

_lib = None


def lib() -> C.CDLL:
    """Load libclane_b200.so (built in-tree by clane_b200/build.py).  Fails loudly."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ClaneError(
                f"{LIB_PATH} is missing: build it with `python -m clane_b200.build` "
                "(nvcc, sm_100a).  clane_b200 has no CPU fallback.")
        L = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code: int, what: str = "") -> int:
    """Raise ClaneError for a non-zero return code of a C-ABI call."""
    if code != 0:
        msg = lib().clane_error_string(int(code)).decode()
        raise ClaneError(f"{what or 'clane call'} failed: {msg} (code {code})")
    return code


def require_cuda():
    """The hot path runs on a B200 or not at all."""
    import torch
    if not torch.cuda.is_available():
        raise ClaneError("clane_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def ptr(t) -> int:
    """data_ptr of a torch tensor (or 0 for None)."""
    return 0 if t is None else t.data_ptr()


def stream_handle() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


class Plan:
    """Owner of a ``clane_plan`` handle (device-side schedule + reduction scratch)."""

    def __init__(self, n: int, e: int, d: int, rowptr_host=None, row_lo: int = 0, row_hi: int | None = None,
                 hub_threshold: int = 0):
        require_cuda()
        self.handle = c_vp()
        self.n, self.e, self.d = int(n), int(e), int(d)
        rp = 0
        if rowptr_host is not None:
            self._rowptr = rowptr_host          # keep alive during the call
            rp = rowptr_host.ctypes.data
        hi = self.n if row_hi is None else int(row_hi)
        check(lib().clane_plan_create(C.byref(self.handle), self.n, self.e, self.d, rp, int(row_lo), hi,
                                      int(hub_threshold)), "clane_plan_create")
        g, ns, nh, nf, fu, la = (C.c_int32() for _ in range(6))
        check(lib().clane_plan_info(self.handle, C.byref(g), C.byref(ns), C.byref(nh), C.byref(nf), C.byref(fu),
                                    C.byref(la)))
        self.group_rows, self.n_spans, self.n_hub_rows, self.n_fix_groups = g.value, ns.value, nh.value, nf.value
        self.fused_l1, self.launches_per_sweep = bool(fu.value), la.value

    def __del__(self):
        try:
            if getattr(self, "handle", None) and self.handle.value:
                lib().clane_plan_destroy(self.handle)
                self.handle = c_vp()
        except Exception:
            pass
