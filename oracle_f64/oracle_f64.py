"""ctypes front-end of the fp64 CPU oracle (oracle_f64/clane_oracle_f64.c).

TEST INFRASTRUCTURE ONLY, like oracle/oracle.py, whose entry points these mirror for content embeddings
that are float64: the reference then runs build_P, the sweeps, the L1 change and both patience loops in
double.  Nothing under ``clane_b200/`` imports this module.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_SRC = _HERE / "clane_oracle_f64.c"
_LIB_PATH = _HERE / "libclane_oracle_f64.so"
_lib = None

_f64p = C.POINTER(C.c_double)
_i64p = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)


def build(force: bool = False) -> Path:
    """Compile with the flags of oracle/Makefile: no contraction, no fast-math."""
    if force or not _LIB_PATH.exists() or _LIB_PATH.stat().st_mtime < _SRC.stat().st_mtime:
        cc = "/usr/bin/gcc" if Path("/usr/bin/gcc").exists() else "gcc"
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-mfma",
                        "-fopenmp", "-fvisibility=hidden", "-Wall", "-Wextra", "-o", str(_LIB_PATH), str(_SRC), "-lm"],
                       check=True)
    return _LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(_LIB_PATH))
        L.clane_oracle64_set_threads.argtypes = [C.c_int]
        L.clane_oracle64_aten_sum.argtypes = [_f64p, C.c_int64]
        L.clane_oracle64_aten_sum.restype = C.c_double
        L.clane_oracle64_l1_diff.argtypes = [_f64p, _f64p, C.c_int64]
        L.clane_oracle64_l1_diff.restype = C.c_double
        L.clane_oracle64_scores_raw.argtypes = [_f64p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p, _f64p, _f64p]
        L.clane_oracle64_exp.argtypes = [_f64p, _f64p, C.c_int64]
        L.clane_oracle64_softmax_rows.argtypes = [_f64p, C.c_int64, _i64p, _f64p]
        L.clane_oracle64_build_p.argtypes = [_f64p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p]
        L.clane_oracle64_sweep.argtypes = [_f64p, _f64p, _f64p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p, C.c_double]
        L.clane_oracle64_propagate.argtypes = [_f64p, _f64p, C.c_int64, C.c_int64, _i64p, _i32p, C.c_double,
                                               C.c_int64, C.c_int64, _f64p, C.c_int64, _f64p]
        L.clane_oracle64_propagate.restype = C.c_int64
        L.clane_oracle64_iterate.argtypes = [_f64p, _f64p, C.c_int64, C.c_int64, _i64p, _i32p, C.c_double,
                                             C.c_int64, C.c_int64, _i64p, _f64p, C.c_int64]
        L.clane_oracle64_iterate.restype = C.c_int64
        _lib = L
    return _lib


def _f64(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(_f64p)


def _i64(a):
    a = np.ascontiguousarray(a, dtype=np.int64)
    return a, a.ctypes.data_as(_i64p)


def _i32(a):
    a = np.ascontiguousarray(a, dtype=np.int32)
    return a, a.ctypes.data_as(_i32p)


def set_threads(t: int) -> None:
    lib().clane_oracle64_set_threads(int(t))


def aten_sum(x) -> np.float64:
    x, p = _f64(np.asarray(x).reshape(-1))
    return np.float64(lib().clane_oracle64_aten_sum(p, x.size))


def l1_diff(a, b) -> np.float64:
    a, pa = _f64(a)
    b, pb = _f64(b)
    assert a.size == b.size
    return np.float64(lib().clane_oracle64_l1_diff(pa, pb, a.size))


def exp(x):
    x, p = _f64(x)
    out = np.empty_like(x)
    lib().clane_oracle64_exp(p, out.ctypes.data_as(_f64p), x.size)
    return out


def scores_raw(Z, rowptr, col):
    """(dots[E], S1, S2): per-edge sequential dots and the two cascade-ordered square sums."""
    Z, pz = _f64(Z)
    rowptr, pr = _i64(rowptr)
    col, pc = _i32(col)
    n, d = Z.shape
    dots = np.empty(len(col), np.float64)
    s1, s2 = C.c_double(), C.c_double()
    lib().clane_oracle64_scores_raw(pz, n, d, pr, pc, dots.ctypes.data_as(_f64p), C.byref(s1), C.byref(s2))
    return dots, np.float64(s1.value), np.float64(s2.value)


def softmax_rows(scores, rowptr):
    scores, ps = _f64(scores)
    rowptr, pr = _i64(rowptr)
    w = np.empty_like(scores)
    lib().clane_oracle64_softmax_rows(ps, len(rowptr) - 1, pr, w.ctypes.data_as(_f64p))
    return w


def build_p(Z, rowptr, col):
    Z, pz = _f64(Z)
    rowptr, pr = _i64(rowptr)
    col, pc = _i32(col)
    n, d = Z.shape
    w = np.empty(len(col), np.float64)
    lib().clane_oracle64_build_p(pz, n, d, pr, pc, w.ctypes.data_as(_f64p))
    return w


def sweep(X, Zcur, rowptr, col, w, gamma: float):
    X, px = _f64(X)
    Zcur, pz = _f64(Zcur)
    rowptr, pr = _i64(rowptr)
    col, pc = _i32(col)
    w, pw = _f64(w)
    n, d = X.shape
    Zn = np.empty_like(Zcur)
    lib().clane_oracle64_sweep(px, pz, Zn.ctypes.data_as(_f64p), n, d, pr, pc, pw, float(gamma))
    return Zn


def propagate(X, Z, rowptr, col, gamma: float, tol: int, max_sweeps: int = 0, cap: int = 100000):
    """One propagate() call.  Returns (Z_new, amounts[sweeps], w[E])."""
    X, px = _f64(X)
    Z = np.array(Z, dtype=np.float64, order="C", copy=True)
    rowptr, pr = _i64(rowptr)
    col, pc = _i32(col)
    n, d = X.shape
    amounts = np.zeros(cap, np.float64)
    w = np.empty(len(col), np.float64)
    s = lib().clane_oracle64_propagate(px, Z.ctypes.data_as(_f64p), n, d, pr, pc, float(gamma), tol, max_sweeps,
                                       amounts.ctypes.data_as(_f64p), cap, w.ctypes.data_as(_f64p))
    return Z, amounts[:min(s, cap)].copy(), w


def iterate(X, rowptr, col, gamma: float, tol: int, Z0=None, max_outer: int = 0, cap: int = 4096):
    """Full iterate().  Returns (Z, sweeps_per_call[outer], outer_amounts[outer])."""
    X, px = _f64(X)
    Z = np.array(X if Z0 is None else Z0, dtype=np.float64, order="C", copy=True)
    rowptr, pr = _i64(rowptr)
    col, pc = _i32(col)
    n, d = X.shape
    spc = np.zeros(cap, np.int64)
    oam = np.zeros(cap, np.float64)
    o = lib().clane_oracle64_iterate(px, Z.ctypes.data_as(_f64p), n, d, pr, pc, float(gamma), tol, max_outer,
                                     spc.ctypes.data_as(_i64p), oam.ctypes.data_as(_f64p), cap)
    return Z, spc[:o].copy(), oam[:o].copy()
