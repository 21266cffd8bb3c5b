"""Host-side checks of the fp64 path that need no GPU: the reduction scratch size of the C-ABI, and the fp64
oracle's softmax pieces against torch's own: the exported Sleef expd u10 and torch's double softmax."""
import ctypes
import os
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from clane_b200 import _lib
from oracle_f64 import oracle_f64 as O


def _ceil_log2(x):
    return 0 if x <= 1 else (x - 1).bit_length()


def _scratch_needed(m):
    """Doubles the level kernels of the fp64 cascade write for a reduction over m elements (16 per node)."""
    ni = m // 16
    step = 1 << max(4, _ceil_log2(ni) // 4)
    m1, m2 = ni // step, ni // step // step
    return (-(-ni // step) + -(-m1 // step) + -(-m2 // step) + 1) * 16


def test_work_f64_covers_every_smaller_reduction():
    """One scratch buffer serves the sweeps' L1 (n*d elements) and build_P's norms (e*d): the size for m must cover
    every m' <= m, also across the step changes at 2^19 and 2^23 cascade rows where the need drops by about half."""
    L = _lib.lib()
    grid = sorted({m for b in (1 << 23, 1 << 27) for k in range(-64, 65) for m in (b + 16 * k, b + 16 * k * 997)} |
                  {int(m) for m in np.geomspace(1, 3e9, 400)})
    sizes = [int(L.clane_work_f64(m)) for m in grid]
    assert all(a <= b for a, b in zip(sizes, sizes[1:])), "clane_work_f64 is not non-decreasing"
    best = 0
    for m, s in zip(grid, sizes):
        best = max(best, _scratch_needed(m))
        assert s >= best, f"m={m}: {s} doubles < {best} needed by a reduction of at most m elements"
    # the graphs where sizing by max(n*d, e*d) alone fell short
    for n, e, d in [(60_000, 100_000, 128), (1_000_000, 1_500_000, 128), (100_000, 80_000, 100), (65_536, 70_000, 128)]:
        w = int(L.clane_work_f64(max(n * d, e * d)))
        assert w >= _scratch_needed(n * d) and w >= _scratch_needed(e * d)


def _sleef_expd():
    """ctypes wrapper around the Sleef_expd*_u10 that libtorch_cpu exports (what torch's double softmax calls)."""
    gcc = shutil.which("gcc") or ("/usr/bin/gcc" if Path("/usr/bin/gcc").exists() else None)
    tlib = Path(torch.__file__).resolve().parent / "lib"
    if gcc is None or not (tlib / "libtorch_cpu.so").exists():
        pytest.skip("needs gcc and libtorch_cpu.so")
    avx512 = "avx512f" in Path("/proc/cpuinfo").read_text()
    width, vec, isa = (8, "__m512d", "-mavx512f") if avx512 else (4, "__m256d", "-mavx2")
    load, store = ("_mm512_loadu_pd", "_mm512_storeu_pd") if avx512 else ("_mm256_loadu_pd", "_mm256_storeu_pd")
    return gcc, tlib, width, vec, isa, load, store


def test_exp_matches_exported_sleef(tmp_path):
    gcc, tlib, width, vec, isa, load, store = _sleef_expd()
    src = tmp_path / "sleefw.c"
    src.write_text(f"#include <immintrin.h>\n#include <stdint.h>\nextern {vec} Sleef_expd{width}_u10({vec});\n"
                   f"void expd(const double* x, double* y, int64_t n) {{\n"
                   f"    for (int64_t i = 0; i < n; i += {width}) {store}(y + i, Sleef_expd{width}_u10({load}(x + i)));\n}}\n")
    so = tmp_path / "libsleefw.so"
    env = dict(os.environ)
    env.pop("CC", None)
    subprocess.run([gcc, "-O1", isa, "-mfma", "-shared", "-fPIC", str(src), "-o", str(so), f"-L{tlib}", "-ltorch_cpu",
                    "-lc10", f"-Wl,-rpath,{tlib}"], check=True, env=env)
    f = ctypes.CDLL(str(so)).expd
    f.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]
    rng = np.random.default_rng(7)
    x = np.concatenate([np.linspace(-1000.0, 0.0, 2_000_001),       # the whole range softmax uses (s - max <= 0)
                        np.linspace(-2.0, 0.0, 1_000_001),          # dense where rows are flat
                        -rng.random(1_000_000) * 1100.0, rng.random(200_000) * 709.0,
                        np.array([0.0, -0.0, -1e-300, -745.13321910194122, -1000.0, -1000.0000000000001, 709.7, 710.0])])
    x = np.ascontiguousarray(np.concatenate([x, np.zeros(-len(x) % width)]))
    want = np.empty_like(x)
    f(x.ctypes.data, want.ctypes.data, len(x))
    got = O.exp(x)
    bad = np.flatnonzero(want.view(np.int64) != got.view(np.int64))
    assert bad.size == 0, f"{bad.size} of {len(x)} differ, first at x={x[bad[0]]!r}"


@pytest.mark.parametrize("k", [8, 9, 15, 16, 17, 23, 24, 31, 40])
def test_softmax_reduce_order_matches_torch(k):
    """Masking-style probe of reduce_all's order: one term of exactly 1 (the row max) at every position among tiny
    terms just under half an ulp of 1, so the result depends on which tiny terms are summed before they meet 1."""
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        for pos in range(k):
            for tiny in (0.45, 0.3, 0.2):
                s = np.full(k, np.log(tiny * 2.0 ** -53))
                s += np.arange(k) * 1e-3 * np.log1p(2.0 ** -40)          # distinct terms, still tiny
                s[pos] = 0.0
                want = torch.from_numpy(s).softmax(0).numpy()
                assert np.array_equal(O.softmax_rows(s, np.array([0, k])), want), f"k={k} pos={pos} tiny={tiny}"
    finally:
        torch.set_num_threads(threads)
