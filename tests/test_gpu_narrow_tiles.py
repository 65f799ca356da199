"""Narrow tiles of the persistent kernel (-m gpu; csrc/mega.cu): a tile of the plan whose columns span less than 65536 streams
them as 16-bit codes relative to the tile's smallest column instead of 32-bit indices.  The choice is made per tile from the
matrix; the arithmetic must not notice it: same accumulation order, bitwise the same SpMV as the stand-alone thread-per-row
kernel.  `mega_tiles` reports how many tiles of the plan are narrow."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

from helpers import METHODS, RR, SMALL_CASES, global_csr

pytestmark = pytest.mark.gpu

TOL = 1e-10
V_P, V_S = 3, 4


@pytest.fixture(autouse=True)
def _opts(B):
    B.set_options(quiet=1, tol=TOL, max_iter=1000, cache=1, mega=1, resident=0)
    yield
    B.set_options(resident=1, tol=1e-15, max_iter=1000, mega=1, spmv_lanes=0)


def _check_solve(B, O, dm, method, n, ptr, col, val, rows=slice(None)):
    kw = RR if method.endswith("rr") else {}
    b = O.spmv(n, ptr, col, val, np.ones(n))
    ref = O.solve(method, n, ptr, col, val, b, tol=TOL, max_iter=1000, **kw)
    x = np.zeros(n)
    it, st = dm.solve(method, x, b.copy(), **kw)
    assert st["kernel_launches"] <= 8                         # the loop ran as the persistent kernel
    h, want = np.sqrt(B.last_history()), np.sqrt(ref["hist"])
    m = min(10, it, ref["iters"])
    assert np.all(np.abs(h[1:m + 1] - want[1:m + 1]) <= 1e-10 * want[1:m + 1] + 1e-15), (method, h[1:m + 1], want[1:m + 1])
    assert abs(it - ref["iters"]) <= max(2, int(0.02 * ref["iters"])), (method, it, ref["iters"])
    assert np.abs(x[rows] - 1).max() < 1e-6


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("name,kind,g,p0", [c for c in SMALL_CASES if c[1] != "random"])
def test_banded_small_cases_are_all_narrow(B, O, name, kind, g, p0, method):
    blk, n, ptr, col, val = global_csr(B, kind, g, p0)
    dm = B.DeviceMatrix(blk)
    try:
        tiles, narrow = dm.mega_tiles()
        assert tiles > 0 and narrow == tiles
        _check_solve(B, O, dm, method, n, ptr, col, val)
    finally:
        dm.destroy()


def _mixed(special_col):
    """Band matrix (offsets +-1, +-300) of 240 000 rows with
      * rows 302 .. 19 999 also referencing column 0, so every tile among the first 20 000 rows has column 0 as its smallest;
      * row 15 000 referencing `special_col`: its tile spans exactly special_col columns;
      * rows 200 000 .. 201 999 referencing a column 150 000 places back: wide tiles;
      * empty rows (single ones and a run of 100), whose columns no row references either, so the system stays regular
        on the other rows.
    Row lengths vary (3 .. 6 entries), so tiles start at entries of every alignment."""
    n = 240000
    rng = np.random.default_rng(5)
    i = np.arange(n)
    r, c = [], []
    for o in (-300, -1, 1, 300):
        k = (i + o >= 0) & (i + o < n)
        r.append(i[k]); c.append(i[k] + o)
    a = np.arange(302, 20000)
    r.append(a); c.append(np.zeros_like(a))
    r.append(np.array([15000])); c.append(np.array([special_col]))
    f = np.arange(200000, 202000)
    r.append(f); c.append(f - 150000)
    r, c = np.concatenate(r), np.concatenate(c)
    empty = np.concatenate([np.arange(100003, 110000, 997), np.arange(120000, 120100)])
    keep = np.ones(n, dtype=bool)
    keep[empty] = False
    m = keep[r] & keep[c]
    r, c = r[m], c[m]
    A = sp.csr_matrix((-(0.2 + 0.6 * rng.random(r.size)), (r, c)), shape=(n, n))
    d = np.where(keep, np.asarray(abs(A).sum(axis=1)).ravel() + 0.5 + rng.random(n), 0.0)
    A = sp.csr_matrix(A + sp.diags(d))
    A.eliminate_zeros()
    A.sort_indices()
    assert np.all(np.diff(A.indptr)[empty] == 0)
    return n, A, keep


def test_mixed_matrix_narrow_and_wide_tiles(B, O):
    """Tiles spanning 65 535 columns are narrow, 65 536 wide: the two variants of the matrix differ in that one entry only
    (same row lengths, same plan) and by exactly one narrow tile.  Both solve like the oracle."""
    counts = []
    for special in (65535, 65536):
        n, A, keep = _mixed(special)
        blk = B.blocks_from_csr(n, A.indptr, A.indices, A.data)
        dm = B.DeviceMatrix(blk)
        try:
            tiles, narrow = dm.mega_tiles()
            assert 0 < narrow < tiles
            counts.append((tiles, narrow))
            _check_solve(B, O, dm, "bicgstab", n, A.indptr, A.indices, A.data, rows=keep)
        finally:
            dm.destroy()
    (t0, n0), (t1, n1) = counts
    assert t0 == t1 and n0 == n1 + 1, counts


def test_mixed_matrix_spmv_is_bitwise_the_thread_per_row_kernel(B):
    """s = A p of a one-iteration persistent-kernel solve equals, bit for bit, the stand-alone SpMV with one thread per row:
    both add a row's products left to right with fma from 0."""
    n, A, keep = _mixed(65535)
    B.set_options(spmv_lanes=1, tol=0.0, max_iter=1)
    blk = B.blocks_from_csr(n, A.indptr, A.indices, A.data)
    dm = B.DeviceMatrix(blk)
    try:
        tiles, narrow = dm.mega_tiles()
        assert 0 < narrow < tiles
        b = dm.spmv(np.ones(n))
        x = np.zeros(n)
        it, st = dm.solve("bicgstab", x, b)
        assert it == 1 and st["kernel_launches"] <= 8
        p, s = np.empty(n), np.empty(n)
        B.lib.bicg_debug_get_vec(dm.h, V_P, p.ctypes.data_as(C.c_void_p))
        B.lib.bicg_debug_get_vec(dm.h, V_S, s.ctypes.data_as(C.c_void_p))
        assert np.abs(p).max() > 0
        want = dm.spmv(p)
        assert np.array_equal(s.view(np.uint64), want.view(np.uint64))
    finally:
        dm.destroy()


def test_random_columns_keep_wide_tiles(B, O):
    """cfg-5 family (random columns over 200 000 rows) forced onto the persistent kernel: every tile spans far more than
    65 536 columns, so all of them stream 32-bit columns.  Their SpMV is bitwise the thread-per-row kernel's, and the solve
    converges like the oracle's.  (No check of the history against the oracle at 1e-10: on this matrix the dot products'
    summation order alone moves it by a few 1e-10 within the first iterations, whichever column width the tiles use.)"""
    B.set_options(mega=2, spmv_lanes=1)
    blk, n, ptr, col, val = global_csr(B, "random", 200000, 8)
    dm = B.DeviceMatrix(blk)
    try:
        tiles, narrow = dm.mega_tiles()
        assert tiles > 0 and narrow == 0
        B.set_options(tol=0.0, max_iter=1)
        b = dm.spmv(np.ones(n))
        x = np.zeros(n)
        it, st = dm.solve("bicgstab", x, b)
        assert it == 1 and st["kernel_launches"] <= 8
        p, s = np.empty(n), np.empty(n)
        B.lib.bicg_debug_get_vec(dm.h, V_P, p.ctypes.data_as(C.c_void_p))
        B.lib.bicg_debug_get_vec(dm.h, V_S, s.ctypes.data_as(C.c_void_p))
        assert np.array_equal(s.view(np.uint64), dm.spmv(p).view(np.uint64))

        B.set_options(tol=TOL, max_iter=1000)
        b = O.spmv(n, ptr, col, val, np.ones(n))
        ref = O.solve("bicgstab", n, ptr, col, val, b, tol=TOL, max_iter=1000)
        x = np.zeros(n)
        it, st = dm.solve("bicgstab", x, b.copy())
        assert st["kernel_launches"] <= 8
        assert abs(it - ref["iters"]) <= 2, (it, ref["iters"])
        assert np.abs(x - 1).max() < 1e-6
    finally:
        dm.destroy()
