"""CPU: the C-ABI library loads, exports every symbol include/bicgstab_b200.h declares, and its host-only entry
points (planning, generators, Matrix-Market loader) work without a GPU."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    txt = open(os.path.join(ROOT, "include", "bicgstab_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    txt = re.sub(r"typedef[^;]*;", "", txt)                       # function-pointer typedefs are not symbols
    names = set(re.findall(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*\([^;{}]*\)\s*;", txt))
    return {n for n in names if not n.startswith("bicg_allgather_fn") and n not in ("defined",)}


def test_every_declared_symbol_is_exported(B):
    declared = _declared_symbols()
    assert {"bicgstab", "ca_bicgstab", "pipe_bicgstab", "pipe_bicgstab_rr", "MPI_csr_spmv_ovlap",
            "MPI_csr_load_matrix_block", "csr_init_matrix", "csr_free_matrix"} <= declared
    out = subprocess.run(["nm", "-D", "--defined-only", B.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if l.strip()}
    missing = sorted(declared - exported)
    assert not missing, f"declared in include/bicgstab_b200.h but not exported: {missing}"
    assert declared <= set(B.SYMBOLS) | {"bicg_plan_push_runs"}, sorted(declared - set(B.SYMBOLS))


def test_struct_layouts_match_reference(B):
    # matrix.h:19-26 / 28-33 (SURVEY.md 8(a) a1, a2)
    assert C.sizeof(B.CSR_Matrix) == 40
    assert [getattr(B.CSR_Matrix, f).offset for f in ("val", "col", "ptr", "nz", "rows", "cols")] == [0, 8, 16, 24, 28, 32]
    assert C.sizeof(B.INFO_Matrix) == 32
    assert [getattr(B.INFO_Matrix, f).offset for f in ("nz", "rows", "cols", "code", "recvcounts", "displs")] == [0, 4, 8, 12, 16, 24]


def test_sass_is_blackwell_native(B):
    """The shipped cubin is sm_100a and the SpMV really uses the TMA bulk-copy path (UBLKCP) + mbarriers."""
    out = subprocess.run(["cuobjdump", "-lelf", B.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump not available")
    assert "sm_100a" in out.stdout
    sass = subprocess.run(["cuobjdump", "-sass", B.LIB_PATH], capture_output=True, text=True).stdout
    assert "UBLKCP" in sass and "SYNCS" in sass and "DFMA" in sass


@pytest.mark.parametrize("n,world", [(10, 3), (1601613, 8), (7, 8), (16, 4)])
def test_partition_rule(B, O, n, world):
    cnt, dsp = B.plan_partition(n, world)
    c2, d2 = O.partition(n, world)                              # oracle restatement of matrix.c:295-308
    assert np.array_equal(cnt, c2) and np.array_equal(dsp, d2)
    assert cnt.sum() == n and dsp[0] == 0 and np.all(np.diff(dsp) == cnt[:-1])
    assert cnt.max() - cnt.min() <= 1 and np.all(np.diff(cnt) <= 0)


def test_tile_plan_covers_rows(B):
    blk = B.gen_block("stencil15", 13, 14.0)
    _, _, ptr = blk.diag_arrays()
    rows = blk.n_loc
    for rpt, cap in ((256, 4000), (128, 1000), (32, 64)):
        tr = (C.c_int * (rows + 2))()
        nt = B.lib.bicg_plan_tiles(ptr.ctypes.data_as(C.POINTER(C.c_uint)), rows, rpt, cap, tr, rows + 2)
        t = np.array(tr[:nt + 1])
        assert t[0] == 0 and t[-1] == rows and np.all(np.diff(t) > 0) and np.all(np.diff(t) <= rpt)
        assert np.all(ptr[t[1:]].astype(np.int64) - ptr[t[:-1]].astype(np.int64) <= cap)
    tr = (C.c_int * (rows + 2))()
    assert B.lib.bicg_plan_tiles(ptr.ctypes.data_as(C.POINTER(C.c_uint)), rows, 32, 5, tr, rows + 2) == -2   # a row > cap


def test_generators_match_block_split_of_global(B):
    """gen_block(rank, world) must equal the reference-style split of the world=1 matrix (matrix.c:380-392)."""
    g1 = B.gen_block("stencil15", 8, 14.0)
    ptr, col, val = B.block_to_global_csr(g1)
    for world in (2, 3):
        for rank in range(world):
            a = B.gen_block("stencil15", 8, 14.0, rank=rank, world=world)
            b = B.blocks_from_csr(g1.n, ptr, col, val, rank, world)
            for x, y in ((a.diag_arrays(), b.diag_arrays()), (a.offd_arrays(), b.offd_arrays())):
                for u, v in zip(x, y):
                    assert np.array_equal(np.asarray(u), np.asarray(v))
            assert np.array_equal(a.recvcounts, b.recvcounts) and np.array_equal(a.displs, b.displs)
            assert a.diag.cols == a.n_loc and a.offd.cols == g1.n                 # matrix.c:344, 351


def _checks():
    return np.load(os.path.join(ROOT, "tests", "golden", "ref_checks.npz"))


def test_matrix_market_loader(B, O, tmp_path):
    """MPI_csr_load_matrix_block: same blocks as the generator the file was written from; in-row order = file order
    (stable row sort).  The reference program itself (main.c unchanged) solves the same file in as many iterations as the
    oracle: its count is golden, and the program is run too where oracle/_ref is built."""
    from helpers import write_mtx
    blk = B.gen_block("convdiff", 12, 1.5)
    n = blk.n
    ptr, col, val = B.block_to_global_csr(blk)
    f = tmp_path / "a.mtx"
    A = write_mtx(f, n, ptr, col, val)
    got = B.load_matrix_block(f, world=1)
    assert (got.n, got.n_loc, int(got.info.nz)) == (n, n, A.nnz) and got.info.code == b"MCRG"
    for u, v in zip(got.diag_arrays(), blk.diag_arrays()):
        assert np.array_equal(np.asarray(u), np.asarray(v))
    assert got.offd.nz == 0 and got.offd.rows == n and got.offd.cols == n
    b = O.spmv(n, ptr, col, val, np.ones(n))
    it = O.solve("bicgstab", n, ptr, col, val, b, tol=1e-10, max_iter=500)["iters"]
    assert it == int(_checks()["mm_cd12|iters"])
    ref_main = os.path.join(ROOT, "oracle", "_ref", "ref_main_hist")
    if os.path.exists(ref_main):
        env = dict(os.environ, REF_EPS="1e-10", REF_MAX_ITER="500", REF_OUT_ITER="1", MALLOC_MMAP_THRESHOLD_="0")
        out = subprocess.run([ref_main, str(f), "bicgstab"], env=env, capture_output=True, text=True, check=True).stdout
        assert it == int(re.search(r"Total iter\s*:\s*(\d+)", out).group(1))


def test_matrix_market_pattern_and_errors(B, tmp_path):
    f = tmp_path / "p.mtx"
    f.write_text("%%MatrixMarket matrix coordinate pattern general\n3 3 4\n1 1\n2 2\n3 3\n1 3\n")
    got = B.load_matrix_block(f, world=1)
    val, col, ptr = got.diag_arrays()
    assert list(ptr) == [0, 2, 3, 4] and list(col) == [0, 2, 1, 2] and np.all(np.asarray(val) == 1.0)
    bad = tmp_path / "bad.mtx"
    bad.write_text("not a banner\n")
    code = ("import sys; sys.path.insert(0, %r); import mpi_bicgstab_b200 as B; B.load_matrix_block(%r, world=1)"
            % (ROOT, str(bad)))
    p = subprocess.run(["python", "-c", code], capture_output=True, text=True)
    assert p.returncode != 0 and "Could not process Matrix Market banner" in p.stderr        # matrix.c:281-284


def test_compute_entry_points_fail_loudly_without_gpu(B):
    """No CPU fallback: on a box without a usable GPU a solve must exit(1) with a message, not return numbers."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    code = ("import sys; sys.path.insert(0, %r); import numpy as np; import mpi_bicgstab_b200 as B; "
            "blk = B.gen_block('laplace5', 8); x = np.zeros(blk.n); b = np.ones(blk.n); B.bicgstab(blk, x, b); print('RETURNED')" % ROOT)
    p = subprocess.run(["python", "-c", code], capture_output=True, text=True)
    assert p.returncode == 1 and "RETURNED" not in p.stdout and "no usable CUDA device" in p.stderr


def _reference_driver(name):
    """oracle/_ref/<name>: one of the reference's drivers, UNCHANGED, compiled against include/compat/mpi.h and linked against
    libbicgstab_b200.so by `make -C oracle ref` (which needs the reference's sources at build time)."""
    exe = os.path.join(ROOT, "oracle", "_ref", name)
    if not os.path.exists(exe):
        pytest.skip(f"oracle/_ref/{name} not built (the reference's sources were absent at build time)")
    ldd = subprocess.run(["ldd", "-r", exe], capture_output=True, text=True)      # binds every symbol against today's library
    out = ldd.stdout + ldd.stderr
    assert ldd.returncode == 0 and "undefined symbol" not in out, out
    lib = re.search(r"libbicgstab_b200\.so => (\S+)", out)
    assert lib and os.path.realpath(lib.group(1)) == os.path.realpath(os.path.join(ROOT, "mpi-bicgstab_b200", "libbicgstab_b200.so")), out
    return exe


def test_reference_main_c_links_against_the_library(B):
    """The drop-in claim itself: the reference's main.c, UNCHANGED, compiles against include/compat/mpi.h and
    links against libbicgstab_b200.so."""
    exe = _reference_driver("ref_main_b200")
    p = subprocess.run([exe], capture_output=True, text=True)              # no arguments -> usage text (main.c:64-75)
    assert "Usage:" in p.stdout and "pipe_bicgstab_rr" in p.stdout
    undefined = subprocess.run(["nm", "-u", exe], capture_output=True, text=True).stdout
    for sym in ("bicgstab", "ca_bicgstab", "pipe_bicgstab", "pipe_bicgstab_rr", "MPI_csr_spmv_ovlap",
                "MPI_csr_load_matrix_block", "csr_init_matrix", "csr_free_matrix"):
        assert re.search(r"\bU %s\b" % sym, undefined), sym


@pytest.mark.parametrize("driver,solver", [("main_shifted.c", "shifted_lopbicg_switching"), ("main_repeat.c", "shifted_lopbicg_switching"),
                                           ("main_seed_diff.c", "shifted_lopbicg_switching")])
def test_reference_shifted_drivers_link_against_the_library(B, driver, solver):
    """The shifted drivers (what the reference's top-level Makefile builds), UNCHANGED: besides the loader / SpMV / solver
    entry points they call vector.h's my_daxpy / my_dcopy on host arrays (main_shifted.c:114-135), which the library exports."""
    exe = _reference_driver("ref_%s_b200" % driver[len("main_"):-len(".c")])
    undefined = subprocess.run(["nm", "-u", exe], capture_output=True, text=True).stdout
    for sym in (solver, "MPI_csr_spmv_ovlap", "MPI_csr_load_matrix_block", "csr_init_matrix", "my_daxpy"):
        assert re.search(r"\bU %s\b" % sym, undefined), sym


def test_unchanged_shifted_driver_reaches_the_library_and_fails_loudly_without_a_gpu(B, tmp_path):
    """main_shifted.c built against the library, run on a small Matrix-Market file: the loader (host code) works, the first
    device call (MPI_csr_spmv_ovlap, main_shifted.c:113) must refuse to run without a GPU -- message + exit(1), no CPU path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible: the driver would really run (covered by the -m gpu tests of its library calls)")
    exe = _reference_driver("ref_shifted_b200")
    mtx = tmp_path / "a.mtx"
    mtx.write_text("%%MatrixMarket matrix coordinate real general\n3 3 5\n1 1 4.0\n2 2 4.0\n3 3 4.0\n1 2 -1.0\n3 2 -1.0\n")
    p = subprocess.run([exe, str(mtx)], capture_output=True, text=True)
    assert p.returncode == 1 and "IO time" in p.stdout and "no usable CUDA device" in p.stderr


def test_host_blas1_entry_points_match_the_oracle_bitwise(B, O):
    """vector.c:3-27 as exported for the drivers (csrc/hostvec.cpp) against the oracle's restatement: same loops, no contraction."""
    rng = np.random.default_rng(5)
    for n in (0, 1, 7, 1000, 4097):
        x, y = rng.standard_normal(n), rng.standard_normal(n)
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        y1, y2 = y.copy(), y.copy()
        B.lib.my_daxpy(n, 0.37, dp(x), dp(y1)); O.daxpy(0.37, x, y2)
        assert np.array_equal(y1, y2)
        assert B.lib.my_ddot(n, dp(x), dp(y)) == O.ddot(x, y)
        x1, x2 = x.copy(), x.copy()
        B.lib.my_dscal(n, -1.25, dp(x1)); O.dscal(-1.25, x2)
        assert np.array_equal(x1, x2)
        z = np.empty(n)
        B.lib.my_dcopy(n, dp(x), dp(z))
        assert np.array_equal(z, x)


def test_csr_shift_diagonal_matches_the_reference(B, O):
    """matrix.h's csr_shift_diagonal (matrix.c:536-551) on host arrays: same values as the reference's own compiled function
    (its golden output, and the function itself when oracle/_ref is there) and as the definition, a missing diagonal is fatal,
    and the cached device copy keyed by the arrays is forgotten (no GPU needed: nothing is cached here)."""
    blk = B.gen_block("convdiff", 12, 1.5)
    n = blk.n
    before = np.array(blk.diag_arrays()[0][:int(blk.diag.nz)], dtype=np.float64)
    col = np.array(blk.diag_arrays()[1][:int(blk.diag.nz)], dtype=np.int64)
    ptr = np.array(blk.diag_arrays()[2][:n + 1], dtype=np.int64)
    want = before.copy()
    rows = np.repeat(np.arange(n), np.diff(ptr))
    want[col == rows] += 0.37
    assert np.array_equal(_checks()["shiftdiag_cd12|val"], want)
    if O.have_ref("libref_strict.so"):
        import ctypes
        L = O.ref_lib("strict")
        v2 = before.copy()
        c2, p2 = col.astype(np.uint32), ptr.astype(np.uint32)
        D = O._RefCSR()
        D.val, D.col, D.ptr = O._p(v2, O._dp), O._p(c2, O._up), O._p(p2, O._up)
        D.nz, D.rows, D.cols = int(ptr[-1]), n, n
        L.csr_shift_diagonal.argtypes = [ctypes.POINTER(O._RefCSR), ctypes.c_double]
        L.csr_shift_diagonal(ctypes.byref(D), 0.37)
        assert np.array_equal(v2, want)
    B.lib.csr_shift_diagonal(C.byref(blk.diag), 0.37)
    got = np.array(blk.diag_arrays()[0][:int(blk.diag.nz)], dtype=np.float64)
    assert np.array_equal(got, want) and not np.array_equal(got, before)
    # a row without a stored diagonal entry: message + exit(EXIT_FAILURE), like the reference
    code = ("import numpy as np, ctypes as C, mpi_bicgstab_b200 as B\n"
            "blk = B.blocks_from_csr(3, [0, 1, 2, 3], [0, 2, 2], [1.0, 2.0, 3.0])\n"
            "B.lib.csr_shift_diagonal(C.byref(blk.diag), 1.0)\nprint('RETURNED')\n")
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT)
    assert p.returncode == 1 and "RETURNED" not in p.stdout and "Diagonal element not found in row 1" in p.stderr


def test_halo_runs_gap_merging(B):
    """plan_halo_runs: gap = 0 gives exactly the referenced columns, a larger gap merges runs and never loses one."""
    blk = B.gen_block("random", 4000, 6, rank=1, world=4)
    cols = np.unique(np.asarray(blk.offd_arrays()[1])[:int(blk.offd.nz)]).astype(np.int64)
    for gap in (0, 3, 64, 10**6):
        out = (C.c_int * (3 * (cols.size + 1)))()
        k = B.lib.bicg_plan_halo_runs(C.byref(blk.offd), C.byref(blk.info), 1, 4, gap, out, len(out))
        runs = np.array(out[:3 * k]).reshape(-1, 3)
        covered = np.concatenate([np.arange(f, f + l) for f, l, _ in runs]) if k else np.zeros(0, dtype=np.int64)
        assert np.all(np.diff(runs[:, 0]) > 0) and set(cols) <= set(covered)
        lo, cnt = blk.displs, blk.recvcounts
        for f, l, o in runs:                       # a run never leaves its owner's row range, never touches rank 1
            assert o != 1 and lo[o] <= f and f + l <= lo[o] + cnt[o]
        if gap == 0:
            assert covered.size == cols.size
        if gap == 10**6:
            assert k <= 3                          # one run per owner


def test_options_and_unknown_keys(B):
    B.set_options(tol=1e-9, max_iter=77, out_iter=5, unroll=4, graph=0, cache=1, mega=1)
    with pytest.raises(KeyError):
        B.set_option("NO_SUCH_OPTION", 1)
    B.set_options(tol=1e-15, max_iter=1000, out_iter=100, unroll=10, graph=1)
    assert B.lib.bicg_comm_rank() == 0 and B.lib.bicg_comm_world() == 1 and B.lib.bicg_comm_selftest() == 0


@pytest.mark.parametrize("rows,ctas,rpt", [(1601613, 148, 512), (200264, 148, 512), (343, 148, 512), (1, 148, 256),
                                            (5000, 7, 256), (148 * 512, 148, 512), (2_000_000, 148, 64)])
@pytest.mark.parametrize("extra", [0, 600])
def test_persistent_kernel_tile_plan(B, rows, ctas, rpt, extra):
    """plan_cta_tiles (mega.cu's work split): contiguous, complete, 16-row aligned, balanced by per-row work
    24*nnz + 216 (+ extra per pushed row), every tile fits the CTA's rows-per-tile."""
    rng = np.random.default_rng(rows)
    ptr = np.concatenate([[0], np.cumsum(rng.integers(0, 20, size=rows))]).astype(np.uint32)
    row_extra = np.zeros(rows, dtype=np.uint8)
    row_extra[: rows // 10] = 1                                   # the first tenth of the rows is pushed to a peer
    cap = rows + ctas + 8
    tr = (C.c_int * cap)(); ct = (C.c_int * (ctas + 1))(); mx = C.c_uint()
    nt = B.lib.bicg_plan_cta_tiles(ptr.ctypes.data_as(C.POINTER(C.c_uint)), rows, ctas, rpt,
                                   row_extra.ctypes.data_as(C.c_void_p) if extra else None, extra, tr, cap, ct, C.byref(mx))
    t = np.array(tr[:nt + 1]); c = np.array(ct[:])
    assert t[0] == 0 and t[-1] == rows and np.all(np.diff(t) > 0) and np.all(np.diff(t) <= rpt)
    assert c[0] == 0 and c[-1] == nt and np.all(np.diff(c) >= 0)
    first = t[c]                                                  # first row of every CTA (then `rows`)
    assert first[0] == 0 and first[-1] == rows and np.all(np.diff(first) >= 0)
    assert np.all(first[:-1] % 16 == 0)                           # 128-byte aligned vector slices
    w = 24 * np.diff(ptr.astype(np.int64)) + 216 + extra * row_extra.astype(np.int64)
    pw = np.concatenate([[0], np.cumsum(w)])
    per_cta = pw[first[1:]] - pw[first[:-1]]
    ideal = pw[-1] / ctas
    assert per_cta.max() <= ideal + 17 * w.max()                  # within one alignment granule of the ideal share
    for g in range(ctas):                                        # tiles of one CTA have (almost) equal height
        h = np.diff(t[c[g]:c[g + 1] + 1])
        assert h.size == 0 or h.max() - h.min() <= 1
    assert mx.value == (ptr[t[1:]].astype(np.int64) - ptr[t[:-1]].astype(np.int64)).max()


@pytest.mark.parametrize("n,world", [(1000, 4), (17, 3), (5, 8), (100000, 8)])
def test_nnz_balanced_partition_rule(B, n, world):
    """bicg_plan_partition_nnz = the reference's archived DYNAMIC_ROWS rule (archive/matrix.c:407-420): ranks take rows
    until their entry count reaches nnz / world, the last rank takes the rest."""
    rng = np.random.default_rng(n + world)
    row_nnz = rng.integers(1, 40, size=n).astype(np.uint32)
    row_nnz[: n // 5] *= 6                                   # a dense head: equal-rows would be badly unbalanced
    cnt = (C.c_int * world)(); dsp = (C.c_int * world)()
    B.lib.bicg_plan_partition_nnz(row_nnz.ctypes.data_as(C.POINTER(C.c_uint)), n, world, cnt, dsp)
    cnt, dsp = np.array(cnt[:]), np.array(dsp[:])
    assert cnt.sum() == n and dsp[0] == 0 and np.all(dsp[1:] == np.cumsum(cnt)[:-1]) and np.all(cnt >= 0)
    target = int(row_nnz.sum()) // world                    # restatement of the archived loop
    start = 0
    for p in range(world):
        end = n
        if p < world - 1:
            cum = 0
            for i in range(start, n):
                cum += int(row_nnz[i])
                if cum >= target:
                    end = i + 1
                    break
        assert (dsp[p], cnt[p]) == (start, end - start)
        start = end
    if n >= 1000:                                            # and it does balance the entries
        per = np.add.reduceat(row_nnz.astype(np.int64), dsp[cnt > 0])
        assert per.max() <= 1.15 * row_nnz.sum() / world + row_nnz.max()


def test_generator_and_loader_honour_nnz_partition(B, tmp_path, monkeypatch):
    monkeypatch.setenv("BICG_PARTITION", "nnz")
    world = 3
    blocks = [B.gen_block("stencil15", 9, 14.0, rank=r, world=world) for r in range(world)]
    monkeypatch.delenv("BICG_PARTITION")
    full = B.gen_block("stencil15", 9, 14.0)
    ptr, col, val = B.block_to_global_csr(full)
    row_nnz = np.diff(ptr).astype(np.uint32)
    cnt = (C.c_int * world)(); dsp = (C.c_int * world)()
    B.lib.bicg_plan_partition_nnz(row_nnz.ctypes.data_as(C.POINTER(C.c_uint)), full.n, world, cnt, dsp)
    for r, blk in enumerate(blocks):
        assert list(blk.recvcounts) == list(cnt[:]) and list(blk.displs) == list(dsp[:])
        p2, c2, v2 = B.block_to_global_csr(blk, rank=r)
        lo, hi = dsp[r], dsp[r] + cnt[r]
        # same rows as the global matrix (entries of a row: diag block first, then offd -- compare as sets per row)
        assert np.array_equal(np.diff(p2), np.diff(ptr[lo:hi + 1]))
        for i in (0, cnt[r] // 2, cnt[r] - 1):
            a = sorted(zip(c2[p2[i]:p2[i + 1]], v2[p2[i]:p2[i + 1]]))
            b = sorted(zip(col[ptr[lo + i]:ptr[lo + i + 1]], val[ptr[lo + i]:ptr[lo + i + 1]]))
            assert a == b


def test_persistent_kernel_plan_cuts_long_rows_into_chunks(B):
    """Cap-limited plan (plan.cpp): tiles hold <= cap entries; a longer row becomes consecutive chunk tiles (flag 1 ... 1 2)
    inside ONE CTA's range; every entry of the matrix is covered exactly once, in order."""
    rng = np.random.default_rng(5)
    rows, ctas, rpt, cap = 6000, 148, 512, 1000
    lens = rng.integers(0, 12, size=rows)
    lens[[0, 17, 2999, 5999]] = [4096, 1000, 1001, 2500]          # 1000 fits exactly, the others are cut
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint32)
    tc = rows + ctas + 64
    tr = (C.c_int * tc)(); nz = (C.c_uint * tc)(); fl = (C.c_int * tc)(); ct = (C.c_int * (ctas + 1))(); mx = C.c_uint()
    nt = B.lib.bicg_plan_cta_tiles_capped(ptr.ctypes.data_as(C.POINTER(C.c_uint)), rows, ctas, rpt, cap, tr, nz, fl, tc, ct, C.byref(mx))
    assert nt > 0 and mx.value <= cap
    t, z, f, c = np.array(tr[:nt + 1]), np.array(nz[:nt + 1]), np.array(fl[:nt + 1]), np.array(ct[:])
    assert t[0] == 0 and t[-1] == rows and z[0] == 0 and z[-1] == ptr[-1]
    assert np.all(np.diff(z.astype(np.int64)) >= 0) and np.all(np.diff(z.astype(np.int64)) <= cap)      # contiguous cover of the entries
    for k in range(nt):
        if f[k] == 0:
            assert t[k + 1] > t[k] or z[k + 1] == z[k]
            assert z[k] == ptr[t[k]] and z[k + 1] == ptr[t[k + 1]] and t[k + 1] - t[k] <= rpt
        else:
            r = t[k]
            assert lens[r] > cap and ptr[r] <= z[k] < ptr[r + 1]
            assert (f[k] == 2) == (z[k + 1] == ptr[r + 1]) and t[k + 1] == (r + 1 if f[k] == 2 else r)
    chunk_rows = set(t[:-1][f[:-1] != 0])
    assert chunk_rows == {0, 2999, 5999}
    for g in range(ctas):                                         # a row's chunks never straddle two CTAs
        if c[g] < nt and c[g] > 0:
            assert f[c[g] - 1] != 1


_BOOT_C = r"""
#include <stdio.h>
int bicg_shm_bootstrap(void); void bicg_shm_shutdown(void); int bicg_comm_rank(void); int bicg_comm_world(void); int bicg_comm_selftest(void);
int main() { bicg_shm_bootstrap(); printf("rank %d of %d selftest %d\n", bicg_comm_rank(), bicg_comm_world(), bicg_comm_selftest());
             bicg_shm_shutdown(); return 0; }
"""


def _boot_exe(tmp_path):
    import subprocess
    src = tmp_path / "boot.c"
    src.write_text(_BOOT_C)
    exe = tmp_path / "boot"
    libdir = os.path.join(ROOT, "mpi-bicgstab_b200")
    subprocess.run(["gcc", "-O1", str(src), f"-L{libdir}", "-lbicgstab_b200", f"-Wl,-rpath,{libdir}", "-o", str(exe)], check=True)
    return str(exe)


def test_shm_bootstrap_four_ranks_and_cleanup(B, tmp_path):
    """csrc/shm_boot.cpp (the MPI_Init of include/compat/mpi.h): 4 processes rendezvous, allgather works, the segment is
    unlinked afterwards.  No GPU involved."""
    import subprocess
    exe = _boot_exe(tmp_path)
    p = subprocess.run([os.path.join(ROOT, "tools", "bicgrun"), "-np", "4", exe], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stdout + p.stderr
    assert sorted(p.stdout.split("\n")[:4]) == [f"rank {r} of 4 selftest 0" for r in range(4)]
    assert not [f for f in os.listdir("/dev/shm") if f.startswith(f"bicg_b200_{os.getuid()}_job")]


def test_shm_bootstrap_survives_a_stale_segment(B, tmp_path):
    """A crashed job left a READY segment with no join tickets; the new job's ranks 1, 2 start BEFORE rank 0.  They must
    not attach to the corpse (round-1 behaviour: hang) but wait for rank 0's fresh segment."""
    import struct, subprocess, time
    exe = _boot_exe(tmp_path)
    job = f"stale{os.getpid()}"
    name = f"/dev/shm/bicg_b200_{os.getuid()}_{job}"
    with open(name, "wb") as f:
        f.truncate(64 + (256 << 20))
        f.write(struct.pack("<iiiiiiQ", 0x42494347, 0, 0, 3, 0, 1, 0))     # READY, joined = 3, creator pid 1 (alive)
    env = dict(os.environ, WORLD_SIZE="3", BICG_JOB_ID=job, BICG_BOOT_TIMEOUT_S="30")
    ps = [subprocess.Popen([exe], env=dict(env, RANK=str(r), LOCAL_RANK=str(r)), stdout=subprocess.PIPE, text=True) for r in (1, 2)]
    time.sleep(0.5)
    ps.append(subprocess.Popen([exe], env=dict(env, RANK="0", LOCAL_RANK="0"), stdout=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=90)[0].strip() for p in ps]
    assert all(p.returncode == 0 for p in ps), outs
    assert sorted(outs) == [f"rank {r} of 3 selftest 0" for r in range(3)]
    assert not os.path.exists(name)


def test_shm_bootstrap_rejects_more_than_eight_ranks(B, tmp_path):
    import subprocess
    exe = _boot_exe(tmp_path)
    p = subprocess.run([exe], env=dict(os.environ, WORLD_SIZE="9", RANK="0", BICG_JOB_ID=f"big{os.getpid()}"), capture_output=True,
                       text=True, timeout=60)
    assert p.returncode == 1 and "more than 8 ranks" in p.stderr        # main.c ignores MPI_Init's return value: must be fatal


_MPI_BOOT_C = r"""
/* The maintainer-side line of INTEGRATION.md section 1: an MPI program registers MPI itself as the library's bootstrap
 * transport.  Compiled here against the oracle's functional mini-MPI (fork + shm, oracle/mini_mpi.c) because the image has
 * no MPI installation; with a real MPI the callback body is MPI_Allgather(s, n, MPI_BYTE, r, n, MPI_BYTE, MPI_COMM_WORLD). */
#include <stdio.h>
#include <mpi.h>
#include "bicgstab_b200.h"
static int ag(void *c, const void *s, void *r, size_t n)
{
    int np, cnt[8], dsp[8]; MPI_Request q; (void)c;
    MPI_Comm_size(MPI_COMM_WORLD, &np);
    for (int p = 0; p < np; ++p) { cnt[p] = (int)n; dsp[p] = (int)(p * n); }
    MPI_Iallgatherv(s, (int)n, MPI_CHAR, r, cnt, dsp, MPI_CHAR, MPI_COMM_WORLD, &q);
    return MPI_Wait(&q, MPI_STATUS_IGNORE);
}
int main(int argc, char **argv)
{
    int np, me;
    MPI_Init(&argc, &argv);
    MPI_Comm_size(MPI_COMM_WORLD, &np); MPI_Comm_rank(MPI_COMM_WORLD, &me);
    int rc = bicg_comm_init(me, np, ag, NULL);
    printf("rank %d of %d init %d selftest %d\n", bicg_comm_rank(), bicg_comm_world(), rc, bicg_comm_selftest());
    fflush(stdout);
    bicg_comm_finalize();
    MPI_Finalize();
    return 0;
}
"""


def test_mpi_program_registers_mpi_as_bootstrap_transport(B, tmp_path):
    """INTEGRATION.md section 1, exercised: bicg_comm_init with an MPI-allgather callback inside an MPI program (the oracle's
    mini-MPI stands in for the absent MPI installation), 4 ranks, the library's self-test round-trips through it.  CPU only."""
    import subprocess
    src = tmp_path / "mpiboot.c"
    src.write_text(_MPI_BOOT_C)
    exe = tmp_path / "mpiboot"
    libdir = os.path.join(ROOT, "mpi-bicgstab_b200")
    subprocess.run(["gcc", "-O1", f"-I{os.path.join(ROOT, 'oracle', 'mpi_stub')}", f"-I{os.path.join(ROOT, 'include')}", str(src),
                    os.path.join(ROOT, "oracle", "mini_mpi.c"), f"-L{libdir}", "-lbicgstab_b200", f"-Wl,-rpath,{libdir}", "-o", str(exe)],
                   check=True)
    p = subprocess.run([str(exe)], env=dict(os.environ, MINI_MPI_NP="4"), capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stdout + p.stderr
    assert sorted(l for l in p.stdout.splitlines() if l.startswith("rank")) == [f"rank {r} of 4 init 0 selftest 0" for r in range(4)]
