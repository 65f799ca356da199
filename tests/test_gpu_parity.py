"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the oracle.

Tolerances (SURVEY.md 8(c), north_star: residual history within 1e-10 relative):
  K-level  SpMV vs long-double oracle                        <= 1e-13 relative (max-norm)
  H-level  sqrt(dot_r/dot_zero), iterations 1..10            <= 1e-10 relative (+ 1e-15 ||r0|| absolute floor)
  C-level  iterations to tol within max(2, 2 %) of the oracle; true residual ||b-Ax||/||b|| <= 10 tol
The summation order of the dots and of each row differs from the reference's scalar loops (parallel
reduction), so bit-exactness is not expected beyond the element-wise updates.
"""
import os

import numpy as np
import pytest

from helpers import METHODS, RR, SMALL_CASES, big_csr, global_csr, rel_err, write_mtx

pytestmark = pytest.mark.gpu

TOL = 1e-10
H_FLOOR = 1e-15


@pytest.fixture(autouse=True, params=[1, 0], ids=["mega", "multikernel"])
def _quiet(B, request):
    """Every test runs twice: iteration loop in the persistent kernel (mega.cu) and as the kernel-per-phase graph."""
    B.set_options(quiet=1, tol=1e-15, max_iter=1000, cache=1, mega=request.param)
    yield
    B.set_options(mega=1)


@pytest.mark.parametrize("name,kind,g,p0", SMALL_CASES)
def test_spmv_matches_oracle(B, O, name, kind, g, p0):
    blk, n, ptr, col, val = global_csr(B, kind, g, p0)
    rng = np.random.default_rng(7)
    x = rng.standard_normal(n)
    y = B.spmv_ovlap(blk, x)
    y_ld = O.spmv(n, ptr, col, val, x, long_double=True)
    assert rel_err(y, y_ld) <= 1e-13
    y_ref = O.spmv(n, ptr, col, val, x)           # the reference's own association
    assert rel_err(y, y_ref) <= 1e-13


@pytest.mark.parametrize("spmv,lanes", [("tma", 1), ("tma", 2), ("tma", 4), ("tma", 8), ("tma", 32),
                                        ("rowsplit", 1), ("rowsplit", 4), ("rowsplit", 32)])
def test_spmv_every_kernel_variant(B, O, spmv, lanes):
    blk, n, ptr, col, val = global_csr(B, "stencil15", 14, 14.0)
    B.set_options(spmv=spmv, spmv_lanes=lanes)
    try:
        dm = B.DeviceMatrix(blk)
        x = np.random.default_rng(3).standard_normal(n)
        y = dm.spmv(x)
        dm.destroy()
    finally:
        B.set_options(spmv="auto", spmv_lanes=0)
    assert rel_err(y, O.spmv(n, ptr, col, val, x, long_double=True)) <= 1e-13


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("name,kind,g,p0", SMALL_CASES)
def test_history_and_convergence(B, O, name, kind, g, p0, method):
    blk, n, ptr, col, val = global_csr(B, kind, g, p0)
    kw = RR if method.endswith("rr") else {}
    B.set_options(tol=TOL, max_iter=600)
    b = B.spmv_ovlap(blk, np.ones(n))                         # main.c:109-113
    b0 = b.copy()
    x = np.zeros(n)
    iters = B.solve(method, blk, x, b, **kw)
    hist = B.last_history()
    ref = O.solve(method, n, ptr, col, val, O.spmv(n, ptr, col, val, np.ones(n)), tol=TOL, max_iter=600, **kw)

    # H-level: first 10 iterations of the residual history
    m = min(10, iters, ref["iters"])
    got, want = np.sqrt(hist[1:m + 1]), np.sqrt(ref["hist"][1:m + 1])
    # 1e-10 relative; the absolute floor (in units of ||r0||) is the fp64 resolution of the residual
    # recursion itself -- once the residual has dropped to ~1e-10 ||r0|| its trailing digits are rounding noise
    # in the reference too (two builds of the reference differ there, SURVEY.md Appendix A)
    assert np.all(np.abs(got - want) <= 1e-10 * want + H_FLOOR), (got, want, np.abs(got - want) / want)
    # C-level
    assert abs(iters - ref["iters"]) <= max(2, int(0.02 * ref["iters"])), (iters, ref["iters"])
    true_res = np.linalg.norm(b0 - O.spmv(n, ptr, col, val, x, long_double=True)) / np.linalg.norm(b0)
    limit = 10 * TOL if "pipe" not in method else 1e3 * TOL       # pipelined variants lose attainable accuracy
    assert true_res <= limit, true_res
    assert np.abs(x - 1.0).max() <= 1e3 * max(np.abs(ref["x"] - 1.0).max(), TOL)
    # the returned r is the recursive residual: its norm matches the last history entry
    assert abs(np.dot(b, b) / np.dot(b0, b0) - hist[iters]) <= 1e-9 * hist[iters]


@pytest.mark.parametrize("method", METHODS[:3])
def test_graph_and_stream_paths_agree(B, method):
    blk = B.gen_block("stencil15", 12, 14.0)
    n = blk.n
    out = {}
    for graph in (1, 0):
        B.set_options(tol=1e-9, max_iter=400, graph=graph, mega=0)
        b = B.spmv_ovlap(blk, np.ones(n))
        x = np.zeros(n)
        it = B.solve(method, blk, x, b)
        out[graph] = (it, x.copy(), B.last_history().copy())
    B.set_options(graph=1)
    assert out[0][0] == out[1][0]
    assert np.array_equal(out[0][1], out[1][1])          # same kernels, same order -> bitwise equal
    assert np.array_equal(out[0][2], out[1][2])


def test_max_iter_stops_exactly(B):
    blk = B.gen_block("stencil15", 12, 14.0)
    n = blk.n
    for mi in (1, 7, 10, 23):
        B.set_options(tol=0.0, max_iter=mi)
        b = B.spmv_ovlap(blk, np.ones(n))
        x = np.zeros(n)
        assert B.bicgstab(blk, x, b) == mi
        assert len(B.last_history()) == mi + 1


def test_zero_rhs_does_no_iterations(B):
    blk = B.gen_block("laplace5", 20)
    x, b = np.zeros(blk.n), np.zeros(blk.n)
    B.set_options(tol=1e-15, max_iter=50)
    assert B.bicgstab(blk, x, b) == 0                    # solver.c:86: 0 > 0 is false


def test_stdout_contract(B, capfd):
    blk = B.gen_block("convdiff", 30, 1.5)
    B.set_options(quiet=0, tol=1e-12, max_iter=300, out_iter=10)
    b = B.spmv_ovlap(blk, np.ones(blk.n))
    x = np.zeros(blk.n)
    it = B.bicgstab(blk, x, b)
    B.lib.bicg_synchronize()
    import ctypes
    ctypes.CDLL(None).fflush(None)
    out = capfd.readouterr().out
    lines = out.strip().splitlines()
    assert lines[0].startswith("Iteration: 10, Residual: ")
    assert f"Total iter   : {it}" in out and "Final r      : " in out
    assert "Total time   : " in out and "Avg time/iter: " in out and "[sec.] " in out
    B.set_options(quiet=1, out_iter=100)


def test_full_size_properties(B):
    """BASELINE config 2 size (T' surrogate, 1.6 M rows / 23.6 M nnz): size-independent checks."""
    blk = B.gen_block("stencil15", 117, 16.0)
    n = blk.n
    dm = B.DeviceMatrix(blk)
    ones = np.ones(n)
    y1 = dm.spmv(ones)
    # row sums: closed form from the CSR arrays
    dv, dc, dp = blk.diag_arrays()
    rowsum = np.add.reduceat(dv, dp[:-1].astype(np.int64))
    assert rel_err(y1, rowsum) <= 1e-13
    # linearity: A(2x + e) = 2Ax + Ae
    rng = np.random.default_rng(0)
    x = rng.standard_normal(n)
    assert rel_err(dm.spmv(2 * x + ones), 2 * dm.spmv(x) + y1) <= 1e-12
    # solve: x* = 1 is recovered, recursive residual equals the true residual at convergence
    B.set_options(tol=1e-8, max_iter=1000)
    b = y1.copy()
    xs = np.zeros(n)
    it, st = dm.solve("bicgstab", xs, b)
    assert st["converged"] == 1 and it < 1000
    true_res = np.linalg.norm(y1 - dm.spmv(xs)) / np.linalg.norm(y1)
    assert true_res <= 1e-7
    assert np.abs(xs - 1).max() <= 1e-5
    dm.destroy()


@pytest.mark.parametrize("method", METHODS[:3])
def test_persistent_and_multikernel_paths_agree(B, method):
    """Same phases, different partial-sum grouping: histories agree to rounding, iteration counts to +-2."""
    blk = B.gen_block("convdiff", 40, 1.5)
    n = blk.n
    out = {}
    for mega in (1, 0):
        B.set_options(tol=1e-10, max_iter=600, mega=mega)
        b = B.spmv_ovlap(blk, np.ones(n))
        x = np.zeros(n)
        it = B.solve(method, blk, x, b)
        out[mega] = (it, x.copy(), B.last_history().copy(), B.last_stats()["kernel_launches"])
    assert abs(out[0][0] - out[1][0]) <= 2
    m = min(10, out[0][0], out[1][0])
    assert np.allclose(np.sqrt(out[0][2][1:m + 1]), np.sqrt(out[1][2][1:m + 1]), rtol=1e-10, atol=1e-15)
    assert np.abs(out[0][1] - out[1][1]).max() < 1e-7
    assert out[1][3] < 10 < out[0][3]            # one launch for the whole loop vs ~5 per iteration


def test_reference_main_c_runs_on_the_library(B, O, tmp_path):
    """The drop-in itself: the reference's UNCHANGED main.c (built in the dev container into oracle/_ref/ref_main_b200,
    linked against libbicgstab_b200.so) loads a Matrix-Market file, forms b = A*1 and solves on the GPU; its stdout
    is the reference's (main.c:52, 93; solver.c:124, 135-139) and its iteration count the oracle's."""
    import re, subprocess
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "ref_main_b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/ref_main_b200 not built (the reference's sources were absent at build time)")
    blk = B.gen_block("convdiff", 36, 1.5)
    f = tmp_path / "cd36.mtx"
    n = blk.n
    ptr, col, val = B.block_to_global_csr(blk)
    write_mtx(f, n, ptr, col, val)
    b = O.spmv(n, ptr, col, val, np.ones(n))
    for method, extra in (("bicgstab", []), ("ca_bicgstab", []), ("pipe_bicgstab_rr", ["10", "3"])):
        kw = dict(krr=10, nrr=3) if extra else {}
        env = dict(os.environ, BICG_TOL="1e-10", BICG_MAX_ITER="600", BICG_OUT_ITER="10")
        p = subprocess.run([exe, str(f), method] + extra, capture_output=True, text=True, env=env, timeout=300)
        assert p.returncode == 0, p.stdout + p.stderr
        out = p.stdout
        assert out.startswith("Node: 1, Proc: 1\n") and "IO time      : " in out
        it = int(re.search(r"Total iter\s*:\s*(\d+)", out).group(1))
        ref = O.solve(method, n, ptr, col, val, b, tol=1e-10, max_iter=600, **kw)
        assert abs(it - ref["iters"]) <= 2, (method, it, ref["iters"])
        assert re.search(r"Iteration: 10, Residual: \d\.\d{6}e[-+]\d\d", out)
        assert float(re.search(r"Final r\s*:\s*(\S+)", out).group(1)) <= 1e-10


def test_bench_matrix_parity(B, O, request):
    """The BASELINE config-2 matrix itself (T' surrogate with the bench's p0 = 14: 1,601,613 rows, 23,616,325 entries),
    tol 1e-8: H-level against the oracle, C-level against the iteration counts of the reference's own sources compiled in
    place (oracle/_ref/ref_driver_fast and _strict, P = 1), stored in tests/golden/ref_checks.npz."""
    f, n, ptr, col, val = big_csr("stencil15", 117, 14.0)
    blk = B.gen_block("stencil15", 117, 14.0)
    assert blk.n == n and blk.nnz_loc == val.size
    b_ref = O.spmv(n, ptr, col, val, np.ones(n))
    dm = B.DeviceMatrix(blk)
    b = dm.spmv(np.ones(n))
    assert rel_err(b, b_ref) <= 1e-13
    B.set_options(tol=1e-8, max_iter=1000)
    x = np.zeros(n)
    r = b.copy()
    it, st = dm.solve("bicgstab", x, r)
    hist = B.last_history()
    assert st["converged"] == 1
    ref10 = O.solve("bicgstab", n, ptr, col, val, b_ref, tol=1e-8, max_iter=10)
    got, want = np.sqrt(hist[1:11]), np.sqrt(ref10["hist"][1:11])
    assert np.all(np.abs(got - want) <= 1e-10 * want + H_FLOOR), np.abs(got - want) / want
    # C-level partner: the reference as a user builds it (gcc -O3: FMA contraction on, like the GPU's fma chain).  At this
    # size and tolerance the reference's own builds disagree by more than the 2 % rule -- the strict IEEE build
    # (-O2 -ffp-contract=off) needs 380 iterations where the -O3 build needs 333 (measured on the same box, round 2) -- so the
    # iteration count is compared with the -O3 build and must in any case lie inside the spread of the reference's builds.
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_checks.npz"))
    fast_it, strict_it = int(gold["tprime|iters_fast"]), int(gold["tprime|iters_strict"])
    lo, hi = min(fast_it, strict_it), max(fast_it, strict_it)
    near_user_build = abs(it - fast_it) <= max(2, int(0.02 * fast_it))
    inside_reference_spread = lo - max(2, int(0.02 * lo)) <= it <= hi + max(2, int(0.02 * hi))
    assert near_user_build or inside_reference_spread, (it, fast_it, strict_it)
    if "mega" in request.node.name:                # the loop the benchmark runs: held to the 2 % rule against the -O3 build
        assert near_user_build, (it, fast_it)
    true_res = np.linalg.norm(b_ref - O.spmv(n, ptr, col, val, x)) / np.linalg.norm(b_ref)
    assert true_res <= 1e-7 and np.abs(x - 1.0).max() <= 1e-5
    dm.destroy()


def test_random_block_parity(B, O, request):
    """A >= 1 M-row block of the config-5 family (random, 32 entries per row, CA-BiCGStab): the long-row path of the
    persistent kernel (LANES > 1, forced with BICG_MEGA=2) and the autotuned kernel-per-phase path at size."""
    f, n, ptr, col, val = big_csr("random", 1_000_003, 32)
    blk = B.gen_block("random", 1_000_003, 32)
    b_ref = O.spmv(n, ptr, col, val, np.ones(n))
    if "mega" in request.node.name:
        B.set_options(mega=2)
    dm = B.DeviceMatrix(blk)
    B.set_options(tol=1e-10, max_iter=200)
    x = np.zeros(n)
    r = dm.spmv(np.ones(n))
    assert rel_err(r, b_ref) <= 1e-13
    it, st = dm.solve("ca_bicgstab", x, r)
    hist = B.last_history()
    ref = O.solve("ca_bicgstab", n, ptr, col, val, b_ref, tol=1e-10, max_iter=200)
    m = min(10, it, ref["iters"])
    got, want = np.sqrt(hist[1:m + 1]), np.sqrt(ref["hist"][1:m + 1])
    # this family converges by ~2 digits per iteration: the recursion's own rounding noise (eps ||r_{k-1}||, i.e. ~100 eps
    # relative to ||r_k||, carried through the CA recurrences) reaches 1e-10 of the residual after a few iterations, hence the
    # absolute floor of 1e-12 ||r0|| next to the 1e-10 relative bound
    assert np.all(np.abs(got - want) <= 1e-10 * want + 1e-12), (got, want, np.abs(got - want) / want)
    assert abs(it - ref["iters"]) <= 2 and np.abs(x - 1.0).max() <= 1e-8, (it, ref["iters"], np.abs(x - 1.0).max())
    if "mega" in request.node.name:
        assert st["kernel_launches"] <= 8          # the loop ran as one persistent kernel
    dm.destroy()
