"""CPU: the oracle restatement (oracle/bicg_oracle.c) against the golden vectors the REFERENCE produced
(tests/golden/ref_histories.npz and ref_checks.npz, generators tests/golden/make_golden*.py) -- bit for bit, for 1, 2
and 3 ranks -- and, where oracle/_ref is built, the compiled reference itself reproduces the golden vectors."""
import os

import numpy as np
import pytest

from helpers import METHODS, RR, SMALL_CASES, global_csr, sha256

GOLD = os.path.join(os.path.dirname(__file__), "golden", "ref_histories.npz")
TOL, MAX_ITER = 1e-10, 600


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.fixture(scope="module")
def checks():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_checks.npz"))


@pytest.mark.parametrize("P", [1, 2, 3])
@pytest.mark.parametrize("name,kind,g,p0", SMALL_CASES)
def test_oracle_reproduces_reference_bitwise(B, O, gold, name, kind, g, p0, P):
    blk, n, ptr, col, val = global_csr(B, kind, g, p0)
    b = O.spmv(n, ptr, col, val, np.ones(n), P=P)              # main.c:109-113 with P ranks
    for method in METHODS:
        kw = RR if method.endswith("rr") else {}
        o = O.solve(method, n, ptr, col, val, b, P=P, tol=TOL, max_iter=MAX_ITER, **kw)
        key = f"{name}|{method}|P{P}"
        assert o["iters"] == int(gold[key + "|iters"]), key
        assert np.array_equal(np.sqrt(o["hist"][1:]), gold[key + "|res"]), key      # every iteration, every bit
        assert np.array_equal(o["x"], gold[key + "|x"]), key
        if key + "|r" in gold:
            assert np.array_equal(o["r"], gold[key + "|r"]), key
        else:                                                    # stored as a digest (make_golden.py: R_DIGEST)
            assert sha256(o["r"]) == str(gold[key + "|r_sha256"]), key


def _same_solve(o, r):
    """oracle result o and reference result r (ref_solve / ref_driver / golden): bit-identical"""
    assert o["iters"] == r["iters"]
    assert np.array_equal(np.sqrt(o["hist"][1:]), r["res"])
    assert np.array_equal(o["x"], r["x"]) and np.array_equal(o["r"], r["r"])


def _gold_solve(checks, prefix):
    return {k: checks[f"{prefix}|{k}"] for k in ("iters", "res", "x", "r")}


def test_oracle_against_compiled_reference_live(B, O, checks):
    """The compiled reference's bicgstab()/... (P = 1, in-process) on another matrix, rank count 1, other tol / krr, nrr."""
    blk, n, ptr, col, val = global_csr(B, "convdiff", 25, 2.0, seed=99)
    b = O.spmv(n, ptr, col, val, np.ones(n))
    for method in METHODS:
        kw = dict(krr=7, nrr=2) if method.endswith("rr") else {}
        o = O.solve(method, n, ptr, col, val, b, tol=1e-11, max_iter=400, **kw)
        _same_solve(o, _gold_solve(checks, f"cd25|{method}"))
        if O.have_ref("libref_strict.so"):
            _same_solve(o, O.ref_solve(method, n, ptr, col, val, b, tol=1e-11, max_iter=400, **kw))


def test_oracle_rhs_ones_multi_rank_live(B, O, checks, tmp_path):
    """README / BASELINE wording "right-hand side = all ones" (main.c itself uses b = A*1): the oracle follows the
    compiled reference for that rhs too, with 1 and 3 ranks."""
    blk, n, ptr, col, val = global_csr(B, "stencil15", 9, 14.0)
    f = str(tmp_path / "a.bin")
    O.write_csr_bin(f, n, ptr, col, val)
    for P in (1, 3):
        for method in METHODS[:3]:
            o = O.solve(method, n, ptr, col, val, np.ones(n), P=P, tol=1e-11, max_iter=400)
            _same_solve(o, _gold_solve(checks, f"ones_s9|{method}|P{P}"))
            if O.have_ref("ref_driver_strict"):
                _same_solve(o, O.ref_driver(method, f, P=P, rhs="ones", tol=1e-11, max_iter=400, flavour="strict"))


def test_oracle_spmv_and_blas1(B, O):
    blk, n, ptr, col, val = global_csr(B, "random", 500, 6)
    import scipy.sparse as sp
    A = sp.csr_matrix((val, col, ptr), shape=(n, n))
    x = np.random.default_rng(1).standard_normal(n)
    for P in (1, 2, 5):
        assert np.allclose(O.spmv(n, ptr, col, val, x, P=P), A @ x, rtol=1e-13, atol=1e-13)
    assert np.allclose(O.spmv(n, ptr, col, val, x, long_double=True), A @ x, rtol=1e-13, atol=1e-13)
    y = np.random.default_rng(2).standard_normal(n)
    assert abs(O.lib().orc_ddot(n, x.ctypes.data_as(O._dp), y.ctypes.data_as(O._dp)) - float(x @ y)) < 1e-12


def test_manufactured_solution(B, O):
    """x* = 1 (main.c:109-117): every variant recovers it."""
    blk, n, ptr, col, val = global_csr(B, "stencil15", 9, 14.0)
    b = O.spmv(n, ptr, col, val, np.ones(n))
    for method in METHODS:
        kw = RR if method.endswith("rr") else {}
        o = O.solve(method, n, ptr, col, val, b, tol=1e-12, max_iter=500, **kw)
        assert np.abs(o["x"] - 1).max() < 1e-8


# ---- shifted family (SURVEY.md 8(f) N4) --------------------------------------------------------------------------
from helpers import SHIFTED_CASES, shifted_problem


@pytest.fixture(scope="module")
def gold_shifted():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_shifted.npz"))


@pytest.mark.parametrize("name,kind,g,p0,L,scale,seed", SHIFTED_CASES)
def test_shifted_oracle_reproduces_reference_bitwise(B, O, gold_shifted, name, kind, g, p0, L, scale, seed):
    """orc_shifted_lopbicg_switching vs the golden outputs of the reference's own shifted_lopbicg_switching
    (shifted_switching_solver.c:260-602, strict build): same return value, bit-identical x_j for every shift, r and history."""
    blk, n, ptr, col, val = global_csr(B, kind, g, p0)
    sigma, b = shifted_problem(O, n, ptr, col, val, L, scale, seed)
    o = O.shifted_solve(n, ptr, col, val, b, sigma, seed, tol=1e-12, max_iter=1000)
    assert o["ret"] == int(gold_shifted[name + "|ret"])
    assert np.array_equal(o["x"], gold_shifted[name + "|x"])
    assert np.array_equal(o["r"], gold_shifted[name + "|r"])
    assert np.array_equal(np.sqrt(o["hist"][1:]), gold_shifted[name + "|res"])
    if "switch" in name:
        assert o["seed"] != seed                                   # the seed-switching branch really ran
    for j in range(L):                                             # and every shifted system is solved
        res = O.spmv(n, ptr, col, val, o["x"][j]) + sigma[j] * o["x"][j] - b
        assert np.linalg.norm(res) <= 1e-10 * np.linalg.norm(b)


def test_shifted_oracle_against_compiled_reference_live(B, O, gold_shifted):
    """The oracle's defaults (tol 1e-12, 1000 iterations) against the compiled reference's: the golden outputs, and the
    live function where oracle/_ref is built."""
    name, kind, g, p0, L, scale, seed = SHIFTED_CASES[1]
    blk, n, ptr, col, val = global_csr(B, kind, g, p0)
    sigma, b = shifted_problem(O, n, ptr, col, val, L, scale, seed)
    o = O.shifted_solve(n, ptr, col, val, b, sigma, seed)
    refs = [{k: gold_shifted[f"{name}|{k}"] for k in ("ret", "x", "r")}]
    if O.have_ref("libref_strict.so"):
        refs.append(O.ref_shifted_solve(n, ptr, col, val, b, sigma, seed))
    for r in refs:
        assert o["ret"] == r["ret"] and np.array_equal(o["x"], r["x"]) and np.array_equal(o["r"], r["r"])


@pytest.mark.parametrize("name,kind,g,p0,L,scale,seed", SHIFTED_CASES)
def test_reference_noovlp_twin_is_the_same_solve(B, O, gold_shifted, checks, name, kind, g, p0, L, scale, seed):
    """shifted_lopbicg_switching_noovlp (shifted_switching_solver.c:611) differs from shifted_lopbicg_switching only in when it waits
    for the halo exchange and in its timers: return value, every x_j, r and the residual history of the two compiled reference
    functions are bit-identical -- which is why the library exports the former as the latter (csrc/abi.cu).  The twin's outputs
    are golden (x and r as digests); the live functions are compared too where oracle/_ref is built."""
    blk, n, ptr, col, val = global_csr(B, kind, g, p0)
    sigma, b = shifted_problem(O, n, ptr, col, val, L, scale, seed)
    a = {k: gold_shifted[f"{name}|{k}"] for k in ("ret", "x", "r", "res")}
    c = {k: checks[f"noovlp|{name}|{k}"] for k in ("ret", "res", "x_sha256", "r_sha256")}
    assert a["ret"] == c["ret"] and sha256(a["x"]) == str(c["x_sha256"]) and sha256(a["r"]) == str(c["r_sha256"])
    assert np.array_equal(a["res"], c["res"])
    o = O.shifted_solve(n, ptr, col, val, b, sigma, seed)                      # and the oracle reproduces the twin
    assert o["ret"] == c["ret"] and sha256(o["x"]) == str(c["x_sha256"]) and sha256(o["r"]) == str(c["r_sha256"])
    if O.have_ref("libref_strict.so"):
        a = O.ref_shifted_solve(n, ptr, col, val, b, sigma, seed)
        c = O.ref_shifted_solve(n, ptr, col, val, b, sigma, seed, variant="shifted_lopbicg_switching_noovlp")
        assert a["ret"] == c["ret"] and np.array_equal(a["x"], c["x"]) and np.array_equal(a["r"], c["r"])
        assert np.array_equal(a["res"], c["res"])
