"""Generate tests/golden/ref_checks.npz: what the reference's own compiled code (oracle/_ref, built by `make -C oracle ref`
from the reference's sources) returns for the remaining comparisons of the test suite, so that the suite compares against
the reference without needing it.  Run where oracle/_ref is built:  python tests/golden/make_golden_checks.py

  cd25|<method>|...          bicgstab()/... in-process (libref_strict.so), convdiff g=25, b = A*1, tol 1e-11
  ones_s9|<method>|P<P>|...  ref_driver_strict with P ranks, stencil15 g=9, b = all ones, tol 1e-11
  noovlp|<case>|...          shifted_lopbicg_switching_noovlp on every SHIFTED_CASES problem (x, r as SHA-256 digests)
  mm_cd12|iters              the reference's main.c (ref_main_hist) on the Matrix-Market file of convdiff g=12
  shiftdiag_cd12|val         csr_shift_diagonal(A, 0.37) on the diagonal block of convdiff g=12
  tprime|iters_fast/_strict  ref_driver_fast / _strict, P = 1, on the benchmark's T' matrix, b = A*1, tol 1e-8
"""
import ctypes
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import mpi_bicgstab_b200 as B
import oracle as O
from helpers import METHODS, SHIFTED_CASES, big_csr, global_csr, sha256, shifted_problem, write_mtx

out = {}
blk, n, ptr, col, val = global_csr(B, "convdiff", 25, 2.0, seed=99)
b = O.spmv(n, ptr, col, val, np.ones(n))
for method in METHODS:
    kw = dict(krr=7, nrr=2) if method.endswith("rr") else {}
    r = O.ref_solve(method, n, ptr, col, val, b, tol=1e-11, max_iter=400, **kw)
    for k in ("iters", "res", "x", "r"):
        out[f"cd25|{method}|{k}"] = np.asarray(r[k])

blk, n, ptr, col, val = global_csr(B, "stencil15", 9, 14.0)
with tempfile.TemporaryDirectory() as td:
    f = os.path.join(td, "a.bin")
    O.write_csr_bin(f, n, ptr, col, val)
    for P in (1, 3):
        for method in METHODS[:3]:
            r = O.ref_driver(method, f, P=P, rhs="ones", tol=1e-11, max_iter=400, flavour="strict")
            for k in ("iters", "res", "x", "r"):
                out[f"ones_s9|{method}|P{P}|{k}"] = np.asarray(r[k])

for name, kind, g, p0, L, scale, seed in SHIFTED_CASES:
    blk, n, ptr, col, val = global_csr(B, kind, g, p0)
    sigma, b = shifted_problem(O, n, ptr, col, val, L, scale, seed)
    r = O.ref_shifted_solve(n, ptr, col, val, b, sigma, seed, variant="shifted_lopbicg_switching_noovlp")
    out[f"noovlp|{name}|ret"] = np.int64(r["ret"])
    out[f"noovlp|{name}|res"] = r["res"]
    out[f"noovlp|{name}|x_sha256"] = np.array(sha256(r["x"]))
    out[f"noovlp|{name}|r_sha256"] = np.array(sha256(r["r"]))

blk = B.gen_block("convdiff", 12, 1.5)
ptr, col, val = B.block_to_global_csr(blk)
with tempfile.TemporaryDirectory() as td:
    f = os.path.join(td, "a.mtx")
    write_mtx(f, blk.n, ptr, col, val)
    env = dict(os.environ, REF_EPS="1e-10", REF_MAX_ITER="500", REF_OUT_ITER="1", MALLOC_MMAP_THRESHOLD_="0")
    p = subprocess.run([os.path.join(O.REF_DIR, "ref_main_hist"), f, "bicgstab"], env=env, capture_output=True, text=True,
                       check=True)
    out["mm_cd12|iters"] = np.int64(re.search(r"Total iter\s*:\s*(\d+)", p.stdout).group(1))

nz = int(blk.diag.nz)
v = np.array(blk.diag_arrays()[0][:nz], dtype=np.float64)
c = np.array(blk.diag_arrays()[1][:nz], dtype=np.uint32)
q = np.array(blk.diag_arrays()[2][:blk.n + 1], dtype=np.uint32)
D = O._RefCSR()
D.val, D.col, D.ptr = O._p(v, O._dp), O._p(c, O._up), O._p(q, O._up)
D.nz, D.rows, D.cols = nz, blk.n, blk.n
L = O.ref_lib("strict")
L.csr_shift_diagonal.argtypes = [ctypes.POINTER(O._RefCSR), ctypes.c_double]
L.csr_shift_diagonal(ctypes.byref(D), 0.37)
out["shiftdiag_cd12|val"] = v

f = big_csr("stencil15", 117, 14.0)[0]
for fl in ("fast", "strict"):
    out[f"tprime|iters_{fl}"] = np.int64(O.ref_driver("bicgstab", f, P=1, rhs="a1", tol=1e-8, max_iter=1000, flavour=fl,
                                                       want_vectors=False, timeout=1200)["iters"])

np.savez_compressed(os.path.join(ROOT, "tests", "golden", "ref_checks.npz"), **out)
for k, a in out.items():
    if a.size == 1:
        print(k, a)
print("written", len(out), "arrays")
