"""Generate tests/golden/ref_histories.npz from the reference's own sources (oracle/_ref, built by `make -C oracle ref`).
Run where oracle/_ref is built:  python tests/golden/make_golden.py

For every small case x method x rank-count it stores what the REFERENCE produced: iteration count, the full
per-iteration sqrt(dot_r/dot_zero) history (captured as doubles before printf formatting), final x and r.  r hardly
compresses: for the cases in R_DIGEST only the SHA-256 of its bytes is kept, which keeps the bit-for-bit check and the
file under 1 MB.
P = 1 runs the reference in-process (libref_strict.so); P > 1 runs ref_driver_strict under the fork+shm
mini-MPI.  Matrices are regenerated from (kind, g, p0, seed) by csrc/gen.cpp, so only the results are stored.
"""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import mpi_bicgstab_b200 as B
import oracle as O
from helpers import METHODS, RR, SMALL_CASES, global_csr, sha256

TOL, MAX_ITER = 1e-10, 600
R_DIGEST = {"laplace5_g37"}
out = {}
for name, kind, g, p0 in SMALL_CASES:
    blk, n, ptr, col, val = global_csr(B, kind, g, p0)
    with tempfile.TemporaryDirectory() as td:
        f = os.path.join(td, "a.bin")
        O.write_csr_bin(f, n, ptr, col, val)
        for P in (1, 2, 3):
            for method in METHODS:
                kw = RR if method.endswith("rr") else {}
                if P == 1:
                    b = O.spmv(n, ptr, col, val, np.ones(n))
                    r = O.ref_solve(method, n, ptr, col, val, b, tol=TOL, max_iter=MAX_ITER, **kw)
                else:
                    r = O.ref_driver(method, f, P=P, rhs="a1", tol=TOL, max_iter=MAX_ITER, flavour="strict", **kw)
                key = f"{name}|{method}|P{P}"
                out[key + "|iters"] = np.int64(r["iters"])
                out[key + "|res"] = r["res"]
                out[key + "|x"] = r["x"]
                if name in R_DIGEST:
                    out[key + "|r_sha256"] = np.array(sha256(r["r"]))
                else:
                    out[key + "|r"] = r["r"]
                print(key, r["iters"], float(r["res"][-1]))
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "ref_histories.npz"), **out)
print("written", len(out), "arrays")
