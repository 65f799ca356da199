"""Shared test inputs: small members of the BASELINE.json matrix families (csrc/gen.cpp)."""
import numpy as np

# (name, kind, g, p0): sizes the oracle finishes in well under a second
SMALL_CASES = [
    ("stencil15_g12", "stencil15", 12, 14.0),      # Transport-like T', not diagonally dominant
    ("convdiff_g40", "convdiff", 40, 1.5),         # nonsymmetric convection-diffusion
    ("laplace5_g37", "laplace5", 37, 0.0),         # cfg 3 family, odd n
    ("random_n3001_k8", "random", 3001, 8),        # cfg 5 family, odd n
]
METHODS = ["bicgstab", "ca_bicgstab", "pipe_bicgstab", "pipe_bicgstab_rr"]
RR = dict(krr=10, nrr=3)


# shifted family (SURVEY.md 8(f) N4): (name, kind, g, p0, number of shifts, shift scale, seed index); sigma_j = (j + 1) * scale.
# The reference drivers use scale = 0.01 / L and seed 0 (main_shifted.c:95-99); the large-scale cases make the seed (the most
# diagonally dominant system) converge first, which exercises seed switching (shifted_switching_solver.c:490-527).
SHIFTED_CASES = [
    ("sh_stencil15_g12_L5", "stencil15", 12, 14.0, 5, 0.01 / 5, 0),
    ("sh_convdiff_g40_L6_switch", "convdiff", 40, 1.5, 6, 0.8, 5),
    ("sh_stencil15_g12_L4_switch", "stencil15", 12, 14.0, 4, 2.0, 3),
    ("sh_laplace5_g37_L16", "laplace5", 37, 0.0, 16, 0.01 / 16, 0),
]


def shifted_problem(O, n, ptr, col, val, L, scale, seed):
    """sigma and b = (A + sigma[seed] I) 1 as main_shifted.c:95-114 builds them."""
    sigma = (np.arange(L) + 1) * scale
    b = O.spmv(n, ptr, col, val, np.ones(n))
    O.daxpy(sigma[seed], np.ones(n), b)
    return sigma, b


def global_csr(B, kind, g, p0, seed=12345):
    blk = B.gen_block(kind, g, p0, seed)
    ptr, col, val = B.block_to_global_csr(blk)
    return blk, blk.n, ptr, col, val


def sha256(a):
    """Digest of a float64 vector's bytes: golden files store it in place of vectors too large to keep whole."""
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<f8").tobytes()).hexdigest()


def write_mtx(path, n, ptr, col, val):
    """Matrix-Market file of a CSR matrix, column-major like SuiteSparse files, with a comment and a blank line."""
    import scipy.sparse as sp
    A = sp.csr_matrix((val, col, ptr), shape=(n, n)).tocsc().tocoo()
    with open(path, "w") as fh:
        fh.write("%%MatrixMarket matrix coordinate real general\n% comment\n\n")
        fh.write(f"{n} {n} {A.nnz}\n")
        for r, c, v in zip(A.row, A.col, A.data):
            fh.write(f"{r + 1} {c + 1} {float(v)!r}\n")
    return A


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


_BIG = {}


def big_csr(kind, g, p0, tmpdir="/dev/shm"):
    """Full-size synthetic matrix as (file, n, ptr, col, val): written once per session by the stand-alone generator
    oracle/gen_csr (binary layout of oracle.py: write_csr_bin), so neither numpy index gymnastics nor a second copy of the
    1.6 M-row matrix is needed.  The file is what oracle/_ref/ref_driver_* reads."""
    import atexit, os, shutil, subprocess, tempfile
    key = (kind, g, p0)
    if key not in _BIG:
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        gen = os.path.join(root, "oracle", "gen_csr")
        if not os.path.exists(gen):
            subprocess.run(["make", "-C", os.path.join(root, "oracle"), "oracle"], check=True)
        d = tempfile.mkdtemp(dir=tmpdir if os.path.isdir(tmpdir) else None)
        atexit.register(shutil.rmtree, d, True)           # a few hundred MB of shared memory per matrix
        f = os.path.join(d, f"{kind}_{g}.bin")
        kinds = {"stencil15": 0, "laplace5": 1, "random": 2, "convdiff": 3}
        subprocess.run([gen, str(kinds[kind]), str(int(g)), repr(float(p0)), f], check=True, capture_output=True)
        with open(f, "rb") as fh:
            n, nnz = (int(v) for v in np.fromfile(fh, dtype=np.int64, count=2))
            ptr = np.fromfile(fh, dtype=np.uint32, count=n + 1)
            col = np.fromfile(fh, dtype=np.uint32, count=nnz)
            if (n + 1 + nnz) % 2:
                np.fromfile(fh, dtype=np.uint32, count=1)
            val = np.fromfile(fh, dtype=np.float64, count=nnz)
        _BIG[key] = (f, n, ptr, col, val)
    return _BIG[key]
