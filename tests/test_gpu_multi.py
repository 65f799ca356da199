"""GPU, N > 1 (skipped on single-GPU boxes): row-partitioned solve over peer memory vs the oracle's P-rank emulation."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ngpu():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_multi_gpu_parity(world):
    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 29700 + world
    cmd = ["timeout", "600", sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "_mgpu_worker.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=700)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    assert f"MGPU_WORKER_OK {world}" in p.stdout


def test_reference_main_c_two_ranks(tmp_path):
    """The reference's unchanged main.c as TWO processes (one per GPU) under tools/bicgrun: MPI_Init of
    include/compat/mpi.h bootstraps through POSIX shm, each rank loads its row block from the .mtx file."""
    import re
    import numpy as np
    if _ngpu() < 2:
        pytest.skip("needs 2 GPUs")
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_main_b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/ref_main_b200 not built")
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
    import mpi_bicgstab_b200 as B
    import oracle as O
    from helpers import write_mtx
    blk = B.gen_block("stencil15", 12, 14.0)
    f = tmp_path / "s12.mtx"
    n = blk.n
    ptr, col, val = B.block_to_global_csr(blk)
    write_mtx(f, n, ptr, col, val)
    env = dict(os.environ, BICG_TOL="1e-10", BICG_MAX_ITER="600")
    p = subprocess.run([os.path.join(ROOT, "tools", "bicgrun"), "-np", "2", exe, str(f), "bicgstab"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    assert "Node: 1, Proc: 2" in p.stdout
    it = int(re.search(r"Total iter\s*:\s*(\d+)", p.stdout).group(1))
    ref = O.solve("bicgstab", n, ptr, col, val, O.spmv(n, ptr, col, val, np.ones(n), P=2), P=2, tol=1e-10, max_iter=600)
    assert abs(it - ref["iters"]) <= 2
