"""Python mirror of the reference's operator interface for the BiCGStab hot path.

Same names, argument meaning and error behaviour as solver.h:10-13 / matrix.h:44-51 of the reference, on
numpy arrays instead of raw pointers; every call goes straight through the C ABI of libbicgstab_b200.so
(include/bicgstab_b200.h) -- nothing is computed in Python.

    blk = gen_block("stencil15", 24, diag=16.0)            # or load_matrix_block("A.mtx"), or blocks_from_csr(...)
    b = spmv_ovlap(blk, np.ones(blk.n_loc))                  # main.c:109-113
    x = np.zeros(blk.n_loc)
    iters = bicgstab(blk, x, b)                              # x: solution, b: final recursive residual
"""
import ctypes as C

import numpy as np

from ._lib import ALLGATHER_FN, CSR_Matrix, INFO_Matrix, bicg_stats, lib

METHODS = {"bicgstab": 0, "ca_bicgstab": 1, "pipe_bicgstab": 2, "pipe_bicgstab_rr": 3}
GEN_KINDS = {"stencil15": 0, "laplace5": 1, "random": 2, "convdiff": 3}


def _dptr(a):
    return a.ctypes.data_as(C.c_void_p)


class MatrixBlock:
    """One rank's (A_loc_diag, A_loc_offd, A_info) triple -- what the reference's entry points take."""

    def __init__(self, world):
        self.diag = CSR_Matrix()
        self.offd = CSR_Matrix()
        self.info = INFO_Matrix()
        self._recvcounts = (C.c_int * world)()
        self._displs = (C.c_int * world)()
        self.info.recvcounts = C.cast(self._recvcounts, C.POINTER(C.c_int))
        self.info.displs = C.cast(self._displs, C.POINTER(C.c_int))
        self.world = world
        self._keep = []            # numpy arrays backing the CSR pointers (when Python owns them)
        self._lib_owned = False    # True: arrays were malloc'ed by the library -> csr_free_matrix

    # -- views ---------------------------------------------------------------------------------------
    @property
    def n_loc(self):
        return int(self.diag.rows)

    @property
    def n(self):
        return int(self.info.rows)

    @property
    def nnz_loc(self):
        return int(self.diag.nz) + int(self.offd.nz)

    @property
    def recvcounts(self):
        return np.array(self._recvcounts[:], dtype=np.int32)

    @property
    def displs(self):
        return np.array(self._displs[:], dtype=np.int32)

    @staticmethod
    def _view(m):
        nz, rows = int(m.nz), int(m.rows)
        val = np.ctypeslib.as_array(m.val, shape=(nz,)) if nz else np.zeros(0)
        col = np.ctypeslib.as_array(m.col, shape=(nz,)) if nz else np.zeros(0, dtype=np.uint32)
        ptr = np.ctypeslib.as_array(m.ptr, shape=(rows + 1,))
        return val, col, ptr

    def diag_arrays(self):
        return self._view(self.diag)

    def offd_arrays(self):
        return self._view(self.offd)

    def free(self):
        if self._lib_owned:
            lib.csr_free_matrix(C.byref(self.diag))
            lib.csr_free_matrix(C.byref(self.offd))
            self._lib_owned = False
        else:
            lib.bicg_matrix_invalidate(C.byref(self.diag))
        self._keep = []

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def plan_partition(n, world):
    """matrix.c:295-308."""
    cnt = (C.c_int * world)()
    dsp = (C.c_int * world)()
    lib.bicg_plan_partition(n, world, cnt, dsp)
    return np.array(cnt[:], dtype=np.int64), np.array(dsp[:], dtype=np.int64)


def _fill_csr(m, val, col, ptr, rows, cols, keep):
    val = np.ascontiguousarray(val, dtype=np.float64)
    col = np.ascontiguousarray(col, dtype=np.uint32)
    ptr = np.ascontiguousarray(ptr, dtype=np.uint32)
    if val.size == 0:               # keep non-null pointers like malloc(0) would
        val = np.zeros(1, dtype=np.float64)
        col = np.zeros(1, dtype=np.uint32)
    keep += [val, col, ptr]
    m.val = val.ctypes.data_as(C.POINTER(C.c_double))
    m.col = col.ctypes.data_as(C.POINTER(C.c_uint))
    m.ptr = ptr.ctypes.data_as(C.POINTER(C.c_uint))
    m.nz = int(ptr[-1])
    m.rows = rows
    m.cols = cols


def blocks_from_csr(n, ptr, col, val, rank=0, world=1):
    """Split a global CSR into rank's diag / offd blocks exactly as the reference's block loader does
    (partition matrix.c:295-308; diag: local columns, offd: global columns, in-row order kept,
    matrix.c:380-392)."""
    ptr = np.asarray(ptr, dtype=np.int64)
    col = np.asarray(col, dtype=np.int64)
    val = np.asarray(val, dtype=np.float64)
    cnt, dsp = plan_partition(n, world)
    lo, nloc = int(dsp[rank]), int(cnt[rank])
    hi = lo + nloc
    a, b = int(ptr[lo]), int(ptr[hi])
    c, v = col[a:b], val[a:b]
    rows = np.repeat(np.arange(nloc), np.diff(ptr[lo:hi + 1]))
    own = (c >= lo) & (c < hi)
    blk = MatrixBlock(world)
    for mask, m, shift, ncols in ((own, blk.diag, lo, nloc), (~own, blk.offd, 0, n)):
        r = rows[mask]
        p = np.zeros(nloc + 1, dtype=np.int64)
        np.add.at(p, r + 1, 1)
        p = np.cumsum(p)
        _fill_csr(m, v[mask], c[mask] - shift, p, nloc, ncols, blk._keep)
    blk.info.nz = int(ptr[-1]) & 0xFFFFFFFF
    blk.info.rows = n
    blk.info.cols = n
    blk.info.code = b"MCRG"
    for p_ in range(world):
        blk._recvcounts[p_] = int(cnt[p_])
        blk._displs[p_] = int(dsp[p_])
    return blk


def gen_block(kind, g, p0=0.0, seed=12345, rank=0, world=1):
    """Synthetic inputs of SURVEY.md 8(d) (csrc/gen.cpp), generated directly as one rank's blocks."""
    blk = MatrixBlock(world)
    rc = lib.bicg_gen_block(GEN_KINDS[kind], int(g), float(p0), int(seed), rank, world,
                            C.byref(blk.diag), C.byref(blk.offd), C.byref(blk.info))
    if rc != 0:
        raise ValueError(f"bicg_gen_block({kind}, g={g}) failed with {rc}")
    blk._lib_owned = True
    return blk


def load_matrix_block(filename, world=None):
    """MPI_csr_load_matrix_block (matrix.h:50): Matrix-Market file -> this rank's blocks."""
    world = world or lib.bicg_comm_world()
    blk = MatrixBlock(world)
    lib.MPI_csr_load_matrix_block(str(filename).encode(), C.byref(blk.diag), C.byref(blk.offd), C.byref(blk.info))
    blk._lib_owned = True
    return blk


def block_to_global_csr(blk, rank=0):
    """(ptr, col, val) of the block's rows with GLOBAL column indices, diag entries first then offd
    (the order the reference accumulates them in, matrix.c:437-440)."""
    dv, dc, dp = blk.diag_arrays()
    ov, oc, op_ = blk.offd_arrays()
    lo = int(blk.displs[rank])
    nloc = blk.n_loc
    ptr = dp.astype(np.int64) + op_.astype(np.int64)
    col = np.empty(int(ptr[-1]), dtype=np.int64)
    val = np.empty(int(ptr[-1]), dtype=np.float64)
    dlen, olen = np.diff(dp.astype(np.int64)), np.diff(op_.astype(np.int64))
    row_d = np.repeat(np.arange(nloc), dlen)
    row_o = np.repeat(np.arange(nloc), olen)
    pos_d = ptr[row_d] + (np.arange(dlen.sum()) - dp.astype(np.int64)[row_d])
    pos_o = ptr[row_o] + dlen[row_o] + (np.arange(olen.sum()) - op_.astype(np.int64)[row_o])
    col[pos_d] = dc.astype(np.int64)[:dlen.sum()] + lo
    val[pos_d] = dv[:dlen.sum()]
    col[pos_o] = oc.astype(np.int64)[:olen.sum()]
    val[pos_o] = ov[:olen.sum()]
    return ptr, col, val


# ---- the reference's entry points ------------------------------------------------------------------------
def _vec(a, n):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"] and a.size >= n, "need a contiguous float64 vector"
    return _dptr(a)


def spmv_ovlap(blk, x_loc, x_scratch=None, y_loc=None):
    """MPI_csr_spmv_ovlap (matrix.h:51): y_loc = A x.  Returns y_loc."""
    if y_loc is None:
        y_loc = np.empty(blk.n_loc)
    if x_scratch is None:
        x_scratch = np.zeros(blk.n)
    lib.MPI_csr_spmv_ovlap(C.byref(blk.diag), C.byref(blk.offd), C.byref(blk.info), _vec(x_loc, blk.n_loc),
                           _vec(x_scratch, blk.n), _vec(y_loc, blk.n_loc))
    return y_loc


def bicgstab(blk, x_loc, r_loc):
    return lib.bicgstab(C.byref(blk.diag), C.byref(blk.offd), C.byref(blk.info), _vec(x_loc, blk.n_loc), _vec(r_loc, blk.n_loc))


def ca_bicgstab(blk, x_loc, r_loc):
    return lib.ca_bicgstab(C.byref(blk.diag), C.byref(blk.offd), C.byref(blk.info), _vec(x_loc, blk.n_loc), _vec(r_loc, blk.n_loc))


def pipe_bicgstab(blk, x_loc, r_loc):
    return lib.pipe_bicgstab(C.byref(blk.diag), C.byref(blk.offd), C.byref(blk.info), _vec(x_loc, blk.n_loc), _vec(r_loc, blk.n_loc))


def pipe_bicgstab_rr(blk, x_loc, r_loc, krr, nrr):
    return lib.pipe_bicgstab_rr(C.byref(blk.diag), C.byref(blk.offd), C.byref(blk.info), _vec(x_loc, blk.n_loc),
                                _vec(r_loc, blk.n_loc), int(krr), int(nrr))


def solve(method, blk, x_loc, r_loc, krr=0, nrr=0):
    if method == "pipe_bicgstab_rr":
        return pipe_bicgstab_rr(blk, x_loc, r_loc, krr, nrr)
    return {"bicgstab": bicgstab, "ca_bicgstab": ca_bicgstab, "pipe_bicgstab": pipe_bicgstab}[method](blk, x_loc, r_loc)


def shifted_lopbicg_switching(blk, x_set, r_loc, sigma, seed):
    """shifted_switching_solver.h:12.  x_set: (sigma_len, n_loc) C-contiguous; returns the reference's k (iterations + 1)."""
    sigma = np.ascontiguousarray(sigma, dtype=np.float64)
    assert x_set.dtype == np.float64 and x_set.flags["C_CONTIGUOUS"] and x_set.shape == (sigma.size, blk.n_loc)
    return lib.shifted_lopbicg_switching(C.byref(blk.diag), C.byref(blk.offd), C.byref(blk.info), _dptr(x_set), _vec(r_loc, blk.n_loc),
                                         _dptr(sigma), int(sigma.size), int(seed))


def last_shift_info(sigma_len):
    seed = C.c_int()
    stop = (C.c_int * sigma_len)()
    lib.bicg_last_shift_info(C.byref(seed), stop, sigma_len)
    return seed.value, np.array(stop[:])


# ---- extensions ------------------------------------------------------------------------------------------
def set_option(key, value):
    if lib.bicg_set_option(str(key).encode(), str(value).encode()) != 0:
        raise KeyError(key)


def set_options(**kw):
    for k, v in kw.items():
        set_option(k.upper(), v)


def last_history():
    """dot_r/dot_zero after every iteration of the last solve on this rank (entry 0 = 1)."""
    n = lib.bicg_last_history(None, 0)
    out = np.empty(max(n, 1))
    lib.bicg_last_history(out.ctypes.data_as(C.POINTER(C.c_double)), n)
    return out[:n]


def _stats_dict(s):
    return {f: getattr(s, f) for f, _ in bicg_stats._fields_}


def last_stats():
    return _stats_dict(lib.bicg_last_stats().contents)


class DeviceMatrix:
    """A device-resident matrix handle (bicg_matrix): upload once, solve / multiply many times."""

    def __init__(self, blk):
        self.blk = blk
        self.h = lib.bicg_matrix_create(C.byref(blk.diag), C.byref(blk.offd), C.byref(blk.info))
        if not self.h:
            raise RuntimeError("bicg_matrix_create failed")

    def solve(self, method, x, r, krr=0, nrr=0):
        st = bicg_stats()
        it = lib.bicg_solve(self.h, METHODS[method], _vec(x, self.blk.n_loc), _vec(r, self.blk.n_loc), krr, nrr, 0, C.byref(st))
        return it, _stats_dict(st)

    def spmv(self, x_loc):
        y = np.empty(self.blk.n_loc)
        lib.bicg_spmv(self.h, _vec(x_loc, self.blk.n_loc), _dptr(y))
        return y

    def resident_ctas(self):
        """CTAs of the last persistent-kernel launch that kept their matrix slice in shared memory (BICG_RESIDENT)."""
        return int(lib.bicg_debug_resident_ctas(self.h))

    def mega_tiles(self):
        """(tiles, narrow): tiles of the persistent-kernel plan and how many of them stream 16-bit column codes."""
        narrow = C.c_int()
        tiles = lib.bicg_debug_mega_tiles(self.h, C.byref(narrow))
        return int(tiles), int(narrow.value)

    def spmv_time(self, reps=20):
        ms, by = C.c_double(), C.c_double()
        lib.bicg_spmv_time(self.h, reps, C.byref(ms), C.byref(by))
        return ms.value, by.value

    def profile(self, method, iters):
        ms = (C.c_double * 3)()
        cnt = (C.c_int * 3)()
        rc = lib.bicg_profile_solve(self.h, METHODS[method], iters, ms, cnt)
        if rc != 0:
            raise RuntimeError("bicg_profile_solve failed")
        return list(ms), list(cnt)

    def destroy(self):
        if self.h:
            lib.bicg_matrix_destroy(self.h)
            self.h = None


_CALLBACK_KEEPALIVE = []


def comm_init(rank, world, allgather_bytes):
    """Register this process as `rank` of `world`.  allgather_bytes(b: bytes) -> list[bytes] (one per rank)."""

    def _cb(_ctx, send, recv, nbytes):
        try:
            mine = C.string_at(send, nbytes)
            parts = allgather_bytes(mine)
            C.memmove(recv, b"".join(parts), nbytes * world)
            return 0
        except Exception as exc:                      # never let an exception unwind through C
            print(f"bicg allgather callback failed: {exc!r}", flush=True)
            return 1

    cb = ALLGATHER_FN(_cb)
    _CALLBACK_KEEPALIVE.append(cb)
    rc = lib.bicg_comm_init(rank, world, cb, None)
    if rc != 0:
        raise ValueError(f"bicg_comm_init({rank}, {world}) failed")


def comm_init_torch(group=None):
    """Bootstrap from an initialised torch.distributed job (one process per GPU, as torchrun starts them).
    Only the bootstrap bytes (IPC handles, halo plans) travel through torch; solver traffic is peer memory."""
    import torch
    import torch.distributed as dist

    rank, world = dist.get_rank(group), dist.get_world_size(group)
    backend = dist.get_backend(group)
    dev = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")

    def allgather_bytes(b):
        t = torch.frombuffer(bytearray(b), dtype=torch.uint8).to(dev)
        outs = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(outs, t, group=group)
        return [o.cpu().numpy().tobytes() for o in outs]

    comm_init(rank, world, allgather_bytes)
    return rank, world


def comm_finalize():
    lib.bicg_comm_finalize()
