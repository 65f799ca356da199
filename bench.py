#!/usr/bin/env python
"""bench.py -- BiCGStab iterations/s on the BASELINE.json configs.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload transport|laplace|random]
                  [--method bicgstab|ca_bicgstab|pipe_bicgstab]

One STEP = one complete solve of the workload (b = A*1, x0 = 0, to BICG_TOL / MAX_ITER of the config).
  value : iterations/s, matrix + vectors resident in HBM when the timed region starts (CUDA events on the
          library's stream around the K solves, max over ranks)
  e2e   : the same metric through the reference-facing call bicgstab(A_diag, A_offd, A_info, x, r) on pinned
          HOST buffers with the upload cache disabled: every step uploads the matrix and the vectors and reads
          x and r back (wall clock around K calls, device idle on both sides).  e2e_pageable: the same with plain
          malloc'ed buffers (what the reference's main.c:81-107 passes).  first_call_ms: the very first upload +
          plan (SpMV autotune included), which the warm-up otherwise hides.
  roofline    : the kernel that runs in the timed region -- the persistent solver kernel (one launch per solve):
                iterations x per-iteration algorithmic bytes (SURVEY.md 8(d)) / the library's CUDA-event time of
                the loop; the fused SpMV + dot kernel is timed live beside it (roofline.spmv_kernel)
  parity      : on EVERY line (every N): H-level max relative error of the first 10 residual-history entries
                against the oracle's P = N emulation on the same matrix, and iterations-to-tolerance against the
                reference's own sources run with P = N ranks (oracle/_ref/ref_driver_*)
  cpu_baseline: the reference's own sources (oracle/_ref, compiled in place) on this box's host cores, bounded
                sample = the first REF_ITERS iterations of the same solve

--impl reference times that CPU build alone (rank 0 only under torchrun); it never loads the product library.

--dump-outputs DIR writes what the last timed solve returned to its caller, so that two builds can be compared output
for output (the inputs depend only on the arguments): x.npy and r.npy (the solution and the recursive residual),
history.npy (dot_r/dot_zero per iteration) and iterations.npy, all float64.  Under torchrun every rank writes its own
row block with a _rank<R> suffix.  Where x and r would exceed 64 MB in all, a fixed seeded sample of rows is written
instead, with their global row numbers in index.npy.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs 2/4: Transport.mtx is not in the image (no network) -> T' surrogate of SURVEY.md 8(d)
    "transport": dict(kind="stencil15", g=117, p0=14.0, tol=1e-8, max_iter=1000, method="bicgstab",
                      label="T' = 15-pt stencil on 117^3 (n=1,601,613, nnz=23,616,325; Transport.mtx surrogate, "
                            "diag=14 variant), b=A*1, x0=0, tol 1e-8"),
    # config 3
    "laplace": dict(kind="laplace5", g=2000, p0=0.0, tol=1e-8, max_iter=1000, method="pipe_bicgstab",
                    label="5-pt Laplacian 2000^2 (n=4,000,000, nnz=19,992,000), b=A*1, x0=0, 1000 iterations max"),
    # config 5 (per-GPU block 2 M rows x 32 nnz/row; n scales with the number of GPUs)
    "random": dict(kind="random", g=2_000_000, p0=32, tol=1e-8, max_iter=1000, method="ca_bicgstab",
                   label="random CSR, 2,000,000 rows per GPU x 32 nnz/row, b=A*1, x0=0, tol 1e-8"),
}
BYTES_PER_ITER_N = {"bicgstab": 160, "ca_bicgstab": 216, "pipe_bicgstab": 232}   # SURVEY.md 8(d)
REF_ITERS = 100        # iterations per reference step: ~1-2 s of CPU work per step, init SpMV amortised over 100
DUMP_BYTES = 60 << 20  # --dump-outputs: x and r of all ranks together stay below this (history and index come on top)


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [t.strip() for t in l.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def pinned_array(B, shape, dtype):
    import ctypes as C
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = B.lib.bicg_host_alloc(max(nbytes, 16))
    buf = (C.c_char * max(nbytes, 16)).from_address(p)
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


def pinned_block(B, blk, rank, world):
    """Copy a generated block into pinned host memory (the e2e leg's inputs live there)."""
    import ctypes as C
    out = B.MatrixBlock(world)
    for src, dst, ncols in ((blk.diag, out.diag, blk.diag.cols), (blk.offd, out.offd, blk.offd.cols)):
        val, col, ptr = B.MatrixBlock._view(src)
        pv, pc, pp = pinned_array(B, max(val.size, 1), np.float64), pinned_array(B, max(col.size, 1), np.uint32), \
            pinned_array(B, ptr.size, np.uint32)
        pv[:val.size] = val; pc[:col.size] = col; pp[:] = ptr
        dst.val = pv.ctypes.data_as(C.POINTER(C.c_double)); dst.col = pc.ctypes.data_as(C.POINTER(C.c_uint))
        dst.ptr = pp.ctypes.data_as(C.POINTER(C.c_uint))
        dst.nz, dst.rows, dst.cols = src.nz, src.rows, ncols
        out._keep += [pv, pc, pp]
    out.info.nz, out.info.rows, out.info.cols, out.info.code = blk.info.nz, blk.info.rows, blk.info.cols, b"MCRG"
    for p in range(world):
        out._recvcounts[p] = int(blk.recvcounts[p]); out._displs[p] = int(blk.displs[p])
    return out


# ---------------------------------------------------------------------------------------------------------
GEN_KIND = {"stencil15": 0, "laplace5": 1, "random": 2, "convdiff": 3}


def _ref_flavour(O, gen):
    """BASELINE.md builds the CPU baseline with -march=native.  oracle/_ref/ref_driver_native was compiled in the dev
    container; if this host's CPU cannot execute it (SIGILL on a tiny real solve) fall back to the portable
    x86-64-v3 build."""
    with tempfile.TemporaryDirectory() as td:
        tiny = os.path.join(td, "tiny.bin")
        try:
            subprocess.run([gen, "0", "8", "14.0", tiny], check=True, capture_output=True, timeout=60)
        except Exception:
            return None
        for flavour in ("native", "fast"):
            if not os.path.exists(os.path.join(O.REF_DIR, f"ref_driver_{flavour}")):
                continue
            try:
                r = O.ref_driver("bicgstab", tiny, P=1, tol=0.0, max_iter=3, flavour=flavour, want_vectors=False, timeout=60)
                if r["iters"] == 3:
                    return flavour
            except Exception:
                pass
    return None


class RefRunner:
    """The reference's own CPU code (oracle/_ref/ref_driver_* + mini-MPI) on the same input.  The matrix is written
    once to a binary file in /dev/shm by the stand-alone generator oracle/gen_csr (same generator source as the
    library, but no product .so is loaded in this arm); every run() is one `ref_driver` process tree."""

    def __init__(self, w, cores=None):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle as O
        self.O, self.w = O, w
        gen = os.path.join(ROOT, "oracle", "gen_csr")
        self.flavour = _ref_flavour(O, gen) if os.path.exists(gen) else None
        self.ok = self.flavour is not None
        if not self.ok:
            return
        self.march = {"native": "-march=native (built in the dev container)", "fast": "-march=x86-64-v3"}[self.flavour]
        self.cores = cores or min(len(os.sched_getaffinity(0)), 64)
        self.td = tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        self.file = os.path.join(self.td.name, "a.bin")
        subprocess.run([gen, str(GEN_KIND[w["kind"]]), str(int(w["g"])), repr(float(w["p0"])), self.file], check=True,
                       capture_output=True, timeout=1800)

    def load_csr(self):
        """(n, ptr, col, val) of the file the reference solves (oracle.py: write_csr_bin layout)."""
        with open(self.file, "rb") as f:
            n, nnz = (int(v) for v in np.fromfile(f, dtype=np.int64, count=2))
            ptr = np.fromfile(f, dtype=np.uint32, count=n + 1)
            col = np.fromfile(f, dtype=np.uint32, count=nnz)
            if (n + 1 + nnz) % 2:
                np.fromfile(f, dtype=np.uint32, count=1)
            val = np.fromfile(f, dtype=np.float64, count=nnz)
        return n, ptr, col, val

    def run(self, n_iters, cores=None):
        cores = cores or self.cores
        res = self.O.ref_driver(self.w["method"], self.file, P=cores, rhs="a1", tol=0.0, max_iter=n_iters,
                                flavour=self.flavour, want_vectors=False, pin=True, timeout=1800)
        res["cores"] = cores
        return res

    def pick_cores(self):
        """The reference replicates the whole x on every rank per SpMV (matrix.c:432), so more ranks is not always
        faster on one host: try the power-of-two rank counts up to the core count (capped at 64, the reference's own
        largest single-node job) for a few iterations each and keep the fastest -- its best foot forward."""
        limit = min(len(os.sched_getaffinity(0)), 64)
        best, tried, p = None, {}, 1
        while p <= limit:
            try:
                r = self.run(4, cores=p)
                tried[p] = r["avg_time_per_iter_s"]
                if best is None or tried[p] < tried[best]:
                    best = p
            except Exception:
                pass
            p *= 2
        self.cores = best or 1
        self.tried = tried
        return self.cores

    def solve_to_tol(self, P, tol, max_iter):
        """Full solve with P ranks: the reference's iteration count for the parity object."""
        return self.O.ref_driver(self.w["method"], self.file, P=P, rhs="a1", tol=tol, max_iter=max_iter,
                                 flavour=self.flavour, want_vectors=False, pin=True, timeout=1800)

    def close(self):
        if self.ok:
            self.td.cleanup()


def reference_sample(rr, n_iters):
    rr.pick_cores()                        # also pages the file in and warms the cores
    res = rr.run(n_iters)
    res["tried"] = rr.tried
    res["march"] = rr.march
    return res


def _first_exceed(a, b, tol=1e-10):
    """first index k (1-based iteration) where |a_k - b_k| / b_k > tol; len + 1 if never"""
    m = min(len(a), len(b))
    bad = np.nonzero(np.abs(a[:m] - b[:m]) > tol * np.abs(b[:m]))[0]
    return int(bad[0]) + 1 if bad.size else m + 1


def parity_object(rr, w, world, hist, iters):
    """Driver-visible parity at the benchmark's own size and rank count.
    H-level: first 10 entries of the residual history vs the oracle's P = world emulation (SURVEY.md 8(c): <= 1e-10 relative);
             plus the WINDOW over which the GPU history agrees with the oracle to 1e-10, next to the window over which the
             reference's own two builds (strict IEEE vs -O3 with FMA contraction) agree with each other -- BiCGStab histories are
             chaotic in the summation order, so agreement beyond the reference's own self-consistency window is not defined.
    C-level: iterations to tol vs the reference's own sources (the -O3 build a user makes) run with P = world ranks: within
             max(2, 2 %).  When that fails, the strict build of the same reference is run as well: at this size the
             reference's builds differ from each other by more than the rule (round 2: 333 vs 380 at P = 1)."""
    O = rr.O
    n, ptr, col, val = rr.load_csr()
    method = w["method"]
    t0 = time.perf_counter()
    b = O.spmv(n, ptr, col, val, np.ones(n), P=world)
    W = min(40, iters)
    ref = O.solve(method, n, ptr, col, val, b, P=world, tol=w["tol"], max_iter=W)
    W = min(W, ref["iters"])
    got, want = np.sqrt(np.asarray(hist[1:W + 1])), np.sqrt(ref["hist"][1:W + 1])
    m = min(10, W)
    rel = float(np.max(np.abs(got[:m] - want[:m]) / want[:m])) if m else 0.0
    out = {"h_level_max_rel": rel, "h_level_iters": int(m), "h_level_tol": 1e-10, "h_level_ok": bool(rel <= 1e-10),
           "h_level_oracle": f"oracle/liboracle.so, P={world} rank emulation (pinned bitwise to the compiled reference)",
           "h_window_gpu_vs_oracle": _first_exceed(got, want) - 1,
           "iters": int(iters), "ref_iters": None, "ref_P": world, "c_level_rule": "max(2, 2 %)"}
    try:
        user = rr.O.ref_driver(method, rr.file, P=world, rhs="a1", tol=0.0, max_iter=W, flavour=rr.flavour, want_vectors=True,
                               pin=True, timeout=900)
        out["h_window_reference_builds"] = _first_exceed(np.asarray(user["res"][:W]), want) - 1
        out["h_window_note"] = ("iterations over which the history agrees to 1e-10: GPU vs oracle, and the reference's own -O3 build "
                                f"vs its strict build (= the oracle), first {W} iterations examined")
    except Exception as exc:
        out["h_window_reference_builds"] = None
        out["h_window_note"] = f"reference history run failed: {exc!r}"
    try:
        full = rr.solve_to_tol(world, w["tol"], w["max_iter"])
        out["ref_iters"] = int(full["iters"])
        out["c_level_ok"] = bool(abs(iters - full["iters"]) <= max(2, int(0.02 * full["iters"])))
        out["ref_source"] = f"oracle/_ref/ref_driver_{rr.flavour} (the reference's own solver.c/matrix.c/vector.c), {world} ranks"
        if not out["c_level_ok"]:
            strict = rr.O.ref_driver(method, rr.file, P=world, rhs="a1", tol=w["tol"], max_iter=w["max_iter"], flavour="strict",
                                     want_vectors=False, pin=True, timeout=1800)
            lo, hi = sorted((int(full["iters"]), int(strict["iters"])))
            out["ref_iters_strict_build"] = int(strict["iters"])
            out["c_level_in_reference_spread"] = bool(lo - max(2, int(0.02 * lo)) <= iters <= hi + max(2, int(0.02 * hi)))
    except Exception as exc:
        out["ref_source"] = f"reference run failed: {exc!r}"
    out["seconds"] = round(time.perf_counter() - t0, 1)
    return out


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rr = RefRunner(w)
    if not rr.ok:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/ref_driver_* or oracle/gen_csr is not built"}))
        return
    steps, times, its = args.steps, [], 0
    try:
        rr.pick_cores()
        for s in range(args.warmup + steps):
            r = rr.run(REF_ITERS)
            if s >= args.warmup:
                times.append(r["total_time_s"]); its += r["iters"]
    finally:
        rr.close()
    total = sum(times)
    val = its / total
    line = {"metric": "BiCGStab iterations/sec", "value": val, "unit": "iterations/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": {"workload": w["label"], "method": w["method"],
                       "sample": f"first {REF_ITERS} iterations of the solve per step (reference's own timed region, solver.c:69-132)"},
            "cpu_baseline": {"value": val, "unit": "iterations/s", "cores": rr.cores, "kind": "reference",
                             "sample": f"{REF_ITERS} iterations/step x {steps} steps, {rr.cores} ranks (fork+shm mini-MPI; fastest of "
                                       f"s/iter by ranks {rr.tried}), gcc -O3 {rr.march}"},
            "e2e": {"value": val, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def bind_near_gpu(index):
    """Pin this process to the cores of the GPU's NUMA node (what `numactl --cpunodebind` would do), so that the
    pinned host buffers of the e2e leg are allocated next to the GPU's PCIe root.  Returns the previous affinity."""
    prev = os.sched_getaffinity(0)
    try:
        bdf = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bdf.count(":") == 2 and len(bdf.split(":")[0]) == 8:
            bdf = bdf[4:]                                     # sysfs uses a 4-digit PCI domain
        with open(f"/sys/bus/pci/devices/{bdf}/local_cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        near = prev & cpus
        if near:
            os.sched_setaffinity(0, near)
    except Exception:
        pass
    return prev


# ---------------------------------------------------------------------------------------------------------
def run_b200(args, w):
    import torch
    import torch.distributed as dist
    import mpi_bicgstab_b200 as B

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("NCCL_DEBUG"):             # keep NCCL's log (the driver reads the rank count from it), but on stderr:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # stdout carries exactly ONE JSON line
    full_affinity = bind_near_gpu(local)
    torch.cuda.set_device(local)
    B.set_options(device=local, quiet=1)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        # the library's own bootstrap transport, as the reference's main.c gets it from MPI_Init of include/compat/mpi.h:
        # POSIX shared memory (csrc/shm_boot.cpp; reads torchrun's RANK / WORLD_SIZE / MASTER_PORT).  BENCH_BOOT=torch routes
        # the bootstrap bytes through torch.distributed instead.  torch itself is only used for this script's barriers.
        if os.environ.get("BENCH_BOOT", "shm") == "torch":
            B.comm_init_torch()
        elif B.lib.bicg_shm_bootstrap() != 0:
            raise RuntimeError("bicg_shm_bootstrap failed")
    method = w["method"]
    n_glob_g = w["g"] * world if w["kind"] == "random" else w["g"]

    blk = B.gen_block(w["kind"], n_glob_g, w["p0"], rank=rank, world=world)
    n_loc, n = blk.n_loc, blk.n
    B.set_options(tol=w["tol"], max_iter=w["max_iter"])
    t_first = time.perf_counter()
    dm = B.DeviceMatrix(blk)                                   # upload + plan (collective); first call: SpMV autotune too
    B.lib.bicg_synchronize()
    first_call_ms = 1e3 * (time.perf_counter() - t_first)
    stream = torch.cuda.ExternalStream(B.lib.bicg_stream(), device=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    import ctypes as C
    st = B.bicg_stats()
    with torch.cuda.stream(stream):
        ones = np.ones(n_loc)
        b_host = dm.spmv(ones)                                  # b = A*1 (main.c:109-113), collective
        b_dev = torch.from_numpy(b_host).cuda()
        x_dev = torch.zeros(n_loc, dtype=torch.float64, device="cuda")
        r_dev = torch.empty_like(b_dev)

        def resident_step():
            x_dev.zero_(); r_dev.copy_(b_dev)
            it = B.lib.bicg_solve(dm.h, B.METHODS[method], C.c_void_p(x_dev.data_ptr()), C.c_void_p(r_dev.data_ptr()),
                                  0, 0, 1, C.byref(st))
            return it, st.kernel_launches, st.loop_ms

        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()                 # nvidia-smi needs a moment to start: begin before the warm-up solves ...
            t_wait = time.perf_counter()    # ... and do not enter the (sub-second) timed region before it delivers samples
            while not sampler.lines and time.perf_counter() - t_wait < 8.0:
                time.sleep(0.05)
        for _ in range(args.warmup):
            resident_step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        iters, launches, loop_ms = 0, 0, 0.0
        for _ in range(args.steps):
            it, nl, lm = resident_step()
            iters += it; launches += nl; loop_ms += lm
        e1.record(stream)
        barrier()
        clocks = sampler.stop() if rank == 0 else None
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        final_res, converged = st.final_res, st.converged
        hist = B.last_history().copy()          # full-precision residual history of the last resident solve (parity object)
        last_iters = int(st.iters)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"x": x_dev.cpu().numpy(), "r": r_dev.cpu().numpy(), "history": hist,
                                             "iterations": np.array([last_iters])}, rank, world, int(blk.displs[rank]))

        # roofline of the dominant kernel, measured live (per rank; rank 0 reported)
        peak, peak_src = measured_peak()
        k_ms, k_bytes = dm.spmv_time(50)
        prof_ms, prof_cnt = dm.profile(method, 50)
        B.set_options(tol=w["tol"], max_iter=w["max_iter"])

    # ---- e2e: reference-facing call on pinned host buffers, upload cache off --------------------------
    B.set_options(cache=0)
    pblk = pinned_block(B, blk, rank, world)
    xh, rh = pinned_array(B, n_loc, np.float64), pinned_array(B, n_loc, np.float64)
    h2d = d2h = 0
    e2e_iters, t_e2e = 0, 0.0
    for s in range(max(1, args.warmup // 2) + args.steps):
        if os.environ.get("BENCH_E2E_VERBOSE"):
            B.set_options(verbose=2 if s == 1 else 0)
        xh[:] = 0.0; rh[:] = b_host
        barrier()
        t0 = time.perf_counter()
        it = B.solve(method, pblk, xh, rh)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if s >= max(1, args.warmup // 2):
            e2e_iters += it; t_e2e += dt
            s_ = B.last_stats(); h2d, d2h = s_["h2d_bytes"], s_["d2h_bytes"]
    if world > 1:
        t = torch.tensor([t_e2e], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_e2e = float(t.item())
    # the same call on plain malloc'ed (pageable) buffers -- what the reference's main.c hands over (main.c:81-107)
    xp, rp = np.zeros(n_loc), np.zeros(n_loc)
    pg_iters, t_pg, pg_steps = 0, 0.0, max(1, min(args.steps, 3))
    for s in range(1 + pg_steps):
        xp[:] = 0.0; rp[:] = b_host
        barrier()
        t0 = time.perf_counter()
        it = B.solve(method, blk, xp, rp)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if s >= 1:
            pg_iters += it; t_pg += dt
    if world > 1:
        t = torch.tensor([t_pg], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_pg = float(t.item())
    B.set_options(cache=1)
    dm.destroy()
    if world > 1:                      # collective teardown first: rank 0 then spends up to a minute in the CPU legs alone
        if os.environ.get("BENCH_BOOT", "shm") == "torch":
            B.comm_finalize()
        else:
            B.lib.bicg_shm_shutdown()
        dist.destroy_process_group()

    if rank == 0:
        nnz_glob = int(blk.info.nz) if w["kind"] != "random" else n * int(w["p0"])
        bytes_iter = 24 * nnz_glob + BYTES_PER_ITER_N[method] * n
        persistent = launches <= 8 * args.steps                   # the loop ran as ONE persistent kernel per solve
        spmv_obj = {"kernel": "spmv_ws_kernel + fused (r#,s) dot" if st.spmv_kind == 0 else "spmv_rowsplit_kernel + dot",
                    "achieved": k_bytes / (k_ms * 1e-3) / 1e9, "frac": k_bytes / (k_ms * 1e-3) / 1e9 / peak, "unit": "GB/s",
                    "algorithmic_bytes_per_launch": k_bytes, "avg_launch_us": k_ms * 1e3,
                    "traffic": read_traffic("dram_bytes_per_launch") if (world == 1 and args.workload == "transport") else None,
                    "in_per_phase_kernels": {"spmv_avg_us": 1e3 * prof_ms[0] / max(prof_cnt[0], 1),
                                             "vector_avg_us": 1e3 * prof_ms[1] / max(prof_cnt[1], 1),
                                             "spmv_share_of_step": prof_ms[0] / max(sum(prof_ms), 1e-12)}}
        if persistent:
            # dominant kernel of the timed region = bicg_mega_kernel (one launch per solve): its algorithmic bytes are the
            # iterations it ran x the per-iteration bytes of SURVEY.md 8(d), per rank; its duration is the library's
            # CUDA-event time of the reference's timed region (init SpMV + the persistent kernel)
            per_rank = bytes_iter / world
            ach = per_rank * iters / (loop_ms * 1e-3) / 1e9
            tpi = read_traffic("mega_dram_bytes_per_iteration")
            roofline = {"bound": "hbm", "kernel": f"bicg_mega_kernel (persistent solver loop of {method}: 2 SpMV phases + the fused "
                                                  "vector phases + 3 reductions and 2 neighbour waits per iteration; one launch per solve)",
                        "achieved": ach, "peak": peak, "unit": "GB/s",
                        "frac": ach / peak, "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": per_rank * iters / args.steps,
                        "avg_launch_us": 1e3 * loop_ms / args.steps,
                        "traffic": (tpi * iters / args.steps) if (tpi and world == 1 and args.workload == "transport"
                                                                   and method == "bicgstab") else None,
                        "traffic_note": "ncu dram bytes per iteration of the same kernel on the same matrix x iterations per launch",
                        "spmv_kernel": spmv_obj}
        else:
            roofline = dict(spmv_obj, bound="hbm", peak=peak, peak_source=peak_src)
        line = {
            "metric": "BiCGStab iterations/sec", "value": iters / (ms * 1e-3), "unit": "iterations/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak" if w["kind"] == "random" else "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": w["label"], "method": method, "iterations_per_step": iters / args.steps,
                       "converged": bool(converged), "final_relative_residual": final_res,
                       "l2": "inputs larger than L2 (matrix stream %.0f MB per SpMV > 126 MB L2)" % (12e-6 * blk.nnz_loc),
                       "spmv_plan": {"kind": ["tma", "rowsplit"][st.spmv_kind], "lanes": st.spmv_lanes},
                       "spmv_effective_GBps_all_gpus": world * (12.0 * blk.nnz_loc + 20.0 * n_loc + 4) / (k_ms * 1e-3) / 1e9,
                       "algorithmic_bytes_per_iteration": bytes_iter,
                       "solver_effective_GBps": bytes_iter * iters / (ms * 1e-3) / 1e9},
            "clocks": clocks,
            "e2e": {"value": e2e_iters / t_e2e, "unit": "iterations/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * t_e2e / args.steps,
                    "host_buffers": "pinned (cudaHostAlloc), upload cache off: matrix + vectors re-uploaded every step"},
            "e2e_pageable": {"value": pg_iters / t_pg, "unit": "iterations/s", "ms_per_step": 1e3 * t_pg / pg_steps,
                             "steps": pg_steps, "host_buffers": "plain malloc (what main.c:81-107 passes), upload cache off"},
            "first_call_ms": first_call_ms,
            "gpu_launches": int(launches),
            "roofline": roofline,
        }
        if world == 1 and args.workload == "transport":
            line["roofline"]["traffic_source"] = ("profiles/spmv_traffic.json (ncu --set full dram__bytes_read + dram__bytes_write of the same kernel on the "
                                                  "same matrix, profiles/r02c_mega_kernel_ncu_full.json), not measured in this run")
        else:
            line["roofline"]["traffic_source"] = "no ncu capture for this workload / rank count: traffic null"
        rr = None
        if not args.no_cpu:
            try:
                os.sched_setaffinity(0, full_affinity)      # the CPU reference may use every core of the box
                rr = RefRunner(w)
                if not rr.ok:
                    rr = None
            except Exception as exc:
                line["parity"] = {"error": f"reference runner unavailable: {exc!r}"}
                rr = None
        if rr is not None:
            try:
                line["parity"] = parity_object(rr, w, world, hist, last_iters)
            except Exception as exc:
                line["parity"] = {"error": repr(exc)}
        if world == 1 and rr is not None:
            try:
                r = reference_sample(rr, REF_ITERS)
                if r:
                    line["cpu_baseline"] = {"value": 1.0 / r["avg_time_per_iter_s"], "unit": "iterations/s",
                                            "cores": r["cores"], "kind": "reference",
                                            "sample": f"first {REF_ITERS} iterations of the same solve, reference sources compiled in place "
                                                      f"(gcc -O3 {r['march']}), {r['cores']} ranks over a fork+shm mini-MPI"}
            except Exception as exc:        # the GPU numbers must not be lost to a CPU-side hiccup
                line["cpu_baseline"] = {"value": None, "unit": "iterations/s", "cores": 0, "kind": "reference",
                                        "sample": f"failed: {exc!r}"}
        if rr is not None:
            rr.close()
        print(json.dumps(line))


def dump_outputs(d, outputs, rank, world, row0):
    """One float64 .npy per output of the rank's last timed solve; x and r shrink to the same seeded rows on every run
    when all ranks' x and r together exceed DUMP_BYTES."""
    os.makedirs(d, exist_ok=True)
    n = outputs["x"].size
    if world * 2 * 8 * n > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(rank).choice(n, size=DUMP_BYTES // (world * 3 * 8), replace=False))
        outputs = dict(outputs, x=outputs["x"][idx], r=outputs["r"][idx], index=row0 + idx)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in outputs.items():
        np.save(os.path.join(d, f"{name}{suffix}.npy"), np.asarray(a, dtype=np.float64))


def read_traffic(key):
    """dram bytes measured by ncu (committed under profiles/spmv_traffic.json), else None."""
    try:
        with open(os.path.join(ROOT, "profiles", "spmv_traffic.json")) as f:
            return json.load(f).get(key)
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="transport", choices=sorted(WORKLOADS))
    ap.add_argument("--method", default=None)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed solve's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    w = dict(WORKLOADS[args.workload])
    if args.method:
        w["method"] = args.method
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_b200(args, w)


if __name__ == "__main__":
    main()
