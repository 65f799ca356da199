/*
 * bicgstab_b200.h -- C ABI of libbicgstab_b200.so, the B200-native drop-in for the BiCGStab hot
 * path of RtrMmmt/MPI-BiCGStab (SpMV + BLAS-1 + iteration loops + their collectives).
 *
 * Part 1 re-declares, with identical signatures and struct layouts, the eight non-libc, non-MPI
 * symbols the reference's main.c needs (reference file:line beside each one), so that main.c
 * compiles UNCHANGED against include/compat/mpi.h + the reference's own solver.h and links against
 * this library instead of solver.c / matrix.c / vector.c.
 * Part 2 is the small extension surface (prefix bicg_) that tests, bench.py and multi-process
 * launchers use: rank/communicator bootstrap, device-resident matrices, solve statistics,
 * synthetic-matrix generators.  No torch / CUDA types appear anywhere in this header.
 *
 * Every entry point drives hand-written sm_100a CUDA kernels; there is no CPU fallback -- if no
 * CUDA device is usable the compute entry points print an error and exit(1) (the reference's own
 * error convention, solver.c:43-46).
 */
#ifndef BICGSTAB_B200_H
#define BICGSTAB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------
 * Part 1 -- the reference's own interface
 * ---------------------------------------------------------------------------------------------- */
#ifndef MATRIX_H /* the reference's matrix.h (include guard MATRIX_H) already defines these types */

typedef char MM_typecode[4];                 /* mmio.h:16 */

/* matrix.h:19-26 -- sizeof 40; val@0 col@8 ptr@16 nz@24 rows@28 cols@32 */
typedef struct {
    double       *val;   /* nz values                                   */
    unsigned int *col;   /* nz column indices (diag: local, offd: global) */
    unsigned int *ptr;   /* rows+1 row starts, ptr[0] == 0              */
    unsigned int  nz, rows, cols;
} CSR_Matrix;

/* matrix.h:28-33 -- sizeof 32; nz@0 rows@4 cols@8 code@12 recvcounts@16 displs@24 */
typedef struct {
    unsigned int nz, rows, cols;  /* global sizes */
    MM_typecode  code;
    int         *recvcounts;      /* rows of rank p            (matrix.c:306) */
    int         *displs;          /* first global row of rank p (matrix.c:307) */
} INFO_Matrix;

/* matrix.h:44-45 (matrix.c:188-204) */
void csr_init_matrix(CSR_Matrix *m);
void csr_free_matrix(CSR_Matrix *m);
/* matrix.h:57 (matrix.c:536-551): A_diag += sigma I in place on the caller's host arrays; drops the cached device copy */
void csr_shift_diagonal(CSR_Matrix *A_diag, double sigma);

/* matrix.h:50 (matrix.c:402-419): Matrix-Market file -> this rank's diag / offd CSR blocks + partition */
void MPI_csr_load_matrix_block(char *filename, CSR_Matrix *matrix_loc_diag, CSR_Matrix *matrix_loc_offd,
                               INFO_Matrix *matrix_info);

/* matrix.h:51 (matrix.c:428-441): y_loc = A_diag x_loc + A_offd x, host pointers; x (length cols) is
 * caller-owned scratch that receives the gathered vector like the reference's allgather does. */
void MPI_csr_spmv_ovlap(CSR_Matrix *matrix_loc_diag, CSR_Matrix *matrix_loc_offd, INFO_Matrix *matrix_info,
                        double *x_loc, double *x, double *y_loc);

/* solver.h:10-13 (solver.c:35-146, 160-278, 292-417, 433-576).  Host pointers.  x_loc: initial guess in,
 * solution out.  r_loc: right-hand side in, final recursive residual out (b is destroyed, as in the
 * reference).  Return value: iterations performed.  Collective over all ranks of the job. */
int bicgstab(CSR_Matrix *A_loc_diag, CSR_Matrix *A_loc_offd, INFO_Matrix *A_info, double *x_loc, double *r_loc);
int ca_bicgstab(CSR_Matrix *A_loc_diag, CSR_Matrix *A_loc_offd, INFO_Matrix *A_info, double *x_loc, double *r_loc);
int pipe_bicgstab(CSR_Matrix *A_loc_diag, CSR_Matrix *A_loc_offd, INFO_Matrix *A_info, double *x_loc, double *r_loc);
int pipe_bicgstab_rr(CSR_Matrix *A_loc_diag, CSR_Matrix *A_loc_offd, INFO_Matrix *A_info, double *x_loc,
                     double *r_loc, int krr, int nrr);

#endif /* MATRIX_H */

/* shifted_switching_solver.h:12 (shifted_switching_solver.c:260-602): seed-switching shifted BiCGStab for (A + sigma_j I) x_j = b.
 * x_loc_set: sigma_len blocks of n_loc doubles (initial guesses in, solutions out); r_loc: b in, seed residual out; returns the
 * reference's k (iterations performed + 1).  EPS / MAX_ITER of the reference (1e-12 / 1000, :5-6) = BICG_SHIFT_TOL /
 * BICG_SHIFT_MAX_ITER.  Not needed by main.c; it is what main_shifted.c / main_repeat.c call (SURVEY.md 8(f) N4). */
int shifted_lopbicg_switching(CSR_Matrix *A_loc_diag, CSR_Matrix *A_loc_offd, INFO_Matrix *A_info, double *x_loc_set,
                              double *r_loc, double *sigma, int sigma_len, int seed);
/* shifted_switching_solver.h:13 (shifted_switching_solver.c:611): the same solve without communication overlap in the reference --
 * identical arithmetic, so the same function here. */
int shifted_lopbicg_switching_noovlp(CSR_Matrix *A_loc_diag, CSR_Matrix *A_loc_offd, INFO_Matrix *A_info, double *x_loc_set,
                                     double *r_loc, double *sigma, int sigma_len, int seed);

/* vector.h:4-7 (vector.c:3-27) on HOST arrays: the shifted drivers build and copy their right-hand sides with these
 * (main_shifted.c:114-135, main_repeat.c:121, main_seed_diff.c:118-121), so they are exported for those programs to link
 * unchanged (csrc/hostvec.cpp).  The solvers do not use them: their vector work is fused into the device kernels. */
void    my_daxpy(int n, double alpha, const double *x, double *y);
double  my_ddot(int n, const double *x, const double *y);
void    my_dscal(int n, double alpha, double *x);
void    my_dcopy(int n, const double *x, double *y);

/* ------------------------------------------------------------------------------------------------
 * Part 2 -- extensions
 * ---------------------------------------------------------------------------------------------- */

#define BICG_ABI_VERSION 1
int bicg_abi_version(void);

/* Runtime options.  The reference fixes these with #defines (solver.c:3-9) and its signatures carry no
 * options, so they come from the environment (read once, on first use) or from bicg_set_option():
 *   BICG_TOL       (1e-15, solver.c:3)   BICG_MAX_ITER (1000, solver.c:4)   BICG_OUT_ITER (100, solver.c:9)
 *   BICG_QUIET=1   suppress the solver.c:124,135-139 stdout lines
 *   BICG_SPMV      auto | tma | rowsplit        BICG_SPMV_LANES  lanes per row (1,2,4,...,32; 0 = choose)
 *   BICG_GRAPH     1 (CUDA-graph replay of iteration batches) | 0 (plain stream launches)
 *   BICG_UNROLL    iterations per graph (default 10)
 *   BICG_CACHE     1 keep uploaded matrices keyed by host pointer (default) | 0 re-upload on every call
 *   BICG_DEVICE    CUDA device ordinal (default: LOCAL_RANK if set, else 0)
 *   BICG_MEGA      1 persistent solver kernel where it wins (thread-per-row plans; default) | 2 always | 0 kernel-per-phase graph
 *   BICG_RESIDENT  1 persistent kernel keeps a CTA's matrix slice in shared memory for the whole solve when it fits (default) | 0
 *   BICG_PARTITION rows (matrix.c:295-308, default) | nnz (archive/matrix.c:407-420) in the loader and the generators
 *   BICG_PEER_TIMEOUT_S  bound of every device-side wait for another CTA / GPU (default 20)
 *   tuning / experiments: BICG_MEGA_THREADS, BICG_MEGA_LANES, BICG_ROW_WEIGHT, BICG_BOUNDARY_WEIGHT, BICG_L2_HINT,
 *   BICG_GATHER_CG, BICG_STAGE_UPLOAD, BICG_AUTOTUNE, BICG_SPMV_THREADS / _STAGES / _CTAS, BICG_HALO_GAP, BICG_VERBOSE,
 *   BICG_MEGA_TRACE (per-phase device timestamps of the persistent kernel on stderr)
 * Returns 0 on success, -1 for an unknown key. */
int bicg_set_option(const char *key, const char *value);

/* Multi-process bootstrap (one process = one rank = one GPU, like one MPI rank in the reference).
 * `allgather` must copy `bytes` bytes from every rank's `send` into `recv` (rank-major) and return 0;
 * the launcher supplies it (bench.py: torch.distributed; include/compat/mpi.h shim: POSIX shm).
 * Without this call the process is a single rank (world = 1). */
typedef int (*bicg_allgather_fn)(void *ctx, const void *send, void *recv, size_t bytes);
int  bicg_comm_init(int rank, int world, bicg_allgather_fn allgather, void *ctx);
void bicg_comm_finalize(void);
int  bicg_comm_rank(void);
int  bicg_comm_world(void);

/* Device-resident matrix (upload + SpMV tiling plan + halo plan); the host-pointer entry points of
 * Part 1 create and cache one of these internally. */
typedef struct bicg_matrix bicg_matrix;
bicg_matrix *bicg_matrix_create(const CSR_Matrix *diag, const CSR_Matrix *offd, const INFO_Matrix *info);
void         bicg_matrix_destroy(bicg_matrix *m);
/* drop the cached upload of a host matrix whose values were changed in place (csr_shift_diagonal,
 * matrix.c:536-551, does that) */
void         bicg_matrix_invalidate(const CSR_Matrix *diag);

enum { BICG_METHOD_BICGSTAB = 0, BICG_METHOD_CA = 1, BICG_METHOD_PIPE = 2, BICG_METHOD_PIPE_RR = 3 };

typedef struct {
    int    iters;          /* iterations performed (the reference's return value)        */
    int    converged;      /* 1 if dot_r <= tol^2 dot_zero stopped the loop               */
    double final_res;      /* sqrt(dot_r / dot_zero)  (solver.c:136)                      */
    double loop_ms;        /* CUDA-event time of the reference's timed region a14 (solver.c:69-71,129-132):
                              initial A x0 ... end of loop, device resident                */
    double h2d_ms, d2h_ms; /* host<->device copies of x, b / x, r done by this call        */
    double upload_ms;      /* matrix upload + planning done by this call (0 when cached)   */
    uint64_t h2d_bytes, d2h_bytes;
    int    kernel_launches;/* kernels launched inside the timed region                      */
    int    spmv_lanes;     /* lanes per row the SpMV plan chose                             */
    int    spmv_kind;      /* 0 = tma tile kernel, 1 = rowsplit kernel                      */
} bicg_stats;

/* Solve on a device-resident matrix.  x and r are HOST pointers unless `device_vectors` != 0, in which
 * case they are device pointers (same in/out meaning as Part 1).  krr/nrr only for BICG_METHOD_PIPE_RR. */
int bicg_solve(bicg_matrix *m, int method, double *x, double *r, int krr, int nrr, int device_vectors,
               bicg_stats *stats);

/* shifted_lopbicg_switching on a resident matrix; bicg_last_shift_info: the seed the last shifted solve ended with and the
 * iteration at which every shift stopped (returns sigma_len). */
int bicg_shifted_solve(bicg_matrix *m, double *x_set, double *r, const double *sigma, int sigma_len, int seed, bicg_stats *stats);
int bicg_last_shift_info(int *seed, int *stop_iter, int cap);

/* y_loc = A x_loc on a resident matrix (host pointers) -- the kernel behind MPI_csr_spmv_ovlap. */
int bicg_spmv(bicg_matrix *m, const double *x_loc, double *y_loc);

/* Time `reps` launches of the fused SpMV + (r_hat, s) dot kernel (the dominant kernel of every
 * variant) with CUDA events on the library's stream; returns average ms per launch in *ms and the
 * algorithmic bytes of one launch (12 nnz + 28 n_loc, SURVEY.md 8(d) phase P1) in *bytes. */
int bicg_spmv_time(bicg_matrix *m, int reps, double *ms, double *bytes);

/* per-kernel-class device time of one solve run WITHOUT graphs, each launch bracketed by events.
 * classes: 0 = SpMV(+dots), 1 = fused vector updates, 2 = other.  ms are totals over the solve. */
int bicg_profile_solve(bicg_matrix *m, int method, int iters, double class_ms[3], int class_launches[3]);

/* Test hooks for kernel-level parity (tests/test_gpu_kernels.py); single rank.  `vecs` holds the 11 arena vectors
 * x r r# p s y|z w v t b ax (n_loc doubles each), in and out.
 *   bicg_debug_vec_phase: ONE fused vector phase (enum Phase of csrc/vec.cuh) with coef = {alpha, beta, omega}; returns the
 *                         number of dot products the phase reduces, their values in dots[].
 *   bicg_debug_spmv_epi : s = A p with the solver's epilogue dots (1: (r#,s); 2: (r,s),(s,s); 3: w = A p with
 *                         (r#,r),(r#,w),(r#,ax),(r#,z)).
 *   bicg_debug_get_vec / _get_scalars: arena vector `id` / {rTr rTr_old rTs rTy yTy rTw wTw rTz dot_r dot_zero alpha
 *                         beta omega} as the last solve on this handle left them.
 *   bicg_debug_resident_ctas: how many CTAs of the last persistent-kernel launch on this handle kept their matrix slice in
 *                         shared memory for the whole solve (BICG_RESIDENT, csrc/mega.cu).
 *   bicg_debug_mega_tiles: the number of tiles of the persistent-kernel plan (0: no usable plan); *narrow = how many of them
 *                         stream their columns as 16-bit tile-relative codes instead of 32-bit indices (csrc/mega.cu). */
int bicg_debug_vec_phase(bicg_matrix *m, int phase, const double coef[3], double *vecs, double dots[8]);
int bicg_debug_spmv_epi(bicg_matrix *m, int epi, double *vecs, double dots[8]);
int bicg_debug_get_vec(bicg_matrix *m, int id, double *out);
int bicg_debug_get_scalars(bicg_matrix *m, double out[13]);
int bicg_debug_resident_ctas(bicg_matrix *m);
int bicg_debug_mega_tiles(bicg_matrix *m, int *narrow);

/* full-precision history of the last solve on this rank: out[k] = dot_r/dot_zero after iteration k
 * (out[0] = 1).  Returns the number of entries available (iters + 1). */
int bicg_last_history(double *out, int cap);
const bicg_stats *bicg_last_stats(void);

/* the library's compute stream (a cudaStream_t) so callers can record their own events on it */
void *bicg_stream(void);
int   bicg_device(void);
void  bicg_synchronize(void);
/* pinned host allocations for callers that want full-rate host<->device copies */
void *bicg_host_alloc(size_t bytes);
void  bicg_host_free(void *p);

/* Host-side planning, exposed for CPU-only tests (no CUDA call inside). */
void bicg_plan_partition(int n, int world, int *counts, int *displs);          /* matrix.c:295-308 */
/* nnz-balanced contiguous partition (archive/matrix.c:407-420, DYNAMIC_ROWS): used by the loader and the generators when
 * BICG_PARTITION=nnz; row_nnz[i] = entries of global row i. */
void bicg_plan_partition_nnz(const unsigned int *row_nnz, int n, int world, int *counts, int *displs);
/* SpMV tile plan for a CSR block: tiles of <= rows_per_tile rows and <= cap_nnz entries.
 * Writes tile_row[0..ntiles] (first row of each tile); returns ntiles, or -1 if tile_row_cap is too small,
 * or -2 if a single row exceeds cap_nnz. */
int  bicg_plan_tiles(const unsigned int *ptr, int rows, int rows_per_tile, int cap_nnz, int *tile_row,
                     int tile_row_cap);
/* Tile plan of the persistent solver kernel: CTA g of `ctas` owns a contiguous row range starting at a multiple of 16
 * rows; ranges are balanced by per-row work 24*nnz(row) + 216 + extra_weight*row_extra[row] (row_extra may be NULL) and
 * cut into tiles of <= rows_per_tile rows of equal height.  tile_row[0..ntiles] (first row of each tile, then `rows`),
 * cta_tile[0..ctas] (first tile of each CTA).  Returns ntiles (or -needed ints), *max_tile_nnz = entries of the fullest tile. */
int  bicg_plan_cta_tiles(const unsigned int *ptr, int rows, int ctas, int rows_per_tile, const unsigned char *row_extra,
                         int extra_weight, int *tile_row, int tile_row_cap, int *cta_tile, unsigned int *max_tile_nnz);
/* The same with a stage capacity: tiles hold <= cap_limit entries; a row longer than cap_limit becomes a run of chunk tiles
 * (tile_flag 1 = more chunks of the row follow, 2 = last chunk, 0 = ordinary tile of whole rows); tile_nz[t] = first entry of
 * tile t.  The three tile arrays need tile_cap ints each. */
int  bicg_plan_cta_tiles_capped(const unsigned int *ptr, int rows, int ctas, int rows_per_tile, int cap_limit, int *tile_row,
                                unsigned int *tile_nz, int *tile_flag, int tile_cap, int *cta_tile, unsigned int *max_tile_nnz);
/* Halo plan of rank `self`: which global columns of the offd block it must receive, as merged runs.
 * runs_out holds triples (first_col, length, owner); returns the number of runs (or -needed if cap is small).
 * gap: runs of one owner separated by <= gap unreferenced columns are merged. */
int  bicg_plan_halo_runs(const CSR_Matrix *offd, const INFO_Matrix *info, int self, int world, int gap,
                         int *runs_out, int runs_cap);

/* The device layout of rank `self`: its diag / offd blocks merged into one CSR over [own columns | ghost slots]
 * (ghost slot g = column ghost_off + g; per row diag entries first, then offd, matrix.c:437-440).  Outputs are
 * caller-allocated: ptr_out[rows+1], col_out/val_out[diag.nz + offd.nz], recv_out quadruples (first_col, len,
 * owner, ghost_idx).  Returns the number of quadruples (or -needed ints if recv_cap is too small). */
long long bicg_plan_merge(const CSR_Matrix *diag, const CSR_Matrix *offd, const INFO_Matrix *info, int self, int world,
                          int gap, int ghost_off, unsigned int *ptr_out, unsigned int *col_out, double *val_out,
                          int *recv_out, int recv_cap, int *n_ghost_out);
/* round trip of a few bytes through the registered allgather callback; 0 = every rank's contribution arrived */
int  bicg_comm_selftest(void);

/* What rank `self` pushes to rank `dest`, derived from every rank's receive list (quadruples first_col, len,
 * owner, ghost_idx; `stride` ints reserved per rank, cnts[p] quadruples valid).  Writes triples
 * (local_src_row, len, ghost_offset_on_dest); returns their number (or -needed). */
int  bicg_plan_push_runs(const int *all_recv, const int *cnts, int stride, int self, int dest, int my_first,
                         int *out, int out_cap);

/* Synthetic inputs of SURVEY.md 8(d) / BASELINE.json configs, generated directly as one rank's blocks
 * (malloc'ed like the reference loader's, so csr_free_matrix() releases them).  info->recvcounts/displs
 * must be caller-allocated with `world` entries (main.c:82-83).
 *   kind 0: 15-point 3-D stencil on a g^3 grid ("Transport-like" T'); p0 = diagonal value
 *   kind 1: 5-point 2-D Laplacian on a g x g grid (diag 4, off -1)
 *   kind 2: random, n = g rows, k = (int)p0 entries per row incl. the diagonal (diag = k+1, off in -(0,1])
 *   kind 3: 2-D convection-diffusion g x g, upwind, p0 = Peclet-like convection strength (nonsymmetric)
 */
int bicg_gen_block(int kind, long long g, double p0, uint64_t seed, int rank, int world,
                   CSR_Matrix *diag, CSR_Matrix *offd, INFO_Matrix *info);

#ifdef __cplusplus
}
#endif
#endif /* BICGSTAB_B200_H */
