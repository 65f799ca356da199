// engine.hpp -- host-side runtime of libbicgstab_b200: process context, device-resident matrix, solver driver.
#pragma once
#include "bicgstab_b200.h"
#include "dev.cuh"
#include "plan.hpp"
#include "spmv.cuh"
#include "vec.cuh"
#include "mega.cuh"

#include <cstdio>
#include <cstdlib>
#include <initializer_list>
#include <map>
#include <string>
#include <vector>

namespace bicg {

[[noreturn]] void fatal(const char *fmt, ...);
#define BICG_CUDA(call)                                                                              \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess)                                                                       \
            ::bicg::fatal("bicgstab_b200: CUDA error %s at %s:%d: %s", cudaGetErrorName(e_), __FILE__, \
                          __LINE__, cudaGetErrorString(e_));                                          \
    } while (0)

struct Config {
    double tol = 1.0e-15;        // solver.c:3
    int max_iter = 1000;         // solver.c:4
    int out_iter = 100;          // solver.c:9
    int quiet = 0;
    int spmv_kind = -1;          // -1 auto, 0 tma, 1 rowsplit
    int spmv_lanes = 0;          // 0 choose
    int spmv_threads = 0;
    int spmv_stages = 0;
    int spmv_ctas = 0;           // CTAs per SM (0 choose)
    int autotune = 1;
    int graph = 1;
    int unroll = 10;
    int cache = 1;
    int mega = 1;                // 1: persistent cooperative kernel for the iteration loop where applicable
    int mega_threads = 0;        // 0 choose (512, else 256)
    int mega_trace = 0;
    int mega_lanes = 0;          // lanes per row of the persistent kernel's SpMV (0 choose from the mean row length)
    int stage_upload = 1;        // large pageable host arrays are uploaded through multi-threaded pinned staging (Context::h2d)
    int resident = 1;            // persistent kernel: keep a CTA's matrix slice in shared memory for the whole solve when it fits
    int gather_cg = -1;          // SpMV gathers of the persistent kernel through L2 only + fence-free neighbour waits (-1: default = off)
    int l2_hint = 1;             // matrix stream loaded with an L2 evict-first policy (persistent kernel)
    int row_weight = 1200;       // per-row cost (byte equivalents) next to 24 B per entry when CTA row ranges are balanced
    int boundary_weight = 300;   // extra work (bytes) charged per pushed row when CTA row ranges are balanced
    int device = -1;
    int halo_gap = 64;
    int verbose = 0;
    double shift_tol = 1.0e-12;  // EPS of the shifted solvers (shifted_switching_solver.c:5)
    int shift_max_iter = 1000;   // their MAX_ITER (:6)
    int peer_timeout_s = 20;     // bound of device-side waits for peers / other CTAs (then: error + exit(1))
    int fence_writers = 0;       // 1: every thread that stored to a peer also fences at system scope itself (debug aid;
                                 // the CTA barrier + one system fence per CTA is sufficient and much cheaper)
};

struct TuneKey {
    int n_loc; size_t nnz; unsigned max_row; int kind;
    bool operator<(const TuneKey &o) const
    {
        if (n_loc != o.n_loc) return n_loc < o.n_loc;
        if (nnz != o.nnz) return nnz < o.nnz;
        if (max_row != o.max_row) return max_row < o.max_row;
        return kind < o.kind;
    }
};
struct TuneVal { int kind, lanes, threads, stages, ctas; };

struct Context {
    bool ready = false;
    Config cfg;
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    // job
    int rank = 0, world = 1;
    bicg_allgather_fn allgather = nullptr;
    void *allgather_ctx = nullptr;
    // results of the last solve
    std::vector<double> last_hist;
    bicg_stats last_stats{};
    std::vector<int> last_shift_stop;     // shifted solver: iteration at which every shift stopped
    int last_shift_seed = 0;              // ... and the seed it ended with
    // host-pointer keyed cache of uploaded matrices
    std::map<const void *, bicg_matrix *> cache;
    std::map<TuneKey, TuneVal> tuned;     // SpMV autotune winners by matrix shape
    // pinned scratch
    int *h_flags = nullptr;      // ring of {k, max_iter, done, converged}
    // profiling of individual launches
    bool prof_on = false;
    std::vector<cudaEvent_t> prof_ev;
    std::vector<int> prof_class;
    int launches = 0;

    void ensure();               // lazy device init; fails loudly if there is no usable GPU
    // device-memory cache: cudaMalloc / cudaFree are synchronising driver calls that cost milliseconds for the
    // 100 MB-class buffers of a matrix; blocks are kept by exact size and reused by the next upload
    void *dev_alloc(size_t bytes);
    void  dev_free(void *p);
    void  dev_release_all();
    void  dev_free_after(std::initializer_list<void *> ptrs, cudaEvent_t ev);   // dev_free once `ev` has completed
    void  dev_sweep(bool wait);
    struct Deferred { cudaEvent_t ev; std::vector<void *> ptrs; };
    std::vector<Deferred> deferred;
    std::multimap<size_t, void *> pool;
    std::map<void *, size_t> live;
    size_t pool_bytes = 0;
    // IPC-exported arenas (world > 1) are never freed between matrices: an un-cached call (BICG_CACHE=0) re-uses a parked
    // arena of the same size, and the peers keep their mappings, so no cudaMalloc / cudaIpcOpenMemHandle /
    // cudaIpcCloseMemHandle sits in the reference-facing call after the first one
    struct ArenaRec { char *ptr; size_t bytes; unsigned long long id; cudaIpcMemHandle_t handle; };
    std::multimap<size_t, ArenaRec> arena_pool;
    std::map<std::pair<int, unsigned long long>, void *> peer_maps;    // (rank, that rank's arena id) -> mapped base
    unsigned long long next_arena_id = 1;
    void release_arenas();       // collective: unmap the peers' arenas, free the parked ones
    void host_allgather(const void *send, void *recv, size_t bytes);
    // Host -> device copy ordered on `stream`.  Pinned sources go straight to cudaMemcpyAsync.  Large PAGEABLE sources (what the
    // reference's main.c passes: plain malloc, main.c:81-107) are staged by a few host threads through pinned bounce buffers, each
    // thread copying and issuing its own chunks -- the driver's own pageable path stages with one thread (~11 GB/s).
    void h2d(void *dst, const void *src, size_t bytes);
    struct Stager { cudaStream_t st = nullptr; cudaEvent_t ev[2] = {nullptr, nullptr}; cudaEvent_t done = nullptr; char *buf[2] = {nullptr, nullptr}; };
    std::vector<Stager> stagers;
    int stage_threads = 4;
};
Context &ctx();
void load_config_from_env(Config &c);
int  set_option(Config &c, const char *key, const char *value);


struct SpmvPlan {
    int kind = 0, lanes = 1, threads = 256, stages = 3, cap = 0, grid = 0, ctas_per_sm = 1;
    size_t smem = 0;
    int ntiles = 0;
    int *d_tile_row = nullptr;
    unsigned *d_tile_nz = nullptr;
    double ms = 0.0;             // measured time of one launch (autotune) or 0
};

struct MegaPlan {
    bool ok = false;
    int threads = 512, lanes = 1, stages = 2, cap = 0, grid = 0;
    size_t smem = 0;
    size_t res_smem = 0;         // > 0: every CTA's slice fits into shared memory (mega_resident_bytes of the largest one)
    int ntiles = 0;
    int *d_tile_row = nullptr;
    unsigned *d_tile_nz = nullptr;
    int *d_cta_tile = nullptr;
    int4 *d_cta_dep = nullptr;
    int *d_tile_flag = nullptr;  // only when rows longer than a stage were cut into chunk tiles
    int narrow = 0;              // tiles whose columns are streamed as 16-bit codes (mega.cu: StageHdr::cbase)
    int *d_tile_cbase = nullptr; // only when narrow > 0: per tile the column base, -1 for a wide tile
    unsigned short *d_col16 = nullptr;   // only when narrow > 0: nnz + 16 codes, those of the narrow tiles filled in
    bool chunked = false;
    std::vector<int> cta_row;    // grid + 1: first row of every CTA
};

} // namespace bicg

// the opaque handle of the C ABI
struct bicg_matrix {
    int rank = 0, world = 1;
    int n_loc = 0, n_glob = 0;
    size_t nnz = 0;              // entries of this rank's rows (diag + offd)
    unsigned max_row = 0;
    double mean_row = 0.0;
    // device CSR over the extended local column space
    double *d_val = nullptr;
    unsigned *d_col = nullptr;
    unsigned *d_ptr = nullptr;
    bicg::SpmvPlan plan;
    bicg::MegaPlan mega;             // persistent-kernel plan (mega.cu)
    bicg::MegaSync *d_msync = nullptr;
    bicg::MegaSync *peer_msync[bicg::MAX_RANKS] = {};
    unsigned long long *d_ll = nullptr;                      // LL halo regions [3][ll_stride][2 words] (world > 1)
    long long ll_stride = 0;
    unsigned long long *peer_ll[bicg::MAX_RANKS] = {};
    long long peer_ll_stride[bicg::MAX_RANKS] = {};
    unsigned long long *d_trace = nullptr;   // BICG_MEGA_TRACE
    // ghost layout
    int ghost_off = 0;           // first ghost column index = roundup(n_loc, 16)
    int n_ghost = 0;
    long long vstride = 0;       // doubles between consecutive arena vectors
    std::vector<int> recv_runs;  // quadruples (first_col, len, owner, ghost_idx)
    // arena (one cudaMalloc, IPC-shared with the peers)
    char *arena = nullptr;
    size_t arena_bytes = 0;
    unsigned long long arena_id = 0;         // world > 1: identity of the exported allocation
    cudaIpcMemHandle_t arena_handle{};
    double *vec_base = nullptr;
    bicg::Scalars *d_sc = nullptr;
    double *d_partials = nullptr;
    double *d_hist = nullptr;
    double *hist_extra = nullptr;   // replaces the arena slot when BICG_MAX_ITER grows
    int hist_cap = 0;
    bicg::Mailbox *d_mail = nullptr;
    bicg::HaloFlag *d_hflag = nullptr;
    bicg::CommDev comm{};
    // peers
    void *peer_base[bicg::MAX_RANKS] = {};
    long long peer_vec_off[bicg::MAX_RANKS] = {}, peer_vstride[bicg::MAX_RANKS] = {}, peer_ghost_off[bicg::MAX_RANKS] = {};
    int npush = 0;                                   // peers this rank sends to
    int push_peer[bicg::MAX_RANKS - 1] = {};
    bicg::PushRun *d_push_runs[bicg::MAX_RANKS - 1] = {};
    int push_nruns[bicg::MAX_RANKS - 1] = {};
    // fused-vector launch shape
    int vgrid = 0, vchunk = 0;
    // captured iteration batches, per method
    cudaGraphExec_t graph[4] = {};
    int graph_unroll[4] = {};
    // cache key
    const void *host_key = nullptr;
    uint64_t host_fp = 0;            // content fingerprint of the caller's arrays at upload time (matrix.cu)
    double upload_ms = 0.0;
    cudaEvent_t ev_upload0 = nullptr, ev_upload1 = nullptr;   // around upload + planning; read lazily (matrix_upload_ms)
    uint64_t upload_bytes = 0;

    double *vec(int id) const { return vec_base + (long long)id * vstride; }
};

namespace bicg {

// matrix.cu
bicg_matrix *matrix_create(const CSR_Matrix *diag, const CSR_Matrix *offd, const INFO_Matrix *info);
void matrix_destroy(bicg_matrix *m);
double matrix_upload_ms(bicg_matrix *m);
bicg_matrix *matrix_get_cached(const CSR_Matrix *diag, const CSR_Matrix *offd, const INFO_Matrix *info, bool *fresh);
// solve.cu
int  solve(bicg_matrix *m, int method, double *x, double *r, int krr, int nrr, int device_vectors, bicg_stats *st);
int  spmv_host(bicg_matrix *m, const double *x_loc, double *y_loc, double *x_full_or_null);
int  spmv_time(bicg_matrix *m, int reps, double *ms, double *bytes);
void print_reference_lines(const bicg_stats &st, const std::vector<double> &hist);
// shifted.cu
int  shifted_solve(bicg_matrix *m, double *x_set, double *r, const double *sigma, int sigma_len, int seed, double tol, int max_iter);
// helpers shared by matrix.cu / solve.cu
SpmvArgs make_spmv_args(const bicg_matrix *m, const SpmvPlan &p, int x_id, int y_id);
void launch_spmv_plan(const bicg_matrix *m, const SpmvPlan &p, const SpmvArgs &a, int prof_class = 0);

} // namespace bicg
