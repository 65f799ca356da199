// mega.cuh -- argument block, synchronisation state and launch interface of the persistent solver kernel (mega.cu)
#pragma once
#include "dev.cuh"
#include "vec.cuh"

namespace bicg {

constexpr int MEGA_MAX_CTAS   = 160;   // >= SM count (148 on B200); one CTA per SM
constexpr int MEGA_RING       = 8;     // generations of arrival slots kept (a CTA is never more than 3 ahead of another)
constexpr int MEGA_SLOT_WORDS = 16;    // 8 doubles as LL words

// What a CTA leaves at a synchronisation point: its partial dot products as self-validating LL words
// {generation | 32 data bits} (dev.cuh).  One 128-byte line per CTA and generation, written once, polled by the CTAs
// that depend on it -- no atomics, no master, no second "release" flag.
struct alignas(128) MegaSlot { unsigned long long w[MEGA_SLOT_WORDS]; };

// counters that survive from one solve to the next (same value in every CTA / on every rank)
struct alignas(128) MegaState {
    unsigned gen;                       // last arrival generation used
    unsigned red_epoch;                 // last cross-GPU reduction posted
    unsigned long long halo_epoch;      // last halo exchange signalled
    int plan_ok[MAX_RANKS];             // written by rank p at plan time: its persistent-kernel plan is usable
    int resident_ctas;                  // CTAs of the last launch that kept their matrix slice in shared memory (test / trace aid)
};

// Lives in the IPC-shared arena: `mail` and `st.plan_ok` are written by the peers.
struct MegaSync {
    MegaState st;
    MegaSlot  slot[MEGA_RING][MEGA_MAX_CTAS];
    MegaSlot  mail[2][MAX_RANKS];                           // [epoch parity][source rank]: that rank's local sums
};

// where the boundary runs of the arena vectors go on the peers (LL halo regions, see LLRegion)
struct PushPlan {
    int npeers;
    int peer[MAX_RANKS - 1];                        // rank of push slot i
    const PushRun *runs[MAX_RANKS - 1];
    int nruns[MAX_RANKS - 1];
    unsigned long long *ll_dst[MAX_RANKS - 1];      // that rank's LL halo regions (region k at + k * 2 * ll_stride words)
    long long ll_stride[MAX_RANKS - 1];             // ... its region length in elements
};

// LL halo regions (one per pushed vector; s has two because the multi-GPU BiCGStab loop double-buffers it)
enum LLRegion : int { LL_S0 = 0, LL_S1, LL_R, LL_P, LL_Z, LL_X, LL_W, LL_REGIONS };

constexpr int MEGA_TRACE_ITERS = 256, MEGA_TRACE_SLOTS = 16;

struct MegaArgs {
    Scalars *sc;
    double  *hist;
    CommDev  comm;              // kernel-per-phase protocol state (only for the halo wait on entry)
    MegaSync *sync;             // this rank's
    MegaSlot *peer_mail[MAX_RANKS];              // rank p's sync->mail[0]
    int n_ghost;                // ghost slots of this rank
    const int4 *cta_dep;        // [grid]: min / max own column, min / max ghost slot referenced by the CTA's rows
    const double   *val;
    const unsigned *col;
    const unsigned *ptr;
    const int      *tile_row;   // ntiles + 1
    const unsigned *tile_nz;    // ntiles + 1
    const int      *cta_tile;   // grid + 1 : first tile of every CTA (contiguous ownership)
    const int      *tile_flag;  // null, or per tile: 0 whole rows, 1 / 2 chunk of ONE long row (more follow / last)
    const int      *tile_cbase; // null, or per tile: >= 0 a narrow tile, its columns are streamed as col16 = col - tile_cbase;
                                //    -1 a wide tile (32-bit col).  Null: every tile is wide
    const unsigned short *col16;
    int cap, stages;
    int ghost_off;
    int l2_hint;                // 1: matrix stream is loaded with an L2 evict-first policy
    int gather_cg;              // 1: SpMV gathers bypass L1 (ld.global.cg) and the neighbour waits skip the acquire fence
    int resident;               // 1: a CTA whose whole matrix slice fits into its shared memory (strong scaling: 8 GPUs x 148 CTAs)
                                //    loads it ONCE per solve (values + 16-bit CTA-relative columns + row pointers) instead of streaming it
                                //    through the TMA ring in every SpMV
    int smem_bytes;             // dynamic shared memory of this launch
    double *vec_base; long long vstride;   // arena vectors: vec(id) = vec_base + id * vstride
    VecPtrs v;
    PushPlan push;
    const unsigned long long *ll;          // this rank's LL halo regions, [LL_REGIONS][ll_stride] pairs
    long long ll_stride;
    int method;                 // 0 bicgstab, 1 ca_bicgstab, 2 pipe_bicgstab, 3 pipe_bicgstab_rr
    int krr, nrr;
    unsigned long long *snap;   // optional [grid][2]: arrival / release of the alpha sync of iteration snap_iter, every CTA
    int snap_iter;
    unsigned long long *trace;  // optional [2][MEGA_TRACE_ITERS][MEGA_TRACE_SLOTS] globaltimer checkpoints (BICG_MEGA_TRACE)
};

int    launch_mega(int threads, int lanes, int grid, size_t smem, const MegaArgs &a, cudaStream_t st);
int    mega_setup_attributes();
bool   mega_has_variant(int threads, int lanes);
size_t mega_smem_bytes(int cap, int stages, int threads, int lanes);
// shared memory a CTA needs to keep `nnz` entries of `rows` rows resident (host and device use the same formula)
__host__ __device__ inline size_t mega_resident_bytes(unsigned nnz, int rows)
{
    const size_t nnzp = ((size_t)nnz + 7u) & ~(size_t)7u;
    return nnzp * 10u + ((size_t)rows + 1u) * 4u;
}
// per-CTA column ranges of the plan (one launch at plan time)
void   launch_mega_dep(const unsigned *col, const unsigned *ptr, const int *tile_row, const int *cta_tile, int grid,
                       int ghost_off, int4 *dep, cudaStream_t st);
// Column width of every tile of the plan (one CTA per tile).  A tile is narrow when it holds whole rows, has entries, none of
// them in the ghost window, and max col - min col < 65536: tile_cbase[t] = min col, else -1.  narrow_count += narrow tiles.
void   launch_mega_tile_base(const unsigned *col, const unsigned *tile_nz, const int *tile_flag, int ntiles, int ghost_off,
                             int *tile_cbase, int *narrow_count, cudaStream_t st);
// col16[j] = col[j] - tile_cbase[t] for the entries of the narrow tiles
void   launch_mega_tile_codes(const unsigned *col, const unsigned *tile_nz, const int *tile_cbase, int ntiles,
                              unsigned short *col16, cudaStream_t st);

} // namespace bicg
