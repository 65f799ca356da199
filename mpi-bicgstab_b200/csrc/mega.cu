// mega.cu -- one persistent, cooperative kernel per solve: the whole iteration loop of solver.c on the device.
//
// Why: with the matrix split over 8 GPUs an iteration is ~13 us of memory traffic; kernel boundaries, atomics and
// master/worker barriers cost several times that.  Here one CTA per SM stays resident for the entire solve and
//   * owns a fixed, contiguous, work-balanced range of rows (plan.cpp: plan_cta_tiles);
//   * runs the SpMV phases as the warp-specialised TMA pipeline of spmv.cu over its own tiles -- the producer warp
//     never stops: while the consumers are in a vector phase or wait at a synchronisation point it is already
//     streaming the first stages of the NEXT SpMV (the matrix never changes), with an L2 evict-first policy so that
//     the once-per-SpMV matrix stream does not push the (re-used) vectors out of the 126 MB L2;
//   * runs the vector phases (vec_body.cuh) on its own rows only, so nothing but the gathered x crosses SMs;
//   * keeps ITS OWN copy of the solver scalars (alpha, beta, omega, the dots, k, the loop test) in shared memory:
//     every CTA evaluates the recurrences of solver.c:93-120 itself from the same reduced values, in the same
//     order, so all CTAs (and all ranks) take bitwise identical decisions and nobody waits for a "master".
//
// Synchronisation (the replacement of MPI_Iallreduce/MPI_Wait and of the grid barriers of round 1):
//   arrive   : a CTA publishes its partial dots as self-validating LL words {generation | 32 data bits} in its own
//              128-byte slot of the generation's ring entry -- plain stores, no atomics (a release fence only where the
//              arrival also publishes rows that other CTAs gather next);
//   reduce   : (1 GPU) every CTA polls all slots of the generation (160 threads, one slot each) and adds them in a
//              fixed order; (N GPUs) only the middle CTA (the reducer) does that, posts the rank's sums into every rank's mailbox over
//              NVLink (LL words again), and every CTA of every rank polls its own GPU's 8 mailboxes and adds them in
//              rank order.  Critical path: one L2 round trip (+ one NVLink hop + one L2 round trip);
//   post / complete : the same, split (MPI_Iallreduce ... SpMV ... MPI_Wait of the pipelined variants);
//   neighbour wait  : where solver.c has no reduction but the next SpMV gathers what other CTAs just wrote (q, p,
//              s, ...), a CTA waits only for the CTAs that own the columns its rows reference (a handful for banded
//              matrices);
//   halo (N GPUs)   : boundary rows travel to the peers as LL words too (16 bytes per value, push_ll): no system-scope
//              fence, no flag -- the consumer polls exactly the ghost slots it needs.  In the BiCGStab loop the pushes
//              ride on the alpha / beta reductions and the ghost copies of q and p are advanced redundantly
//              (run_bicgstab_multi); the CA / pipelined loops unpack the LL words into the ghost tails (halo_ll, post).
// Coherence: gathered vectors are read with plain (L1-cached) loads; every neighbour wait ends in an acquire fence at gpu
// scope (SASS: MEMBAR + CCTL.IVALL), so rows rewritten by other SMs are re-fetched from L2; values from peers are taken
// from the LL words with system-scope loads and re-stored locally by the consuming CTA.
// Every wait is bounded by CommDev::timeout_ns (BICG_PEER_TIMEOUT_S): a lost CTA or rank raises Scalars::error instead of hanging the GPU.
#include "mega.cuh"
#include "vec_body.cuh"

namespace bicg {

namespace {

constexpr int PROW_PAD = 8;
constexpr int RED_THREADS = MEGA_MAX_CTAS;          // one polled slot per thread
constexpr int RED_WARPS = RED_THREADS / 32;
// lo, hi: the tile's entries relative to a0.  cbase >= 0: a narrow tile -- the column region of the stage holds 16-bit codes
// col - cbase from entry (a0 & ~7) on (TMA wants 16-byte windows), so entry a0 + i has its code at index i + (a0 & 4)
struct StageHdr { int row0, row1; unsigned a0; int rowa; unsigned lo, hi; int flag; int cbase; };

__device__ __forceinline__ void mbar_arrive(unsigned bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void nbar(int id, int nthreads)  // named CTA barrier (the producer warp free-runs)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ unsigned long long l2_evict_first_policy()
{
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void tma_load_1d_hint(unsigned dst_smem, const void *src, unsigned bytes, unsigned bar,
                                                 unsigned long long pol)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}
// Polling etiquette: the first probes go out back to back (the last arriver normally finds everything in place), after
// that the thread sleeps 64 .. 256 ns between probes -- 148 CTAs spinning flat out on the same 148 cache lines delay the
// very stores they are waiting for.
__device__ __forceinline__ void poll_pause(unsigned spins)
{
    if (spins > 2u) __nanosleep(spins > 16u ? 256u : (spins > 6u ? 128u : 64u));
}
template <int LANES>
__device__ __forceinline__ double lanes_sum(double v)
{
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// CTA-wide sum over the consumer threads only; result valid in every lane of warp 0
template <int N, int CT>
__device__ __forceinline__ void cblock_sum(double (&v)[N], double *scratch)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int NW = CT / 32;
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] = warp_sum(v[k]);
    nbar(1, CT);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < N; ++k) scratch[warp * N + k] = v[k];
    }
    nbar(1, CT);
    if (warp == 0) {
#pragma unroll
        for (int k = 0; k < N; ++k) {
            double t = (lane < NW) ? scratch[lane * N + k] : 0.0;
            v[k] = warp_sum(t);
        }
    }
}

enum Epi : int { EPI_NONE = 0, EPI_RH_Y, EPI_QY_YY, EPI_CA4 };

struct MegaShared {
    Scalars sc;                               // this CTA's copy of the solver scalars
    double tot[MAIL_VALS];                    // reduced values of the current synchronisation point
    double red[RED_WARPS][MAIL_VALS];
    double contrib[MAX_RANKS][MAIL_VALS];
    double scratch[32 * MAX_DOTS];
    unsigned long long full_bar[4], empty_bar[4];
    StageHdr hdr[4];
    volatile int flags[4];                    // [1] producer stop, [2] consumed visits, [3] a wait timed out
};

// Resident mode (MegaArgs::resident; strong scaling, e.g. T' over 8 GPUs x 148 CTAs = 20 k entries per CTA): a CTA whose whole
// slice fits into its shared memory -- 8-byte values, columns as 16-bit offsets into the CTA's own / ghost column windows
// (mega_dep_kernel), row pointers -- loads it ONCE per solve; its SpMV phases then touch neither L2 nor the TMA ring for
// the matrix.  Decided per CTA, identically by the producer thread and by every consumer thread.
struct ResidentPlan { bool on; int row_lo, rows; unsigned nz_lo, nnz, ospan; int obase, gbase; };
__device__ __forceinline__ ResidentPlan resident_plan(const MegaArgs &a, int t0, int t1, int lanes)
{
    ResidentPlan p;
    p.on = false; p.row_lo = 0; p.rows = 0; p.nz_lo = 0u; p.nnz = 0u; p.ospan = 0u; p.obase = 0; p.gbase = 0;
    if (!a.resident || lanes != 1 || t1 <= t0 || a.tile_flag != nullptr) return p;
    p.row_lo = a.tile_row[t0];
    p.rows = a.tile_row[t1] - p.row_lo;
    if (p.rows <= 0) return p;
    p.nz_lo = a.ptr[p.row_lo];
    p.nnz = a.ptr[p.row_lo + p.rows] - p.nz_lo;
    if (mega_resident_bytes(p.nnz, p.rows) > (size_t)a.smem_bytes) return p;
    const int4 dep = a.cta_dep[blockIdx.x];
    const bool own = dep.x <= dep.y, gh = dep.z <= dep.w;
    p.ospan = own ? (unsigned)(dep.y - dep.x + 1) : 0u;
    const unsigned gspan = gh ? (unsigned)(dep.w - dep.z + 1) : 0u;
    if (p.ospan + gspan > 65536u) return p;             // the columns of this CTA do not fit 16-bit offsets: it streams
    p.obase = own ? dep.x : 0;
    p.gbase = a.ghost_off + (gh ? dep.z : 0) - (int)p.ospan;   // column = gbase + code for codes >= ospan
    p.on = true;
    return p;
}

template <int CT, int LANES>
struct Mega {
    static constexpr int RPT = CT / LANES, PROW = RPT + PROW_PAD, NCW = CT / 32, UNR = (LANES == 1) ? 16 : 8;
    static_assert(CT >= RED_THREADS, "the slot reduction uses one thread per CTA slot");

    const MegaArgs &a;
    MegaShared &sh;
    unsigned char *dyn;
    int tid, lane, my_tiles, row_lo, row_hi;
    unsigned vis;                 // SpMV tile visits consumed so far (mirrors the producer's counter)
    unsigned gen;                 // arrival generation (same value in every CTA)
    unsigned red_epoch;           // cross-GPU reductions posted (same value on every rank)
    unsigned posted_gen;          // generation of the reduction posted and not yet completed
    unsigned long long halo_epoch;
    int dep_lo, dep_hi;           // CTAs owning the own columns this CTA's rows reference
    unsigned push_slots;          // push slots (peers) that need rows of this CTA
    int ghost_lo, ghost_hi;       // ghost slots this CTA's rows gather [lo, hi)
    int gs_lo, gs_hi;             // ghost slots this CTA keeps up to date itself (multi-GPU bicgstab: redundant recurrences)
    bool reads_ghost;             // this CTA's rows gather ghost columns
    bool is_reducer;              // N > 1: the CTA that adds up this GPU's slots and posts them to the peers' mailboxes
    size_t stage_bytes;
    int trace_it, trace_who;
    bool resident;                // this CTA keeps its matrix slice in shared memory (ResidentPlan)
    ResidentPlan rp;
    const double *rs_val; const unsigned short *rs_col; const unsigned *rs_ptr;

    __device__ Mega(const MegaArgs &args, MegaShared &s) : a(args), sh(s) {}

    __device__ bool stop_now() const { return sh.sc.done != 0 || sh.sc.error != 0; }
    __device__ void fail() { sh.flags[3] = 1; }
    // one iteration's alpha sync seen by EVERY CTA: [G][2] = arrival, release (globaltimer, per GPU)
    __device__ void snap(int which)
    {
        if (a.snap && tid == 0 && sh.sc.k == a.snap_iter) a.snap[2 * blockIdx.x + which] = globaltimer_ns();
    }
    __device__ void mark(int slot)
    {
        if (a.trace && trace_who >= 0 && tid == 0 && trace_it < MEGA_TRACE_ITERS)
            a.trace[((size_t)trace_who * MEGA_TRACE_ITERS + trace_it) * MEGA_TRACE_SLOTS + slot] = globaltimer_ns();
    }

    // ---------------------------------------------------------------- arrive ------------------------------
    // Publish NV partial sums (NV = 0: presence only) for generation ++gen.
    // release: the arrival also PUBLISHES this CTA's stores of the phase (rows that other CTAs gather after waiting for
    // it): CTA barrier + release fence before the words go out.  A pure reduction arrival does not need it: the reduced
    // values travel inside the words, nobody gathers this CTA's rows before its next releasing arrival (a neighbour wait
    // always precedes a gather), and its own earlier gathers completed before the dots that depend on them.
    template <int NV>
    __device__ void arrive(double (&dot)[NV > 0 ? NV : 1], bool release)
    {
        // a CTA barrier (inside cblock_sum, or the explicit one) puts every consumer's stores of the phase before the fence
        if (NV > 0) cblock_sum<(NV > 0 ? NV : 1), CT>(dot, sh.scratch);
        else nbar(1, CT);
        ++gen;
        if (tid < 32) {
            if (release) fence_gpu();
            MegaSlot *s = &a.sync->slot[gen & (MEGA_RING - 1)][blockIdx.x];
            constexpr int NW = NV > 0 ? 2 * NV : 1;
            if (lane < NW) {
                unsigned data = 0u;
                if (NV > 0) {
                    double v = dot[0];
#pragma unroll
                    for (int k = 1; k < NV; ++k) v = ((lane >> 1) == k) ? dot[k] : v;
                    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
                    data = (lane & 1) ? (unsigned)(b >> 32) : (unsigned)b;
                }
                st_ll_gpu(&s->w[lane], ll_pack(data, gen));
            }
        }
    }

    // ---------------------------------------------------------------- neighbour wait ----------------------
    // wait for the CTAs (of this GPU) that own the columns this CTA's rows gather
    __device__ void wait_nbr()
    {
        if (tid < 32) {
            bool ok = true;
            const unsigned long long t0 = globaltimer_ns();
            const MegaSlot *ring = a.sync->slot[gen & (MEGA_RING - 1)];
            for (int c = dep_lo + lane; c <= dep_hi; c += 32) {
                if (c == (int)blockIdx.x) continue;
                unsigned spins = 0;
                while ((unsigned)(ld_ll_gpu(&ring[c].w[0]) >> 32) != gen) {
                    poll_pause(++spins);
                    if ((spins & 255u) == 0u && globaltimer_ns() - t0 > a.comm.timeout_ns) { ok = false; break; }
                }
            }
            if (!a.gather_cg) fence_gpu();                   // acquire (+ L1 invalidate): the gathers that follow see the data
            if (!__all_sync(0xffffffffu, ok) && lane == 0) fail();
        }
        nbar(1, CT);
        if (sh.flags[3]) { if (tid == 0) { sh.sc.error = 1; sh.sc.done = 1; } nbar(1, CT); }
    }
    __device__ void sync_nbr()
    {
        double d0[1] = {0.0};
        arrive<0>(d0, true);
        wait_nbr();
    }

    // ---------------------------------------------------------------- reductions --------------------------
    // All slots of generation g -> sh.tot (fixed order: thread c takes CTA c, butterfly inside each of the five
    // warps, then warp 0..4 left to right).  Called by every consumer thread; sh.tot is valid for tid 0 on return.
    template <int NV>
    __device__ void local_reduce(unsigned g)
    {
        if (tid < RED_THREADS) {
            double v[NV];
#pragma unroll
            for (int k = 0; k < NV; ++k) v[k] = 0.0;
            if (tid < (int)gridDim.x) {
                const unsigned long long *w = a.sync->slot[g & (MEGA_RING - 1)][tid].w;
                const unsigned long long t0 = globaltimer_ns();
                unsigned long long w0[NV], w1[NV];
                unsigned spins = 0;
                for (;;) {
                    bool all = true;
#pragma unroll
                    for (int k = 0; k < NV; ++k) { ld_ll_gpu2(w + 2 * k, w0[k], w1[k]); all = all && ll_valid(w0[k], w1[k], g); }
                    if (all) break;
                    ++spins;
                    if (a.comm.world == 1) poll_pause(spins);        // N > 1: only the reducer CTA polls the slots -- no crowd, no pause
                    if ((spins & 255u) == 0u && globaltimer_ns() - t0 > a.comm.timeout_ns) { fail(); break; }
                }
#pragma unroll
                for (int k = 0; k < NV; ++k) v[k] = ll_decode(w0[k], w1[k]);
            }
#pragma unroll
            for (int k = 0; k < NV; ++k) v[k] = warp_sum(v[k]);
            if (lane == 0) {
#pragma unroll
                for (int k = 0; k < NV; ++k) sh.red[tid >> 5][k] = v[k];
            }
            nbar(2, RED_THREADS);
            if (tid == 0) {
#pragma unroll
                for (int k = 0; k < NV; ++k) {
                    double t = sh.red[0][k];
#pragma unroll
                    for (int wq = 1; wq < RED_WARPS; ++wq) t += sh.red[wq][k];
                    sh.tot[k] = t;
                }
            }
        }
    }
    // warp 0 of the reducer CTA: this rank's sums -> every rank's mailbox[parity][me]
    template <int NV>
    __device__ void post_mail()
    {
        __syncwarp();
        if (lane < a.comm.world) {
            MegaSlot *mb = a.peer_mail[0];
#pragma unroll
            for (int p = 1; p < MAX_RANKS; ++p) mb = (lane == p) ? a.peer_mail[p] : mb;
            mb += (size_t)(red_epoch & 1u) * MAX_RANKS + a.comm.rank;
#pragma unroll
            for (int k = 0; k < NV; ++k) {
                unsigned long long w0, w1;
                ll_encode(sh.tot[k], red_epoch, w0, w1);
                st_ll_sys(&mb->w[2 * k], w0, w1);
            }
        }
        __syncwarp();
    }
    // warp 0 of every CTA: the ranks' sums from this GPU's own mailboxes, added in rank order -> sh.tot
    template <int NV>
    __device__ void mail_reduce()
    {
        if (lane < a.comm.world) {
            const unsigned long long *w = a.sync->mail[red_epoch & 1u][lane].w;
            const unsigned long long t0 = globaltimer_ns();
            unsigned long long w0[NV], w1[NV];
            unsigned spins = 0;
            for (;;) {
                bool all = true;
#pragma unroll
                for (int k = 0; k < NV; ++k) { ld_ll_sys(w + 2 * k, w0[k], w1[k]); all = all && ll_valid(w0[k], w1[k], red_epoch); }
                if (all) break;
                if (++spins > 4u) __nanosleep(48);                   // 8 lines polled by 148 x 8 threads: a short pause is enough
                if ((spins & 255u) == 0u && globaltimer_ns() - t0 > a.comm.timeout_ns) { fail(); break; }
            }
#pragma unroll
            for (int k = 0; k < NV; ++k) sh.contrib[lane][k] = ll_decode(w0[k], w1[k]);
        }
        __syncwarp();
        if (lane < NV) {
            double acc = sh.contrib[0][lane];
            for (int p = 1; p < a.comm.world; ++p) acc += sh.contrib[p][lane];
            sh.tot[lane] = acc;
        }
        __syncwarp();
    }
    // complete the reduction published at generation g and evaluate the scalar recurrence `fin` in this CTA's copy
    template <int NV>
    __device__ void finish(unsigned g, int fin, bool posted, bool tr = false)
    {
        if (a.comm.world == 1) { local_reduce<NV>(g); if (tr) mark(12); }
        else {
            if (is_reducer && !posted) { local_reduce<NV>(g); if (tr) mark(12); if (tid < 32) post_mail<NV>(); if (tr) mark(13); }
            if (tid < 32) mail_reduce<NV>();
            if (tr) mark(14);
        }
        if (tid == 0) {
            // no acquire fence here: a reduction is never directly followed by a gather of other CTAs' rows (a neighbour
            // wait with its own fence always sits in between), and the writes that follow are control-dependent on the
            // polls above
            if (sh.flags[3]) { sh.sc.error = 1; sh.sc.done = 1; }
            else finalize(fin, &sh.sc, blockIdx.x == 0 ? a.hist : nullptr, sh.tot);
        }
        nbar(1, CT);
    }
    // push_id >= 0: the boundary rows of that vector leave as LL words (push_ll) right AFTER this CTA's reduction words --
    // the consumers poll the LL words themselves, so the push need not delay the arrival; it overlaps with the reduction's
    // NVLink latency instead of preceding it
    template <int NV>
    __device__ void reduce(double (&dot)[NV], int fin, bool tr = false, int push_id = -1, int region = 0, unsigned epoch = 0u)
    {
        arrive<NV>(dot, false);
        if (tr) { mark(11); snap(0); }
        if (push_id >= 0) push_ll(push_id, region, epoch);
        if (a.comm.world > 1) ++red_epoch;
        finish<NV>(gen, fin, false, tr);
        if (tr) snap(1);
    }
    // MPI_Iallreduce + the halo of vector `id` that the SpMV hiding the reduction gathers (LL region `region`)
    template <int NV>
    __device__ void post(double (&dot)[NV], int id, int region)
    {
        const bool multi = a.comm.world > 1;
        const unsigned ep = multi ? (unsigned)(++halo_epoch) : 0u;
        arrive<NV>(dot, true);
        posted_gen = gen;
        if (multi) {
            ++red_epoch;
            if (is_reducer) { local_reduce<NV>(gen); if (tid < 32) post_mail<NV>(); }
            push_ll(id, region, ep);
        }
        wait_nbr();
        if (multi) unpack_ll(id, region, ep);
    }
    // MPI_Wait.  after_spmv: the SpMV that hid the reduction gathered a vector that the NEXT phase overwrites in place
    // (pipelined loops: y = w - alpha z is stored over w right after t = A w): the reduction was published BEFORE that
    // SpMV, so its completion says nothing about the other CTAs having finished their gathers.  A second, data-free
    // arrival after the SpMV, awaited from every CTA of this GPU (peers never gather own rows), closes the window.
    template <int NV>
    __device__ void complete(int fin, bool after_spmv)
    {
        if (after_spmv) {
            double d0[1] = {0.0};
            arrive<0>(d0, false);
            if (tid < RED_THREADS && tid < (int)gridDim.x && tid != (int)blockIdx.x) {
                const unsigned long long *w = a.sync->slot[gen & (MEGA_RING - 1)][tid].w;
                const unsigned long long t0 = globaltimer_ns();
                unsigned spins = 0;
                while ((unsigned)(ld_ll_gpu(w) >> 32) != gen) {
                    poll_pause(++spins);
                    if ((spins & 255u) == 0u && globaltimer_ns() - t0 > a.comm.timeout_ns) { fail(); break; }
                }
            }
        }
        finish<NV>(posted_gen, fin, true);
    }

    // ---------------------------------------------------------------- SpMV over this CTA's tiles ----------
    // gather_cg (BICG_GATHER_CG=1, multi-GPU experiments): x is gathered with L2-only loads; the neighbour waits then need no
    // acquire fence (no L1 line can be stale), which takes a MEMBAR + CCTL.IVALL off every neighbour wait
    template <int EPI>
    __device__ void spmv(const double *x, double *y, double (&dot)[4])
    {
        if constexpr (LANES == 1) {
            if (resident) {
                if (a.gather_cg) spmv_res<EPI, true>(x, y, dot); else spmv_res<EPI, false>(x, y, dot);
                return;
            }
        }
        if (a.gather_cg) spmv_impl<EPI, true>(x, y, dot); else spmv_impl<EPI, false>(x, y, dot);
    }
    // one row's epilogue: y and the dots fused into the SpMV (same operations, same order as the streaming path)
    template <int EPI>
    __device__ __forceinline__ void row_done(int row, double acc, double e0, double e1, double e2, double e3, double *y, double (&dot)[4])
    {
        y[row] = acc;
        if (EPI == EPI_RH_Y) dot[0] = fma(e0, acc, dot[0]);
        if (EPI == EPI_QY_YY) { dot[0] = fma(e0, acc, dot[0]); dot[1] = fma(acc, acc, dot[1]); }
        if (EPI == EPI_CA4) {
            dot[0] = fma(e0, e1, dot[0]); dot[1] = fma(e0, acc, dot[1]);
            dot[2] = fma(e0, e2, dot[2]); dot[3] = fma(e0, e3, dot[3]);
        }
    }
    // SpMV over a shared-memory-resident slice: thread-per-row (rows tid + k CT, so neighbouring threads gather neighbouring
    // columns); a row's entries are accumulated in storage order, like spmv_impl.  Loads are unconditional on clamped indices
    // (always a valid entry of this slice; no predicate per load, so the U gathers of a pass are in flight together), only the
    // multiply-adds are guarded.
    template <int EPI, bool CG>
    __device__ void spmv_res(const double *x, double *y, double (&dot)[4])
    {
        constexpr int U = 16;
        const double *xo = x + rp.obase, *xg = x + rp.gbase;
        const unsigned ospan = rp.ospan;
        const int rows = rp.rows;
        const bool empty = rp.nnz == 0u;                      // a slice of empty rows: y = 0, the dots see acc = 0
        const unsigned last = empty ? 0u : rp.nnz - 1u;
        for (int r = tid; r < rows; r += CT) {
            const int row = rp.row_lo + r;
            unsigned j = rs_ptr[r];
            const unsigned e = rs_ptr[r + 1];
            double e0 = 0.0, e1 = 0.0, e2 = 0.0, e3 = 0.0;     // epilogue operands: in flight during the gathers
            if (EPI == EPI_RH_Y) e0 = a.v.rh[row];
            if (EPI == EPI_QY_YY) e0 = a.v.r[row];
            if (EPI == EPI_CA4) { e0 = a.v.rh[row]; e1 = a.v.r[row]; e2 = a.v.s[row]; e3 = a.v.z[row]; }
            double acc = 0.0;
            while (j < e) {                                    // never entered when the slice is empty
                double xv[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const unsigned c = rs_col[min(min(j + (unsigned)u, e - 1u), last)];
                    const double *src = (c < ospan ? xo : xg) + c;
                    xv[u] = CG ? ld_l2(src) : ld_coherent(src);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {                  // the values come from shared memory when they are needed
                    const double v = rs_val[min(min(j + (unsigned)u, e - 1u), last)];
                    if (j + (unsigned)u < e) acc = fma(v, xv[u], acc);
                }
                j += (unsigned)U;
            }
            row_done<EPI>(row, acc, e0, e1, e2, e3, y, dot);
        }
    }

    template <int EPI, bool CG>
    __device__ void spmv_impl(const double *x, double *y, double (&dot)[4])
    {
        const int stages = a.stages, cap = a.cap;
        const int sub = tid % LANES, row_in_tile = tid / LANES;
        double carry = 0.0;
        for (int lt = 0; lt < my_tiles; ++lt, ++vis) {
            const int s = (int)(vis % (unsigned)stages);
            mbar_wait(smem_u32(&sh.full_bar[s]), (vis / (unsigned)stages) & 1u);
            const unsigned char *st = dyn + (size_t)s * stage_bytes;
            const double   *sval = reinterpret_cast<const double *>(st);
            const unsigned *scol = reinterpret_cast<const unsigned *>(sval + cap);
            const unsigned *sptr = scol + cap;
            const StageHdr h = sh.hdr[s];
            if (h.flag != 0) {
                // one chunk of a row longer than a stage: the whole CTA multiplies it, the row's partial sum is carried
                // from chunk to chunk in `carry` (same value in every thread) and the row is finished by its last chunk
                double part[1] = {0.0};
                for (unsigned jj = h.lo + (unsigned)tid; jj < h.hi; jj += 4u * CT) {
                    double pv[4], px[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const unsigned idx = min(jj + (unsigned)(u * CT), h.hi - 1u);
                        pv[u] = sval[idx]; px[u] = CG ? ld_l2(x + scol[idx]) : ld_coherent(x + scol[idx]);
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (jj + (unsigned)(u * CT) < h.hi) part[0] = fma(pv[u], px[u], part[0]);
                }
                cblock_sum<1, CT>(part, sh.scratch);                   // fixed order; result in every lane of warp 0
                if (tid == 0) sh.red[0][0] = part[0];
                nbar(1, CT);
                carry += sh.red[0][0];
                if (h.flag == 2) {
                    if (tid == 0) {
                        const int row = h.row0;
                        const double acc = carry;
                        y[row] = acc;
                        if (EPI == EPI_RH_Y) dot[0] = fma(a.v.rh[row], acc, dot[0]);
                        if (EPI == EPI_QY_YY) { dot[0] = fma(a.v.r[row], acc, dot[0]); dot[1] = fma(acc, acc, dot[1]); }
                        if (EPI == EPI_CA4) {
                            const double rh = a.v.rh[row];
                            dot[0] = fma(rh, a.v.r[row], dot[0]); dot[1] = fma(rh, acc, dot[1]);
                            dot[2] = fma(rh, a.v.s[row], dot[2]); dot[3] = fma(rh, a.v.z[row], dot[3]);
                        }
                    }
                    carry = 0.0;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(smem_u32(&sh.empty_bar[s]));
                continue;
            }
            // the branch is uniform over the CTA (one header per stage)
            if (h.cbase >= 0)
                tile_rows<EPI, CG>(h, sval, reinterpret_cast<const unsigned short *>(scol) + (h.a0 & 4u), sptr, x + h.cbase, y,
                                   dot, sub, row_in_tile);
            else
                tile_rows<EPI, CG>(h, sval, scol, sptr, x, y, dot, sub, row_in_tile);
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&sh.empty_bar[s]));
        }
    }
    // one tile of whole rows: LANES threads per row, a row's entries accumulated in storage order.  ColT = unsigned short (narrow
    // tile): scol holds the codes col - cbase and xb = x + cbase; ColT = unsigned: scol holds the columns and xb = x.
    template <int EPI, bool CG, typename ColT>
    __device__ __forceinline__ void tile_rows(const StageHdr &h, const double *sval, const ColT *scol, const unsigned *sptr,
                                              const double *xb, double *y, double (&dot)[4], int sub, int row_in_tile)
    {
        const int row = h.row0 + row_in_tile;
        const bool valid = row < h.row1;
        int j = 0, e = 0;
        double e0 = 0.0, e1 = 0.0, e2 = 0.0, e3 = 0.0;     // epilogue operands: in flight during the gathers
        if (valid) {
            j = (int)(sptr[row - h.rowa] - h.a0) + sub;
            e = (int)(sptr[row - h.rowa + 1] - h.a0);
            if (sub == 0) {
                if (EPI == EPI_RH_Y) e0 = a.v.rh[row];
                if (EPI == EPI_QY_YY) e0 = a.v.r[row];
                if (EPI == EPI_CA4) { e0 = a.v.rh[row]; e1 = a.v.r[row]; e2 = a.v.s[row]; e3 = a.v.z[row]; }
            }
        }
        double acc = 0.0;
        while (j < e) {
            unsigned c[UNR];
            double v[UNR], xv[UNR];
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                const int idx = min(j + u * LANES, e - 1);
                c[u] = scol[idx];
                v[u] = sval[idx];
            }
#pragma unroll
            for (int u = 0; u < UNR; ++u) xv[u] = CG ? ld_l2(xb + c[u]) : ld_coherent(xb + c[u]);
#pragma unroll
            for (int u = 0; u < UNR; ++u)
                if (j + u * LANES < e) acc = fma(v[u], xv[u], acc);
            j += UNR * LANES;
        }
        acc = lanes_sum<LANES>(acc);
        if (valid && sub == 0) {
            y[row] = acc;
            if (EPI == EPI_RH_Y) dot[0] = fma(e0, acc, dot[0]);
            if (EPI == EPI_QY_YY) { dot[0] = fma(e0, acc, dot[0]); dot[1] = fma(acc, acc, dot[1]); }
            if (EPI == EPI_CA4) {
                dot[0] = fma(e0, e1, dot[0]); dot[1] = fma(e0, acc, dot[1]);
                dot[2] = fma(e0, e2, dot[2]); dot[3] = fma(e0, e3, dot[3]);
            }
        }
    }

    // ---------------------------------------------------------------- vector phase over the CTA's own rows --
    // row_lo is a multiple of 16 and every arena vector is 128-byte aligned: 16-byte accesses, two in flight per
    // vector and thread
    template <int PH>
    __device__ void vec(double *dot)
    {
        Coef c;
        c.al = sh.sc.alpha; c.be = sh.sc.beta; c.om = sh.sc.omega;
        c.nbo = -c.be * c.om;
        const int hi2 = row_lo + ((row_hi - row_lo) & ~1);
        int i = row_lo + 2 * tid;
        for (; i + 2 * CT < hi2; i += 4 * CT) body<PH, Pairs<2, 2 * CT>>(a.v, i, c, dot);
        for (; i < hi2; i += 2 * CT) body<PH, Pairs<1, 2 * CT>>(a.v, i, c, dot);
        if (tid == 0 && hi2 < row_hi) body<PH, Contig<1>>(a.v, hi2, c, dot);
    }
    // ---------------------------------------------------------------- multi-GPU helpers ---------------------
    // releasing arrival + wait for EVERY CTA of this GPU (all == true) or for the CTAs owning the gathered columns
    __device__ void sync_local(bool all)
    {
        double d0[1] = {0.0};
        arrive<0>(d0, true);
        if (!all) { wait_nbr(); return; }
        if (tid < RED_THREADS) {
            if (tid < (int)gridDim.x && tid != (int)blockIdx.x) {
                const unsigned long long *w = a.sync->slot[gen & (MEGA_RING - 1)][tid].w;
                const unsigned long long t0 = globaltimer_ns();
                unsigned spins = 0;
                while ((unsigned)(ld_ll_gpu(w) >> 32) != gen) {
                    poll_pause(++spins);
                    if ((spins & 255u) == 0u && globaltimer_ns() - t0 > a.comm.timeout_ns) { fail(); break; }
                }
            }
            nbar(2, RED_THREADS);
            if (tid < 32 && !a.gather_cg) fence_gpu(); // acquire (+ L1 invalidate) after ALL pollers are through
        }
        nbar(1, CT);
        if (sh.flags[3]) { if (tid == 0) { sh.sc.error = 1; sh.sc.done = 1; } nbar(1, CT); }
    }
    // Boundary rows of vector `id` -> LL region `region` of the peers that gather them: every element travels as one
    // 16-byte pair of self-validating words {lo | epoch, hi | epoch} (dev.cuh), so the receiver needs neither a flag nor
    // a system-scope fence on the sender's side -- it polls the words of the elements it consumes.
    __device__ void push_ll(int id, int region, unsigned epoch)
    {
        if (push_slots == 0u) return;
        nbar(1, CT);                                  // the rows being pushed are final
        const double *src = a.vec_base + (long long)id * a.vstride;
#pragma unroll
        for (int s = 0; s < MAX_RANKS - 1; ++s) {
            if (!((push_slots >> s) & 1u)) continue;
            unsigned long long *dst = a.push.ll_dst[s] + 2ll * (long long)region * a.push.ll_stride[s];
            const PushRun *runs = a.push.runs[s];
            const int nr = a.push.nruns[s];
            int lo = 0, hi = nr;                      // first run that ends after row_lo
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (runs[mid].src + runs[mid].len <= row_lo) lo = mid + 1; else hi = mid; }
            for (int ri = lo; ri < nr; ++ri) {
                const PushRun r = runs[ri];
                if (r.src >= row_hi) break;
                const int b = max(r.src, row_lo), e = min(r.src + r.len, row_hi);
                for (int i = b + tid; i < e; i += CT) {
                    unsigned long long w0, w1;
                    ll_encode(src[i], epoch, w0, w1);
                    st_ll_sys(dst + 2ll * (long long)(r.dst_off + (i - r.src)), w0, w1);
                }
            }
        }
    }
    __device__ double ll_take(const unsigned long long *w, unsigned epoch, unsigned long long t0)
    {
        unsigned long long w0, w1;
        unsigned spins = 0;
        for (;;) {
            ld_ll_sys(w, w0, w1);
            if (ll_valid(w0, w1, epoch)) break;
            poll_pause(++spins);
            if ((spins & 255u) == 0u && globaltimer_ns() - t0 > a.comm.timeout_ns) { fail(); break; }
        }
        return ll_decode(w0, w1);
    }
    // LL region -> plain ghost tail of vector `id`, for exactly the ghost slots this CTA's rows gather (several CTAs may
    // unpack the same slot: the copy is out of place and writes the same bits).  Ends with a CTA barrier.
    __device__ void unpack_ll(int id, int region, unsigned epoch)
    {
        if (ghost_hi > ghost_lo) {
            double *g = a.vec_base + (long long)id * a.vstride + a.ghost_off;
            const unsigned long long *ll = a.ll + 2ll * region * a.ll_stride;
            const unsigned long long t0 = globaltimer_ns();
            for (int i = ghost_lo + tid; i < ghost_hi; i += CT) g[i] = ll_take(ll + 2ll * i, epoch, t0);
        }
        nbar(1, CT);
    }
    // halo exchange of the CA / pipelined loops where solver.c has no reduction: boundary rows leave as LL words, the CTA waits
    // for the CTAs owning the gathered columns, then unpacks the ghost slots it gathers
    __device__ void halo_ll(int id, int region)
    {
        if (a.comm.world == 1) { sync_nbr(); return; }
        const unsigned ep = (unsigned)(++halo_epoch);
        double d0[1] = {0.0};
        arrive<0>(d0, true);
        push_ll(id, region, ep);
        wait_nbr();
        unpack_ll(id, region, ep);
    }
    // this CTA's share of the ghost slots, element-wise exactly like the owner's rows (same operands, same operation
    // order -> bitwise the values the owner computes)
    __device__ void ghost_q(int sregion, unsigned s_epoch)                 // q = r - alpha s            solver.c:94
    {
        const double al = sh.sc.alpha;
        double *r = a.v.r + a.ghost_off;
        const unsigned long long *sll = a.ll + 2ll * sregion * a.ll_stride;
        const unsigned long long t0 = globaltimer_ns();
        for (int i = gs_lo + tid; i < gs_hi; i += CT) r[i] = fma(-al, ll_take(sll + 2ll * i, s_epoch, t0), r[i]);
    }
    __device__ void ghost_p(int sregion, unsigned s_epoch, unsigned r_epoch)   // p = r + beta (p - omega s)  solver.c:117-119
    {
        const double be = sh.sc.beta, nbo = -sh.sc.beta * sh.sc.omega;
        double *p = a.v.p + a.ghost_off, *r = a.v.r + a.ghost_off;
        const unsigned long long *sll = a.ll + 2ll * sregion * a.ll_stride, *rll = a.ll + 2ll * LL_R * a.ll_stride;
        const unsigned long long t0 = globaltimer_ns();
        for (int i = gs_lo + tid; i < gs_hi; i += CT) {
            const double rn = ll_take(rll + 2ll * i, r_epoch, t0);      // the owner's new r (pushed with the beta reduction)
            const double sg = ll_take(sll + 2ll * i, s_epoch, t0);      // the same s the ghost q used (already validated)
            double t = be * p[i];
            t = fma(1.0, rn, t);
            p[i] = fma(nbo, sg, t);
            r[i] = rn;                                                   // ghost r for the next q and for nothing else
        }
    }
    // ---------------------------------------------------------------- solver.c:86-127, several GPUs ---------
    // Two halo exchanges per iteration instead of the reference's two allgathers -- and neither is waited for on its own:
    // the boundary rows of s leave with the alpha reduction, those of the new r with the beta reduction (both are known
    // before the reduction they ride on), and every rank advances its ghost copies of q and p itself with the
    // recurrences q = r - alpha s, p = r + beta (p - omega s) applied to the ghost slots (bitwise what the owner
    // computes).  So an iteration costs three NVLink-latency sync points, not five.  The boundary values travel as LL
    // words (push_ll): no system-scope fence and no flag on the sender's side (a fence.sys after NVLink stores was
    // measured at ~4.5 us), the consumer polls exactly the elements it needs.  The LL copy of s alternates between
    // two regions: a peer may already push s of iteration k + 1 while this rank still applies s of iteration k to its
    // ghost p; r needs one region (its next push follows a reduction that this rank enters after consuming it).
    __device__ void run_bicgstab_multi()
    {
        double d4[4], d2[2], d1[1], d0[1];
        d0[0] = 0.0;
        unsigned par = 0u;
        while (true) {
            mark(0);
            d4[0] = d4[1] = d4[2] = d4[3] = 0.0;
            spmv<EPI_RH_Y>(a.v.p, a.v.s, d4);                               // s = A p, (r#,s)           :88-91
            const unsigned s_epoch = (unsigned)(++halo_epoch);
            mark(1);
            d1[0] = d4[0];
            reduce<1>(d1, FIN_BICG_ALPHA, true, V_S, LL_S0 + (int)par, s_epoch);    // alpha (+ boundary rows of s) :93
            mark(2);
            if (stop_now()) break;
            vec<PH_BICG_Q>(d0);                                             // q = r - alpha s            :94
            ghost_q(LL_S0 + (int)par, s_epoch);
            mark(3);
            sync_local(reads_ghost);
            mark(4);
            d4[0] = d4[1] = 0.0;
            spmv<EPI_QY_YY>(a.v.r, a.v.y, d4);                              // y = A q, (q,y), (y,y)      :96-102
            mark(5);
            d2[0] = d4[0]; d2[1] = d4[1];
            reduce<2>(d2, FIN_BICG_OMEGA);                                  // omega                      :104
            mark(6);
            d2[0] = d2[1] = 0.0;
            vec<PH_BICG_XR>(d2);                                            // x, r, (r,r), (r#,r)        :105-114
            const unsigned r_epoch = (unsigned)(++halo_epoch);
            mark(7);
            reduce<2>(d2, FIN_BICG_BETA, false, V_R, LL_R, r_epoch);          // beta, k++, loop test (+ boundary rows of r) :116-120
            mark(8);
            if (stop_now()) break;
            vec<PH_BICG_P>(d0);                                             // p                          :117-119
            ghost_p(LL_S0 + (int)par, s_epoch, r_epoch);
            mark(9);
            sync_local(reads_ghost);
            mark(10);
            par ^= 1u;
            ++trace_it;
        }
    }
    // ---------------------------------------------------------------- solver.c:86-127 -----------------------
    __device__ void run_bicgstab()
    {
        double d4[4], d2[2], d1[1], d0[1];
        d0[0] = 0.0;
        while (true) {
            mark(0);
            d4[0] = d4[1] = d4[2] = d4[3] = 0.0;
            spmv<EPI_RH_Y>(a.v.p, a.v.s, d4);                               // s = A p, (r#,s)           :88-91
            mark(1);
            d1[0] = d4[0];
            reduce<1>(d1, FIN_BICG_ALPHA, true);                            // alpha                      :93
            mark(2);
            if (stop_now()) break;
            vec<PH_BICG_Q>(d0);                                             // q = r - alpha s            :94
            mark(3);
            sync_nbr();
            mark(4);
            d4[0] = d4[1] = 0.0;
            spmv<EPI_QY_YY>(a.v.r, a.v.y, d4);                              // y = A q, (q,y), (y,y)      :96-102
            mark(5);
            d2[0] = d4[0]; d2[1] = d4[1];
            reduce<2>(d2, FIN_BICG_OMEGA);                                  // omega                      :104
            mark(6);
            d2[0] = d2[1] = 0.0;
            vec<PH_BICG_XR>(d2);                                            // x, r, (r,r), (r#,r)        :105-114
            mark(7);
            reduce<2>(d2, FIN_BICG_BETA);                                   // beta, k++, loop test       :116-120
            mark(8);
            if (stop_now()) break;
            vec<PH_BICG_P>(d0);                                             // p                          :117-119
            mark(9);
            sync_nbr();
            mark(10);
            ++trace_it;
        }
    }
    // ---------------------------------------------------------------- solver.c:216-259 ----------------------
    __device__ void run_ca()
    {
        double d5[5], d4[4], d2[2], d1[1], d0[1];
        d0[0] = 0.0;
        while (true) {
            vec<PH_CA_PS>(d0);                                              // p, s                       :217-222
            halo_ll(V_S, LL_S0);
            d4[0] = 0.0;
            spmv<EPI_NONE>(a.v.s, a.v.z, d4);                               // z = A s                    :224
            nbar(1, CT);                                                    // own rows of z written by other warps
            d2[0] = d2[1] = 0.0;
            vec<PH_QY>(d2);                                                 // q, y, (q,y), (y,y)         :225-230
            reduce<2>(d2, FIN_OMEGA2);                                      // omega                      :232
            if (stop_now()) break;
            d1[0] = 0.0;
            vec<PH_CA_XR>(d1);                                              // x, r, local (r,r)          :233-236
            halo_ll(V_R, LL_R);
            d4[0] = d4[1] = d4[2] = d4[3] = 0.0;
            spmv<EPI_CA4>(a.v.r, a.v.w, d4);                                // w = A r, 4 dots            :238-247
            d5[0] = d4[0]; d5[1] = d4[1]; d5[2] = d4[2]; d5[3] = d4[3]; d5[4] = d1[0];
            reduce<5>(d5, FIN_CAPIPE_END);                                  // beta, alpha, k++, test     :248-253
            if (stop_now()) break;
        }
    }
    // ---------------------------------------------------------------- solver.c:351-398 / 494-547 ------------
    __device__ void run_pipe(bool rr)
    {
        double d5[5], d4[4], d2[2], d0[1];
        d0[0] = 0.0; d4[0] = d4[1] = d4[2] = d4[3] = 0.0;
        while (true) {
            const int k = sh.sc.k;
            const bool replace = rr && (k % a.krr == 0) && k > 0 && k <= a.krr * a.nrr;   // solver.c:498, 522
            d2[0] = d2[1] = 0.0;
            if (!replace) {
                vec<PH_PIPE_1>(d2);                                         // p,s,z,q,y + (q,y),(y,y)    :352-364
            } else {
                vec<PH_RR_P>(d0);                                           // p                          :494-496
                halo_ll(V_P, LL_P);
                spmv<EPI_NONE>(a.v.p, a.v.s, d4);                           // s = A p                    :499
                halo_ll(V_S, LL_S0);
                spmv<EPI_NONE>(a.v.s, a.v.z, d4);                           // z = A s                    :500
                nbar(1, CT);
                vec<PH_QY>(d2);                                             // q, y, (q,y), (y,y)         :509-512
            }
            post<2>(d2, V_Z, LL_Z);                                         // MPI_Iallreduce x2 (+ halo of z)
            spmv<EPI_NONE>(a.v.z, a.v.v, d4);                               // v = A z hides it           :365 / 513
            complete<2>(FIN_OMEGA2, false);                                 // MPI_Wait x2 -> omega       :366-369
            if (stop_now()) break;
            d5[0] = d5[1] = d5[2] = d5[3] = d5[4] = 0.0;
            if (!replace) {
                vec<PH_PIPE_3>(d5);                                         // x, r, w + 5 dots           :370-380
            } else {
                vec<PH_RR_X>(d0);                                           // x                          :518-519
                halo_ll(V_X, LL_X);
                spmv<EPI_NONE>(a.v.x, a.v.ax, d4);                          // Ax = A x                   :523
                nbar(1, CT);
                vec<PH_RR_R>(d0);                                           // r = b - Ax                 :524-525
                halo_ll(V_R, LL_R);
                spmv<EPI_NONE>(a.v.r, a.v.w, d4);                           // w = A r                    :526
                nbar(1, CT);
                vec<PH_RR_DOTS>(d5);                                        // 5 dots                     :533-539
            }
            post<5>(d5, V_W, LL_W);                                         // MPI_Iallreduce x5 (+ halo of w)
            spmv<EPI_NONE>(a.v.w, a.v.t, d4);                               // t = A w hides it           :381 / 540
            complete<5>(FIN_CAPIPE_END, true);                              // MPI_Wait x5 -> beta, alpha :382-388
            if (stop_now()) break;
        }
    }
};

template <int CT, int LANES>
__global__ void __launch_bounds__(CT + 32, 1) bicg_mega_kernel(const __grid_constant__ MegaArgs a)
{
    using M = Mega<CT, LANES>;
    extern __shared__ __align__(128) unsigned char dyn_smem[];
    __shared__ __align__(16) MegaShared sh;

    const int tid = threadIdx.x;
    const int stages = a.stages, cap = a.cap;
    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(smem_u32(&sh.full_bar[s]), 1u);
            mbar_init(smem_u32(&sh.empty_bar[s]), (unsigned)M::NCW);
        }
        sh.flags[0] = sh.flags[1] = sh.flags[2] = sh.flags[3] = 0;
        mbar_fence_init();
    }
    __syncthreads();

    const int t0 = a.cta_tile[blockIdx.x], t1 = a.cta_tile[blockIdx.x + 1];
    const int my_tiles = t1 - t0;
    const size_t stage_bytes = (size_t)cap * 12 + (size_t)M::PROW * 4;

    if (tid >= CT) {
        // ============================ producer warp: streams this CTA's tiles round and round ==============
        if (tid == CT && my_tiles > 0 && !resident_plan(a, t0, t1, LANES).on) {
            volatile int *flags = sh.flags;
            const unsigned long long pol = l2_evict_first_policy();
            const bool hint = a.l2_hint != 0;
            unsigned v = 0;
            bool stop = false;
            for (;; ++v) {
                const int s = (int)(v % (unsigned)stages);
                if (v >= (unsigned)stages) {
                    const unsigned par = (v / (unsigned)stages - 1u) & 1u;
                    while (!mbar_try_wait(smem_u32(&sh.empty_bar[s]), par)) {
                        if (flags[1]) { stop = true; break; }
                    }
                }
                if (stop || flags[1]) break;
                const int t = t0 + (int)(v % (unsigned)my_tiles);
                const int row0 = a.tile_row[t], row1 = a.tile_row[t + 1];
                const unsigned p0 = a.tile_nz[t], p1 = a.tile_nz[t + 1];
                const unsigned a0 = p0 & ~3u, cnt = ((p1 + 3u) & ~3u) - a0;
                const int rowa = row0 & ~3, cntp = ((row1 + 1 + 3) & ~3) - rowa;
                // narrow tile: codes from entry p0 & ~7 to p1 rounded up to 8 -- at most 2 (tile entries + 14) bytes, which
                // the 4 cap bytes of the column region always hold (cap >= tile entries + 8).  A narrow tile has entries.
                const int cbase = a.tile_cbase ? a.tile_cbase[t] : -1;
                const unsigned c0 = p0 & ~7u;
                const void *csrc = cbase >= 0 ? (const void *)(a.col16 + c0) : (const void *)(a.col + a0);
                const unsigned cbytes = cbase >= 0 ? (((p1 + 7u) & ~7u) - c0) * 2u : cnt * 4u;
                unsigned char *st = dyn_smem + (size_t)s * stage_bytes;
                double   *sval = reinterpret_cast<double *>(st);
                unsigned *scol = reinterpret_cast<unsigned *>(sval + cap);
                unsigned *sptr = scol + cap;
                sh.hdr[s] = StageHdr{row0, row1, a0, rowa, p0 - a0, p1 - a0, a.tile_flag ? a.tile_flag[t] : 0, cbase};
                const unsigned bar = smem_u32(&sh.full_bar[s]);
                mbar_arrive_expect_tx(bar, cnt * 8u + cbytes + (unsigned)cntp * 4u);
                if (cnt) {
                    if (hint) {
                        tma_load_1d_hint(smem_u32(sval), a.val + a0, cnt * 8u, bar, pol);
                        tma_load_1d_hint(smem_u32(scol), csrc, cbytes, bar, pol);
                    } else {
                        tma_load_1d(smem_u32(sval), a.val + a0, cnt * 8u, bar);
                        tma_load_1d(smem_u32(scol), csrc, cbytes, bar);
                    }
                }
                tma_load_1d(smem_u32(sptr), a.ptr + rowa, (unsigned)cntp * 4u, bar);
            }
            // drain: bulk copies already issued must land before the CTA may retire its shared memory
            const unsigned consumed = (unsigned)flags[2];
            for (unsigned w = consumed; w < v; ++w)
                mbar_wait(smem_u32(&sh.full_bar[w % (unsigned)stages]), (w / (unsigned)stages) & 1u);
        }
    } else {
        // ============================ consumer warps: the solver ============================================
        M m(a, sh);
        m.dyn = dyn_smem; m.tid = tid; m.lane = tid & 31; m.my_tiles = my_tiles; m.vis = 0u; m.stage_bytes = stage_bytes;
        m.row_lo = a.tile_row[t0]; m.row_hi = a.tile_row[t1];
        m.trace_it = 0;
        m.trace_who = blockIdx.x == 0 ? 0 : (blockIdx.x == gridDim.x / 2 ? 1 : -1);
        // counters left by the previous solve; nobody advances them before every CTA has passed its first arrive
        m.gen = a.sync->st.gen; m.red_epoch = a.sync->st.red_epoch; m.halo_epoch = a.sync->st.halo_epoch;
        m.posted_gen = m.gen;
        if (tid == 0) sh.sc = *a.sc;                  // the scalars the init kernels left (solver.c:74-83, 200-213)

        // which CTAs own the columns my rows gather, which ranks fill the ghost slots they gather
        const int4 dep = a.cta_dep[blockIdx.x];
        const int G = (int)gridDim.x;
        auto cta_of_row = [&](int r) {              // last CTA whose first row is <= r
            int lo = 0, hi = G;                     // first rows are non-decreasing; a.tile_row[a.cta_tile[G]] = rows
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (a.tile_row[a.cta_tile[mid]] <= r) lo = mid + 1; else hi = mid; }
            return lo - 1;
        };
        m.dep_lo = 1; m.dep_hi = 0;
        if (dep.x <= dep.y) { m.dep_lo = max(0, cta_of_row(dep.x)); m.dep_hi = min(G - 1, cta_of_row(dep.y)); }
        m.reads_ghost = a.comm.world > 1 && dep.z <= dep.w;
        m.ghost_lo = m.reads_ghost ? dep.z : 0; m.ghost_hi = m.reads_ghost ? dep.w + 1 : 0;
        // the reducer sits in the middle of the row range: on banded matrices the CTAs at the ends are busy pushing boundary
        // rows over NVLink (slow per SM) right before the reductions, and everybody would wait for them twice
        m.is_reducer = (int)blockIdx.x == G / 2;
        m.gs_lo = m.gs_hi = 0;
        if (a.comm.world > 1) {
            // ghost slots are shared out evenly (16-slot granules) over the CTAs
            const int ng = a.n_ghost;
            const int chunk = ((ng + G - 1) / G + 15) & ~15;
            m.gs_lo = min(ng, (int)blockIdx.x * chunk);
            m.gs_hi = min(ng, m.gs_lo + chunk);
        }
        m.push_slots = 0u;
        if (a.comm.world > 1) {
            PushDesc pd;
            pd.npeers = 1;
            for (int s = 0; s < a.push.npeers; ++s) {
                pd.runs[0] = a.push.runs[s]; pd.nruns[0] = a.push.nruns[s];
                if (m.row_hi > m.row_lo && push_touches(pd, m.row_lo, m.row_hi)) m.push_slots |= 1u << s;
            }
        }
        // resident mode: the slice goes into shared memory once (plain coalesced loads; the ring is not used by this CTA)
        m.rp = resident_plan(a, t0, t1, LANES);
        m.resident = m.rp.on;
        if (m.resident) {
            const size_t nnzp = ((size_t)m.rp.nnz + 7u) & ~(size_t)7u;
            double *sv = reinterpret_cast<double *>(dyn_smem);
            unsigned short *sc16 = reinterpret_cast<unsigned short *>(sv + nnzp);
            unsigned *sp = reinterpret_cast<unsigned *>(sc16 + nnzp);
            const int gh0 = a.ghost_off + (dep.z <= dep.w ? dep.z : 0);
            for (unsigned i = (unsigned)tid; i < m.rp.nnz; i += (unsigned)CT) {
                sv[i] = a.val[m.rp.nz_lo + i];
                const int cc = (int)a.col[m.rp.nz_lo + i];
                sc16[i] = (unsigned short)(cc < a.ghost_off ? cc - m.rp.obase : cc - gh0 + (int)m.rp.ospan);
            }
            for (int r = tid; r <= m.rp.rows; r += CT) sp[r] = a.ptr[m.rp.row_lo + r] - m.rp.nz_lo;
            m.rs_val = sv; m.rs_col = sc16; m.rs_ptr = sp;
            if (tid == 0) atomicAdd(&a.sync->st.resident_ctas, 1);
        }
        nbar(1, CT);
        if (a.comm.world > 1 && (m.reads_ghost || m.gs_hi > m.gs_lo)) {
            // the vectors the first phases read were pushed by the init kernels (kernel-per-phase protocol)
            if (tid < 32 && !halo_wait(a.comm, sh.sc.halo_epoch) && tid == 0) { sh.sc.error = 1; sh.sc.done = 1; }
            if (tid < 32) fence_sys();
            nbar(1, CT);
        }
        if (!m.stop_now()) {                                             // solver.c:86 before the first pass
            if (a.method == 0) { if (a.comm.world > 1) m.run_bicgstab_multi(); else m.run_bicgstab(); }
            else if (a.method == 1) m.run_ca();
            else m.run_pipe(a.method == 3);
        }
        nbar(1, CT);
        if (tid == 0) {
            sh.flags[2] = (int)m.vis; __threadfence_block(); sh.flags[1] = 1;
            if (blockIdx.x == 0) {
                *a.sc = sh.sc;
                a.sync->st.gen = m.gen; a.sync->st.red_epoch = m.red_epoch; a.sync->st.halo_epoch = m.halo_epoch;
            } else if (sh.sc.error) a.sc->error = 1;
        }
    }
}

// per-CTA column ranges: min / max own column and min / max ghost slot over the CTA's entries
__global__ void __launch_bounds__(256) mega_dep_kernel(const unsigned *__restrict__ col, const unsigned *__restrict__ ptr,
                                                       const int *__restrict__ tile_row, const int *__restrict__ cta_tile,
                                                       int ghost_off, int4 *dep)
{
    __shared__ int s[4];
    if (threadIdx.x == 0) { s[0] = 0x7fffffff; s[1] = -1; s[2] = 0x7fffffff; s[3] = -1; }
    __syncthreads();
    const int r0 = tile_row[cta_tile[blockIdx.x]], r1 = tile_row[cta_tile[blockIdx.x + 1]];
    int omin = 0x7fffffff, omax = -1, gmin = 0x7fffffff, gmax = -1;
    if (r1 > r0) {
        const unsigned e0 = ptr[r0], e1 = ptr[r1];
        for (unsigned j = e0 + threadIdx.x; j < e1; j += blockDim.x) {
            const int c = (int)col[j];
            if (c < ghost_off) { omin = min(omin, c); omax = max(omax, c); }
            else { gmin = min(gmin, c - ghost_off); gmax = max(gmax, c - ghost_off); }
        }
    }
    atomicMin(&s[0], omin); atomicMax(&s[1], omax); atomicMin(&s[2], gmin); atomicMax(&s[3], gmax);
    __syncthreads();
    if (threadIdx.x == 0) dep[blockIdx.x] = make_int4(s[0], s[1], s[2], s[3]);
}

// one CTA per tile: column base of a narrow tile, -1 for a wide one (see launch_mega_tile_base)
__global__ void __launch_bounds__(256) mega_tile_base_kernel(const unsigned *__restrict__ col, const unsigned *__restrict__ tile_nz,
                                                             const int *__restrict__ tile_flag, int ghost_off, int *tile_cbase,
                                                             int *narrow_count)
{
    __shared__ int s[2];
    if (threadIdx.x == 0) { s[0] = 0x7fffffff; s[1] = -1; }
    __syncthreads();
    const int t = blockIdx.x;
    const unsigned p0 = tile_nz[t], p1 = tile_nz[t + 1];
    int lo = 0x7fffffff, hi = -1;
    for (unsigned j = p0 + threadIdx.x; j < p1; j += blockDim.x) {
        const int c = (int)col[j];
        lo = min(lo, c); hi = max(hi, c);
    }
    atomicMin(&s[0], lo); atomicMax(&s[1], hi);
    __syncthreads();
    if (threadIdx.x == 0) {
        const bool narrow = (tile_flag == nullptr || tile_flag[t] == 0) && p1 > p0 && s[1] < ghost_off && s[1] - s[0] < 65536;
        tile_cbase[t] = narrow ? s[0] : -1;
        if (narrow) atomicAdd(narrow_count, 1);
    }
}

__global__ void __launch_bounds__(256) mega_tile_codes_kernel(const unsigned *__restrict__ col, const unsigned *__restrict__ tile_nz,
                                                              const int *__restrict__ tile_cbase, unsigned short *__restrict__ col16)
{
    const int t = blockIdx.x;
    const int base = tile_cbase[t];
    if (base < 0) return;
    for (unsigned j = tile_nz[t] + threadIdx.x; j < tile_nz[t + 1]; j += blockDim.x) col16[j] = (unsigned short)((int)col[j] - base);
}

template <int CT, int LANES>
cudaError_t launch(const MegaArgs &a, int grid, size_t smem, cudaStream_t st)
{
    void *params[1] = {(void *)&a};
    return cudaLaunchCooperativeKernel((const void *)bicg_mega_kernel<CT, LANES>, dim3(grid), dim3(CT + 32), params, smem, st);
}
template <int CT, int LANES>
cudaError_t set_attr()
{
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, bicg_mega_kernel<CT, LANES>);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(bicg_mega_kernel<CT, LANES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                227 * 1024 - (int)fa.sharedSizeBytes);
}

} // namespace

size_t mega_smem_bytes(int cap, int stages, int threads, int lanes)
{
    return (size_t)stages * ((size_t)cap * 12u + (size_t)(threads / lanes + PROW_PAD) * 4u);
}

bool mega_has_variant(int threads, int lanes)
{
    if (threads == 256) return lanes == 1;
    return threads == 512 && (lanes == 1 || lanes == 4 || lanes == 8 || lanes == 32);
}

int mega_setup_attributes()
{
    cudaError_t e;
    if ((e = set_attr<256, 1>()) != cudaSuccess) return (int)e;
    if ((e = set_attr<512, 1>()) != cudaSuccess) return (int)e;
    if ((e = set_attr<512, 4>()) != cudaSuccess) return (int)e;
    if ((e = set_attr<512, 8>()) != cudaSuccess) return (int)e;
    if ((e = set_attr<512, 32>()) != cudaSuccess) return (int)e;
    return 0;
}

int launch_mega(int threads, int lanes, int grid, size_t smem, const MegaArgs &a, cudaStream_t st)
{
    if (threads == 256 && lanes == 1) return (int)launch<256, 1>(a, grid, smem, st);
    if (threads != 512) return (int)cudaErrorInvalidValue;
    switch (lanes) {
    case 1:  return (int)launch<512, 1>(a, grid, smem, st);
    case 4:  return (int)launch<512, 4>(a, grid, smem, st);
    case 8:  return (int)launch<512, 8>(a, grid, smem, st);
    case 32: return (int)launch<512, 32>(a, grid, smem, st);
    default: return (int)cudaErrorInvalidValue;
    }
}

void launch_mega_dep(const unsigned *col, const unsigned *ptr, const int *tile_row, const int *cta_tile, int grid,
                     int ghost_off, int4 *dep, cudaStream_t st)
{
    mega_dep_kernel<<<grid, 256, 0, st>>>(col, ptr, tile_row, cta_tile, ghost_off, dep);
}

void launch_mega_tile_base(const unsigned *col, const unsigned *tile_nz, const int *tile_flag, int ntiles, int ghost_off,
                           int *tile_cbase, int *narrow_count, cudaStream_t st)
{
    mega_tile_base_kernel<<<ntiles, 256, 0, st>>>(col, tile_nz, tile_flag, ghost_off, tile_cbase, narrow_count);
}

void launch_mega_tile_codes(const unsigned *col, const unsigned *tile_nz, const int *tile_cbase, int ntiles,
                            unsigned short *col16, cudaStream_t st)
{
    mega_tile_codes_kernel<<<ntiles, 256, 0, st>>>(col, tile_nz, tile_cbase, col16);
}

} // namespace bicg
