// solve.cu -- the four iteration loops of solver.c re-expressed as device-resident kernel sequences.
//
// The reference's host loop (solver.c:86-127 etc.) launches nothing but CPU loops and blocks on five to
// seven one-double MPI_Iallreduce/MPI_Wait pairs per iteration.  Here the host only *enqueues*: every
// scalar (alpha, beta, omega, the dot products, k, the loop test) lives in HBM, is produced by the tail of
// the kernel that reduces it and is read by the kernels that follow, so an iteration is a fixed list of 4-5
// kernel launches with no host round trip.  BICG_UNROLL iterations are captured once into a CUDA graph and
// replayed; when the device-side loop test fails it raises Scalars::done and all later kernels of a batch
// return immediately, so the iteration count is exact although the host looks at the flag only once per batch.
//
//   bicgstab       K1 SpMV s=Ap (+ (r#,s))  K2 q  K3 SpMV y=Aq (+ (q,y),(y,y))  K4 x,r (+ 2 dots)  K5 p
//   ca_bicgstab    C1 p,s  C2 SpMV z=As  C3 q,y (+ 2 dots)  C4 x,r (+ local (r,r))  C5 SpMV w=Ar (+ 4 dots, 5-value reduction)
//   pipe_bicgstab  P1 p,s,z,q,y (+ post 2 dots)  P2 SpMV v=Az (completes it)  P3 x,r,w (+ post 5 dots)  P4 SpMV t=Aw (completes it)
//   pipe_bicgstab_rr  = pipe, with the replacement iterations of solver.c:498-501, 522-527 as extra SpMVs
#include "engine.hpp"
#include "vec_body.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>

namespace bicg {

namespace {

__global__ void reset_state_kernel(Scalars *s, double tol, int max_iter)
{
    s->rTr = s->rTr_old = s->rTs = s->rTy = s->yTy = s->rTw = s->wTw = s->rTz = 0.0;
    s->dot_r = s->dot_zero = 0.0;
    s->alpha = s->beta = s->omega = 0.0;
    s->tol2 = tol * tol;                   // solver.c:86  tol * tol * dot_zero
    for (int k = 0; k < MAX_DOTS; ++k) s->pend[k] = 0.0;
    s->k = 0; s->max_iter = max_iter; s->done = 0; s->converged = 0; s->error = 0; s->ticket = 0u;
    // red_epoch / red_done / halo_epoch are job-long sequence numbers and are NOT reset
}

__global__ void fill_kernel(double *p, int n, double v)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = v;
}

__global__ void set_coef_kernel(Scalars *s, double al, double be, double om) { s->alpha = al; s->beta = be; s->omega = om; }

inline TailDesc tail_none() { return TailDesc{TAIL_NONE, FIN_NONE, 0, 0, 0, 0, 0}; }
inline TailDesc tail_allreduce(int fin, int ndot, int npend = 0) { return TailDesc{TAIL_ALLREDUCE, fin, ndot, npend, 0, 0, 0}; }
inline TailDesc tail_post(int ndot) { return TailDesc{TAIL_POST, FIN_NONE, ndot, 0, 0, 0, 0}; }
inline TailDesc tail_complete(int fin, int nred) { return TailDesc{TAIL_COMPLETE, fin, 0, 0, 0, nred, 0}; }
inline TailDesc tail_pend(int ndot, int off) { return TailDesc{TAIL_PEND, FIN_NONE, ndot, 0, off, 0, 0}; }

struct Seq {
    bicg_matrix *m;
    Context &c;
    int launches = 0;

    explicit Seq(bicg_matrix *mm) : m(mm), c(ctx()) {}

    VecPtrs ptrs() const
    {
        VecPtrs v;
        v.x = m->vec(V_X); v.r = m->vec(V_R); v.rh = m->vec(V_RH); v.p = m->vec(V_P); v.s = m->vec(V_S);
        v.y = m->vec(V_Y); v.z = m->vec(V_Z); v.w = m->vec(V_W); v.v = m->vec(V_V); v.t = m->vec(V_T);
        v.b = m->vec(V_B); v.ax = m->vec(V_AX);
        return v;
    }

    // where the runs of vector `id` that peers need go: their ghost slots, addressed through the IPC mappings
    PushDesc make_push(int id) const
    {
        PushDesc pd{};
        if (m->world == 1) return pd;
        pd.npeers = m->npush;
        pd.fence_writers = c.cfg.fence_writers;
        pd.src = m->vec(id);
        for (int s = 0; s < m->npush; ++s) {
            const int d = m->push_peer[s];
            pd.dst[s] = (double *)((char *)m->peer_base[d] + m->peer_vec_off[d]) + (long long)id * m->peer_vstride[d] +
                        m->peer_ghost_off[d];
            pd.runs[s] = m->d_push_runs[s];
            pd.nruns[s] = m->push_nruns[s];
        }
        return pd;
    }

    // the persistent kernel runs the whole loop (mega.cu); false: it could not be launched
    bool mega(int method, int krr, int nrr)
    {
        MegaArgs a{};
        a.sc = m->d_sc; a.hist = m->d_hist; a.comm = m->comm; a.sync = m->d_msync;
        for (int p = 0; p < MAX_RANKS; ++p) a.peer_mail[p] = &m->peer_msync[p]->mail[0][0];
        a.n_ghost = m->n_ghost; a.cta_dep = m->mega.d_cta_dep;
        a.val = m->d_val; a.col = m->d_col; a.ptr = m->d_ptr;
        a.tile_row = m->mega.d_tile_row; a.tile_nz = m->mega.d_tile_nz; a.cta_tile = m->mega.d_cta_tile;
        a.tile_flag = m->mega.d_tile_flag;
        a.tile_cbase = m->mega.d_tile_cbase; a.col16 = m->mega.d_col16;
        a.cap = m->mega.cap; a.stages = m->mega.stages;
        a.ghost_off = m->ghost_off; a.l2_hint = c.cfg.l2_hint;
        a.gather_cg = c.cfg.gather_cg >= 0 ? c.cfg.gather_cg : 0;
        size_t smem = m->mega.smem;
        a.resident = (c.cfg.resident && m->mega.res_smem) ? 1 : 0;
        if (a.resident) smem = std::max(smem, m->mega.res_smem);
        a.smem_bytes = (int)smem;
        a.vec_base = m->vec_base; a.vstride = m->vstride;
        a.v = ptrs();
        a.push.npeers = m->world > 1 ? m->npush : 0;
        for (int s = 0; s < a.push.npeers; ++s) {
            const int d = m->push_peer[s];
            a.push.peer[s] = d;
            a.push.runs[s] = m->d_push_runs[s];
            a.push.nruns[s] = m->push_nruns[s];
            a.push.ll_dst[s] = m->peer_ll[d];
            a.push.ll_stride[s] = m->peer_ll_stride[d];
        }
        a.ll = m->d_ll; a.ll_stride = m->ll_stride;
        a.method = method; a.krr = krr; a.nrr = nrr;
        a.trace = m->d_trace;
        a.snap = m->d_trace ? m->d_trace + (size_t)2 * MEGA_TRACE_ITERS * MEGA_TRACE_SLOTS : nullptr;
        a.snap_iter = 50;
        BICG_CUDA(cudaMemsetAsync(&m->d_msync->st.resident_ctas, 0, sizeof(int), c.stream));
        int rc = launch_mega(m->mega.threads, m->mega.lanes, m->mega.grid, smem, a, c.stream);
        if (rc) {
            // e.g. the grid cannot be co-resident because something else holds SMs.  Single rank: not an error, the
            // kernel-per-phase path below does the same job.  With peers the ranks must agree on the loop
            // implementation (its synchronisation protocol), so a local failure is fatal.
            (void)cudaGetLastError();
            if (m->world > 1) fatal("bicgstab_b200: rank %d could not launch the persistent kernel: %s", m->rank,
                                    cudaGetErrorString((cudaError_t)rc));
            if (c.cfg.verbose) fprintf(stderr, "[bicg] persistent kernel not launched (%s); using the per-phase kernels\n",
                                       cudaGetErrorString((cudaError_t)rc));
            m->mega.ok = false;
            return false;
        }
        ++launches; ++c.launches;
        return true;
    }

    // one fused vector kernel; push_vec >= 0: that vector is the next SpMV's input
    void vec(int phase, TailDesc tail, int push_vec = -1)
    {
        VecArgs a{};
        a.kc.sc = m->d_sc; a.kc.partials = m->d_partials; a.kc.hist = m->d_hist; a.kc.comm = m->comm;
        a.kc.tail = tail;
        a.v = ptrs(); a.n = m->n_loc; a.chunk = m->vchunk;
        a.push.npeers = 0; a.push.src = nullptr;
        if (push_vec >= 0 && m->world > 1) {
            a.kc.tail.signal_halo = 1;               // every rank advances its halo epoch, senders also signal
            a.push = make_push(push_vec);
        } else if (phase == PH_PUSH) {
            return;                                   // single rank: nothing to exchange
        }
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (c.prof_on) { BICG_CUDA(cudaEventCreate(&e0)); BICG_CUDA(cudaEventCreate(&e1)); BICG_CUDA(cudaEventRecord(e0, c.stream)); }
        int rc = launch_vec(phase, m->vgrid, a, c.stream);
        if (rc) fatal("bicgstab_b200: vector kernel launch failed (phase %d): %s", phase, cudaGetErrorString((cudaError_t)rc));
        if (c.prof_on) {
            BICG_CUDA(cudaEventRecord(e1, c.stream));
            c.prof_ev.push_back(e0); c.prof_ev.push_back(e1); c.prof_class.push_back(phase == PH_PUSH ? 2 : 1);
        }
        ++launches; ++c.launches;
    }

    void spmv(int x_id, int y_id, TailDesc tail, int ndot = 0, const double *a0 = nullptr, const double *b0 = nullptr,
              const double *a1 = nullptr, const double *b1 = nullptr, const double *a2 = nullptr, const double *b2 = nullptr,
              const double *a3 = nullptr, const double *b3 = nullptr)
    {
        SpmvArgs a = make_spmv_args(m, m->plan, x_id, y_id);
        a.kc.tail = tail;
        const double *as[4] = {a0, a1, a2, a3}, *bs[4] = {b0, b1, b2, b3};
        for (int k = 0; k < ndot; ++k) epi_add_dot(a.epi, as[k], bs[k]);
        launch_spmv_plan(m, m->plan, a, 0);
        ++launches;
    }

    // ---- solver.c:74-83 --------------------------------------------------------------------------------
    void bicgstab_init()
    {
        vec(PH_PUSH, tail_none(), V_X);
        spmv(V_X, V_AX, tail_none());                                            // Ax = A x0
        vec(PH_BICG_INIT, tail_allreduce(FIN_BICG_INIT, 1), V_P);                // r, r#, p, (r,r)
        // several GPUs, persistent kernel: it keeps ghost copies of r and p up to date itself (mega.cu: run_bicgstab_multi)
        // and therefore starts from the ghost values of r0 as well (p0 = r0 was pushed just now)
        if (m->world > 1 && c.cfg.mega && m->mega.ok && !c.prof_on) vec(PH_PUSH, tail_none(), V_R);
    }
    // ---- solver.c:88-120 -------------------------------------------------------------------------------
    void bicgstab_iter()
    {
        const double *Y = nullptr;   // "the y this SpMV just produced"
        spmv(V_P, V_S, tail_allreduce(FIN_BICG_ALPHA, 1), 1, m->vec(V_RH), Y);                    // s = A p, (r#,s)
        vec(PH_BICG_Q, tail_none(), V_R);                                                         // q = r - alpha s
        spmv(V_R, V_Y, tail_allreduce(FIN_BICG_OMEGA, 2), 2, m->vec(V_R), Y, Y, Y);               // y = A q, (q,y), (y,y)
        vec(PH_BICG_XR, tail_allreduce(FIN_BICG_BETA, 2));                                        // x, r, (r,r), (r#,r)
        vec(PH_BICG_P, tail_none(), V_P);                                                         // p
    }

    // ---- solver.c:200-213 / 333-347 ----------------------------------------------------------------------
    void capipe_init(bool pipe)
    {
        vec(PH_PUSH, tail_none(), V_X);
        spmv(V_X, V_AX, tail_none());
        vec(PH_INIT_R, tail_allreduce(FIN_STORE_RTR, 1), V_R);                                    // r, r#, (r,r)
        spmv(V_R, V_W, tail_allreduce(FIN_CAPIPE_INIT, 1), 1, m->vec(V_R), nullptr);              // w = A r, (r,w)
        if (pipe) {
            vec(PH_PUSH, tail_none(), V_W);
            spmv(V_W, V_T, tail_none());                                                          // t = A w
        }
    }
    // ---- solver.c:217-253 --------------------------------------------------------------------------------
    void ca_iter()
    {
        const double *Y = nullptr;
        vec(PH_CA_PS, tail_none(), V_S);                                                          // p, s
        spmv(V_S, V_Z, tail_none());                                                              // z = A s
        vec(PH_QY, tail_allreduce(FIN_OMEGA2, 2));                                                // q, y, (q,y), (y,y)
        vec(PH_CA_XR, tail_pend(1, 0), V_R);                                                      // x, r, local (r,r)
        spmv(V_R, V_W, tail_allreduce(FIN_CAPIPE_END, 4, 1), 4,                                   // w = A r
             m->vec(V_RH), m->vec(V_R), m->vec(V_RH), Y, m->vec(V_RH), m->vec(V_S), m->vec(V_RH), m->vec(V_Z));
    }
    // ---- solver.c:352-388 --------------------------------------------------------------------------------
    void pipe_iter()
    {
        vec(PH_PIPE_1, tail_post(2), V_Z);                                                        // post (q,y),(y,y)
        spmv(V_Z, V_V, tail_complete(FIN_OMEGA2, 2));                                             // v = A z hides it
        vec(PH_PIPE_3, tail_post(5), V_W);                                                        // post 5 dots
        spmv(V_W, V_T, tail_complete(FIN_CAPIPE_END, 5));                                         // t = A w hides it
    }
    // ---- solver.c:494-547, replacement branch ----------------------------------------------------------
    void rr_replace_iter()
    {
        vec(PH_RR_P, tail_none(), V_P);
        spmv(V_P, V_S, tail_none());                                                              // s = A p   :499
        vec(PH_PUSH, tail_none(), V_S);
        spmv(V_S, V_Z, tail_none());                                                              // z = A s   :500
        vec(PH_QY, tail_post(2), V_Z);
        spmv(V_Z, V_V, tail_complete(FIN_OMEGA2, 2));                                             // v = A z
        vec(PH_RR_X, tail_none(), V_X);
        spmv(V_X, V_AX, tail_none());                                                             // Ax        :523
        vec(PH_RR_R, tail_none(), V_R);                                                           // r = b - Ax :524-525
        spmv(V_R, V_W, tail_none());                                                              // w = A r   :526
        vec(PH_RR_DOTS, tail_post(5), V_W);
        spmv(V_W, V_T, tail_complete(FIN_CAPIPE_END, 5));                                         // t = A w
    }
};

int kernels_per_iter(int method, int world)
{
    (void)world;
    switch (method) {
    case BICG_METHOD_BICGSTAB: return 5;
    case BICG_METHOD_CA: return 5;
    default: return 4;
    }
}

void ensure_graph(bicg_matrix *m, int method, int unroll)
{
    Context &c = ctx();
    if (m->graph[method] && m->graph_unroll[method] == unroll) return;
    if (m->graph[method]) { cudaGraphExecDestroy(m->graph[method]); m->graph[method] = nullptr; }
    cudaGraph_t g = nullptr;
    BICG_CUDA(cudaStreamBeginCapture(c.stream, cudaStreamCaptureModeThreadLocal));
    Seq s(m);
    for (int u = 0; u < unroll; ++u) {
        if (method == BICG_METHOD_BICGSTAB) s.bicgstab_iter();
        else if (method == BICG_METHOD_CA) s.ca_iter();
        else s.pipe_iter();
    }
    BICG_CUDA(cudaStreamEndCapture(c.stream, &g));
    BICG_CUDA(cudaGraphInstantiate(&m->graph[method], g, 0));
    BICG_CUDA(cudaGraphDestroy(g));
    m->graph_unroll[method] = unroll;
    c.launches -= s.launches;       // capture is not execution
}

} // namespace

void print_reference_lines(const bicg_stats &st, const std::vector<double> &hist)
{
    const Context &c = ctx();
    if (c.rank != 0 || c.cfg.quiet) return;
    const int out = std::max(1, c.cfg.out_iter);
    for (int k = out; k <= st.iters && k < (int)hist.size(); k += out)
        printf("Iteration: %d, Residual: %e\n", k, sqrt(hist[(size_t)k]));                  // solver.c:124
    const double t = st.loop_ms * 1e-3;
    printf("Total iter   : %d\n", st.iters);                                                // solver.c:135
    printf("Final r      : %e\n", st.final_res);                                            // solver.c:136
    printf("Total time   : %e [sec.] \n", t);                                               // solver.c:138
    printf("Avg time/iter: %e [sec.] \n", t / st.iters);                                    // solver.c:139
    fflush(stdout);
}

int solve(bicg_matrix *m, int method, double *x, double *r, int krr, int nrr, int device_vectors, bicg_stats *out)
{
    Context &c = ctx();
    c.ensure();
    if (method < 0 || method > 3) return -1;
    if (method == BICG_METHOD_PIPE_RR && krr <= 0) method = BICG_METHOD_PIPE;
    const Config &cfg = c.cfg;
    const int max_iter = cfg.max_iter;
    if (max_iter + 2 > m->hist_cap) {
        // BICG_MAX_ITER was raised after the handle was created: move the history out of the arena and
        // drop the captured graphs (their kernel arguments hold the old pointer)
        BICG_CUDA(cudaStreamSynchronize(c.stream));
        if (m->hist_extra) cudaFree(m->hist_extra);
        BICG_CUDA(cudaMalloc((void **)&m->hist_extra, ((size_t)max_iter + 2) * sizeof(double)));
        m->d_hist = m->hist_extra; m->hist_cap = max_iter + 2;
        for (int g = 0; g < 4; ++g) if (m->graph[g]) { cudaGraphExecDestroy(m->graph[g]); m->graph[g] = nullptr; }
    }
    const size_t vbytes = (size_t)m->n_loc * sizeof(double);
    const cudaMemcpyKind in_kind = device_vectors ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    const cudaMemcpyKind out_kind = device_vectors ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;

    cudaEvent_t e_in0, e_in1, e_loop1, e_out1;
    BICG_CUDA(cudaEventCreate(&e_in0)); BICG_CUDA(cudaEventCreate(&e_in1));
    BICG_CUDA(cudaEventCreate(&e_loop1)); BICG_CUDA(cudaEventCreate(&e_out1));

    // ---- inputs (outside the reference's timed region, solver.c:61-71) ---------------------------------
    BICG_CUDA(cudaEventRecord(e_in0, c.stream));
    BICG_CUDA(cudaMemcpyAsync(m->vec(V_X), x, vbytes, in_kind, c.stream));
    BICG_CUDA(cudaMemcpyAsync(m->vec(V_R), r, vbytes, in_kind, c.stream));
    reset_state_kernel<<<1, 1, 0, c.stream>>>(m->d_sc, cfg.tol, max_iter);
    if (method != BICG_METHOD_BICGSTAB) {
        // p, s, z, v, t start at zero: the defined version of the reference's uninitialised reads (SURVEY 5)
        const int zero_ids[5] = {(int)V_P, (int)V_S, (int)V_Z, (int)V_V, (int)V_T};
        for (int id : zero_ids)
            BICG_CUDA(cudaMemsetAsync(m->vec(id), 0, (size_t)m->ghost_off * sizeof(double), c.stream));   // own part only:
            // the ghost tail belongs to the peers, who may already be pushing into it
    }
    if (method == BICG_METHOD_PIPE_RR)
        BICG_CUDA(cudaMemcpyAsync(m->vec(V_B), m->vec(V_R), vbytes, cudaMemcpyDeviceToDevice, c.stream));   // solver.c:475
    BICG_CUDA(cudaEventRecord(e_in1, c.stream));

    // ---- the reference's timed region a14 (solver.c:69-132) ------------------------------------------------
    const int launches0 = c.launches;
    Seq seq(m);
    if (method == BICG_METHOD_BICGSTAB) seq.bicgstab_init();
    else seq.capipe_init(method != BICG_METHOD_CA);

    bool use_mega = cfg.mega && m->mega.ok && !c.prof_on;
    if (use_mega) use_mega = seq.mega(method, krr, nrr);
    const bool use_graph = cfg.graph && !c.prof_on && method != BICG_METHOD_PIPE_RR;   // replacement iterations are host-scheduled
    const int U = std::max(1, cfg.unroll);
    const int batches = (max_iter + U - 1) / U;
    const int DEPTH = 3, RING = 64;
    std::vector<cudaEvent_t> ring((size_t)RING, nullptr);
    if (use_graph && !use_mega) ensure_graph(m, method, U);
    int launched_batches = 0;
    for (int b = 0; b < batches && !use_mega; ++b) {
        if (b >= DEPTH) {
            const int o = (b - DEPTH) % RING;
            BICG_CUDA(cudaEventSynchronize(ring[(size_t)o]));
            if (c.h_flags[o * 4 + 2]) break;                     // done was raised in batch b - DEPTH
        }
        if (use_graph) {
            BICG_CUDA(cudaGraphLaunch(m->graph[method], c.stream));
            c.launches += U * kernels_per_iter(method, m->world);
        } else {
            for (int u = 0; u < U; ++u) {
                const int k = b * U + u;
                if (k >= max_iter) break;
                if (method == BICG_METHOD_BICGSTAB) seq.bicgstab_iter();
                else if (method == BICG_METHOD_CA) seq.ca_iter();
                else if (method == BICG_METHOD_PIPE) seq.pipe_iter();
                else {
                    const bool replace = (k % krr == 0) && k > 0 && k <= krr * nrr;       // solver.c:498, 522
                    if (replace) seq.rr_replace_iter(); else seq.pipe_iter();
                }
            }
        }
        const int o = b % RING;
        BICG_CUDA(cudaMemcpyAsync(&c.h_flags[o * 4], &m->d_sc->k, 4 * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        if (!ring[(size_t)o]) BICG_CUDA(cudaEventCreateWithFlags(&ring[(size_t)o], cudaEventDisableTiming));
        BICG_CUDA(cudaEventRecord(ring[(size_t)o], c.stream));
        ++launched_batches;
    }
    BICG_CUDA(cudaEventRecord(e_loop1, c.stream));

    // ---- outputs ---------------------------------------------------------------------------------------
    BICG_CUDA(cudaMemcpyAsync(x, m->vec(V_X), vbytes, out_kind, c.stream));
    BICG_CUDA(cudaMemcpyAsync(r, m->vec(V_R), vbytes, out_kind, c.stream));
    BICG_CUDA(cudaEventRecord(e_out1, c.stream));
    Scalars hs;
    BICG_CUDA(cudaMemcpyAsync(&hs, m->d_sc, sizeof(Scalars), cudaMemcpyDeviceToHost, c.stream));
    BICG_CUDA(cudaStreamSynchronize(c.stream));
    for (cudaEvent_t e : ring) if (e) cudaEventDestroy(e);
    (void)launched_batches;

    if (hs.error) fatal("bicgstab_b200: rank %d timed out after %d s waiting for a peer GPU / another CTA (halo flag or reduction "
                        "mailbox; BICG_PEER_TIMEOUT_S raises the bound)", m->rank, cfg.peer_timeout_s);
    if (m->d_trace && use_mega && method == BICG_METHOD_BICGSTAB) {
        // BICG_MEGA_TRACE=1: where CTA 0 and the middle CTA of the persistent kernel spent their time, averaged over the iterations
        const int iters = std::min(hs.k - 1, (int)MEGA_TRACE_ITERS);
        std::vector<unsigned long long> tr((size_t)2 * MEGA_TRACE_ITERS * MEGA_TRACE_SLOTS);
        BICG_CUDA(cudaMemcpy(tr.data(), m->d_trace, tr.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        static const char *names[10] = {"spmv s=Ap", "sync alpha", "vec q +push", "nbr/halo q", "spmv y=Aq", "sync omega",
                                        "vec x,r", "sync beta", "vec p +push", "nbr/halo p"};
        for (int who = 0; who < 2; ++who) {
            double sum[10] = {0};
            const size_t base = (size_t)who * MEGA_TRACE_ITERS * MEGA_TRACE_SLOTS;
            for (int it = 1; it < iters; ++it)
                for (int k = 0; k < 10; ++k)
                    sum[k] += (double)(tr[base + (size_t)it * MEGA_TRACE_SLOTS + k + 1] - tr[base + (size_t)it * MEGA_TRACE_SLOTS + k]);
            char line[1536]; int o = 0;
            o += snprintf(line + o, sizeof(line) - o, "[bicg mega trace r%d] us per iteration (CTA %s):", m->rank, who ? "mid" : "0");
            double tot = 0;
            for (int k = 0; k < 10; ++k) { o += snprintf(line + o, sizeof(line) - o, " %s %.2f |", names[k], sum[k] / std::max(1, iters - 1) * 1e-3); tot += sum[k]; }
            o += snprintf(line + o, sizeof(line) - o, " total %.2f", tot / std::max(1, iters - 1) * 1e-3);
            // inside the alpha sync point: arrive (CTA sum + release fence + slot store) | all local slots seen | posted to the
            // peers' mailboxes (reducer = middle CTA, N > 1) | every rank's sums seen
            double sub[4] = {0};
            const int mk[5] = {1, 11, 12, 13, 14};
            for (int it = 1; it < iters; ++it) {
                unsigned long long prev = tr[base + (size_t)it * MEGA_TRACE_SLOTS + mk[0]];
                for (int k = 1; k < 5; ++k) {
                    const unsigned long long t = tr[base + (size_t)it * MEGA_TRACE_SLOTS + mk[k]];
                    if (t) { sub[k - 1] += (double)(t - prev); prev = t; }
                }
            }
            snprintf(line + o, sizeof(line) - o, " || alpha sync: arrive %.2f local %.2f post %.2f mail %.2f\n", sub[0] / std::max(1, iters - 1) * 1e-3,
                     sub[1] / std::max(1, iters - 1) * 1e-3, sub[2] / std::max(1, iters - 1) * 1e-3, sub[3] / std::max(1, iters - 1) * 1e-3);
            fputs(line, stderr);
        }
        {   // the alpha sync of iteration 50 as every CTA saw it: spread of the arrivals, and how long after the LAST arrival
            // (this GPU's) the CTAs were released
            std::vector<unsigned long long> sn((size_t)2 * MEGA_MAX_CTAS);
            BICG_CUDA(cudaMemcpy(sn.data(), m->d_trace + (size_t)2 * MEGA_TRACE_ITERS * MEGA_TRACE_SLOTS, sn.size() * sizeof(unsigned long long),
                                 cudaMemcpyDeviceToHost));
            unsigned long long a_min = ~0ull, a_max = 0, r_min = ~0ull, r_max = 0; int last = -1;
            for (int g = 0; g < m->mega.grid; ++g) {
                if (!sn[2 * (size_t)g]) continue;
                if (sn[2 * (size_t)g] > a_max) { a_max = sn[2 * (size_t)g]; last = g; }
                a_min = std::min(a_min, sn[2 * (size_t)g]);
                r_min = std::min(r_min, sn[2 * (size_t)g + 1]); r_max = std::max(r_max, sn[2 * (size_t)g + 1]);
            }
            if (last >= 0)
                fprintf(stderr, "[bicg mega snap r%d] alpha sync @ iteration 50: arrivals spread %.2f us (last: CTA %d), first release %.2f us / last release "
                                "%.2f us after the last local arrival\n", m->rank, (double)(a_max - a_min) * 1e-3, last,
                        ((double)r_min - (double)a_max) * 1e-3, ((double)r_max - (double)a_max) * 1e-3);
        }
    }

    bicg_stats st{};
    st.iters = hs.k;
    st.converged = hs.converged;
    st.final_res = sqrt(hs.dot_r / hs.dot_zero);
    float ms = 0.f;
    BICG_CUDA(cudaEventElapsedTime(&ms, e_in1, e_loop1)); st.loop_ms = ms;
    BICG_CUDA(cudaEventElapsedTime(&ms, e_in0, e_in1));   st.h2d_ms = ms;
    BICG_CUDA(cudaEventElapsedTime(&ms, e_loop1, e_out1)); st.d2h_ms = ms;
    st.h2d_bytes = device_vectors ? 0 : 2 * vbytes;
    st.d2h_bytes = device_vectors ? 0 : 2 * vbytes;
    st.kernel_launches = c.launches - launches0;
    st.spmv_lanes = m->plan.lanes; st.spmv_kind = m->plan.kind;
    cudaEventDestroy(e_in0); cudaEventDestroy(e_in1); cudaEventDestroy(e_loop1); cudaEventDestroy(e_out1);

    c.last_hist.assign((size_t)st.iters + 1, 0.0);
    BICG_CUDA(cudaMemcpy(c.last_hist.data(), m->d_hist, ((size_t)st.iters + 1) * sizeof(double), cudaMemcpyDeviceToHost));
    c.last_stats = st;
    if (out) *out = st;
    return st.iters;
}

// y_loc = A x_loc with host pointers (the kernel behind MPI_csr_spmv_ovlap, matrix.c:428-441)
int spmv_host(bicg_matrix *m, const double *x_loc, double *y_loc, double *x_full)
{
    Context &c = ctx();
    c.ensure();
    const size_t vbytes = (size_t)m->n_loc * sizeof(double);
    BICG_CUDA(cudaMemcpyAsync(m->vec(V_X), x_loc, vbytes, cudaMemcpyHostToDevice, c.stream));
    reset_state_kernel<<<1, 1, 0, c.stream>>>(m->d_sc, c.cfg.tol, c.cfg.max_iter);
    Seq seq(m);
    seq.vec(PH_PUSH, tail_none(), V_X);
    // With peers the SpMV ends in an (empty) cross-GPU reduction = a barrier: nobody may push the next x into a
    // neighbour's ghost slots while that neighbour is still gathering from them.  Inside the solvers the dot
    // reductions provide this ordering; a bare SpMV (main.c:113) needs it explicitly, like the collective
    // MPI_Iallgatherv it replaces (matrix.c:432).
    seq.spmv(V_X, V_AX, m->world > 1 ? tail_allreduce(FIN_NONE, 0) : tail_none());
    BICG_CUDA(cudaMemcpyAsync(y_loc, m->vec(V_AX), vbytes, cudaMemcpyDeviceToHost, c.stream));
    BICG_CUDA(cudaStreamSynchronize(c.stream));
    Scalars hs;
    BICG_CUDA(cudaMemcpy(&hs, m->d_sc, sizeof(Scalars), cudaMemcpyDeviceToHost));
    if (hs.error) fatal("bicgstab_b200: rank %d timed out waiting for a peer GPU during SpMV", m->rank);
    if (x_full) {
        // the reference leaves the gathered vector in the caller's scratch (matrix.c:432); we only ever hold
        // the own part plus the halo, so fill what we have: own rows, then the received ghost runs
        const int first = 0;
        (void)first;
        if (m->world == 1) memcpy(x_full, x_loc, vbytes);
        else {
            std::vector<double> ghost((size_t)std::max(1, m->n_ghost));
            BICG_CUDA(cudaMemcpy(ghost.data(), m->vec(V_X) + m->ghost_off, (size_t)m->n_ghost * sizeof(double), cudaMemcpyDeviceToHost));
            for (size_t i = 0; i + 3 < m->recv_runs.size(); i += 4)
                memcpy(x_full + m->recv_runs[i], ghost.data() + m->recv_runs[i + 3], (size_t)m->recv_runs[i + 1] * sizeof(double));
        }
    }
    return 0;
}

int spmv_time(bicg_matrix *m, int reps, double *ms_out, double *bytes_out)
{
    Context &c = ctx();
    c.ensure();
    reset_state_kernel<<<1, 1, 0, c.stream>>>(m->d_sc, c.cfg.tol, c.cfg.max_iter);
    fill_kernel<<<256, 256, 0, c.stream>>>(m->vec(V_P), (int)m->vstride, 1.0);
    fill_kernel<<<256, 256, 0, c.stream>>>(m->vec(V_RH), m->n_loc, 1.0);
    SpmvArgs a = make_spmv_args(m, m->plan, V_P, V_S);
    a.wait_halo = 0;
    epi_add_dot(a.epi, m->vec(V_RH), nullptr);
    a.kc.tail = tail_pend(1, 0);               // full in-kernel reduction of the dot, no peer traffic
    cudaEvent_t e0, e1;
    BICG_CUDA(cudaEventCreate(&e0)); BICG_CUDA(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) launch_spmv_plan(m, m->plan, a);
    BICG_CUDA(cudaEventRecord(e0, c.stream));
    for (int i = 0; i < reps; ++i) launch_spmv_plan(m, m->plan, a);
    BICG_CUDA(cudaEventRecord(e1, c.stream));
    BICG_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    BICG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (ms_out) *ms_out = (double)ms / reps;
    // SURVEY.md 8(d) phase P1: matrix 12 nnz + 4 n, x read 8 n, y write 8 n, r# read 8 n
    if (bytes_out) *bytes_out = 12.0 * (double)m->nnz + 28.0 * (double)m->n_loc;
    return 0;
}

} // namespace bicg

// ------------------------------------------------------------------------------------------------
// test hooks (K-level parity: single fused phases and epilogue dots on caller-supplied vectors; single rank)
// ------------------------------------------------------------------------------------------------
extern "C" int bicg_debug_vec_phase(bicg_matrix *m, int phase, const double coef[3], double *vecs, double dots[8])
{
    using namespace bicg;
    Context &c = ctx();
    c.ensure();
    if (m->world != 1 || phase < 0 || phase >= PH_PUSH) return -1;
    const size_t vb = (size_t)m->n_loc * sizeof(double);
    for (int id = 0; id < V_COUNT; ++id)
        BICG_CUDA(cudaMemcpyAsync(m->vec(id), vecs + (size_t)id * m->n_loc, vb, cudaMemcpyHostToDevice, c.stream));
    reset_state_kernel<<<1, 1, 0, c.stream>>>(m->d_sc, c.cfg.tol, c.cfg.max_iter);
    set_coef_kernel<<<1, 1, 0, c.stream>>>(m->d_sc, coef[0], coef[1], coef[2]);
    static const int ndots[PH_PUSH] = {phase_ndot(PH_BICG_INIT), phase_ndot(PH_BICG_Q), phase_ndot(PH_BICG_XR), phase_ndot(PH_BICG_P),
                                       phase_ndot(PH_INIT_R), phase_ndot(PH_CA_PS), phase_ndot(PH_QY), phase_ndot(PH_CA_XR),
                                       phase_ndot(PH_PIPE_1), phase_ndot(PH_PIPE_3), phase_ndot(PH_RR_P), phase_ndot(PH_RR_X),
                                       phase_ndot(PH_RR_R), phase_ndot(PH_RR_DOTS)};
    const int nd = ndots[phase];
    Seq seq(m);
    seq.vec(phase, nd > 0 ? tail_pend(nd, 0) : tail_none());
    for (int id = 0; id < V_COUNT; ++id)
        BICG_CUDA(cudaMemcpyAsync(vecs + (size_t)id * m->n_loc, m->vec(id), vb, cudaMemcpyDeviceToHost, c.stream));
    Scalars hs;
    BICG_CUDA(cudaMemcpyAsync(&hs, m->d_sc, sizeof(Scalars), cudaMemcpyDeviceToHost, c.stream));
    BICG_CUDA(cudaStreamSynchronize(c.stream));
    for (int k = 0; k < 8; ++k) dots[k] = k < nd ? hs.pend[k] : 0.0;
    return nd;
}

// y (arena vector V_S) = A x (V_P) with the solver's fused epilogue dots.  epi 1: (r#,y); 2: (r,y),(y,y); 3: (r#,r),(r#,y),(r#,s),(r#,z)
// with s, z read from V_S' = V_AX and V_Z (y itself goes to V_W for epi 3, as in ca_bicgstab).  vecs: V_COUNT x n_loc in/out.
extern "C" int bicg_debug_spmv_epi(bicg_matrix *m, int epi, double *vecs, double dots[8])
{
    using namespace bicg;
    Context &c = ctx();
    c.ensure();
    if (m->world != 1 || epi < 0 || epi > 3) return -1;
    const size_t vb = (size_t)m->n_loc * sizeof(double);
    for (int id = 0; id < V_COUNT; ++id)
        BICG_CUDA(cudaMemcpyAsync(m->vec(id), vecs + (size_t)id * m->n_loc, vb, cudaMemcpyHostToDevice, c.stream));
    reset_state_kernel<<<1, 1, 0, c.stream>>>(m->d_sc, c.cfg.tol, c.cfg.max_iter);
    Seq seq(m);
    const double *Y = nullptr;
    int nd = 0;
    if (epi == 0) seq.spmv(V_P, V_S, tail_none());
    else if (epi == 1) { nd = 1; seq.spmv(V_P, V_S, tail_pend(1, 0), 1, m->vec(V_RH), Y); }
    else if (epi == 2) { nd = 2; seq.spmv(V_P, V_S, tail_pend(2, 0), 2, m->vec(V_R), Y, Y, Y); }
    else { nd = 4; seq.spmv(V_P, V_W, tail_pend(4, 0), 4, m->vec(V_RH), m->vec(V_R), m->vec(V_RH), Y, m->vec(V_RH), m->vec(V_AX),
                            m->vec(V_RH), m->vec(V_Z)); }
    for (int id = 0; id < V_COUNT; ++id)
        BICG_CUDA(cudaMemcpyAsync(vecs + (size_t)id * m->n_loc, m->vec(id), vb, cudaMemcpyDeviceToHost, c.stream));
    Scalars hs;
    BICG_CUDA(cudaMemcpyAsync(&hs, m->d_sc, sizeof(Scalars), cudaMemcpyDeviceToHost, c.stream));
    BICG_CUDA(cudaStreamSynchronize(c.stream));
    for (int k = 0; k < 8; ++k) dots[k] = k < nd ? hs.pend[k] : 0.0;
    return nd;
}

// own part of arena vector `id` / the solver scalars as the last solve left them
extern "C" int bicg_debug_get_vec(bicg_matrix *m, int id, double *out)
{
    using namespace bicg;
    Context &c = ctx();
    c.ensure();
    if (id < 0 || id >= V_COUNT) return -1;
    BICG_CUDA(cudaMemcpyAsync(out, m->vec(id), (size_t)m->n_loc * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    BICG_CUDA(cudaStreamSynchronize(c.stream));
    return 0;
}
extern "C" int bicg_debug_get_scalars(bicg_matrix *m, double out[13])
{
    using namespace bicg;
    Context &c = ctx();
    c.ensure();
    Scalars hs;
    BICG_CUDA(cudaMemcpyAsync(&hs, m->d_sc, sizeof(Scalars), cudaMemcpyDeviceToHost, c.stream));
    BICG_CUDA(cudaStreamSynchronize(c.stream));
    const double v[13] = {hs.rTr, hs.rTr_old, hs.rTs, hs.rTy, hs.yTy, hs.rTw, hs.wTw, hs.rTz, hs.dot_r, hs.dot_zero, hs.alpha, hs.beta, hs.omega};
    for (int k = 0; k < 13; ++k) out[k] = v[k];
    return 0;
}

extern "C" int bicg_debug_resident_ctas(bicg_matrix *m)
{
    using namespace bicg;
    Context &c = ctx();
    c.ensure();
    int n = 0;
    BICG_CUDA(cudaMemcpyAsync(&n, &m->d_msync->st.resident_ctas, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    BICG_CUDA(cudaStreamSynchronize(c.stream));
    return n;
}

extern "C" int bicg_debug_mega_tiles(bicg_matrix *m, int *narrow)
{
    if (narrow) *narrow = m->mega.ok ? m->mega.narrow : 0;
    return m->mega.ok ? m->mega.ntiles : 0;
}

// ------------------------------------------------------------------------------------------------
// profile: one solve with plain stream launches, every launch bracketed by events
// ------------------------------------------------------------------------------------------------
extern "C" int bicg_profile_solve(bicg_matrix *m, int method, int iters, double class_ms[3], int class_launches[3])
{
    using namespace bicg;
    Context &c = ctx();
    c.ensure();
    Config saved = c.cfg;
    c.cfg.tol = 0.0; c.cfg.max_iter = iters; c.cfg.quiet = 1;
    if (iters + 2 > m->hist_cap) { c.cfg = saved; return -1; }
    std::vector<double> x((size_t)m->n_loc, 0.0), b((size_t)m->n_loc, 1.0);
    c.prof_on = true; c.prof_ev.clear(); c.prof_class.clear();
    solve(m, method, x.data(), b.data(), 0, 0, 0, nullptr);
    c.prof_on = false;
    for (int k = 0; k < 3; ++k) { class_ms[k] = 0.0; class_launches[k] = 0; }
    for (size_t i = 0; i < c.prof_class.size(); ++i) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, c.prof_ev[2 * i], c.prof_ev[2 * i + 1]);
        class_ms[c.prof_class[i]] += ms; class_launches[c.prof_class[i]] += 1;
        cudaEventDestroy(c.prof_ev[2 * i]); cudaEventDestroy(c.prof_ev[2 * i + 1]);
    }
    c.prof_ev.clear(); c.prof_class.clear();
    c.cfg = saved;
    return 0;
}
