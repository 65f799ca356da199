// matrix.cu -- process context, configuration, and the device-resident matrix:
//   * merge of the reference's diag / offd blocks (matrix.c:380-392) into one CSR over the extended local
//     column space [own columns | ghost columns], upload into padded HBM arrays;
//   * halo plan exchange between the ranks and the IPC-shared arena (vectors with ghost tails, reduction
//     mailboxes, halo flags) that the kernels address directly over NVLink;
//   * SpMV plan: tile plan for the TMA kernel, candidate configurations, on-device autotune.
#include "engine.hpp"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstring>
#include <ctime>
#include <thread>

namespace bicg {

void fatal(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vfprintf(stderr, fmt, ap);
    va_end(ap);
    fputc('\n', stderr);
    exit(1);                       // the reference's error convention (solver.c:43-46, matrix.c:281-288)
}

// ------------------------------------------------------------------------------------------------
// configuration
// ------------------------------------------------------------------------------------------------
int set_option(Config &c, const char *key, const char *value)
{
    std::string k(key);
    if (k.rfind("BICG_", 0) == 0) k = k.substr(5);
    auto as_int = [&] { return atoi(value); };
    if (k == "TOL") c.tol = atof(value);
    else if (k == "MAX_ITER") c.max_iter = as_int();
    else if (k == "OUT_ITER") c.out_iter = as_int();
    else if (k == "QUIET") c.quiet = as_int();
    else if (k == "SPMV") {
        std::string v(value);
        c.spmv_kind = (v == "tma") ? 0 : (v == "rowsplit") ? 1 : -1;
    }
    else if (k == "SPMV_LANES") c.spmv_lanes = as_int();
    else if (k == "SPMV_THREADS") c.spmv_threads = as_int();
    else if (k == "SPMV_STAGES") c.spmv_stages = as_int();
    else if (k == "SPMV_CTAS") c.spmv_ctas = as_int();
    else if (k == "AUTOTUNE") c.autotune = as_int();
    else if (k == "GRAPH") c.graph = as_int();
    else if (k == "UNROLL") c.unroll = std::max(1, as_int());
    else if (k == "CACHE") c.cache = as_int();
    else if (k == "MEGA") c.mega = as_int();
    else if (k == "MEGA_THREADS") c.mega_threads = as_int();
    else if (k == "MEGA_TRACE") c.mega_trace = as_int();
    else if (k == "MEGA_LANES") c.mega_lanes = as_int();
    else if (k == "L2_HINT") c.l2_hint = as_int();
    else if (k == "GATHER_CG") c.gather_cg = as_int();
    else if (k == "RESIDENT") c.resident = as_int();
    else if (k == "STAGE_UPLOAD") c.stage_upload = as_int();
    else if (k == "BOUNDARY_WEIGHT") c.boundary_weight = std::max(0, as_int());
    else if (k == "ROW_WEIGHT") c.row_weight = std::max(1, as_int());
    else if (k == "DEVICE") c.device = as_int();
    else if (k == "HALO_GAP") c.halo_gap = std::max(0, as_int());
    else if (k == "VERBOSE") c.verbose = as_int();
    else if (k == "PEER_TIMEOUT_S") c.peer_timeout_s = std::max(1, as_int());
    else if (k == "SHIFT_TOL") c.shift_tol = atof(value);
    else if (k == "SHIFT_MAX_ITER") c.shift_max_iter = std::max(1, as_int());
    else if (k == "FENCE_WRITERS") c.fence_writers = as_int();
    else return -1;
    return 0;
}

void load_config_from_env(Config &c)
{
    static const char *keys[] = {"BICG_TOL", "BICG_MAX_ITER", "BICG_OUT_ITER", "BICG_QUIET", "BICG_SPMV",
                                 "BICG_SPMV_LANES", "BICG_SPMV_THREADS", "BICG_SPMV_STAGES", "BICG_SPMV_CTAS",
                                 "BICG_AUTOTUNE", "BICG_GRAPH", "BICG_UNROLL", "BICG_CACHE", "BICG_MEGA", "BICG_MEGA_THREADS", "BICG_MEGA_TRACE", "BICG_MEGA_LANES", "BICG_L2_HINT", "BICG_GATHER_CG", "BICG_RESIDENT", "BICG_STAGE_UPLOAD", "BICG_BOUNDARY_WEIGHT", "BICG_ROW_WEIGHT", "BICG_DEVICE",
                                 "BICG_HALO_GAP", "BICG_VERBOSE", "BICG_PEER_TIMEOUT_S", "BICG_SHIFT_TOL", "BICG_SHIFT_MAX_ITER", "BICG_FENCE_WRITERS"};
    for (const char *k : keys)
        if (const char *v = getenv(k)) set_option(c, k, v);
}

Context &ctx()
{
    static Context *c = [] {
        Context *p = new Context();
        load_config_from_env(p->cfg);
        return p;
    }();
    return *c;
}

void Context::ensure()
{
    if (ready) return;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        fatal("bicgstab_b200: no usable CUDA device (%s). This library has no CPU path.",
              e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    int dev = cfg.device;
    if (dev < 0) {
        const char *lr = getenv("LOCAL_RANK");
        dev = lr ? atoi(lr) : 0;
    }
    if (dev >= ndev) {
        // two ranks on one GPU cannot both keep a cooperative one-CTA-per-SM kernel resident: refuse instead of wrapping
        if (world > 1) fatal("bicgstab_b200: rank %d wants device %d but only %d device(s) are visible (one rank per GPU)", rank, dev, ndev);
        dev = dev % ndev;
    }
    BICG_CUDA(cudaSetDevice(dev));
    device = dev;
    cudaDeviceProp prop;
    BICG_CUDA(cudaGetDeviceProperties(&prop, dev));
    sm_count = prop.multiProcessorCount;
    if (prop.major < 10)
        fatal("bicgstab_b200: device %d (%s, sm_%d%d) is not a Blackwell GPU; this library ships sm_100a code only",
              dev, prop.name, prop.major, prop.minor);
    BICG_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    int rc = spmv_setup_attributes();
    if (rc == 0) rc = mega_setup_attributes();
    if (rc != 0) fatal("bicgstab_b200: cudaFuncSetAttribute failed: %s", cudaGetErrorString((cudaError_t)rc));
    BICG_CUDA(cudaHostAlloc((void **)&h_flags, 64 * 4 * sizeof(int), cudaHostAllocDefault));
    ready = true;
}

void Context::dev_free_after(std::initializer_list<void *> ptrs, cudaEvent_t ev)
{
    deferred.push_back(Deferred{ev, std::vector<void *>(ptrs)});
}

// blocks whose last use has completed go back to the pool
void Context::dev_sweep(bool wait)
{
    for (size_t i = 0; i < deferred.size();) {
        const cudaError_t e = wait ? cudaEventSynchronize(deferred[i].ev) : cudaEventQuery(deferred[i].ev);
        if (e == cudaSuccess) {
            for (void *p : deferred[i].ptrs) dev_free(p);
            cudaEventDestroy(deferred[i].ev);
            deferred.erase(deferred.begin() + (long)i);
        } else {
            if (e != cudaErrorNotReady) (void)cudaGetLastError();
            ++i;
        }
    }
}

void *Context::dev_alloc(size_t bytes)
{
    if (!deferred.empty()) dev_sweep(false);
    bytes = (bytes + 511) & ~(size_t)511;
    void *p = nullptr;
    auto it = pool.find(bytes);
    if (it != pool.end()) {
        p = it->second;
        pool.erase(it);
        pool_bytes -= bytes;
    } else {
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess && (pool_bytes || !deferred.empty())) {          // give the cached blocks back and retry once
            (void)cudaGetLastError();
            dev_sweep(true);
            dev_release_all();
            e = cudaMalloc(&p, bytes);
        }
        if (e != cudaSuccess) fatal("bicgstab_b200: cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    }
    live[p] = bytes;
    return p;
}

void Context::dev_free(void *p)
{
    if (!p) return;
    auto it = live.find(p);
    if (it == live.end()) { cudaFree(p); return; }
    const size_t bytes = it->second;
    live.erase(it);
    const size_t LIMIT = (size_t)16 << 30;             // keep at most 16 GB parked
    if (pool_bytes + bytes > LIMIT) { cudaFree(p); return; }
    pool.emplace(bytes, p);
    pool_bytes += bytes;
}

void Context::dev_release_all()
{
    for (auto &kv : pool) cudaFree(kv.second);
    pool.clear();
    pool_bytes = 0;
}

void Context::h2d(void *dst, const void *src, size_t bytes)
{
    constexpr size_t CHUNK = (size_t)8 << 20, MIN_STAGED = (size_t)16 << 20;
    bool pageable = false;
    if (bytes >= MIN_STAGED && cfg.stage_upload) {
        cudaPointerAttributes at{};
        const cudaError_t e = cudaPointerGetAttributes(&at, src);
        if (e != cudaSuccess) (void)cudaGetLastError();
        pageable = (e != cudaSuccess) || at.type == cudaMemoryTypeUnregistered;
    }
    if (!pageable) { BICG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream)); return; }
    const int T = std::max(1, std::min(stage_threads, 8));
    if ((int)stagers.size() < T) {
        const size_t old = stagers.size();
        stagers.resize((size_t)T);
        for (size_t t = old; t < (size_t)T; ++t) {
            Stager &s = stagers[t];
            BICG_CUDA(cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking));
            BICG_CUDA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
            for (int b = 0; b < 2; ++b) {
                BICG_CUDA(cudaEventCreateWithFlags(&s.ev[b], cudaEventDisableTiming));
                BICG_CUDA(cudaHostAlloc((void **)&s.buf[b], CHUNK, cudaHostAllocDefault));
            }
        }
    }
    // the staged copies run on side streams: they must start after whatever `stream` has queued for dst, and `stream` continues after them
    cudaEvent_t start;
    BICG_CUDA(cudaEventCreateWithFlags(&start, cudaEventDisableTiming));
    BICG_CUDA(cudaEventRecord(start, stream));
    const size_t nchunks = (bytes + CHUNK - 1) / CHUNK;
    const int dev = device;
    std::vector<std::thread> th;
    std::vector<int> rc((size_t)T, 0);
    for (int t = 0; t < T; ++t) {
        th.emplace_back([&, t] {
            if (cudaSetDevice(dev) != cudaSuccess) { rc[(size_t)t] = 1; return; }
            Stager &s = stagers[(size_t)t];
            if (cudaStreamWaitEvent(s.st, start, 0) != cudaSuccess) { rc[(size_t)t] = 1; return; }
            int b = 0;
            for (size_t ck = (size_t)t; ck < nchunks; ck += (size_t)T, b ^= 1) {
                const size_t off = ck * CHUNK, len = std::min(CHUNK, bytes - off);
                if (cudaEventSynchronize(s.ev[b]) != cudaSuccess) { rc[(size_t)t] = 1; return; }      // bounce buffer free again
                memcpy(s.buf[b], (const char *)src + off, len);
                if (cudaMemcpyAsync((char *)dst + off, s.buf[b], len, cudaMemcpyHostToDevice, s.st) != cudaSuccess ||
                    cudaEventRecord(s.ev[b], s.st) != cudaSuccess) { rc[(size_t)t] = 1; return; }
            }
            if (cudaEventRecord(s.done, s.st) != cudaSuccess) rc[(size_t)t] = 1;
        });
    }
    for (auto &x : th) x.join();
    for (int t = 0; t < T; ++t) {
        if (rc[(size_t)t]) fatal("bicgstab_b200: staged host-to-device upload failed: %s", cudaGetErrorString(cudaGetLastError()));
        BICG_CUDA(cudaStreamWaitEvent(stream, stagers[(size_t)t].done, 0));
    }
    cudaEventDestroy(start);
}

void Context::host_allgather(const void *send, void *recv, size_t bytes)
{
    if (world == 1) { memcpy(recv, send, bytes); return; }
    if (!allgather) fatal("bicgstab_b200: world > 1 but no allgather callback (call bicg_comm_init)");
    if (allgather(allgather_ctx, send, recv, bytes) != 0) fatal("bicgstab_b200: host allgather failed");
}

// ------------------------------------------------------------------------------------------------
// SpMV planning
// ------------------------------------------------------------------------------------------------
static inline int round_up(long long v, int m) { return (int)(((v + m - 1) / m) * m); }

static void free_plan(SpmvPlan &p)
{
    ctx().dev_free(p.d_tile_row);
    ctx().dev_free(p.d_tile_nz);
    p.d_tile_row = nullptr; p.d_tile_nz = nullptr;
}

// Fill cap / smem / grid of a TMA-kernel candidate and build + upload its tile plan.  false: not feasible.
static bool build_tma_plan(const bicg_matrix *m, const unsigned *h_ptr, int lanes, int threads, int stages,
                           int want_ctas, SpmvPlan &out)
{
    Context &c = ctx();
    const int rpt = threads / lanes;
    const long long SMEM_MAX = 224 * 1024;
    const long long fixed = (long long)(rpt + 8) * 36;        // ptr slice + 4 epilogue slices per stage (spmv.cu)
    // stage capacity: a full tile of average rows with 25 % head-room, never less than the longest row
    long long cap = (long long)std::ceil(rpt * m->mean_row * 1.25) + 64;
    cap = std::max<long long>(cap, (long long)m->max_row + 16);
    cap = round_up(cap, 32);
    int ctas = want_ctas > 0 ? want_ctas : 2;
    // shrink towards the shared-memory budget of `ctas` CTAs per SM
    const long long budget = SMEM_MAX / ctas - 1536;
    if ((long long)stages * (cap * 12 + fixed) > budget) {
        long long fit = (budget / stages - fixed) / 12;
        fit = (fit / 32) * 32;
        if (fit < (long long)m->max_row + 16) return false;
        cap = fit;
    }
    std::vector<int> tile_row;
    int nt = plan_tiles(h_ptr, m->n_loc, rpt, (int)cap - 8, tile_row);
    if (nt < 0) return false;
    std::vector<unsigned> tile_nz(tile_row.size());
    for (size_t i = 0; i < tile_row.size(); ++i) tile_nz[i] = h_ptr[tile_row[i]];

    out.kind = 0; out.lanes = lanes; out.threads = threads; out.stages = stages; out.cap = (int)cap;
    out.smem = spmv_tma_smem_bytes((int)cap, stages, threads, lanes);
    int by_smem = (int)std::max<long long>(1, SMEM_MAX / (long long)(out.smem + 1536));
    out.ctas_per_sm = std::max(1, std::min({by_smem, 2048 / (threads + 32), want_ctas > 0 ? want_ctas : 8}));
    out.ntiles = nt;
    out.grid = std::max(1, std::min(nt, c.sm_count * out.ctas_per_sm));
    out.d_tile_row = (decltype(out.d_tile_row))c.dev_alloc(tile_row.size() * sizeof(int));
    out.d_tile_nz = (decltype(out.d_tile_nz))c.dev_alloc(tile_nz.size() * sizeof(unsigned));
    // synchronous copies (legacy stream; c.stream is non-blocking): they do not queue behind the matrix upload on c.stream
    BICG_CUDA(cudaMemcpy(out.d_tile_row, tile_row.data(), tile_row.size() * sizeof(int), cudaMemcpyHostToDevice));
    BICG_CUDA(cudaMemcpy(out.d_tile_nz, tile_nz.data(), tile_nz.size() * sizeof(unsigned), cudaMemcpyHostToDevice));
    return true;
}

static void build_rowsplit_plan(const bicg_matrix *m, int lanes, SpmvPlan &out)
{
    Context &c = ctx();
    out = SpmvPlan();
    out.kind = 1; out.lanes = lanes; out.threads = 256; out.stages = 0; out.cap = 0; out.smem = 0;
    const int rpb = 256 / lanes;
    long long blocks = ((long long)m->n_loc + rpb - 1) / rpb;
    out.grid = (int)std::max<long long>(1, std::min<long long>(blocks, (long long)c.sm_count * 8));
}

static int heuristic_lanes(double mean_row)
{
    if (mean_row <= 24.0) return 1;
    if (mean_row <= 48.0) return 8;
    if (mean_row <= 128.0) return 16;
    return 32;
}

SpmvArgs make_spmv_args(const bicg_matrix *m, const SpmvPlan &p, int x_id, int y_id)
{
    SpmvArgs a{};
    a.kc.sc = m->d_sc; a.kc.partials = m->d_partials; a.kc.hist = m->d_hist; a.kc.comm = m->comm;
    a.kc.tail = TailDesc{TAIL_NONE, FIN_NONE, 0, 0, 0, 0, 0};
    a.val = m->d_val; a.col = m->d_col; a.ptr = m->d_ptr; a.rows = m->n_loc;
    a.tile_row = p.d_tile_row; a.tile_nz = p.d_tile_nz; a.ntiles = p.ntiles; a.cap = p.cap; a.stages = p.stages;
    a.x = m->vec(x_id); a.y = m->vec(y_id);
    a.epi = EpiArgs{};
    a.wait_halo = (m->world > 1 && m->comm.recv_mask != 0) ? 1 : 0;
    return a;
}

void launch_spmv_plan(const bicg_matrix *m, const SpmvPlan &p, const SpmvArgs &a, int prof_class)
{
    Context &c = ctx();
    (void)m;
    if (c.prof_on) {
        cudaEvent_t e0, e1;
        BICG_CUDA(cudaEventCreate(&e0)); BICG_CUDA(cudaEventCreate(&e1));
        BICG_CUDA(cudaEventRecord(e0, c.stream));
        int rc = launch_spmv(p.kind, p.lanes, p.threads, p.grid, p.smem, a, c.stream);
        if (rc) fatal("bicgstab_b200: SpMV launch failed: %s", cudaGetErrorString((cudaError_t)rc));
        BICG_CUDA(cudaEventRecord(e1, c.stream));
        c.prof_ev.push_back(e0); c.prof_ev.push_back(e1); c.prof_class.push_back(prof_class);
    } else {
        int rc = launch_spmv(p.kind, p.lanes, p.threads, p.grid, p.smem, a, c.stream);
        if (rc) fatal("bicgstab_b200: SpMV launch failed (kind %d lanes %d threads %d grid %d smem %zu): %s",
                      p.kind, p.lanes, p.threads, p.grid, p.smem, cudaGetErrorString((cudaError_t)rc));
    }
    ++c.launches;
}

// time one candidate on the real matrix: x = V_P (whatever it holds), y = V_S, dot (r#, s) fused, no tail
static double time_plan(bicg_matrix *m, const SpmvPlan &p, int reps)
{
    Context &c = ctx();
    SpmvArgs a = make_spmv_args(m, p, V_P, V_S);
    a.wait_halo = 0;
    epi_add_dot(a.epi, m->vec(V_RH), nullptr);
    cudaEvent_t e0, e1;
    BICG_CUDA(cudaEventCreate(&e0)); BICG_CUDA(cudaEventCreate(&e1));
    for (int i = 0; i < 2; ++i) launch_spmv_plan(m, p, a);
    BICG_CUDA(cudaEventRecord(e0, c.stream));
    for (int i = 0; i < reps; ++i) launch_spmv_plan(m, p, a);
    BICG_CUDA(cudaEventRecord(e1, c.stream));
    BICG_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    BICG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return (double)ms / reps;
}

static void choose_spmv_plan(bicg_matrix *m, const unsigned *h_ptr)
{
    Context &c = ctx();
    const Config &cfg = c.cfg;
    const int LANES[6] = {1, 2, 4, 8, 16, 32};

    auto fixed = [&](SpmvPlan &p) -> bool {
        int lanes = cfg.spmv_lanes > 0 ? cfg.spmv_lanes : heuristic_lanes(m->mean_row);
        if (cfg.spmv_kind == 1) { build_rowsplit_plan(m, lanes, p); return true; }
        int threads = cfg.spmv_threads > 0 ? cfg.spmv_threads : 256;
        int stages = cfg.spmv_stages > 0 ? cfg.spmv_stages : 3;
        if (build_tma_plan(m, h_ptr, lanes, threads, stages, cfg.spmv_ctas, p)) return true;
        if (build_tma_plan(m, h_ptr, lanes, threads, 2, 1, p)) return true;
        if (cfg.spmv_kind == 0) return false;
        build_rowsplit_plan(m, std::max(lanes, 8), p);
        return true;
    };

    const bool pinned = cfg.spmv_lanes > 0 || cfg.spmv_threads > 0 || cfg.spmv_stages > 0 || cfg.spmv_ctas > 0;
    if (!cfg.autotune || pinned || m->n_loc < 4096) {
        if (!fixed(m->plan)) fatal("bicgstab_b200: requested SpMV configuration is not feasible for this matrix");
        return;
    }
    // a matrix of the same shape was tuned before in this process: reuse the winner
    const TuneKey key{m->n_loc, m->nnz, m->max_row, cfg.spmv_kind};
    auto hit = c.tuned.find(key);
    if (hit != c.tuned.end()) {
        const TuneVal &t = hit->second;
        if (t.kind == 1) { build_rowsplit_plan(m, t.lanes, m->plan); return; }
        if (build_tma_plan(m, h_ptr, t.lanes, t.threads, t.stages, t.ctas, m->plan)) return;
    }

    // candidates: lanes around the mean row length x {128,256,512} threads x {2,3,4} stages x {1,2,3,4} CTAs/SM
    std::vector<SpmvPlan> cands;
    const int hl = heuristic_lanes(m->mean_row);
    for (int li = 0; li < 6; ++li) {
        const int lanes = LANES[li];
        if (lanes > 2 * std::max(1.0, m->mean_row)) continue;
        if (lanes < hl / 8) continue;
        if (cfg.spmv_kind != 1) {
            for (int threads : {128, 256, 512})
                for (int stages : {2, 3, 4})
                    for (int ctas : {1, 2, 4}) {
                        if ((threads + 32) * ctas > 2048) continue;
                        SpmvPlan p;
                        if (!build_tma_plan(m, h_ptr, lanes, threads, stages, ctas, p)) continue;
                        if (p.ctas_per_sm != ctas) { free_plan(p); continue; }   // duplicate of another entry
                        cands.push_back(p);
                    }
        }
        if (cfg.spmv_kind != 0) {
            SpmvPlan p; build_rowsplit_plan(m, lanes, p); cands.push_back(p);
        }
    }
    if (cands.empty()) { if (!fixed(m->plan)) fatal("bicgstab_b200: no feasible SpMV configuration"); return; }

    int best = -1;
    for (size_t i = 0; i < cands.size(); ++i) {
        cands[i].ms = time_plan(m, cands[i], 5);
        if (cfg.verbose)
            fprintf(stderr, "[bicg autotune r%d] kind=%d lanes=%2d threads=%3d stages=%d ctas=%d cap=%5d grid=%4d smem=%6zu : %.4f ms\n",
                    m->rank, cands[i].kind, cands[i].lanes, cands[i].threads, cands[i].stages, cands[i].ctas_per_sm,
                    cands[i].cap, cands[i].grid, cands[i].smem, cands[i].ms);
        if (best < 0 || cands[i].ms < cands[best].ms) best = (int)i;
    }
    for (size_t i = 0; i < cands.size(); ++i)
        if ((int)i != best) free_plan(cands[i]);
    m->plan = cands[best];
    c.tuned[key] = TuneVal{m->plan.kind, m->plan.lanes, m->plan.threads, m->plan.stages, m->plan.ctas_per_sm};
    if (cfg.verbose)
        fprintf(stderr, "[bicg autotune r%d] chose kind=%d lanes=%d threads=%d stages=%d ctas=%d (%.4f ms)\n", m->rank,
                m->plan.kind, m->plan.lanes, m->plan.threads, m->plan.stages, m->plan.ctas_per_sm, m->plan.ms);
}

// lanes per row of the persistent kernel's SpMV (instantiated: 1, 4, 8, 32)
static int mega_lanes_for(double mean_row)
{
    if (mean_row <= 20.0) return 1;
    if (mean_row <= 40.0) return 4;
    if (mean_row <= 128.0) return 8;
    return 32;
}

// Plan of the persistent solver kernel (mega.cu): one CTA per SM, every CTA owns a contiguous, work-balanced range of rows
// (plan.cpp: plan_cta_tiles), cut into tiles of <= threads / lanes rows.  row_extra[i] = number of peers row i is pushed to.
static void build_mega_plan(bicg_matrix *m, const unsigned *h_ptr, const std::vector<unsigned char> &row_extra)
{
    Context &c = ctx();
    MegaPlan &mp = m->mega;
    mp.ok = false;
    if (m->n_loc < 1) return;                       // the plan is always built; BICG_MEGA gates its use per solve
    const int G = std::min(c.sm_count, MEGA_MAX_CTAS);
    const long long SMEM_MAX = 222 * 1024;
    const int lanes = c.cfg.mega_lanes > 0 ? c.cfg.mega_lanes : mega_lanes_for(m->mean_row);
    // BICG_MEGA=1 (default): the persistent kernel where it wins -- thread-per-row plans (banded matrices, short rows).  On
    // long-row matrices (cfg 5: 32 random entries per row) the loop is bound by L2 sector throughput of the gathers, not by
    // launch / barrier latency, and the autotuned kernel-per-phase SpMV is faster (profiles/r02a_n1_random_block.log);
    // BICG_MEGA=2 or an explicit BICG_MEGA_LANES forces the persistent kernel there too.
    if (lanes != 1 && c.cfg.mega != 2 && c.cfg.mega_lanes == 0) return;
    for (int threads : {512, 256}) {
        if (c.cfg.mega_threads && c.cfg.mega_threads != threads) continue;
        if (!mega_has_variant(threads, lanes)) continue;
        const int rpt = threads / lanes;
        std::vector<int> tile_row, cta_tile, tile_flag;
        std::vector<unsigned> tile_nz;
        // a stage must hold one tile; at least two stages must fit.  Tiles (or single rows) with more entries than that
        // are cut by the planner: greedy tiles + chunked long rows (plan.cpp)
        const int cap_limit = (int)(((SMEM_MAX / 2 - (long long)(rpt + 8) * 4) / 12) / 32 * 32) - 64;   // cap = roundup(max + 8, 32) must still fit twice
        const unsigned max_tile_nnz = plan_cta_tiles(h_ptr, m->n_loc, G, rpt, row_extra.empty() ? nullptr : row_extra.data(),
                                                     c.cfg.boundary_weight, tile_row, cta_tile, cap_limit, &tile_nz, &tile_flag, c.cfg.row_weight);
        const int cap = round_up((long long)max_tile_nnz + 8, 32);
        const long long stage = (long long)cap * 12 + (long long)(rpt + 8) * 4;
        int stages = (int)std::min<long long>(4, SMEM_MAX / stage);
        if (stages < 2) continue;                       // cannot happen with the cap-limited plan; kept as a guard
        bool chunked = false;
        for (int f : tile_flag) chunked = chunked || f != 0;
        mp.chunked = chunked;
        mp.threads = threads; mp.lanes = lanes; mp.stages = stages; mp.cap = cap; mp.grid = G;
        mp.smem = mega_smem_bytes(cap, stages, threads, lanes);
        // strong-scaling regime: if EVERY CTA's slice (8-byte values, 16-bit CTA-relative columns, row pointers) fits into its
        // shared memory the kernel may keep the matrix there for the whole solve (mega.cu: resident mode)
        mp.res_smem = 0;
        if (lanes == 1 && !chunked) {
            size_t need = 0;
            for (int g = 0; g < G; ++g) {
                const int r0 = tile_row[(size_t)cta_tile[(size_t)g]], r1 = tile_row[(size_t)cta_tile[(size_t)g + 1]];
                need = std::max(need, mega_resident_bytes(h_ptr[r1] - h_ptr[r0], r1 - r0));
            }
            if (need <= (size_t)SMEM_MAX) mp.res_smem = std::max<size_t>(need, 16);
        }
        mp.ntiles = (int)tile_row.size() - 1;
        mp.cta_row.assign((size_t)G + 1, m->n_loc);
        for (int g = 0; g <= G; ++g) mp.cta_row[(size_t)g] = tile_row[(size_t)cta_tile[(size_t)g]];
        mp.d_tile_row = (decltype(mp.d_tile_row))c.dev_alloc(tile_row.size() * sizeof(int));
        mp.d_tile_nz = (decltype(mp.d_tile_nz))c.dev_alloc(tile_nz.size() * sizeof(unsigned));
        mp.d_cta_tile = (decltype(mp.d_cta_tile))c.dev_alloc(cta_tile.size() * sizeof(int));
        mp.d_cta_dep = (decltype(mp.d_cta_dep))c.dev_alloc((size_t)G * sizeof(int4));
        mp.d_tile_flag = nullptr;
        if (chunked) {
            mp.d_tile_flag = (int *)c.dev_alloc(tile_flag.size() * sizeof(int));
            BICG_CUDA(cudaMemcpy(mp.d_tile_flag, tile_flag.data(), tile_flag.size() * sizeof(int), cudaMemcpyHostToDevice));
        }
        BICG_CUDA(cudaMemcpy(mp.d_tile_row, tile_row.data(), tile_row.size() * sizeof(int), cudaMemcpyHostToDevice));
        BICG_CUDA(cudaMemcpy(mp.d_tile_nz, tile_nz.data(), tile_nz.size() * sizeof(unsigned), cudaMemcpyHostToDevice));
        BICG_CUDA(cudaMemcpy(mp.d_cta_tile, cta_tile.data(), cta_tile.size() * sizeof(int), cudaMemcpyHostToDevice));
        launch_mega_dep(m->d_col, m->d_ptr, mp.d_tile_row, mp.d_cta_tile, G, m->ghost_off, mp.d_cta_dep, c.stream);   // behind the upload
        BICG_CUDA(cudaGetLastError());
        // the column width of every tile, from the merged columns on the device; the 16-bit copy of the columns only exists
        // when some tile can use it.  Its padding (like d_col's) covers the 8-entry windows the kernel copies.
        int *d_cbase = (int *)c.dev_alloc(((size_t)mp.ntiles + 1) * sizeof(int));
        BICG_CUDA(cudaMemsetAsync(d_cbase + mp.ntiles, 0, sizeof(int), c.stream));
        launch_mega_tile_base(m->d_col, mp.d_tile_nz, mp.d_tile_flag, mp.ntiles, m->ghost_off, d_cbase, d_cbase + mp.ntiles, c.stream);
        BICG_CUDA(cudaGetLastError());
        BICG_CUDA(cudaMemcpyAsync(&mp.narrow, d_cbase + mp.ntiles, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        BICG_CUDA(cudaStreamSynchronize(c.stream));
        if (mp.narrow > 0) {
            mp.d_tile_cbase = d_cbase;
            mp.d_col16 = (unsigned short *)c.dev_alloc((m->nnz + 16) * sizeof(unsigned short));
            BICG_CUDA(cudaMemsetAsync(mp.d_col16, 0, (m->nnz + 16) * sizeof(unsigned short), c.stream));
            launch_mega_tile_codes(m->d_col, mp.d_tile_nz, mp.d_tile_cbase, mp.ntiles, mp.d_col16, c.stream);
            BICG_CUDA(cudaGetLastError());
        } else {
            c.dev_free(d_cbase);
        }
        mp.ok = true;
        if (c.cfg.verbose)
            fprintf(stderr, "[bicg mega r%d] threads=%d lanes=%d stages=%d cap=%d tiles=%d narrow=%d smem=%zu resident_smem=%zu\n", m->rank,
                    threads, lanes, stages, cap, mp.ntiles, mp.narrow, mp.smem, mp.res_smem);
        return;
    }
}

// ------------------------------------------------------------------------------------------------
// device-side merge of the reference's diag / offd blocks (matrix.c:380-392) into one CSR over [own | ghost] columns
// ------------------------------------------------------------------------------------------------
// One thread per row: diag entries first, then offd entries (the reference's accumulation order, matrix.c:437-440);
// an offd entry's global column becomes ghost_off + ghost slot of the receive run that contains it.
__global__ void __launch_bounds__(256) merge_rows_kernel(int n_loc, const unsigned *__restrict__ dptr, const unsigned *__restrict__ optr,
                                                         const double *__restrict__ dval, const unsigned *__restrict__ dcol,
                                                         const double *__restrict__ oval, const unsigned *__restrict__ ocol,
                                                         const int *__restrict__ runs /* quadruples */, int nruns, int ghost_off,
                                                         double *__restrict__ mval, unsigned *__restrict__ mcol)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_loc; i += gridDim.x * blockDim.x) {
        const unsigned d0 = dptr[i], d1 = dptr[i + 1], o0 = optr[i], o1 = optr[i + 1];
        unsigned k = d0 + o0;
        for (unsigned j = d0; j < d1; ++j, ++k) { mval[k] = dval[j]; mcol[k] = dcol[j]; }
        for (unsigned j = o0; j < o1; ++j, ++k) {
            const int gc = (int)ocol[j];
            int a = 0, b = nruns;                          // last run whose first column is <= gc
            while (b - a > 1) { const int mid = (a + b) >> 1; if (runs[4 * mid] <= gc) a = mid; else b = mid; }
            mval[k] = oval[j];
            mcol[k] = (unsigned)(ghost_off + runs[4 * a + 3] + (gc - runs[4 * a]));
        }
    }
}

void Context::release_arenas()
{
    if (world > 1 && (!arena_pool.empty() || !peer_maps.empty())) {
        int token = 0; std::vector<int> all((size_t)world);
        if (ready) cudaStreamSynchronize(stream);
        host_allgather(&token, all.data(), sizeof(int));       // every rank is done with every arena
        for (auto &kv : peer_maps) cudaIpcCloseMemHandle(kv.second);
        peer_maps.clear();
        host_allgather(&token, all.data(), sizeof(int));       // nobody still maps what is freed next
    }
    for (auto &kv : arena_pool) cudaFree(kv.second.ptr);
    arena_pool.clear();
}

// ------------------------------------------------------------------------------------------------
// matrix creation
// ------------------------------------------------------------------------------------------------
constexpr int INLINE_RUNS = 48;      // receive runs that travel inside the bootstrap header (banded matrices: 2 per neighbour)
struct ArenaHdr {
    cudaIpcMemHandle_t handle;
    unsigned long long arena_id;
    long long vec_off, vstride, ghost_off, mail_off, hflag_off, msync_off, ll_off, ll_stride;
    int n_loc, n_ghost, n_runs, pad_;
    int runs[4 * INLINE_RUNS];
};

static double now_ms()
{
    struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
    return 1e3 * (double)ts.tv_sec + 1e-6 * (double)ts.tv_nsec;
}

bicg_matrix *matrix_create(const CSR_Matrix *diag, const CSR_Matrix *offd, const INFO_Matrix *info)
{
    Context &c = ctx();
    c.ensure();
    const double t_begin = now_ms();
    double t_mark = t_begin;
    auto lap = [&](const char *what) {
        if (c.cfg.verbose < 2) return;
        cudaStreamSynchronize(c.stream);
        const double t = now_ms();
        fprintf(stderr, "[bicg create r%d] %-28s %8.3f ms\n", c.rank, what, t - t_mark);
        t_mark = t;
    };
    if (info->cols != info->rows) {                       // solver.c:43-46
        printf("Error: matrix is not square.\n");
        exit(1);
    }
    cudaEvent_t ev0, ev1;
    BICG_CUDA(cudaEventCreate(&ev0)); BICG_CUDA(cudaEventCreate(&ev1));
    BICG_CUDA(cudaEventRecord(ev0, c.stream));

    bicg_matrix *m = new bicg_matrix();
    m->rank = c.rank; m->world = c.world;
    m->n_loc = (int)diag->rows; m->n_glob = (int)info->rows;
    const size_t nd = diag->nz, no = (offd && m->world > 1) ? offd->nz : 0;
    m->nnz = nd + no;
    m->host_key = diag->val ? (const void *)diag->val : (const void *)diag;
    m->ghost_off = round_up(m->n_loc, 16);

    // ---- halo plan + merged CSR over [own | ghost] columns --------------------------------------------------
    // The layout (receive runs, ghost slots, merged row pointer) is planned on the host from ptr[] and the offd
    // columns (plan.cpp); the entries of the two blocks are uploaded as the caller holds them and merged on the
    // GPU -- no O(nnz) host pass sits in the reference-facing call.
    const unsigned *h_ptr = diag->ptr;
    std::vector<unsigned> mptr;
    if (no) {
        plan_merged_layout(diag, offd, info, m->rank, m->world, c.cfg.halo_gap, mptr, m->recv_runs, m->n_ghost);
        h_ptr = mptr.data();
    }
    m->vstride = (long long)m->ghost_off + round_up(std::max(m->n_ghost, 1), 16);
    unsigned max_row = 0;
    for (int i = 0; i < m->n_loc; ++i) max_row = std::max(max_row, h_ptr[i + 1] - h_ptr[i]);
    m->max_row = max_row;
    m->mean_row = m->n_loc ? (double)m->nnz / m->n_loc : 0.0;

    // ---- arena -------------------------------------------------------------------------------------
    m->hist_cap = std::max(c.cfg.max_iter, 1000) + 2;
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    size_t off = 0;
    const size_t vec_off = off;   off = align(off + (size_t)V_COUNT * (size_t)m->vstride * sizeof(double));
    const size_t sc_off = off;    off = align(off + sizeof(Scalars));
    const size_t part_off = off;  off = align(off + (size_t)4096 * MAX_DOTS * sizeof(double));
    const size_t hist_off = off;  off = align(off + (size_t)m->hist_cap * sizeof(double));
    const size_t mail_off = off;  off = align(off + 2 * MAX_RANKS * sizeof(Mailbox));
    const size_t hflag_off = off; off = align(off + MAX_RANKS * sizeof(HaloFlag));
    const size_t msync_off = off; off = align(off + sizeof(MegaSync));
    // LL halo of the persistent kernel's multi-GPU loops (mega.cu): LL_REGIONS ghost-sized regions of 16-byte
    // {lo | epoch, hi | epoch} pairs, one per pushed vector, written by the peers, polled by the consumers
    const size_t ll_stride = (size_t)round_up(std::max(m->n_ghost, 1), 16);
    const bool want_ll = m->world > 1 && (c.cfg.mega == 2 || c.cfg.mega_lanes > 0 || mega_lanes_for(m->mean_row) == 1);
    const size_t ll_off = off;    off = align(off + (want_ll ? (size_t)LL_REGIONS * ll_stride * 16 : 0));
    m->arena_bytes = std::max<size_t>(off, (size_t)4 << 20);     // its own allocation granule: the IPC handle maps exactly this
    if (m->world > 1) {
        // exported through CUDA IPC: an allocation of its own (peers map exactly this one), parked and re-used by size
        auto it = c.arena_pool.find(m->arena_bytes);
        if (it != c.arena_pool.end()) {
            m->arena = it->second.ptr; m->arena_id = it->second.id; m->arena_handle = it->second.handle;
            c.arena_pool.erase(it);
        } else {
            BICG_CUDA(cudaMalloc((void **)&m->arena, m->arena_bytes));
            BICG_CUDA(cudaIpcGetMemHandle(&m->arena_handle, m->arena));
            m->arena_id = c.next_arena_id++;
        }
    } else {
        m->arena = (char *)c.dev_alloc(m->arena_bytes);
    }
    BICG_CUDA(cudaMemsetAsync(m->arena, 0, m->arena_bytes, c.stream));
    m->vec_base = (double *)(m->arena + vec_off);
    m->d_sc = (Scalars *)(m->arena + sc_off);
    m->d_partials = (double *)(m->arena + part_off);
    m->d_hist = (double *)(m->arena + hist_off);
    m->d_mail = (Mailbox *)(m->arena + mail_off);
    m->d_hflag = (HaloFlag *)(m->arena + hflag_off);
    m->d_msync = (MegaSync *)(m->arena + msync_off);
    m->d_ll = want_ll ? (unsigned long long *)(m->arena + ll_off) : nullptr;
    m->ll_stride = (long long)ll_stride;
    BICG_CUDA(cudaStreamSynchronize(c.stream));            // arena zeroed before any peer may write into it

    lap("arena alloc + zero");
    // ---- upload: asynchronous from here on, so that planning and the bootstrap exchange below overlap with the copies ----
    const size_t pad = 16;
    m->d_val = (decltype(m->d_val))c.dev_alloc((m->nnz + pad) * sizeof(double));
    m->d_col = (decltype(m->d_col))c.dev_alloc((m->nnz + pad) * sizeof(unsigned));
    m->d_ptr = (decltype(m->d_ptr))c.dev_alloc(((size_t)m->n_loc + 1 + pad) * sizeof(unsigned));
    BICG_CUDA(cudaMemsetAsync(m->d_ptr + m->n_loc + 1, 0, pad * sizeof(unsigned), c.stream));
    BICG_CUDA(cudaMemsetAsync(m->d_val + m->nnz, 0, pad * sizeof(double), c.stream));
    BICG_CUDA(cudaMemsetAsync(m->d_col + m->nnz, 0, pad * sizeof(unsigned), c.stream));
    BICG_CUDA(cudaMemcpyAsync(m->d_ptr, h_ptr, ((size_t)m->n_loc + 1) * sizeof(unsigned), cudaMemcpyHostToDevice, c.stream));
    if (!no) {
        if (nd) {
            c.h2d(m->d_val, diag->val, nd * sizeof(double));
            c.h2d(m->d_col, diag->col, nd * sizeof(unsigned));
        }
    } else {
        const size_t np1 = (size_t)m->n_loc + 1;
        double *t_dval = (double *)c.dev_alloc(std::max<size_t>(nd, 1) * sizeof(double));
        double *t_oval = (double *)c.dev_alloc(no * sizeof(double));
        unsigned *t_dcol = (unsigned *)c.dev_alloc(std::max<size_t>(nd, 1) * sizeof(unsigned));
        unsigned *t_ocol = (unsigned *)c.dev_alloc(no * sizeof(unsigned));
        unsigned *t_ptr = (unsigned *)c.dev_alloc(2 * np1 * sizeof(unsigned));
        int *t_runs = (int *)c.dev_alloc(m->recv_runs.size() * sizeof(int));
        // small arrays first: a cudaMemcpyAsync from pageable memory synchronises the stream before it starts, so it must not
        // queue behind the big copies
        BICG_CUDA(cudaMemcpyAsync(t_runs, m->recv_runs.data(), m->recv_runs.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
        BICG_CUDA(cudaMemcpyAsync(t_ptr, diag->ptr, np1 * sizeof(unsigned), cudaMemcpyHostToDevice, c.stream));
        BICG_CUDA(cudaMemcpyAsync(t_ptr + np1, offd->ptr, np1 * sizeof(unsigned), cudaMemcpyHostToDevice, c.stream));
        if (nd) {
            c.h2d(t_dval, diag->val, nd * sizeof(double));
            c.h2d(t_dcol, diag->col, nd * sizeof(unsigned));
        }
        c.h2d(t_oval, offd->val, no * sizeof(double));
        c.h2d(t_ocol, offd->col, no * sizeof(unsigned));
        const int blocks = std::max(1, std::min((m->n_loc + 255) / 256, c.sm_count * 8));
        merge_rows_kernel<<<blocks, 256, 0, c.stream>>>(m->n_loc, t_ptr, t_ptr + np1, t_dval, t_dcol, t_oval, t_ocol, t_runs,
                                                        (int)(m->recv_runs.size() / 4), m->ghost_off, m->d_val, m->d_col);
        BICG_CUDA(cudaGetLastError());
        // back to the pool -- but only once the merge has run: planning below fills freshly allocated blocks with SYNCHRONOUS
        // copies that are not ordered behind this stream
        cudaEvent_t merged;
        BICG_CUDA(cudaEventCreateWithFlags(&merged, cudaEventDisableTiming));
        BICG_CUDA(cudaEventRecord(merged, c.stream));
        c.dev_free_after({t_dval, t_oval, t_dcol, t_ocol, t_ptr, t_runs}, merged);
    }
    m->upload_bytes = m->nnz * 12 + ((size_t)m->n_loc + 1) * 4 * (no ? 2 : 1);

    lap("merge + alloc + H2D matrix");
    // ---- peers: exchange arena handles + layouts, then the halo runs -------------------------------
    m->comm.rank = m->rank; m->comm.world = m->world;
    m->comm.timeout_ns = (unsigned long long)c.cfg.peer_timeout_s * 1000000000ull;
    for (int p = 0; p < MAX_RANKS; ++p) { m->comm.mail[p] = m->d_mail; m->comm.hflag[p] = m->d_hflag; m->peer_msync[p] = m->d_msync; }
    std::vector<unsigned char> row_extra;                  // per row: number of peers it is pushed to
    if (m->world > 1) {
        ArenaHdr mine{};
        mine.handle = m->arena_handle; mine.arena_id = m->arena_id;
        mine.vec_off = (long long)vec_off; mine.vstride = m->vstride; mine.ghost_off = m->ghost_off;
        mine.mail_off = (long long)mail_off; mine.hflag_off = (long long)hflag_off; mine.msync_off = (long long)msync_off;
        mine.ll_off = want_ll ? (long long)ll_off : -1; mine.ll_stride = (long long)ll_stride;
        mine.n_loc = m->n_loc; mine.n_ghost = m->n_ghost;
        const int my_cnt = (int)(m->recv_runs.size() / 4);
        mine.n_runs = my_cnt;
        if (my_cnt <= INLINE_RUNS) std::copy(m->recv_runs.begin(), m->recv_runs.end(), mine.runs);
        std::vector<ArenaHdr> all((size_t)m->world);
        c.host_allgather(&mine, all.data(), sizeof(ArenaHdr));           // ONE bootstrap round in the common case
        for (int p = 0; p < m->world; ++p) {
            if (p == m->rank) { m->peer_base[p] = m->arena; }
            else {
                const auto key = std::make_pair(p, all[(size_t)p].arena_id);
                auto hit = c.peer_maps.find(key);
                if (hit == c.peer_maps.end()) {
                    void *base = nullptr;
                    BICG_CUDA(cudaIpcOpenMemHandle(&base, all[(size_t)p].handle, cudaIpcMemLazyEnablePeerAccess));
                    hit = c.peer_maps.emplace(key, base).first;
                }
                m->peer_base[p] = hit->second;
            }
            m->peer_vec_off[p] = all[(size_t)p].vec_off; m->peer_vstride[p] = all[(size_t)p].vstride;
            m->peer_ghost_off[p] = all[(size_t)p].ghost_off;
            m->comm.mail[p] = (Mailbox *)((char *)m->peer_base[p] + all[(size_t)p].mail_off);
            m->comm.hflag[p] = (HaloFlag *)((char *)m->peer_base[p] + all[(size_t)p].hflag_off);
            m->peer_msync[p] = (MegaSync *)((char *)m->peer_base[p] + all[(size_t)p].msync_off);
            m->peer_ll[p] = all[(size_t)p].ll_off >= 0 ? (unsigned long long *)((char *)m->peer_base[p] + all[(size_t)p].ll_off) : nullptr;
            m->peer_ll_stride[p] = all[(size_t)p].ll_stride;
        }
        // receive lists of every rank: inline in the header, or (irregular matrices with many runs) a second round
        std::vector<int> cnts((size_t)m->world);
        int max_cnt = 1;
        for (int p = 0; p < m->world; ++p) { cnts[(size_t)p] = all[(size_t)p].n_runs; max_cnt = std::max(max_cnt, cnts[(size_t)p]); }
        std::vector<int> recv((size_t)max_cnt * 4 * (size_t)m->world, 0);
        if (max_cnt <= INLINE_RUNS) {
            for (int p = 0; p < m->world; ++p)
                std::copy(all[(size_t)p].runs, all[(size_t)p].runs + 4 * cnts[(size_t)p], recv.begin() + (size_t)p * max_cnt * 4);
        } else {
            std::vector<int> send((size_t)max_cnt * 4, 0);
            std::copy(m->recv_runs.begin(), m->recv_runs.end(), send.begin());
            c.host_allgather(send.data(), recv.data(), send.size() * sizeof(int));
        }

        unsigned recv_mask = 0, send_mask = 0;
        row_extra.assign((size_t)m->n_loc, 0);
        for (int i = 0; i < my_cnt; ++i) recv_mask |= 1u << m->recv_runs[4 * (size_t)i + 2];
        const int my_first = info->displs[m->rank];
        for (int p = 0; p < m->world; ++p) {
            if (p == m->rank) continue;
            std::vector<PushRunHost> ph;
            plan_push_runs(recv.data(), cnts.data(), max_cnt * 4, m->rank, p, my_first, ph);
            if (ph.empty()) continue;
            std::vector<PushRun> pr(ph.size());
            for (size_t i = 0; i < ph.size(); ++i) pr[i] = PushRun{ph[i].src, ph[i].len, ph[i].dst_off};
            send_mask |= 1u << p;
            const int slot = m->npush++;
            m->push_peer[slot] = p; m->push_nruns[slot] = (int)pr.size();
            m->d_push_runs[slot] = (PushRun *)c.dev_alloc(pr.size() * sizeof(PushRun));
            BICG_CUDA(cudaMemcpy(m->d_push_runs[slot], pr.data(), pr.size() * sizeof(PushRun), cudaMemcpyHostToDevice));
            for (const PushRunHost &r : ph)
                for (int i = r.src; i < r.src + r.len; ++i) if (row_extra[(size_t)i] < 255) ++row_extra[(size_t)i];
        }
        m->comm.recv_mask = recv_mask; m->comm.send_mask = send_mask;
    }

    lap("peer exchange");
    // ---- fused-vector launch shape --------------------------------------------------------------------
    m->vgrid = std::min(4096, std::max(1, std::min(c.sm_count * 6, (m->n_loc + 1023) / 1024)));
    m->vchunk = round_up((m->n_loc + m->vgrid - 1) / m->vgrid, 4);
    if (m->vchunk < 4) m->vchunk = 4;

    // ---- SpMV plan ------------------------------------------------------------------------------------
    choose_spmv_plan(m, h_ptr);
    build_mega_plan(m, h_ptr, row_extra);
    if (m->world > 1) {
        // everybody must know whether every rank's persistent-kernel plan is usable (the choice of loop implementation, and
        // with it the synchronisation protocol, must be the same on all ranks): written straight into the peers' arenas
        if (!m->d_ll) m->mega.ok = false;                 // the multi-GPU loops of the persistent kernel need the LL halo regions
        const int ok = m->mega.ok ? 1 : 0;
        for (int p = 0; p < m->world; ++p)
            BICG_CUDA(cudaMemcpy(&m->peer_msync[p]->st.plan_ok[m->rank], &ok, sizeof(int), cudaMemcpyDefault));
    }
    if (c.cfg.mega_trace) {
        const size_t tb = ((size_t)2 * MEGA_TRACE_ITERS * MEGA_TRACE_SLOTS + (size_t)2 * MEGA_MAX_CTAS) * sizeof(unsigned long long);
        m->d_trace = (decltype(m->d_trace))c.dev_alloc(tb);
        BICG_CUDA(cudaMemset(m->d_trace, 0, tb));
    }

    lap("spmv plan");
    BICG_CUDA(cudaEventRecord(ev1, c.stream));
    m->ev_upload0 = ev0; m->ev_upload1 = ev1;              // elapsed time is read after the first solve (matrix_upload_ms): no wait here
    if (m->world > 1) {          // nobody may start pushing before every rank has mapped every arena
        int token = 0; std::vector<int> all((size_t)m->world);
        c.host_allgather(&token, all.data(), sizeof(int));
        int oks[MAX_RANKS] = {};
        BICG_CUDA(cudaMemcpy(oks, m->d_msync->st.plan_ok, sizeof(oks), cudaMemcpyDeviceToHost));
        for (int p = 0; p < m->world; ++p) if (!oks[p]) m->mega.ok = false;
    }
    return m;
}

double matrix_upload_ms(bicg_matrix *m)
{
    if (m->ev_upload0) {
        float ms = 0.f;
        if (cudaEventSynchronize(m->ev_upload1) == cudaSuccess && cudaEventElapsedTime(&ms, m->ev_upload0, m->ev_upload1) == cudaSuccess)
            m->upload_ms = ms;
        cudaEventDestroy(m->ev_upload0); cudaEventDestroy(m->ev_upload1);
        m->ev_upload0 = m->ev_upload1 = nullptr;
    }
    return m->upload_ms;
}

void matrix_destroy(bicg_matrix *m)
{
    if (!m) return;
    Context &c = ctx();
    if (c.ready) cudaStreamSynchronize(c.stream);
    (void)matrix_upload_ms(m);
    for (auto it = c.cache.begin(); it != c.cache.end();) {
        if (it->second == m) it = c.cache.erase(it); else ++it;
    }
    for (int g = 0; g < 4; ++g) if (m->graph[g]) cudaGraphExecDestroy(m->graph[g]);
    // world > 1: nothing collective here.  The arena is parked, not freed (the peers keep their mappings), and a rank
    // that has finished its solve has received everything its peers will ever write into this arena: the last
    // reduction completes only after every rank's last push and post (DESIGN.md 4).
    for (int s = 0; s < m->npush; ++s) c.dev_free(m->d_push_runs[s]);
    free_plan(m->plan);
    c.dev_free(m->d_trace);
    c.dev_free(m->mega.d_tile_row); c.dev_free(m->mega.d_tile_nz); c.dev_free(m->mega.d_cta_tile); c.dev_free(m->mega.d_cta_dep);
    c.dev_free(m->mega.d_tile_flag); c.dev_free(m->mega.d_tile_cbase); c.dev_free(m->mega.d_col16);
    if (m->hist_extra) cudaFree(m->hist_extra);
    c.dev_free(m->d_val); c.dev_free(m->d_col); c.dev_free(m->d_ptr);
    if (m->world > 1) c.arena_pool.emplace(m->arena_bytes, Context::ArenaRec{m->arena, m->arena_bytes, m->arena_id, m->arena_handle});
    else c.dev_free(m->arena);
    delete m;
}

// Content fingerprint of the caller's blocks: sizes + up to 8192 evenly spaced samples of val / col / ptr of both blocks
// (FNV-1a).  The upload cache is keyed by the host pointer; the fingerprint catches what the pointer cannot -- a
// different matrix in a recycled allocation, or values changed in place everywhere (diagonal shift, rescaling:
// csr_shift_diagonal, matrix.c:536-551).  A sparse in-place edit that misses every sample still needs
// bicg_matrix_invalidate() (or BICG_CACHE=0, which re-reads the caller's arrays on every call like the reference does).
static uint64_t block_fingerprint(const CSR_Matrix *b, uint64_t h)
{
    auto mix = [&](uint64_t v) { h = (h ^ v) * 0x100000001b3ull; };
    if (!b) { mix(0x9e3779b97f4a7c15ull); return h; }
    mix(b->nz); mix(b->rows); mix(b->cols);
    const size_t S = 8192;
    if (b->nz && b->val && b->col) {
        const size_t step = std::max<size_t>(1, b->nz / S);
        for (size_t i = 0; i < b->nz; i += step) {
            uint64_t bits; memcpy(&bits, &b->val[i], 8);
            mix(bits); mix(b->col[i]);
        }
        uint64_t bits; memcpy(&bits, &b->val[b->nz - 1], 8);
        mix(bits); mix(b->col[b->nz - 1]);
    }
    if (b->ptr) {
        const size_t np1 = (size_t)b->rows + 1, step = std::max<size_t>(1, np1 / S);
        for (size_t i = 0; i < np1; i += step) mix(b->ptr[i]);
        mix(b->ptr[b->rows]);
    }
    return h;
}
static uint64_t host_fingerprint(const CSR_Matrix *diag, const CSR_Matrix *offd, bool with_offd)
{
    uint64_t h = block_fingerprint(diag, 0xcbf29ce484222325ull);
    return with_offd ? block_fingerprint(offd, h) : h;
}

bicg_matrix *matrix_get_cached(const CSR_Matrix *diag, const CSR_Matrix *offd, const INFO_Matrix *info, bool *fresh)
{
    Context &c = ctx();
    const void *key = diag->val ? (const void *)diag->val : (const void *)diag;
    const uint64_t fp = c.cfg.cache ? host_fingerprint(diag, offd, c.world > 1) : 0;
    if (c.cfg.cache) {
        auto it = c.cache.find(key);
        if (it != c.cache.end()) {
            bicg_matrix *old = it->second;
            if (old->host_fp == fp && old->n_loc == (int)diag->rows && old->n_glob == (int)info->rows &&
                old->nnz == (size_t)diag->nz + (c.world > 1 && offd ? offd->nz : 0)) {
                if (fresh) *fresh = false;
                return old;
            }
            matrix_destroy(old);            // same arrays, different matrix: the caller reused the allocation
        }
    }
    bicg_matrix *m = matrix_create(diag, offd, info);
    m->host_fp = fp;
    if (fresh) *fresh = true;
    if (c.cfg.cache) c.cache[key] = m;
    return m;
}

} // namespace bicg
