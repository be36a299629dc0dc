// abi.cu — the extern "C" surface of libeasylp_b200.so (declared in include/easylp_abi.h).
// Every entry point converts C++ exceptions into a nonzero return code + elp_last_error() text.
#include "common.cuh"
#include "comm.cuh"
#include "../../include/easylp_abi.h"
#include <algorithm>
#include <cmath>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>

namespace elp {

std::atomic<int64_t> g_launches{0};
thread_local std::string g_last_error;

// implemented in the other translation units
struct Pdlp;
struct AsmIo {
    int32_t *row, *col, *out_ptr, *out_col;
    double *val, *out_val;
};
AsmIo asm_io_buffers(size_t T, size_t m);
void asm_workspace_release();
struct AsmLowered {
    int32_t* grp;
    int32_t* itab;
    double* dtab;
    elp_fold_group* groups;
};
AsmLowered asm_lowered_buffers(size_t T, size_t n_itab, size_t n_dtab, size_t n_groups);
void asm_expand_families(int n_families, const elp_term_family* fam, const int32_t* d_itab, const double* d_dtab,
                         int64_t stream_offset, int32_t* d_row, int32_t* d_col, double* d_val, int32_t* d_grp,
                         cudaStream_t st);
int64_t assemble_csr_device(int64_t T, const int32_t* d_row, const int32_t* d_col, const double* d_val, int32_t m,
                            int32_t n, int32_t* d_row_ptr, int32_t* d_col_idx, double* d_vals, cudaStream_t st,
                            const int32_t* d_grp = nullptr, const elp_fold_group* d_groups = nullptr,
                            const double* d_dtab = nullptr);
Pdlp* pdlp_create(int m, int n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                  const int8_t* sense, const double* rhs, const double* c, int maximize, const double* lb,
                  const double* ub, const elp_options& opt, bool dist, elp_stats* stats, int64_t nnz_device = -1);
void pdlp_run(Pdlp* p, int max_new_iters, elp_stats* stats);
void pdlp_reset(Pdlp* p);
void pdlp_solution(Pdlp* p, double* x, double* y, double* obj, bool collective_x = false);
void pdlp_probe(Pdlp* p, int reps, double* a, double* b);
void pdlp_probe_step(Pdlp* p, int reps, double* a, double* b);
int pdlp_transpose(Pdlp* p);
void pdlp_destroy(Pdlp* p);
void spmv_host(int m, int n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals, const double* x,
               double* out, const int8_t* sense, const double* rhs, double tol, uint8_t* feasible);
bool simplex_auto_prefers(int m, int n);
int simplex_batch_device(int64_t B, int m, int n, const double* A, const double* b, const double* c, const double* lb,
                         const double* ub, const int8_t* sense, int maximize, int max_pivots, int32_t* status,
                         double* obj, double* x, double* y, int32_t* pivots, cudaStream_t st, int shared_model = 0,
                         int32_t* basis = nullptr);
void densify_device(int m, int n, const int* ptr, const int* idx, const double* val, double* A, cudaStream_t st);
void sensitivity(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                 const int8_t* sense, const double* rhs, const double* c, int32_t maximize, const double* lb,
                 const double* ub, const elp_options& o, int32_t* status, double* objval, double* x, double* obj_from,
                 double* obj_till, double* rhs_from, double* rhs_till, double* duals);
void solve_mip(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals, const int8_t* sense,
               const double* rhs, const double* c, int32_t maximize, const double* lb, const double* ub,
               const uint8_t* is_int, const elp_options& o, int32_t* status, double* objval, double* x, elp_stats* stats);

void pool_release();            // shuts the multi-GPU worker pool down (defined next to it, below)
// a pair of timing events that cannot leak when something between create and destroy throws
struct EventPair {
    cudaEvent_t a = nullptr, b = nullptr;
    EventPair() { ELP_CUDA(cudaEventCreate(&a)); if (cudaEventCreate(&b) != cudaSuccess) { cudaEventDestroy(a); throw Error("cudaEventCreate failed"); } }
    ~EventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
    EventPair(const EventPair&) = delete;
    EventPair& operator=(const EventPair&) = delete;
    float ms() const { float t = 0; cudaEventElapsedTime(&t, a, b); return t; }
};

static void require_device() {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        throw Error(format("no CUDA device available (%s); libeasylp_b200 has no CPU fallback",
                           e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e)));
}

static elp_options effective_options(const elp_options* opt) {
    elp_options o;
    elp_default_options(&o);
    if (opt) {
        o = *opt;
        elp_options d;
        elp_default_options(&d);
        if (!(o.eps_rel > 0)) o.eps_rel = d.eps_rel;
        if (o.check_every <= 1) o.check_every = d.check_every;
        if (o.ruiz_iters < 0) o.ruiz_iters = d.ruiz_iters;
        if (o.devices < 0) o.devices = 0;
    }
    if (o.devices == 0) {
        if (const char* e = getenv("ELP_DEVICES")) o.devices = std::max(0, atoi(e));    // site-wide default (R: gpu.devices=)
    }
    return o;
}

struct Batch {
    int64_t B = 0;
    int m = 0, n = 0, maximize = 0;
    DevBuf<double> A, b, c, lb, ub, obj, x;
    DevBuf<int8_t> sense;
    DevBuf<int32_t> status, pivots;
    bool has_lb = false, has_ub = false, has_sense = false;
    int64_t h2d = 0;
};

// Grow-only workspace of the streamed elp_solve_batch (per host thread; re-created when the thread switches device).
struct BatchStreamWorkspace {
    static constexpr int NS = 3;
    int device = -1;
    cudaStream_t st[NS] = {};
    cudaEvent_t done[NS] = {};
    DevBuf<double> A[NS], b[NS], c[NS], lb[NS], ub[NS], obj[NS], x[NS];
    DevBuf<int8_t> sense[NS];
    DevBuf<int32_t> status[NS], piv[NS];
    int32_t* piv_host = nullptr;       // page-locked, one counter per LP of the whole batch
    size_t piv_cap = 0;
    void release() {
        for (int s = 0; s < NS; ++s) {
            if (st[s]) { cudaStreamSynchronize(st[s]); cudaStreamDestroy(st[s]); st[s] = nullptr; }
            if (done[s]) { cudaEventDestroy(done[s]); done[s] = nullptr; }
            A[s].release(); b[s].release(); c[s].release(); lb[s].release(); ub[s].release(); obj[s].release();
            x[s].release(); sense[s].release(); status[s].release(); piv[s].release();
        }
        if (piv_host) cudaFreeHost(piv_host);
        piv_host = nullptr; piv_cap = 0; device = -1;
    }
    ~BatchStreamWorkspace() { release(); }
    void ensure(size_t chunk, size_t B, int m, int n, bool has_lb, bool has_ub, bool has_sense) {
        int dev = 0;
        ELP_CUDA(cudaGetDevice(&dev));
        if (dev != device) { release(); device = dev; }
        auto grow = [](auto& buf, size_t cnt) { if (buf.n < cnt) buf.alloc(cnt + cnt / 8); };
        for (int s = 0; s < NS; ++s) {
            if (!st[s]) ELP_CUDA(cudaStreamCreateWithFlags(&st[s], cudaStreamNonBlocking));
            if (!done[s]) ELP_CUDA(cudaEventCreateWithFlags(&done[s], cudaEventDisableTiming));
            grow(A[s], chunk * (size_t)std::max(m, 1) * n); grow(b[s], chunk * (size_t)std::max(m, 1)); grow(c[s], chunk * n);
            if (has_lb) grow(lb[s], chunk * n);
            if (has_ub) grow(ub[s], chunk * n);
            if (has_sense) grow(sense[s], chunk * (size_t)std::max(m, 1));
            grow(obj[s], chunk); grow(x[s], chunk * n); grow(status[s], chunk); grow(piv[s], chunk);
        }
        if (piv_cap < B) {
            if (piv_host) cudaFreeHost(piv_host);
            piv_host = nullptr; piv_cap = 0;
            ELP_CUDA(cudaMallocHost(&piv_host, (B + B / 8) * sizeof(int32_t)));
            piv_cap = B + B / 8;
        }
    }
};
BatchStreamWorkspace& batch_stream_workspace() {
    static thread_local BatchStreamWorkspace w;
    return w;
}

}  // namespace elp

using namespace elp;

#define ELP_TRY try {
#define ELP_CATCH                                   \
    }                                               \
    catch (const std::exception& e) {               \
        elp::g_last_error = e.what();               \
        return 1;                                   \
    }                                               \
    catch (...) {                                   \
        elp::g_last_error = "unknown C++ exception"; \
        return 1;                                   \
    }                                               \
    return 0;

// ---- single-process multi-GPU: one persistent worker thread per GPU ---------------------------------------------
// `$solve()` is ONE blocking call from ONE R thread (/root/reference/R/class.R:251-302).  With elp_options.devices = N
// the call partitions the LP by row blocks (balanced by non-zeros), hands block r to worker r — a host thread bound to
// GPU r that owns rank r of an in-process NCCL communicator — and every worker runs the same distributed PDLP a
// process-per-GPU launch runs (pdlp.cu; peers are mapped with cudaDeviceEnablePeerAccess instead of CUDA IPC).  The
// workers and their communicator live until elp_release_workspace(): NCCL initialisation costs more than a solve.
struct DevicePool {
    int N = 0;
    std::vector<int> devs;
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_job, cv_done;
    uint64_t generation = 0;
    int remaining = 0;
    bool stop = false;
    std::function<void(int)> job;
    std::vector<std::string> errors;

    void worker(int r) {
        uint64_t seen = 0;
        for (;;) {
            std::function<void(int)> fn;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_job.wait(lk, [&] { return stop || generation != seen; });
                if (stop) return;
                seen = generation;
                fn = job;
            }
            std::string err;
            try { fn(r); }
            catch (const std::exception& e) { err = e.what(); }
            catch (...) { err = "unknown C++ exception"; }
            {
                std::lock_guard<std::mutex> lk(mu);
                if (!err.empty()) errors[r] = err;
                if (--remaining == 0) cv_done.notify_all();
            }
        }
    }
    // runs fn(rank) on every worker and waits; rethrows the first error
    void run(std::function<void(int)> fn) {
        {
            std::lock_guard<std::mutex> lk(mu);
            job = std::move(fn);
            errors.assign(N, std::string());
            remaining = N;
            ++generation;
        }
        cv_job.notify_all();
        std::unique_lock<std::mutex> lk(mu);
        cv_done.wait(lk, [&] { return remaining == 0; });
        for (int r = 0; r < N; ++r)
            if (!errors[r].empty()) throw Error(format("GPU worker %d (device %d): %s", r, devs[r], errors[r].c_str()));
    }
    void start(int n_dev, int first_dev, int dev_count) {
        N = n_dev;
        devs.resize(N);
        for (int r = 0; r < N; ++r) devs[r] = (first_dev + r) % dev_count;
        for (int r = 0; r < N; ++r) workers.emplace_back([this, r] { worker(r); });
        unsigned char id[ELP_UNIQUE_ID_BYTES];
        comm_unique_id(id);
        run([&](int r) {
            ELP_CUDA(cudaSetDevice(devs[r]));
            comm_init(N, r, id);
        });
    }
    void shutdown() {
        if (workers.empty()) return;
        try { run([](int) { cudaDeviceSynchronize(); comm_destroy(); g_arena_cache.clear(); }); } catch (...) {}
        {
            std::lock_guard<std::mutex> lk(mu);
            stop = true;
        }
        cv_job.notify_all();
        for (auto& t : workers) t.join();
        workers.clear();
        N = 0;
    }
};
static std::mutex g_pool_mutex;          // one multi-GPU solve at a time per process
static DevicePool* g_pool = nullptr;     // deliberately never destroyed at exit (worker threads blocked on a condition
                                         // variable are reaped with the process; tearing NCCL down after CUDA is not safe)

void elp::pool_release() {
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (g_pool) { g_pool->shutdown(); delete g_pool; g_pool = nullptr; }
}

// rows [cut[r], cut[r+1]) for rank r: contiguous, balanced by non-zeros (the rule of easylp_b200/partition.py::row_cuts)
static std::vector<int32_t> row_cuts_by_nnz(int32_t m, const int32_t* row_ptr, int N) {
    std::vector<int32_t> cut(N + 1, 0);
    const int64_t nnz = m > 0 ? row_ptr[m] : 0;
    for (int g = 1; g < N; ++g) {
        const double target = (double)nnz * g / N;
        const int32_t* it = std::lower_bound(row_ptr, row_ptr + m + 1, target, [](int32_t a, double t) { return (double)a < t; });
        cut[g] = (int32_t)(it - row_ptr);
    }
    cut[N] = m;
    for (int g = 1; g <= N; ++g) cut[g] = std::min(std::max(cut[g], cut[g - 1]), m);
    return cut;
}

static void solve_multi(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                        const int8_t* sense, const double* rhs, const double* c, int32_t maximize, const double* lb,
                        const double* ub, const elp_options& o, int32_t* status, double* objval, double* x, double* y,
                        elp_stats* stats) {
    WallTimer wall;
    int dev_count = 0, cur = 0;
    ELP_CUDA(cudaGetDeviceCount(&dev_count));
    ELP_CUDA(cudaGetDevice(&cur));
    ELP_REQUIRE(o.devices <= dev_count, "devices = %d but only %d CUDA device(s) are visible", o.devices, dev_count);
    ELP_REQUIRE(o.devices <= 8, "devices = %d: at most 8 GPUs of one box", o.devices);
    bool bad_bounds = false;
    for (int j = 0; j < n; ++j) if (lb[j] > ub[j]) { bad_bounds = true; break; }
    const int N = o.devices;
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (g_pool && (g_pool->N != N || g_pool->devs[0] != cur)) { g_pool->shutdown(); delete g_pool; g_pool = nullptr; }
    if (!g_pool) {
        g_pool = new DevicePool();
        try { g_pool->start(N, cur, dev_count); }
        catch (...) { g_pool->shutdown(); delete g_pool; g_pool = nullptr; throw; }
    }
    const std::vector<int32_t> cut = row_cuts_by_nnz(m, row_ptr, N);
    std::vector<elp_stats> s_setup(N), s_run(N);
    const int64_t l0 = g_launches.load();
    elp_options od = o;
    od.devices = 0;
    g_pool->run([&](int r) {
        const int32_t r0 = cut[r], r1 = cut[r + 1], ml = r1 - r0;
        const int64_t off = m > 0 ? row_ptr[r0] : 0;
        std::vector<int32_t> rp((size_t)ml + 1);
        for (int32_t i = 0; i <= ml; ++i) rp[i] = (int32_t)((m > 0 ? row_ptr[r0 + i] : 0) - off);
        memset(&s_setup[r], 0, sizeof(elp_stats));
        memset(&s_run[r], 0, sizeof(elp_stats));
        Pdlp* p = pdlp_create(ml, n, rp.data(), col_idx + off, vals + off, sense + r0, rhs + r0, c, maximize, lb, ub, od, true,
                              &s_setup[r]);
        try {
            if (!bad_bounds) pdlp_run(p, 0, &s_run[r]);
            double obj = 0.0;
            pdlp_solution(p, r == 0 ? x : nullptr, y ? y + r0 : nullptr, &obj, true);
            if (r == 0) *objval = obj;
        } catch (...) {
            pdlp_destroy(p);
            throw;
        }
        pdlp_destroy(p);
    });
    *status = bad_bounds ? ELP_STATUS_INFEASIBLE : s_run[0].status;
    if (*status == ELP_STATUS_UNBOUNDED) *objval = maximize ? INFINITY : -INFINITY;
    if (stats) {
        *stats = s_run[0];
        stats->status = *status;
        stats->setup_ms = s_setup[0].setup_ms;
        stats->total_ms = wall.ms();
        stats->kernel_launches = g_launches.load() - l0;
        stats->h2d_bytes = 0; stats->d2h_bytes = 0;
        for (int r = 0; r < N; ++r) {
            stats->h2d_bytes += s_run[r].h2d_bytes;
            stats->d2h_bytes += s_run[r].d2h_bytes;
            stats->solve_ms = std::max(stats->solve_ms, s_run[r].solve_ms);     // device time: the slowest rank
        }
    }
}

extern "C" {

const char* elp_version(void) { return "easylp_b200 0.1 (sm_100a)"; }

int elp_last_error(char* buf, int32_t len) {
    if (!buf || len <= 0) return 1;
    snprintf(buf, (size_t)len, "%s", elp::g_last_error.c_str());
    return 0;
}

int elp_device_count(int32_t* count) {
    ELP_TRY
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) { c = 0; cudaGetLastError(); }
    *count = c;
    ELP_CATCH
}

int elp_set_device(int32_t device) {
    ELP_TRY
    ELP_CUDA(cudaSetDevice(device));
    ELP_CATCH
}

int elp_default_options(elp_options* o) {
    if (!o) return 1;
    o->eps_rel = 1e-6;
    o->time_limit_s = 0.0;
    o->max_iter = 0;
    o->check_every = 64;
    o->method = ELP_METHOD_AUTO;
    o->verbose = 0;
    o->use_graph = 1;
    o->ruiz_iters = 10;
    o->transpose = ELP_TRANSPOSE_AUTO;
    o->devices = 0;
    return 0;
}

const char* elp_status_string(int32_t status) {
    switch (status) {   // /root/reference/R/class.R:279-295
        case 0: return "optimal";
        case 1: return "sub-optimal";
        case 2: return "unfeasible";
        case 3: return "unbounded";
        case 4: return "degenerate model";
        case 5: return "numerical failure encountered";
        case 6: return "process aborted";
        case 7: return "timeout";
        case 9: return "the model was solved by presolve";
        case 10: return "the branch and bound routine failed";
        case 11: return "the branch and bound was stopped because of a break-at-first or break-at-value";
        case 12: return "a feasible branch and bound solution was found";
        case 13: return "no feasible branch and bound solution was found";
        default: return "undocumented status";
    }
}

int64_t elp_kernel_launches(void) { return elp::g_launches.load(); }

int elp_release_workspace(void) {
    ELP_TRY
    asm_workspace_release();
    batch_stream_workspace().release();
    pool_release();
    g_arena_cache.clear();              // parked arenas of this thread (the pool's workers empty theirs when they shut down)
    ELP_CATCH
}

int elp_assemble_csr(int64_t n_terms, const int32_t* term_row, const int32_t* term_col, const double* term_val,
                     int32_t m, int32_t n, int32_t* row_ptr, int32_t* col_idx, double* vals, int64_t* nnz_out,
                     elp_stats* stats) {
    ELP_TRY
    require_device();
    WallTimer wall;
    const int64_t l0 = g_launches.load();
    ELP_REQUIRE(n_terms >= 0 && m >= 0 && n >= 0, "assemble: negative size");
    cudaStream_t st = 0;
    const size_t T = (size_t)n_terms;
    const AsmIo io = asm_io_buffers(std::max<size_t>(T, 1), (size_t)m);      // cached staging (grow-only workspace)
    if (T) {
        ELP_CUDA(cudaMemcpyAsync(io.row, term_row, T * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        ELP_CUDA(cudaMemcpyAsync(io.col, term_col, T * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        ELP_CUDA(cudaMemcpyAsync(io.val, term_val, T * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    EventPair ev;
    cudaEvent_t e0 = ev.a, e1 = ev.b;
    ELP_CUDA(cudaEventRecord(e0, st));
    const int64_t nnz = assemble_csr_device(n_terms, io.row, io.col, io.val, m, n, io.out_ptr, io.out_col, io.out_val, st);
    ELP_CUDA(cudaEventRecord(e1, st));
    ELP_CUDA(cudaMemcpyAsync(row_ptr, io.out_ptr, ((size_t)m + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (nnz) {
        ELP_CUDA(cudaMemcpyAsync(col_idx, io.out_col, (size_t)nnz * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaMemcpyAsync(vals, io.out_val, (size_t)nnz * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    ELP_CUDA(cudaStreamSynchronize(st));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    *nnz_out = nnz;
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->solve_ms = ms;
        stats->total_ms = wall.ms();
        stats->kernel_launches = g_launches.load() - l0;
        stats->h2d_bytes = (int64_t)T * 16;
        stats->d2h_bytes = nnz * 12 + ((int64_t)m + 1) * 4;
    }
    ELP_CATCH
}

// checks a family against the table sizes and returns the number of terms it emits
static int64_t check_family(const elp_term_family& f, int64_t n_itab, int64_t n_dtab, int32_t n_groups, int32_t m,
                            const int32_t* itab = nullptr, int64_t* row_lo = nullptr, int64_t* row_hi = nullptr) {
    ELP_REQUIRE(f.n_loops >= 0 && f.n_loops <= ELP_MAX_LOOPS, "lowered: family with %d loops (max %d)", f.n_loops, ELP_MAX_LOOPS);
    ELP_REQUIRE(f.group >= 0 && f.group < std::max(n_groups, 1), "lowered: family names group %d of %d", f.group, n_groups);
    ELP_REQUIRE(f.out_stride >= 1 && f.out_offset >= 0, "lowered: bad stream placement");
    int64_t count = 1, coef_max = f.coef_tab, row_max = f.row0;
    for (int l = 0; l < f.n_loops; ++l) {
        ELP_REQUIRE(f.extent[l] >= 0, "lowered: negative loop extent");
        count *= f.extent[l];
        ELP_REQUIRE(count < (1ll << 40), "lowered: family too large");
        if (f.extent[l] > 0) {
            ELP_REQUIRE(f.col_tab[l] < 0 || f.col_tab[l] + f.extent[l] <= n_itab, "lowered: column table outside itab");
            ELP_REQUIRE(f.row_tab[l] < 0 || f.row_tab[l] + f.extent[l] <= n_itab, "lowered: row table outside itab");
            ELP_REQUIRE(f.coef_stride[l] >= 0 && f.row_stride[l] >= 0, "lowered: negative stride");
            coef_max += f.coef_stride[l] * (int64_t)(f.extent[l] - 1);
            if (f.row_tab[l] < 0) row_max += (int64_t)f.row_stride[l] * (f.extent[l] - 1);   // table rows: checked by the assembly (out-of-range terms are reported)
        }
    }
    ELP_REQUIRE(count == f.count, "lowered: family count %lld is not the product of its extents (%lld)", (long long)f.count, (long long)count);
    if (count > 0) {
        ELP_REQUIRE(f.coef_tab >= 0 && coef_max < n_dtab, "lowered: coefficient table outside dtab");
        ELP_REQUIRE(f.row0 >= 0 && row_max < m, "lowered: family rows outside the matrix");
    }
    // rows this family touches: row0 plus, per loop, a stride term or an entry of its row table
    if (row_lo && row_hi && count > 0) {
        int64_t lo = f.row0, hi = f.row0;
        for (int l = 0; l < f.n_loops; ++l) {
            if (f.extent[l] <= 0) continue;
            if (f.row_tab[l] >= 0 && itab) {
                int32_t a = itab[f.row_tab[l]], b = a;
                for (int32_t q = 1; q < f.extent[l]; ++q) { a = std::min(a, itab[f.row_tab[l] + q]); b = std::max(b, itab[f.row_tab[l] + q]); }
                lo += a; hi += b;
            } else if (f.row_tab[l] < 0) {
                hi += (int64_t)f.row_stride[l] * (f.extent[l] - 1);
            }
        }
        *row_lo = lo; *row_hi = hi;
    }
    return count;
}

// explicit terms + families -> device term stream (row, col, val, grp); returns the stream length
static int64_t stage_lowered(int64_t n_terms, const int32_t* term_row, const int32_t* term_col, const double* term_val,
                             int32_t n_families, const elp_term_family* families, int64_t n_itab, const int32_t* itab,
                             int64_t n_dtab, const double* dtab, int32_t n_groups, const elp_fold_group* groups, int32_t m,
                             AsmIo* io_out, AsmLowered* lo_out, cudaStream_t st, bool rows_unbounded = false) {
    // rows_unbounded: the caller only wants the stream (elp_expand_terms): no row limit, no row_ptr staging
    const int32_t m_alloc = rows_unbounded ? 0 : m;
    if (rows_unbounded) m = 0x7fffffff;
    ELP_REQUIRE(n_terms >= 0 && n_families >= 0 && n_itab >= 0 && n_dtab >= 0 && n_groups >= 0, "lowered: negative size");
    int64_t total = 0;
    std::vector<int> order;
    const size_t n_g = (groups && n_groups != 0x7fffffff) ? (size_t)std::max(n_groups, 1) : 1;
    std::vector<int64_t> g_lo(n_g, INT64_MAX), g_hi(n_g, -1);
    for (int i = 0; i < n_families; ++i) {
        int64_t lo = 0, hi = -1;
        const int64_t cnt = check_family(families[i], n_itab, n_dtab, n_groups, m, itab, &lo, &hi);
        total += cnt;
        if (cnt > 0) {
            order.push_back(i);
            if ((size_t)families[i].group < n_g && n_g > 1) {
                g_lo[families[i].group] = std::min(g_lo[families[i].group], lo);
                g_hi[families[i].group] = std::max(g_hi[families[i].group], hi);
            }
        }
    }
    // The families must tile the stream exactly: a group of k families with stride k interleaves the k body terms of
    // each cell over one region; regions follow one another without holes or overlap (every slot is written once).
    std::sort(order.begin(), order.end(), [&](int a, int b) { return families[a].out_offset < families[b].out_offset; });
    int64_t pos = 0;
    for (size_t i = 0; i < order.size();) {
        const elp_term_family& f = families[order[i]];
        const int k = f.out_stride;
        bool ok = f.out_offset == pos && i + (size_t)k <= order.size();
        for (int t = 0; ok && t < k; ++t) {
            const elp_term_family& g = families[order[i + t]];
            ok = g.out_offset == pos + t && g.out_stride == k && g.count == f.count;
        }
        ELP_REQUIRE(ok, "lowered: the families do not tile the stream (at position %lld)", (long long)pos);
        pos += f.count * k;
        i += (size_t)k;
    }
    ELP_REQUIRE(pos == total, "lowered: the families do not tile the stream (%lld of %lld slots)", (long long)pos, (long long)total);
    ELP_REQUIRE(groups != nullptr || n_groups == 0 || n_groups == 0x7fffffff, "lowered: groups missing");
    for (int g = 0; groups && g < n_groups; ++g) {
        ELP_REQUIRE(groups[g].n_mul >= 0 && groups[g].n_mul <= ELP_MAX_GROUP_MUL, "lowered: group with %d multipliers", groups[g].n_mul);
        for (int k = 0; k < groups[g].n_mul; ++k) {
            ELP_REQUIRE(groups[g].mul_tab[k] >= 0 && groups[g].mul_tab[k] < std::max<int64_t>(n_dtab, 1), "lowered: multiplier outside dtab");
            if (groups[g].mul_per_row[k] && (size_t)g < n_g && g_hi[g] >= 0) {
                // asm_finish_group reads dtab[mul_tab + (row - row0)]: the table must cover every row the group's families touch
                ELP_REQUIRE(groups[g].row0 <= g_lo[g], "lowered: group %d has a per-row multiplier but starts at row %d, after its first term row %lld",
                            g, groups[g].row0, (long long)g_lo[g]);
                ELP_REQUIRE(groups[g].mul_tab[k] + (g_hi[g] - groups[g].row0) < n_dtab,
                            "lowered: per-row multiplier table of group %d ends before row %lld", g, (long long)g_hi[g]);
            }
        }
    }
    const size_t T = (size_t)(n_terms + total);
    ELP_REQUIRE(T < 0xffffffffull, "lowered: too many terms");
    const AsmIo io = asm_io_buffers(std::max<size_t>(T, 1), (size_t)m_alloc);
    const AsmLowered lo = asm_lowered_buffers(T, (size_t)n_itab, (size_t)n_dtab, groups ? (size_t)n_groups : 0);
    if (n_terms) {
        ELP_CUDA(cudaMemcpyAsync(io.row, term_row, (size_t)n_terms * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        ELP_CUDA(cudaMemcpyAsync(io.col, term_col, (size_t)n_terms * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        ELP_CUDA(cudaMemcpyAsync(io.val, term_val, (size_t)n_terms * sizeof(double), cudaMemcpyHostToDevice, st));
        ELP_CUDA(cudaMemsetAsync(lo.grp, 0, (size_t)n_terms * sizeof(int32_t), st));
    }
    if (n_itab) ELP_CUDA(cudaMemcpyAsync(lo.itab, itab, (size_t)n_itab * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (n_dtab) ELP_CUDA(cudaMemcpyAsync(lo.dtab, dtab, (size_t)n_dtab * sizeof(double), cudaMemcpyHostToDevice, st));
    if (n_groups && groups) ELP_CUDA(cudaMemcpyAsync(lo.groups, groups, (size_t)n_groups * sizeof(elp_fold_group), cudaMemcpyHostToDevice, st));
    asm_expand_families(n_families, families, lo.itab, lo.dtab, n_terms, io.row, io.col, io.val, lo.grp, st);
    *io_out = io; *lo_out = lo;
    return (int64_t)T;
}

int elp_assemble_lowered(int64_t n_terms, const int32_t* term_row, const int32_t* term_col, const double* term_val,
                         int32_t n_families, const elp_term_family* families, int64_t n_itab, const int32_t* itab,
                         int64_t n_dtab, const double* dtab, int32_t n_groups, const elp_fold_group* groups, int32_t m,
                         int32_t n, int32_t* row_ptr, int32_t* col_idx, double* vals, int64_t capacity, int64_t* nnz_out,
                         elp_stats* stats) {
    ELP_TRY
    require_device();
    WallTimer wall;
    const int64_t l0 = g_launches.load();
    ELP_REQUIRE(m >= 0 && n >= 0 && row_ptr && nnz_out, "lowered: bad arguments");
    cudaStream_t st = 0;
    EventPair ev;
    cudaEvent_t e0 = ev.a, e1 = ev.b;
    AsmIo io; AsmLowered lo;
    ELP_CUDA(cudaEventRecord(e0, st));
    const int64_t T = stage_lowered(n_terms, term_row, term_col, term_val, n_families, families, n_itab, itab, n_dtab, dtab,
                                    n_groups, groups, m, &io, &lo, st);
    const int64_t nnz = assemble_csr_device(T, io.row, io.col, io.val, m, n, io.out_ptr, io.out_col, io.out_val, st,
                                            lo.grp, lo.groups, lo.dtab);
    ELP_CUDA(cudaEventRecord(e1, st));
    ELP_REQUIRE(nnz <= capacity, "lowered: %lld non-zeros but room for %lld", (long long)nnz, (long long)capacity);
    ELP_CUDA(cudaMemcpyAsync(row_ptr, io.out_ptr, ((size_t)m + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (nnz) {
        ELP_CUDA(cudaMemcpyAsync(col_idx, io.out_col, (size_t)nnz * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaMemcpyAsync(vals, io.out_val, (size_t)nnz * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    ELP_CUDA(cudaStreamSynchronize(st));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    *nnz_out = nnz;
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->solve_ms = ms;                      // expansion + assembly (uploads of the descriptor tables included)
        stats->total_ms = wall.ms();
        stats->kernel_launches = g_launches.load() - l0;
        stats->iterations = (int32_t)std::min<int64_t>(T, 0x7fffffff);     // terms that went through the fold
        stats->h2d_bytes = n_terms * 16 + n_itab * 4 + n_dtab * 8 + (int64_t)n_groups * (int64_t)sizeof(elp_fold_group);
        stats->d2h_bytes = nnz * 12 + ((int64_t)m + 1) * 4;
    }
    ELP_CATCH
}

int elp_expand_terms(int32_t n_families, const elp_term_family* families, int64_t n_itab, const int32_t* itab,
                     int64_t n_dtab, const double* dtab, int32_t* row, int32_t* col, double* val, int32_t* group) {
    ELP_TRY
    require_device();
    cudaStream_t st = 0;
    AsmIo io; AsmLowered lo;
    const int64_t T = stage_lowered(0, nullptr, nullptr, nullptr, n_families, families, n_itab, itab, n_dtab, dtab,
                                    0x7fffffff, nullptr, 0, &io, &lo, st, true);
    if (T) {
        ELP_CUDA(cudaMemcpyAsync(row, io.row, (size_t)T * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaMemcpyAsync(col, io.col, (size_t)T * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaMemcpyAsync(val, io.val, (size_t)T * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (group) ELP_CUDA(cudaMemcpyAsync(group, lo.grp, (size_t)T * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        ELP_CUDA(cudaStreamSynchronize(st));
    }
    ELP_CATCH
}

static void solve_small(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                        const int8_t* sense, const double* rhs, const double* c, int32_t maximize, const double* lb,
                        const double* ub, const elp_options& o, int32_t* status, double* objval, double* x, double* y,
                        elp_stats* stats) {
    WallTimer wall;
    const int64_t l0 = g_launches.load();
    cudaStream_t st = 0;
    const int64_t nnz = m > 0 ? row_ptr[m] : 0;
    // a dozen small buffers: one allocation (cudaMalloc costs milliseconds per call, more than this whole solve)
    Arena arena;
    arena.reserve((size_t)8 * ((size_t)std::max(m, 1) * n + 2 * (size_t)std::max<int64_t>(nnz, 1) + 4 * (size_t)std::max(m, 1) + 5 * (size_t)n) + 16 * 512);
    ArenaScope scope(arena.base ? &arena : nullptr);
    DevBuf<int> ptr((size_t)m + 1), idx(std::max<int64_t>(nnz, 1));
    DevBuf<double> val(std::max<int64_t>(nnz, 1)), A((size_t)std::max(m, 1) * n), b(std::max(m, 1)), cd(n), lbd(n), ubd(n),
        obj(1), xd(n), yd(std::max(m, 1));
    DevBuf<int8_t> sd(std::max(m, 1));
    DevBuf<int32_t> stat(1), piv(1);
    if (m > 0) { ptr.upload(row_ptr, (size_t)m + 1, st); idx.upload(col_idx, nnz, st); val.upload(vals, nnz, st);
                 b.upload(rhs, m, st); sd.upload(sense, m, st); }
    cd.upload(c, n, st); lbd.upload(lb, n, st); ubd.upload(ub, n, st);
    EventPair ev;
    cudaEvent_t e0 = ev.a, e1 = ev.b;
    ELP_CUDA(cudaEventRecord(e0, st));
    densify_device(m, n, ptr.p, idx.p, val.p, A.p, st);
    const int ctas = simplex_batch_device(1, m, n, A.p, b.p, cd.p, lbd.p, ubd.p, sd.p, maximize, o.max_iter, stat.p, obj.p,
                                          xd.p, yd.p, piv.p, st);
    ELP_CUDA(cudaEventRecord(e1, st));
    int32_t s = 0, pv = 0;
    stat.download(&s, 1, st); piv.download(&pv, 1, st); obj.download(objval, 1, st); xd.download(x, n, st);
    if (y && m > 0) yd.download(y, m, st);
    ELP_CUDA(cudaStreamSynchronize(st));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    *status = s;
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->status = s;
        stats->method_used = ELP_METHOD_SIMPLEX;
        stats->iterations = pv;
        stats->primal_obj = *objval;
        stats->dual_obj = *objval;
        stats->solve_ms = ms;
        stats->total_ms = wall.ms();
        stats->kernel_launches = g_launches.load() - l0;
        stats->h2d_bytes = nnz * 12 + (int64_t)m * 13 + (int64_t)n * 24;
        stats->d2h_bytes = (int64_t)n * 8 + (int64_t)m * 8 + 16;
        stats->simplex_ctas = ctas;
    }
}

// PDLP on one GPU.  nnz_device >= 0: the CSR arrays are device pointers (elp_model_*).
static void solve_large(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                        int64_t nnz_device, const int8_t* sense, const double* rhs, const double* c, int32_t maximize,
                        const double* lb, const double* ub, const elp_options& o, int32_t* status, double* objval,
                        double* x, double* y, elp_stats* stats) {
    WallTimer wall;
    bool bad_bounds = false;
    for (int j = 0; j < n; ++j) if (lb[j] > ub[j]) { bad_bounds = true; break; }
    elp_stats s1;
    memset(&s1, 0, sizeof s1);
    Pdlp* p = pdlp_create(m, n, row_ptr, col_idx, vals, sense, rhs, c, maximize, lb, ub, o, false, &s1, nnz_device);
    try {
        elp_stats s2;
        memset(&s2, 0, sizeof s2);
        if (!bad_bounds) pdlp_run(p, 0, &s2);
        pdlp_solution(p, x, y, objval);
        *status = bad_bounds ? ELP_STATUS_INFEASIBLE : s2.status;
        if (*status == ELP_STATUS_UNBOUNDED) *objval = maximize ? INFINITY : -INFINITY;
        if (stats) {
            *stats = s2;
            stats->status = *status;
            stats->setup_ms = s1.setup_ms;
            stats->total_ms = wall.ms();
        }
    } catch (...) {
        pdlp_destroy(p);
        throw;
    }
    pdlp_destroy(p);
}

int elp_solve_lp(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                 const int8_t* sense, const double* rhs, const double* c, int32_t maximize, const double* lb,
                 const double* ub, const elp_options* opt, int32_t* status, double* objval, double* x, double* y,
                 elp_stats* stats) {
    ELP_TRY
    require_device();
    ELP_REQUIRE(n > 0, "Problem contains no variables.");   // R/class.R:253-254
    ELP_REQUIRE(m >= 0 && status && objval && x && c && lb && ub, "elp_solve_lp: bad arguments");
    const elp_options o = effective_options(opt);
    int method = o.method;
    if (method == ELP_METHOD_AUTO)   // size rule, not a backend switch: does the dense tableau fit in one SM?
        method = simplex_auto_prefers(m, n) ? ELP_METHOD_SIMPLEX : ELP_METHOD_PDLP;
    // any block with lower > upper forces "unfeasible" (R/class.R:297-298); both solvers also detect it
    if (method == ELP_METHOD_SIMPLEX)
        solve_small(m, n, row_ptr, col_idx, vals, sense, rhs, c, maximize, lb, ub, o, status, objval, x, y, stats);
    else if (o.devices > 1)      // the large-LP path over several GPUs of the box, still one blocking call
        solve_multi(m, n, row_ptr, col_idx, vals, sense, rhs, c, maximize, lb, ub, o, status, objval, x, y, stats);
    else
        solve_large(m, n, row_ptr, col_idx, vals, -1, sense, rhs, c, maximize, lb, ub, o, status, objval, x, y, stats);
    ELP_CATCH
}

int elp_solve_mip(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                  const int8_t* sense, const double* rhs, const double* c, int32_t maximize, const double* lb,
                  const double* ub, const uint8_t* is_integer, const elp_options* opt, int32_t* status, double* objval,
                  double* x, elp_stats* stats) {
    ELP_TRY
    require_device();
    ELP_REQUIRE(n > 0, "Problem contains no variables.");   // R/class.R:253-254
    ELP_REQUIRE(m >= 0 && status && objval && x && c && lb && ub && is_integer, "elp_solve_mip: bad arguments");
    const elp_options o = effective_options(opt);
    bool any = false, bad_bounds = false;
    for (int j = 0; j < n; ++j) { any = any || is_integer[j] != 0; bad_bounds = bad_bounds || lb[j] > ub[j]; }
    if (bad_bounds) {                                        // R/class.R:297-298
        *status = ELP_STATUS_INFEASIBLE; *objval = 0.0;
        for (int j = 0; j < n; ++j) x[j] = 0.0;
        if (stats) { memset(stats, 0, sizeof *stats); stats->status = *status; stats->method_used = ELP_METHOD_SIMPLEX; }
    } else if (!any) {                                       // no integer column after all: the plain LP path
        solve_small(m, n, row_ptr, col_idx, vals, sense, rhs, c, maximize, lb, ub, o, status, objval, x, nullptr, stats);
    } else {
        solve_mip(m, n, row_ptr, col_idx, vals, sense, rhs, c, maximize, lb, ub, is_integer, o, status, objval, x, stats);
    }
    ELP_CATCH
}

int elp_sensitivity(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                    const int8_t* sense, const double* rhs, const double* c, int32_t maximize, const double* lb,
                    const double* ub, const elp_options* opt, int32_t* status, double* objval, double* x, double* obj_from,
                    double* obj_till, double* rhs_from, double* rhs_till, double* duals) {
    ELP_TRY
    require_device();
    ELP_REQUIRE(n > 0, "Problem contains no variables.");
    ELP_REQUIRE(m >= 0 && status && objval && x && c && lb && ub && obj_from && obj_till && (m == 0 || (rhs_from && rhs_till && duals)),
                "elp_sensitivity: bad arguments");
    const elp_options o = effective_options(opt);
    sensitivity(m, n, row_ptr, col_idx, vals, sense, rhs, c, maximize, lb, ub, o, status, objval, x, obj_from, obj_till, rhs_from,
                rhs_till, duals);
    ELP_CATCH
}

/* ---- device-resident model: assembled once, solved (and re-solved) without the CSR crossing PCIe again ---- */
struct Model {
    int32_t m = 0, n = 0;
    int64_t nnz = 0;
    DevBuf<unsigned char> slab;          // ONE allocation (cudaMalloc costs 2-13 ms per call on these boxes, with outliers):
    DevBuf<int32_t> ptr, idx;            // ptr, idx and val are views into it
    DevBuf<double> val;
    void alloc(size_t m1, size_t nz) {
        auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t b_val = up(nz * sizeof(double)), b_idx = up(nz * sizeof(int32_t)), b_ptr = up(m1 * sizeof(int32_t));
        slab.alloc(b_val + b_idx + b_ptr);
        val.p = reinterpret_cast<double*>(slab.p); val.n = nz; val.owned = false;
        idx.p = reinterpret_cast<int32_t*>(slab.p + b_val); idx.n = nz; idx.owned = false;
        ptr.p = reinterpret_cast<int32_t*>(slab.p + b_val + b_idx); ptr.n = m1; ptr.owned = false;
    }
};

int elp_model_assemble(int64_t n_terms, const int32_t* term_row, const int32_t* term_col, const double* term_val,
                       int32_t n_families, const elp_term_family* families, int64_t n_itab, const int32_t* itab,
                       int64_t n_dtab, const double* dtab, int32_t n_groups, const elp_fold_group* groups, int32_t m,
                       int32_t n, elp_model** out, int64_t* nnz_out, elp_stats* stats) {
    ELP_TRY
    require_device();
    WallTimer wall;
    const int64_t l0 = g_launches.load();
    ELP_REQUIRE(m >= 0 && n >= 0 && out, "elp_model_assemble: bad arguments");
    cudaStream_t st = 0;
    EventPair ev;
    cudaEvent_t e0 = ev.a, e1 = ev.b;
    AsmIo io; AsmLowered lo;
    ELP_CUDA(cudaEventRecord(e0, st));
    const int64_t T = stage_lowered(n_terms, term_row, term_col, term_val, n_families, families, n_itab, itab, n_dtab, dtab,
                                    n_groups, groups, m, &io, &lo, st);
    const int64_t nnz = assemble_csr_device(T, io.row, io.col, io.val, m, n, io.out_ptr, io.out_col, io.out_val, st,
                                            lo.grp, lo.groups, lo.dtab);
    auto* h = new Model();
    try {
        h->m = m; h->n = n; h->nnz = nnz;
        h->alloc((size_t)m + 1, (size_t)std::max<int64_t>(nnz, 1));
        ELP_CUDA(cudaMemcpyAsync(h->ptr.p, io.out_ptr, ((size_t)m + 1) * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        if (nnz) {
            ELP_CUDA(cudaMemcpyAsync(h->idx.p, io.out_col, (size_t)nnz * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
            ELP_CUDA(cudaMemcpyAsync(h->val.p, io.out_val, (size_t)nnz * sizeof(double), cudaMemcpyDeviceToDevice, st));
        }
        ELP_CUDA(cudaEventRecord(e1, st));
        ELP_CUDA(cudaStreamSynchronize(st));
    } catch (...) {
        delete h;
        throw;
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    *out = reinterpret_cast<elp_model*>(h);
    if (nnz_out) *nnz_out = nnz;
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->solve_ms = ms;
        stats->total_ms = wall.ms();
        stats->kernel_launches = g_launches.load() - l0;
        stats->iterations = (int32_t)std::min<int64_t>(T, 0x7fffffff);
        stats->h2d_bytes = n_terms * 16 + n_itab * 4 + n_dtab * 8 + (int64_t)n_groups * (int64_t)sizeof(elp_fold_group);
    }
    ELP_CATCH
}

int elp_model_dims(const elp_model* hh, int32_t* m, int32_t* n, int64_t* nnz) {
    ELP_TRY
    auto* h = reinterpret_cast<const Model*>(hh);
    ELP_REQUIRE(h, "elp_model_dims: null handle");
    if (m) *m = h->m;
    if (n) *n = h->n;
    if (nnz) *nnz = h->nnz;
    ELP_CATCH
}

int elp_model_csr(const elp_model* hh, int32_t* row_ptr, int32_t* col_idx, double* vals) {
    ELP_TRY
    auto* h = reinterpret_cast<const Model*>(hh);
    ELP_REQUIRE(h && row_ptr, "elp_model_csr: bad arguments");
    cudaStream_t st = 0;
    ELP_CUDA(cudaMemcpyAsync(row_ptr, h->ptr.p, ((size_t)h->m + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (h->nnz && col_idx) ELP_CUDA(cudaMemcpyAsync(col_idx, h->idx.p, (size_t)h->nnz * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (h->nnz && vals) ELP_CUDA(cudaMemcpyAsync(vals, h->val.p, (size_t)h->nnz * sizeof(double), cudaMemcpyDeviceToHost, st));
    ELP_CUDA(cudaStreamSynchronize(st));
    ELP_CATCH
}

int elp_model_solve(const elp_model* hh, const int8_t* sense, const double* rhs, const double* c, int32_t maximize,
                    const double* lb, const double* ub, const elp_options* opt, int32_t* status, double* objval, double* x,
                    double* y, elp_stats* stats) {
    ELP_TRY
    require_device();
    auto* h = reinterpret_cast<const Model*>(hh);
    ELP_REQUIRE(h && status && objval && x && c && lb && ub, "elp_model_solve: bad arguments");
    ELP_REQUIRE(h->n > 0, "Problem contains no variables.");
    const elp_options o = effective_options(opt);
    int method = o.method;
    if (method == ELP_METHOD_AUTO)
        method = simplex_auto_prefers(h->m, h->n) ? ELP_METHOD_SIMPLEX : ELP_METHOD_PDLP;
    if (method == ELP_METHOD_SIMPLEX) {          // a tableau that fits one SM: the few KB of CSR go through the host path
        std::vector<int32_t> rp((size_t)h->m + 1), ci((size_t)std::max<int64_t>(h->nnz, 1));
        std::vector<double> v((size_t)std::max<int64_t>(h->nnz, 1));
        ELP_REQUIRE(elp_model_csr(hh, rp.data(), ci.data(), v.data()) == 0, "%s", g_last_error.c_str());
        solve_small(h->m, h->n, rp.data(), ci.data(), v.data(), sense, rhs, c, maximize, lb, ub, o, status, objval, x, y, stats);
    } else if (o.devices > 1) {
        // several GPUs: the row blocks travel from this device's copy through the host (one D2H of the CSR; the blocks
        // then go straight to their GPUs)
        std::vector<int32_t> rp((size_t)h->m + 1), ci((size_t)std::max<int64_t>(h->nnz, 1));
        std::vector<double> v((size_t)std::max<int64_t>(h->nnz, 1));
        ELP_REQUIRE(elp_model_csr(hh, rp.data(), ci.data(), v.data()) == 0, "%s", g_last_error.c_str());
        solve_multi(h->m, h->n, rp.data(), ci.data(), v.data(), sense, rhs, c, maximize, lb, ub, o, status, objval, x, y, stats);
    } else {
        solve_large(h->m, h->n, h->ptr.p, h->idx.p, h->val.p, h->nnz, sense, rhs, c, maximize, lb, ub, o, status, objval, x, y,
                    stats);
    }
    ELP_CATCH
}

int elp_model_destroy(elp_model* hh) {
    ELP_TRY
    delete reinterpret_cast<Model*>(hh);
    ELP_CATCH
}

int elp_batch_create(int64_t B, int32_t m, int32_t n, const double* A, const double* b, const double* c,
                     const double* lb, const double* ub, const int8_t* sense, int32_t maximize, elp_batch** out) {
    ELP_TRY
    require_device();
    ELP_REQUIRE(B > 0 && m >= 0 && n > 0 && A && b && c && out, "elp_batch_create: bad arguments");
    auto* h = new Batch();
    try {
        cudaStream_t st = 0;
        h->B = B; h->m = m; h->n = n; h->maximize = maximize;
        h->A.alloc((size_t)B * m * n); h->b.alloc((size_t)B * m); h->c.alloc((size_t)B * n);
        h->A.upload(A, (size_t)B * m * n, st); h->b.upload(b, (size_t)B * m, st); h->c.upload(c, (size_t)B * n, st);
        h->h2d = (int64_t)B * (m * n + m + n) * 8;
        if (lb) { h->lb.alloc((size_t)B * n); h->lb.upload(lb, (size_t)B * n, st); h->has_lb = true; h->h2d += (int64_t)B * n * 8; }
        if (ub) { h->ub.alloc((size_t)B * n); h->ub.upload(ub, (size_t)B * n, st); h->has_ub = true; h->h2d += (int64_t)B * n * 8; }
        if (sense) { h->sense.alloc((size_t)B * m); h->sense.upload(sense, (size_t)B * m, st); h->has_sense = true; h->h2d += (int64_t)B * m; }
        h->obj.alloc(B); h->x.alloc((size_t)B * n); h->status.alloc(B); h->pivots.alloc(B);
        ELP_CUDA(cudaStreamSynchronize(st));
    } catch (...) {
        delete h;
        throw;
    }
    *out = reinterpret_cast<elp_batch*>(h);
    ELP_CATCH
}

int elp_batch_run(elp_batch* hh, const elp_options* opt, elp_stats* stats) {
    ELP_TRY
    auto* h = reinterpret_cast<Batch*>(hh);
    ELP_REQUIRE(h, "elp_batch_run: null handle");
    const elp_options o = effective_options(opt);
    WallTimer wall;
    const int64_t l0 = g_launches.load();
    cudaStream_t st = 0;
    EventPair ev;
    cudaEvent_t e0 = ev.a, e1 = ev.b;
    ELP_CUDA(cudaEventRecord(e0, st));
    const int ctas = simplex_batch_device(h->B, h->m, h->n, h->A.p, h->b.p, h->c.p, h->has_lb ? h->lb.p : nullptr,
                                          h->has_ub ? h->ub.p : nullptr, h->has_sense ? h->sense.p : nullptr, h->maximize,
                                          o.max_iter, h->status.p, h->obj.p, h->x.p, nullptr, h->pivots.p, st);
    ELP_CUDA(cudaEventRecord(e1, st));
    ELP_CUDA(cudaStreamSynchronize(st));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->method_used = ELP_METHOD_SIMPLEX;
        stats->solve_ms = ms;
        stats->total_ms = wall.ms();
        stats->kernel_launches = g_launches.load() - l0;
        stats->simplex_ctas = ctas;
    }
    ELP_CATCH
}

int elp_batch_fetch(elp_batch* hh, int32_t* status, double* obj, double* x) {
    ELP_TRY
    auto* h = reinterpret_cast<Batch*>(hh);
    ELP_REQUIRE(h, "elp_batch_fetch: null handle");
    cudaStream_t st = 0;
    if (status) h->status.download(status, h->B, st);
    if (obj) h->obj.download(obj, h->B, st);
    if (x) h->x.download(x, (size_t)h->B * h->n, st);
    ELP_CUDA(cudaStreamSynchronize(st));
    ELP_CATCH
}

int elp_batch_destroy(elp_batch* hh) {
    ELP_TRY
    delete reinterpret_cast<Batch*>(hh);
    ELP_CATCH
}

// Host-buffer entry point: the batch is streamed through the GPU in chunks.  Chunk i's host->device copies, its kernel
// and its device->host copies are queued on stream i % 3, each slot with its own device buffers, so the copy engines
// (both directions) and the SMs work on different chunks at the same time; with page-locked caller buffers the call runs
// at PCIe speed (5.7 KB per 20x30 LP in, 0.25 KB out).  Device buffers, streams and the pinned pivot counters come from
// a grow-only per-thread workspace (elp_release_workspace frees it).
int elp_solve_batch(int64_t B, int32_t m, int32_t n, const double* A, const double* b, const double* c,
                    const double* lb, const double* ub, const int8_t* sense, int32_t maximize, const elp_options* opt,
                    int32_t* status, double* obj, double* x, elp_stats* stats) {
    ELP_TRY
    WallTimer wall;
    require_device();
    ELP_REQUIRE(B > 0 && m >= 0 && n > 0 && A && b && c, "elp_solve_batch: bad arguments");
    ELP_REQUIRE(status && obj && x, "elp_solve_batch: status, obj and x must be provided");
    const elp_options o = effective_options(opt);
    const int64_t l0 = g_launches.load();
    BatchStreamWorkspace& w = batch_stream_workspace();
    // chunk size: ~64 MB of input per chunk, at least 3 chunks when the batch is worth splitting, at most B
    const int64_t in_per_lp = (int64_t)8 * ((int64_t)m * n + m + n) + (lb ? 8 * n : 0) + (ub ? 8 * n : 0) + (sense ? m : 0);
    int64_t chunk = std::max<int64_t>(1, (64ll << 20) / std::max<int64_t>(in_per_lp, 1));
    if (B >= 3 * 4096) chunk = std::min(chunk, (B + 2) / 3);
    chunk = std::min(chunk, B);
    const int64_t nchunks = (B + chunk - 1) / chunk;
    w.ensure((size_t)chunk, (size_t)B, m, n, lb != nullptr, ub != nullptr, sense != nullptr);
    EventPair ev;
    cudaEvent_t e0 = ev.a, e1 = ev.b;
    ELP_CUDA(cudaEventRecord(e0, w.st[0]));
    int ctas = 0;
    for (int64_t i = 0; i < nchunks; ++i) {
        const int s = (int)(i % BatchStreamWorkspace::NS);
        cudaStream_t st = w.st[s];
        const int64_t lo = i * chunk, cnt = std::min(chunk, B - lo);
        const size_t mn = (size_t)m * n;
        w.A[s].upload(A + lo * mn, (size_t)cnt * mn, st);
        w.b[s].upload(b + lo * m, (size_t)cnt * m, st);
        w.c[s].upload(c + lo * n, (size_t)cnt * n, st);
        if (lb) w.lb[s].upload(lb + lo * n, (size_t)cnt * n, st);
        if (ub) w.ub[s].upload(ub + lo * n, (size_t)cnt * n, st);
        if (sense) w.sense[s].upload(sense + lo * m, (size_t)cnt * m, st);
        ctas = simplex_batch_device(cnt, m, n, w.A[s].p, w.b[s].p, w.c[s].p, lb ? w.lb[s].p : nullptr,
                                    ub ? w.ub[s].p : nullptr, sense ? w.sense[s].p : nullptr, maximize, o.max_iter,
                                    w.status[s].p, w.obj[s].p, w.x[s].p, nullptr, w.piv[s].p, st);
        w.status[s].download(status + lo, (size_t)cnt, st);
        w.obj[s].download(obj + lo, (size_t)cnt, st);
        w.x[s].download(x + lo * n, (size_t)cnt * n, st);
        ELP_CUDA(cudaMemcpyAsync(w.piv_host + lo, w.piv[s].p, (size_t)cnt * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    }
    for (int s = 1; s < BatchStreamWorkspace::NS; ++s) {     // join the other slots into stream 0 for the closing event
        ELP_CUDA(cudaEventRecord(w.done[s], w.st[s]));
        ELP_CUDA(cudaStreamWaitEvent(w.st[0], w.done[s], 0));
    }
    ELP_CUDA(cudaEventRecord(e1, w.st[0]));
    ELP_CUDA(cudaStreamSynchronize(w.st[0]));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->method_used = ELP_METHOD_SIMPLEX;
        stats->solve_ms = ms;                       // device time of the whole streamed call (copies included)
        stats->kernel_launches = g_launches.load() - l0;
        stats->h2d_bytes = B * in_per_lp;
        stats->d2h_bytes = B * ((int64_t)n * 8 + 16);
        int64_t piv = 0;
        for (int64_t i = 0; i < B; ++i) piv += w.piv_host[i];
        stats->iterations = (int32_t)std::min<int64_t>(piv, 0x7fffffff);
        stats->total_ms = wall.ms();
        stats->simplex_ctas = ctas;
    }
    ELP_CATCH
}

int elp_spmv(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals, const double* x,
             double* out) {
    ELP_TRY
    require_device();
    spmv_host(m, n, row_ptr, col_idx, vals, x, out, nullptr, nullptr, 0.0, nullptr);
    ELP_CATCH
}

int elp_check_feasible(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                       const double* x, const int8_t* sense, const double* rhs, double tol, uint8_t* feasible) {
    ELP_TRY
    require_device();
    spmv_host(m, n, row_ptr, col_idx, vals, x, nullptr, sense, rhs, tol, feasible);
    ELP_CATCH
}

int elp_pdlp_create(int32_t m_local, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                    const int8_t* sense, const double* rhs, const double* c, int32_t maximize, const double* lb,
                    const double* ub, const elp_options* opt, int32_t dist, elp_pdlp** out, elp_stats* stats) {
    ELP_TRY
    require_device();
    ELP_REQUIRE(out, "elp_pdlp_create: null out");
    if (stats) memset(stats, 0, sizeof *stats);
    const elp_options o = effective_options(opt);
    *out = reinterpret_cast<elp_pdlp*>(
        pdlp_create(m_local, n, row_ptr, col_idx, vals, sense, rhs, c, maximize, lb, ub, o, dist != 0, stats));
    ELP_CATCH
}
int elp_model_pdlp_create(const elp_model* hh, const int8_t* sense, const double* rhs, const double* c, int32_t maximize,
                          const double* lb, const double* ub, const elp_options* opt, elp_pdlp** out, elp_stats* stats) {
    ELP_TRY
    require_device();
    auto* h = reinterpret_cast<const Model*>(hh);
    ELP_REQUIRE(h && out && c && lb && ub, "elp_model_pdlp_create: bad arguments");
    ELP_REQUIRE(h->n > 0, "Problem contains no variables.");
    if (stats) memset(stats, 0, sizeof *stats);
    const elp_options o = effective_options(opt);
    *out = reinterpret_cast<elp_pdlp*>(pdlp_create(h->m, h->n, h->ptr.p, h->idx.p, h->val.p, sense, rhs, c, maximize, lb, ub, o,
                                                   false, stats, h->nnz));
    ELP_CATCH
}
int elp_pdlp_run(elp_pdlp* h, int32_t max_new_iters, elp_stats* stats) {
    ELP_TRY
    ELP_REQUIRE(h, "null handle");
    if (stats) memset(stats, 0, sizeof *stats);
    pdlp_run(reinterpret_cast<Pdlp*>(h), max_new_iters, stats);
    ELP_CATCH
}
int elp_pdlp_reset(elp_pdlp* h) {
    ELP_TRY
    ELP_REQUIRE(h, "null handle");
    pdlp_reset(reinterpret_cast<Pdlp*>(h));
    ELP_CATCH
}
int elp_pdlp_solution(elp_pdlp* h, double* x, double* y, double* objval) {
    ELP_TRY
    ELP_REQUIRE(h, "null handle");
    pdlp_solution(reinterpret_cast<Pdlp*>(h), x, y, objval);
    ELP_CATCH
}
int elp_pdlp_probe_spmv(elp_pdlp* h, int32_t reps, double* ms_csr, double* ms_csc) {
    ELP_TRY
    ELP_REQUIRE(h && reps > 0, "bad arguments");
    pdlp_probe(reinterpret_cast<Pdlp*>(h), reps, ms_csr, ms_csc);
    ELP_CATCH
}
int elp_pdlp_probe_step(elp_pdlp* h, int32_t reps, double* ms_primal, double* ms_dual) {
    ELP_TRY
    ELP_REQUIRE(h && reps > 0, "bad arguments");
    pdlp_probe_step(reinterpret_cast<Pdlp*>(h), reps, ms_primal, ms_dual);
    ELP_CATCH
}
int elp_pdlp_transpose(elp_pdlp* h, int32_t* mode) {
    ELP_TRY
    ELP_REQUIRE(h && mode, "bad arguments");
    *mode = pdlp_transpose(reinterpret_cast<Pdlp*>(h));
    ELP_CATCH
}
int elp_pdlp_destroy(elp_pdlp* h) {
    ELP_TRY
    if (h) pdlp_destroy(reinterpret_cast<Pdlp*>(h));
    ELP_CATCH
}

int elp_comm_unique_id(void* id) {
    ELP_TRY
    comm_unique_id(id);
    ELP_CATCH
}
int elp_comm_init(int32_t nranks, int32_t rank, const void* id) {
    ELP_TRY
    require_device();
    comm_init(nranks, rank, id);
    ELP_CATCH
}
int elp_comm_size(int32_t* nranks, int32_t* rank) {
    ELP_TRY
    if (nranks) *nranks = comm().nranks;
    if (rank) *rank = comm().rank;
    ELP_CATCH
}
int elp_comm_destroy(void) {
    ELP_TRY
    comm_destroy();
    ELP_CATCH
}

}  // extern "C"
