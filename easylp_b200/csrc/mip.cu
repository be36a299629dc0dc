// mip.cu — branch and bound for models with integer / binary variables, on top of the batched simplex kernel.
//
// Replaces what `status <- solve(prob)` does after `set.type(prob, columns, "integer" | "binary")`
// (/root/reference/R/class.R:264-276): lp_solve's branch and bound.  The reference's own tests and vignettes use it
// (tests/testthat/test-cyingair.R:8-9, test-investments.R:28, test-students.R:31, test-associate.R:5-6,
// vignettes/easylp.Rmd:55).
//
// B200 formulation: the open nodes of the tree are LPs that share A, b, c and the row senses and differ only in the
// variable bounds, so a whole FRONTIER is one launch of the batched simplex kernel (simplex.cu, shared_model = 1: one
// LP per warp, CTA or cluster, the tableau in shared memory; the matrix is read once per node from the L2-resident copy).  The host
// keeps the tree: best-bound-first order, up to `wave` nodes per launch, prune by bound against the incumbent,
// branch on the lowest-indexed fractional integer column (lp_solve's default NODE_FIRSTSELECT) into
// x_j <= floor(v) and x_j >= ceil(v).  Integrality tolerance 1e-7 (lp_solve's default epsint), pruning gaps 1e-11
// absolute / 1e-9 relative (lp_solve's default mip_gap).  Status codes are lp_solve's: 0 optimal, 2 unfeasible,
// 3 unbounded, 1 sub-optimal (a node / time limit stopped the search with an incumbent), 7 timeout (without one).
//
// Scope: models whose dense tableau fits one SM's shared memory, or beyond that a thread-block cluster of up to 16
// CTAs (simplex.cu: simplex_ctas decides); larger MILPs are refused with an error naming the shape and the capacity.
#include "common.cuh"
#include "../../include/easylp_abi.h"
#include <algorithm>
#include <cmath>
#include <queue>
#include <vector>

namespace elp {

int simplex_ctas(int m, int n);
int simplex_batch_device(int64_t B, int m, int n, const double* A, const double* b, const double* c, const double* lb,
                         const double* ub, const int8_t* sense, int maximize, int max_pivots, int32_t* status,
                         double* obj, double* x, double* y, int32_t* pivots, cudaStream_t st, int shared_model,
                         int32_t* basis = nullptr);
void densify_device(int m, int n, const int* ptr, const int* idx, const double* val, double* A, cudaStream_t st);

namespace {
struct Node {
    std::vector<double> lb, ub;
    double bound;          // LP value of the parent, in "min" sense: no descendant can do better
    int depth;
};
struct NodeOrder {         // best bound first; deeper first among equals (finds incumbents sooner)
    bool operator()(const Node* a, const Node* b) const {
        if (a->bound != b->bound) return a->bound > b->bound;
        return a->depth < b->depth;
    }
};
}  // namespace

void solve_mip(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals, const int8_t* sense,
               const double* rhs, const double* c, int32_t maximize, const double* lb, const double* ub,
               const uint8_t* is_int, const elp_options& o, int32_t* status, double* objval, double* x, elp_stats* stats) {
    WallTimer wall;
    const int64_t l0 = g_launches.load();
    const int ctas = simplex_ctas(m, n);       // refuses a tableau larger than the largest cluster before any work
    cudaStream_t st = 0;
    const int64_t nnz = m > 0 ? row_ptr[m] : 0;
    const int WAVE = 4096;
    const double EPS_INT = 1e-7, GAP_ABS = 1e-11, GAP_REL = 1e-9;
    const int64_t node_limit = o.max_iter > 0 ? (int64_t)o.max_iter : 2000000;   // nodes, for this entry point

    // ---- the shared model, once ----------------------------------------------------------------------------------
    DevBuf<int> ptr((size_t)m + 1), idx(std::max<int64_t>(nnz, 1));
    DevBuf<double> val(std::max<int64_t>(nnz, 1)), A((size_t)std::max(m, 1) * n), b(std::max(m, 1)), cd(n);
    DevBuf<int8_t> sd(std::max(m, 1));
    if (m > 0) {
        ptr.upload(row_ptr, (size_t)m + 1, st); idx.upload(col_idx, nnz, st); val.upload(vals, nnz, st);
        b.upload(rhs, m, st); sd.upload(sense, m, st);
    }
    cd.upload(c, n, st);
    densify_device(m, n, ptr.p, idx.p, val.p, A.p, st);
    // ---- per-wave buffers ------------------------------------------------------------------------------------------
    DevBuf<double> lbd((size_t)WAVE * n), ubd((size_t)WAVE * n), objd(WAVE), xd((size_t)WAVE * n);
    DevBuf<int32_t> statd(WAVE), pivd(WAVE);
    std::vector<double> h_lb((size_t)WAVE * n), h_ub((size_t)WAVE * n), h_obj(WAVE), h_x((size_t)WAVE * n);
    std::vector<int32_t> h_stat(WAVE), h_piv(WAVE);

    std::priority_queue<Node*, std::vector<Node*>, NodeOrder> open;
    auto drop_all = [&]() { while (!open.empty()) { delete open.top(); open.pop(); } };
    {
        Node* root = new Node{std::vector<double>(lb, lb + n), std::vector<double>(ub, ub + n), -INFINITY, 0};
        for (int j = 0; j < n; ++j)
            if (is_int[j]) {                    // integer columns: bounds tightened to integers once
                if (std::isfinite(root->lb[j])) root->lb[j] = std::ceil(root->lb[j] - EPS_INT);
                if (std::isfinite(root->ub[j])) root->ub[j] = std::floor(root->ub[j] + EPS_INT);
            }
        open.push(root);
    }
    bool have = false, unbounded = false, failed = false, stopped = false;
    double best = INFINITY;                     // incumbent, "min" sense
    std::vector<double> best_x(n, 0.0);
    int64_t nodes = 0, pivots = 0;
    float dev_ms = 0.f;
    cudaEvent_t e0, e1;
    ELP_CUDA(cudaEventCreate(&e0)); ELP_CUDA(cudaEventCreate(&e1));
    try {
        while (!open.empty() && !unbounded && !failed) {
            if (nodes >= node_limit || (o.time_limit_s > 0 && wall.ms() > o.time_limit_s * 1e3)) { stopped = true; break; }
            const double cut = have ? best - std::max(GAP_ABS, GAP_REL * std::fabs(best)) : INFINITY;
            std::vector<Node*> wave;
            while (!open.empty() && (int)wave.size() < WAVE) {
                Node* nd = open.top();
                open.pop();
                if (nd->bound >= cut) { delete nd; continue; }          // pruned by bound while it waited
                wave.push_back(nd);
            }
            if (wave.empty()) break;
            const int W = (int)wave.size();
            for (int w = 0; w < W; ++w) {
                std::copy(wave[w]->lb.begin(), wave[w]->lb.end(), h_lb.begin() + (size_t)w * n);
                std::copy(wave[w]->ub.begin(), wave[w]->ub.end(), h_ub.begin() + (size_t)w * n);
            }
            lbd.upload(h_lb.data(), (size_t)W * n, st); ubd.upload(h_ub.data(), (size_t)W * n, st);
            ELP_CUDA(cudaEventRecord(e0, st));
            simplex_batch_device(W, m, n, A.p, b.p, cd.p, lbd.p, ubd.p, sd.p, maximize, 0, statd.p, objd.p, xd.p, nullptr,
                                 pivd.p, st, /*shared_model=*/1);
            ELP_CUDA(cudaEventRecord(e1, st));
            statd.download(h_stat.data(), W, st); objd.download(h_obj.data(), W, st); xd.download(h_x.data(), (size_t)W * n, st);
            pivd.download(h_piv.data(), W, st);
            ELP_CUDA(cudaStreamSynchronize(st));
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0, e1);
            dev_ms += ms;
            nodes += W;
            for (int w = 0; w < W; ++w) {
                Node* nd = wave[w];
                pivots += h_piv[w];
                const int s = h_stat[w];
                if (s == ELP_STATUS_INFEASIBLE) { delete nd; continue; }
                if (s == ELP_STATUS_UNBOUNDED) { unbounded = true; delete nd; continue; }     // lp_solve: UNBOUNDED
                if (s != ELP_STATUS_OPTIMAL) { failed = true; delete nd; continue; }
                const double v = maximize ? -h_obj[w] : h_obj[w];
                const double cut_now = have ? best - std::max(GAP_ABS, GAP_REL * std::fabs(best)) : INFINITY;
                if (v >= cut_now) { delete nd; continue; }
                const double* xs = h_x.data() + (size_t)w * n;
                int jf = -1;
                for (int j = 0; j < n; ++j)
                    if (is_int[j] && std::fabs(xs[j] - std::nearbyint(xs[j])) > EPS_INT) { jf = j; break; }
                if (jf < 0) {                       // integral: new incumbent
                    have = true; best = v;
                    std::copy(xs, xs + n, best_x.begin());
                    delete nd;
                    continue;
                }
                Node* up = new Node{nd->lb, nd->ub, v, nd->depth + 1};
                nd->ub[jf] = std::floor(xs[jf]);    // the node itself becomes the "down" child
                nd->bound = v; nd->depth += 1;
                up->lb[jf] = std::ceil(xs[jf]);
                open.push(nd);
                open.push(up);
            }
        }
    } catch (...) {
        drop_all();
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        throw;
    }
    drop_all();
    cudaEventDestroy(e0); cudaEventDestroy(e1);

    if (unbounded) {
        *status = ELP_STATUS_UNBOUNDED;
        *objval = maximize ? INFINITY : -INFINITY;
        for (int j = 0; j < n; ++j) x[j] = 0.0;
    } else if (failed) {
        *status = ELP_STATUS_NUMFAILURE;
        *objval = 0.0;
        for (int j = 0; j < n; ++j) x[j] = 0.0;
    } else if (have) {
        *status = stopped ? ELP_STATUS_SUBOPTIMAL : ELP_STATUS_OPTIMAL;
        *objval = maximize ? -best : best;
        std::copy(best_x.begin(), best_x.end(), x);
    } else {
        *status = stopped ? ELP_STATUS_TIMEOUT : ELP_STATUS_INFEASIBLE;
        *objval = 0.0;
        for (int j = 0; j < n; ++j) x[j] = 0.0;
    }
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->status = *status;
        stats->method_used = ELP_METHOD_SIMPLEX;
        stats->iterations = (int32_t)std::min<int64_t>(pivots, 0x7fffffff);
        stats->restarts = (int32_t)std::min<int64_t>(nodes, 0x7fffffff);        // branch-and-bound nodes solved
        stats->simplex_ctas = ctas;
        stats->primal_obj = *objval;
        stats->dual_obj = *objval;
        stats->solve_ms = dev_ms;
        stats->total_ms = wall.ms();
        stats->kernel_launches = g_launches.load() - l0;
        stats->h2d_bytes = nnz * 12 + (int64_t)m * 13 + (int64_t)n * 8 + nodes * (int64_t)n * 16;
        stats->d2h_bytes = nodes * ((int64_t)n * 8 + 16);
        stats->limit_reached = stopped ? (nodes >= node_limit ? 1 : 2) : 0;
    }
}

}  // namespace elp
