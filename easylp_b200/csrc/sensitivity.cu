// sensitivity.cu — objective and right-hand-side ranging of an LP solved by the simplex path (SURVEY §8f N3).
//
// Replaces lpSolveAPI::get.sensitivity.obj / get.sensitivity.rhs behind `$sensitivity_objective` and `$sensitivity_rhs`
// (/root/reference/R/class.R:613-646: arrays Lower | Current | Upper per variable / per constraint).
// The LP is solved by the simplex kernel (simplex.cu), which also returns its final basis; the ranging itself is a few
// dense operations on the host, O(m^3) for the basis inverse and O(m^2 (m + n)) for the objective ranging (the simplex
// path takes tableaus up to one thread-block cluster's shared memory, a few hundred rows):
//   objective ranging  the interval of c_j over which the optimal basis stays optimal (reduced costs keep their sign),
//   rhs ranging        the interval of b_i over which the optimal basis stays feasible (basic variables keep inside
//                      their bounds), i.e. over which the dual value of the row is valid.
// Parity note: lp_solve is not in this image and the reference's tests hold no sensitivity values, so these are the
// textbook basis-invariance ranges, pinned to HiGHS' ranging on non-degenerate models (tests/test_sensitivity.py);
// lp_solve's conventions for degenerate vertices and for what it reports on non-basic columns are NOT pinned.
#include "common.cuh"
#include "../../include/easylp_abi.h"
#include <algorithm>
#include <cmath>
#include <vector>

namespace elp {

int simplex_batch_device(int64_t B, int m, int n, const double* A, const double* b, const double* c, const double* lb,
                         const double* ub, const int8_t* sense, int maximize, int max_pivots, int32_t* status,
                         double* obj, double* x, double* y, int32_t* pivots, cudaStream_t st, int shared_model,
                         int32_t* basis);
void densify_device(int m, int n, const int* ptr, const int* idx, const double* val, double* A, cudaStream_t st);

// Gauss-Jordan inverse with partial pivoting; returns false when singular
static bool invert(std::vector<double>& a, int m, std::vector<double>& inv) {
    inv.assign((size_t)m * m, 0.0);
    for (int i = 0; i < m; ++i) inv[(size_t)i * m + i] = 1.0;
    for (int col = 0; col < m; ++col) {
        int piv = col;
        for (int r = col + 1; r < m; ++r)
            if (std::fabs(a[(size_t)r * m + col]) > std::fabs(a[(size_t)piv * m + col])) piv = r;
        if (std::fabs(a[(size_t)piv * m + col]) < 1e-13) return false;
        if (piv != col)
            for (int k = 0; k < m; ++k) {
                std::swap(a[(size_t)piv * m + k], a[(size_t)col * m + k]);
                std::swap(inv[(size_t)piv * m + k], inv[(size_t)col * m + k]);
            }
        const double d = 1.0 / a[(size_t)col * m + col];
        for (int k = 0; k < m; ++k) { a[(size_t)col * m + k] *= d; inv[(size_t)col * m + k] *= d; }
        for (int r = 0; r < m; ++r) {
            if (r == col) continue;
            const double f = a[(size_t)r * m + col];
            if (f == 0.0) continue;
            for (int k = 0; k < m; ++k) { a[(size_t)r * m + k] -= f * a[(size_t)col * m + k]; inv[(size_t)r * m + k] -= f * inv[(size_t)col * m + k]; }
        }
    }
    return true;
}

void sensitivity(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                 const int8_t* sense, const double* rhs, const double* c, int32_t maximize, const double* lb,
                 const double* ub, const elp_options& o, int32_t* status, double* objval, double* x, double* obj_from,
                 double* obj_till, double* rhs_from, double* rhs_till, double* duals) {
    cudaStream_t st = 0;
    const int64_t nnz = m > 0 ? row_ptr[m] : 0;
    DevBuf<int> ptr((size_t)m + 1), idx(std::max<int64_t>(nnz, 1));
    DevBuf<double> val(std::max<int64_t>(nnz, 1)), Ad((size_t)std::max(m, 1) * n), b(std::max(m, 1)), cd(n), lbd(n), ubd(n),
        objd(1), xd(n), yd(std::max(m, 1));
    DevBuf<int8_t> sd(std::max(m, 1));
    DevBuf<int32_t> statd(1), pivd(1), basd(std::max(m, 1));
    if (m > 0) {
        ptr.upload(row_ptr, (size_t)m + 1, st); idx.upload(col_idx, nnz, st); val.upload(vals, nnz, st);
        b.upload(rhs, m, st); sd.upload(sense, m, st);
    }
    cd.upload(c, n, st); lbd.upload(lb, n, st); ubd.upload(ub, n, st);
    densify_device(m, n, ptr.p, idx.p, val.p, Ad.p, st);
    simplex_batch_device(1, m, n, Ad.p, b.p, cd.p, lbd.p, ubd.p, sd.p, maximize, o.max_iter, statd.p, objd.p, xd.p, yd.p, pivd.p,
                         st, 0, basd.p);
    std::vector<int32_t> basis(std::max(m, 1));
    std::vector<double> y(std::max(m, 1));
    statd.download(status, 1, st); objd.download(objval, 1, st); xd.download(x, n, st);
    if (m > 0) { basd.download(basis.data(), m, st); yd.download(y.data(), m, st); }
    ELP_CUDA(cudaStreamSynchronize(st));
    if (*status != ELP_STATUS_OPTIMAL) return;

    const double sgn = maximize ? -1.0 : 1.0;            // work in "min" sense: cm = sgn * c
    const int N = n + m;
    // dense [A | I]
    std::vector<double> A((size_t)m * n, 0.0);
    for (int i = 0; i < m; ++i)
        for (int k = row_ptr[i]; k < row_ptr[i + 1]; ++k) A[(size_t)i * n + col_idx[k]] = vals[k];
    auto col_entry = [&](int i, int q) { return q < n ? A[(size_t)i * n + q] : (q - n == i ? 1.0 : 0.0); };
    // bounds and values of every column of [A | I]: slack of row i is s_i = b_i - a_i x in [0, inf) (<=), (-inf, 0] (>=), {0} (==)
    std::vector<double> lo(N), up(N), xv(N), cm(N, 0.0);
    for (int j = 0; j < n; ++j) { lo[j] = lb[j]; up[j] = ub[j]; xv[j] = x[j]; cm[j] = sgn * c[j]; }
    for (int i = 0; i < m; ++i) {
        double ax = 0.0;
        for (int k = row_ptr[i]; k < row_ptr[i + 1]; ++k) ax += vals[k] * x[col_idx[k]];
        xv[n + i] = rhs[i] - ax;
        lo[n + i] = sense[i] == ELP_GE ? -INFINITY : 0.0;
        up[n + i] = sense[i] == ELP_LE ? INFINITY : 0.0;
    }
    std::vector<char> is_basic(N, 0);
    for (int k = 0; k < m; ++k) { ELP_REQUIRE(basis[k] >= 0 && basis[k] < N, "sensitivity: bad basis"); is_basic[basis[k]] = 1; }
    std::vector<double> Bm((size_t)m * m), Binv;
    for (int i = 0; i < m; ++i)
        for (int k = 0; k < m; ++k) Bm[(size_t)i * m + k] = col_entry(i, basis[k]);
    ELP_REQUIRE(m == 0 || invert(Bm, m, Binv), "sensitivity: the final basis is numerically singular");
    // multipliers pi = cB' B^-1 and reduced costs d_q = cm_q - pi a_q
    std::vector<double> pi(m, 0.0), d(N, 0.0);
    for (int i = 0; i < m; ++i) {
        double s = 0.0;
        for (int k = 0; k < m; ++k) s += cm[basis[k]] * Binv[(size_t)k * m + i];
        pi[i] = s;
    }
    for (int q = 0; q < N; ++q) {
        double s = cm[q];
        for (int i = 0; i < m; ++i) s -= pi[i] * col_entry(i, q);
        d[q] = is_basic[q] ? 0.0 : s;
    }
    // where the non-basic columns sit: -1 at lower, +1 at upper, 0 fixed / free (never constrains a range)
    const double tol = 1e-9;
    std::vector<int> at(N, 0);
    for (int q = 0; q < N; ++q) {
        if (is_basic[q]) continue;
        const bool fixed = std::isfinite(lo[q]) && std::isfinite(up[q]) && up[q] - lo[q] <= tol;
        if (fixed) at[q] = 0;
        else if (std::isfinite(lo[q]) && std::fabs(xv[q] - lo[q]) <= tol * (1 + std::fabs(lo[q]))) at[q] = -1;
        else if (std::isfinite(up[q]) && std::fabs(xv[q] - up[q]) <= tol * (1 + std::fabs(up[q]))) at[q] = 1;
    }
    // ---- objective ranging ------------------------------------------------------------------------------------
    for (int j = 0; j < n; ++j) {
        double dmin = -INFINITY, dmax = INFINITY;          // admissible change of cm_j
        if (!is_basic[j]) {
            if (at[j] < 0) dmin = -d[j];                    // at lower: cost may fall by its reduced cost
            else if (at[j] > 0) dmax = -d[j];               // at upper: may rise by -d_j
            else if (!(std::isfinite(lo[j]) && std::isfinite(up[j]) && up[j] - lo[j] <= tol)) { dmin = 0.0; dmax = 0.0; }  // free, non-basic
        } else {
            int k = 0;
            while (basis[k] != j) ++k;
            for (int q = 0; q < N; ++q) {
                if (is_basic[q] || at[q] == 0) continue;
                double alpha = 0.0;                         // (B^-1 a_q)_k
                for (int i = 0; i < m; ++i) alpha += Binv[(size_t)k * m + i] * col_entry(i, q);
                if (std::fabs(alpha) <= 1e-12) continue;
                const double ratio = d[q] / alpha;          // d_q - delta * alpha keeps the sign of d_q up to here
                if ((at[q] < 0 && alpha > 0) || (at[q] > 0 && alpha < 0)) dmax = std::min(dmax, ratio);
                else dmin = std::max(dmin, ratio);
            }
        }
        const double a = cm[j] + dmin, bq = cm[j] + dmax;
        obj_from[j] = maximize ? -bq : a;
        obj_till[j] = maximize ? -a : bq;
    }
    // ---- right-hand-side ranging ---------------------------------------------------------------------------------
    for (int i = 0; i < m; ++i) {
        double dmin = -INFINITY, dmax = INFINITY;          // admissible change of b_i: xB + delta * Binv[:, i] stays in bounds
        for (int k = 0; k < m; ++k) {
            const double g = Binv[(size_t)k * m + i];
            if (std::fabs(g) <= 1e-12) continue;
            const int q = basis[k];
            const double room_dn = xv[q] - lo[q], room_up = up[q] - xv[q];      // >= 0 (inf when unbounded)
            if (g > 0) { dmax = std::min(dmax, room_up / g); dmin = std::max(dmin, -room_dn / g); }
            else { dmax = std::min(dmax, room_dn / -g); dmin = std::max(dmin, -room_up / -g); }
        }
        rhs_from[i] = rhs[i] + dmin;
        rhs_till[i] = rhs[i] + dmax;
        duals[i] = y[i];
    }
}

}  // namespace elp
