// simplex.cu — batched dense simplex: one LP per warp for small shapes, else one LP per CTA or per thread-block cluster;
// tableau resident in shared memory.
//
// Replaces `status <- solve(prob)` (/root/reference/R/class.R:276) for LPs whose dense tableau fits in
// the shared memory of one SM or of a cluster, and is the engine of the additive batch entry point (BASELINE config 3:
// 200k LPs of 20x30).  Method: bounded-variable primal simplex on  A x + s = b  with a composite
// phase 1 (minimise the sum of infeasibilities), Dantzig pricing, a two-pass ratio test and Bland's
// rule after a run of degenerate pivots.  The CPU restatement is oracle/simplex_ref.c.
//
// Data movement: each LP's A (m*n doubles) is read ONCE from HBM with 1-D TMA bulk copies, one per row
// (cp.async.bulk -> mbarrier complete_tx), straight into its shared-memory home, b, c, lb, ub by plain loads; results
// (status, objective, x) are written once.  Everything in between — pricing argmax, ratio-test
// argmin (warp shuffles), the rank-1 pivot update — runs out of shared memory in fp64.
// Algorithmic HBM bytes per LP: 8 (m n + m + 3 n) + m   in,   8 (n + 1) + 4   out.
// The serial pivot chain, not HBM, bounds this kernel; bench.py reports LPs/s, pivots/s and the HBM
// fraction side by side (SURVEY §8d).
#include "common.cuh"
#include "tma.cuh"
#include "../../include/easylp_abi.h"
#include <cooperative_groups.h>
#include <algorithm>
#include <cmath>

namespace elp {

#define ST_BASIC 0
#define ST_LOWER 1
#define ST_UPPER 2
#define ST_FREE 3

constexpr double TOL_PRIMAL = 1e-9;
constexpr double TOL_DUAL = 1e-9;
constexpr double TOL_PIVOT = 1e-9;

__device__ __forceinline__ double ptol(double bound) { return TOL_PRIMAL * fmax(1.0, fabs(bound)); }

// ---- block-wide reductions (value, index) ----------------------------------------------------
struct ValIdx {
    double v;
    int i;
};
// "better" = larger v, ties -> smaller index.  Use negated values for argmin.
__device__ __forceinline__ ValIdx better(ValIdx a, ValIdx b) {
    if (b.i < 0) return a;
    if (a.i < 0) return b;
    if (b.v > a.v || (b.v == a.v && b.i < a.i)) return b;
    return a;
}
template <int THREADS>
__device__ __forceinline__ ValIdx block_argmax(ValIdx x, double* red_v, int* red_i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ValIdx y;
        y.v = __shfl_xor_sync(0xffffffffu, x.v, o);
        y.i = __shfl_xor_sync(0xffffffffu, x.i, o);
        x = better(x, y);
    }
    if (THREADS == 32) return x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();   // protect scratch reuse
    if (lane == 0) { red_v[warp] = x.v; red_i[warp] = x.i; }
    __syncthreads();
    ValIdx r{red_v[0], red_i[0]};
#pragma unroll
    for (int w = 1; w < THREADS / 32; ++w) r = better(r, ValIdx{red_v[w], red_i[w]});
    return r;
}
template <int THREADS>
__device__ __forceinline__ double block_sum(double x, double* red_v) {
    x = warp_sum(x);
    if (THREADS == 32) return x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red_v[warp] = x;
    __syncthreads();
    double r = 0.0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; ++w) r += red_v[w];
    return r;
}
// ------------------------------------------------------------------------------------------------
// Warp-per-LP kernel for small LPs (m <= 32, m + n <= 96) — the batched path of BASELINE config 3.
// One WARP solves one LP; a CTA is four independent warps.  The tableau T[MR][NS] (NS = 32*CPL + 2 doubles
// per row, MR = m rounded up to 4: both compile-time, so every tableau access is `base + immediate`) lives
// in the warp's slice of shared memory and is filled ONCE per LP by 1-D TMA bulk copies, one per row, issued
// by the lanes in parallel (cp.async.bulk -> mbarrier complete_tx); b, c, lb, ub arrive by coalesced loads.
// Lane l owns the tableau columns l, l+32, (l+64) and keeps their bounds / cost / non-basic value / state
// in registers; row-indexed data (basic values, basis heads, bounds of the basic variables, the entering
// column) sits beside the tableau.  A pivot is warp-synchronous end to end:
//   pricing     d_j = c_j - sum_i cb_i T[i][j]      one column per lane per pass, conflict-free row reads
//   argmax      three 32-bit hardware reductions (REDUX) on the bit pattern of |d_j| and on the index
//   ratio test  row i on lane i, REDUX min, second pass picks the largest pivot among the ties
//   update      T[i][j] -= colq[i] * rr[j]: MR fused multiply-adds per column straight on shared memory;
//               the dynamic pivot row is a plain address here (registers could not be indexed by it)
// There is no block-wide barrier, no address arithmetic in the loops and ~60 registers per thread, so many
// LPs are resident per SM.  Arithmetic order per entry equals simplex_kernel / oracle/simplex_ref.c.
// ------------------------------------------------------------------------------------------------
constexpr int SW_WARPS = 4;

struct WarpSimplexLayout {      // per-warp shared memory, in bytes
    int ns, off_rows, total;
    __host__ __device__ WarpSimplexLayout(int MR, int CPL) {
        ns = 32 * CPL + 2;                                   // even (16-byte rows for TMA), not a multiple of 32
        off_rows = MR * ns * 8;
        // beta blo bhi bcost cb colq [MR each] | xs[96] | mbarrier | basis[MR]
        total = off_rows + 6 * MR * 8 + 96 * 8 + 16 + MR * 4;
        total = (total + 15) & ~15;
    }
};

struct WVI {
    double v;
    int i;
};
// Warp argmax of (v, i) with v >= 0 (or i < 0 = no candidate): larger v wins, ties go to the smaller i — the
// "better" above.  Non-negative doubles order like their bit patterns, so the maximum is two
// 32-bit hardware reductions (REDUX) on the high and low words and the tie-break a third on the index.
__device__ __forceinline__ WVI warp_best_nonneg(WVI x) {
    const unsigned long long bits = x.i < 0 ? 0ull : (unsigned long long)__double_as_longlong(x.v + 0.0);
    const unsigned hi = (unsigned)(bits >> 32), lo = (unsigned)bits;
    const unsigned mhi = __reduce_max_sync(0xffffffffu, hi);
    const unsigned mlo = __reduce_max_sync(0xffffffffu, hi == mhi ? lo : 0u);
    const bool top = x.i >= 0 && hi == mhi && lo == mlo;
    const unsigned mi = __reduce_min_sync(0xffffffffu, top ? (unsigned)x.i : 0xffffffffu);
    WVI r;
    r.i = (mi == 0xffffffffu) ? -1 : (int)mi;
    r.v = __longlong_as_double((long long)(((unsigned long long)mhi << 32) | mlo));
    return r;
}
// Bland's rule: the candidate with the smallest key (a variable id), index i travels with it.
__device__ __forceinline__ int warp_best_bland(int key, int i) {
    const unsigned k = i < 0 ? 0xffffffffu : (unsigned)key;
    const unsigned mk = __reduce_min_sync(0xffffffffu, k);
    const unsigned mi = __reduce_min_sync(0xffffffffu, (i >= 0 && k == mk) ? (unsigned)i : 0xffffffffu);
    return mi == 0xffffffffu ? -1 : (int)mi;
}
// Warp minimum of non-negative doubles (+inf allowed)
__device__ __forceinline__ double warp_min_nonneg(double v) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(v + 0.0);
    const unsigned hi = (unsigned)(bits >> 32), lo = (unsigned)bits;
    const unsigned mhi = __reduce_min_sync(0xffffffffu, hi);
    const unsigned mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xffffffffu);
    return __longlong_as_double((long long)(((unsigned long long)mhi << 32) | mlo));
}

template <int MR, int CPL>
__global__ void __launch_bounds__(SW_WARPS * 32)
simplex_warp_kernel(int64_t B, int m, int n, const double* __restrict__ Ag, const double* __restrict__ bg,
                    const double* __restrict__ cg, const double* __restrict__ lbg, const double* __restrict__ ubg,
                    const int8_t* __restrict__ senseg, int maximize, int max_pivots, int shared_model, int use_tma,
                    int32_t* __restrict__ status_out, double* __restrict__ obj_out, double* __restrict__ x_out,
                    double* __restrict__ y_out, int32_t* __restrict__ pivots_out, int32_t* __restrict__ basis_out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int NS = 32 * CPL + 2;
    const WarpSimplexLayout lay(MR, CPL);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* wbase = smem_raw + (size_t)warp * lay.total;
    double* Ts = reinterpret_cast<double*>(wbase);               // [MR][NS]
    double* Tl = Ts + lane;                                      // my columns: Tl[i * NS + 32 * c]
    double* rows = reinterpret_cast<double*>(wbase + lay.off_rows);
    double* beta = rows;
    double* blo = rows + MR;
    double* bhi = rows + 2 * MR;
    double* bcost = rows + 3 * MR;
    double* cb = rows + 4 * MR;
    double* colq = rows + 5 * MR;
    double* xs = rows + 6 * MR;                                  // [96] non-basic values by column (setup only)
    uint64_t* bar = reinterpret_cast<uint64_t*>(xs + 96);
    int* basis = reinterpret_cast<int*>(bar + 2);                // [MR]
    const int N = n + m;
    const int64_t gw = (int64_t)blockIdx.x * SW_WARPS + warp, nw = (int64_t)gridDim.x * SW_WARPS;
    if (max_pivots <= 0) max_pivots = 50 * (m + n) + 1000;

    if (lane == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    // padding rows / columns stay zero for the whole kernel (updates of zero entries by zero factors)
    for (int e = lane; e < MR * NS; e += 32) Ts[e] = 0.0;
    __syncwarp();
    uint32_t phase = 0;

    for (int64_t lp = gw; lp < B; lp += nw) {
        const int64_t mlp = shared_model ? 0 : lp;  // branch and bound: every node shares A, b, c, sense; bounds differ
        const double* A = Ag + mlp * (int64_t)m * n;
        const int8_t* sense = senseg ? senseg + mlp * (int64_t)m : nullptr;
        // ---- tableau rows of A: one bulk copy per row, issued by the lanes in parallel ----------------
        if (use_tma && m > 0) {
            // generic-proxy writes to the tableau (previous LP) must be ordered before the async-proxy copies
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_expect_tx(bar, (uint32_t)m * (uint32_t)n * 8u);
            __syncwarp();
            for (int i = lane; i < m; i += 32) tma_load_1d(Ts + i * NS, A + (size_t)i * n, (uint32_t)n * 8u, bar);
        } else {
            for (int i = 0; i < m; ++i)
                for (int j = lane; j < n; j += 32) Ts[i * NS + j] = A[(size_t)i * n + j];
        }
        // ---- registers: scalars of my columns; slack block of the tableau -----------------------------
        double clo[CPL], chi[CPL], ccost[CPL], cxn[CPL];
        int cstate[CPL];
        int bad = 0;
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            const int col = lane + 32 * c;
            clo[c] = 0.0; chi[c] = 0.0; ccost[c] = 0.0; cxn[c] = 0.0; cstate[c] = ST_BASIC;
            if (col < n) {
                const double l = lbg ? lbg[lp * (int64_t)n + col] : 0.0, u = ubg ? ubg[lp * (int64_t)n + col] : INFINITY;
                const double cj = cg[mlp * (int64_t)n + col];
                clo[c] = l; chi[c] = u;
                ccost[c] = maximize ? -cj : cj;
                if (l > u) bad = 1;
                if (isfinite(l)) { cstate[c] = ST_LOWER; cxn[c] = l; }
                else if (isfinite(u)) { cstate[c] = ST_UPPER; cxn[c] = u; }
                else { cstate[c] = ST_FREE; cxn[c] = 0.0; }
                xs[col] = cxn[c];
            } else if (col < N) {
                const int i0 = col - n;
                const int s = sense ? sense[i0] : 0;
#pragma unroll
                for (int i = 0; i < MR; ++i) Tl[i * NS + 32 * c] = (i == i0) ? 1.0 : 0.0;
                clo[c] = (s == ELP_GE) ? -INFINITY : 0.0;
                chi[c] = (s == ELP_LE) ? INFINITY : 0.0;
                basis[i0] = col;
                blo[i0] = clo[c]; bhi[i0] = chi[c]; bcost[i0] = 0.0;
            }
        }
        bad = __any_sync(0xffffffffu, bad);
        if (use_tma && m > 0) { mbar_wait(bar, phase); phase ^= 1u; }
        __syncwarp();
        // beta = b - A xN   (row i on lane i; sequential in j like the reference loop)
        if (lane < MR) {
            double r = 0.0;
            if (lane < m) {
                r = bg[mlp * (int64_t)m + lane];
                const double* Ti = Ts + lane * NS;
                for (int j = 0; j < n; ++j) r -= Ti[j] * xs[j];
            } else { blo[lane] = -INFINITY; bhi[lane] = INFINITY; bcost[lane] = 0.0; basis[lane] = -1; }
            beta[lane] = r;
            cb[lane] = 0.0; colq[lane] = 0.0;
        }
        __syncwarp();

        int status = ELP_STATUS_TIMEOUT, pivots = 0, degenerate_run = 0, bland = 0, qfinal = -1;
        if (bad) status = ELP_STATUS_INFEASIBLE;
        double d[CPL];                       // reduced costs of my columns (phase 2: carried across pivots)
        bool d_fresh_enough = false;
        int d_age = 0;
#pragma unroll
        for (int c = 0; c < CPL; ++c) d[c] = 0.0;

        while (!bad) {
            // ---- phase detection: row i on lane i --------------------------------------------------
            double g = 0.0;
            if (lane < m) {
                const double bi = beta[lane], l = blo[lane], u = bhi[lane];
                if (bi < l - ptol(l)) g = -1.0;
                else if (bi > u + ptol(u)) g = 1.0;
            }
            // the sum of infeasibilities is positive iff some row is infeasible (every term is positive)
            const bool phase1 = __any_sync(0xffffffffu, g != 0.0);
            if (lane < m) cb[lane] = phase1 ? g : bcost[lane];
            __syncwarp();
            // ---- pricing on my columns.  In phase 2 the reduced costs d_j = c_j - cb' T_j are carried in registers
            // from pivot to pivot (d -= d_q * pivot row, the objective row of the textbook tableau) and recomputed
            // from the tableau every 32 pivots, on a phase change, and before optimality is declared. -----------
            WVI cand{0.0, -1};
            for (int attempt = 0; attempt < 2; ++attempt) {
                if (phase1 || !d_fresh_enough) {
#pragma unroll
                    for (int c = 0; c < CPL; ++c) d[c] = phase1 ? 0.0 : ccost[c];
#pragma unroll
                    for (int i = 0; i < MR; ++i) {
                        const double cbi = cb[i];
#pragma unroll
                        for (int c = 0; c < CPL; ++c) d[c] -= cbi * Tl[i * NS + 32 * c];
                    }
                    d_age = 0;
                }
                d_fresh_enough = !phase1;
                cand.v = 0.0; cand.i = -1;
#pragma unroll
                for (int c = 0; c < CPL; ++c) {
                    const int col = lane + 32 * c;
                    const int st = cstate[c];
                    if (col >= N || st == ST_BASIC || !(clo[c] < chi[c])) continue;
                    int dd = 0;
                    if ((st == ST_LOWER || st == ST_FREE) && d[c] < -TOL_DUAL) dd = 1;
                    else if ((st == ST_UPPER || st == ST_FREE) && d[c] > TOL_DUAL) dd = -1;
                    if (!dd) continue;
                    const double key = bland ? (double)col : fabs(d[c]);
                    const int id = 2 * col + (dd < 0 ? 1 : 0);
                    const bool take = cand.i < 0 || (bland ? key < cand.v : (key > cand.v || (key == cand.v && id < cand.i)));
                    if (take) { cand.v = key; cand.i = id; }
                }
                if (bland) cand.i = warp_best_bland((int)cand.v, cand.i);
                else cand = warp_best_nonneg(cand);
                if (cand.i >= 0 || d_age == 0) break;      // a candidate, or no candidate on freshly computed costs
                d_fresh_enough = false;                    // optimality is only declared on recomputed costs
            }
            if (cand.i < 0) { status = phase1 ? ELP_STATUS_INFEASIBLE : ELP_STATUS_OPTIMAL; break; }
            if (pivots >= max_pivots) { status = ELP_STATUS_TIMEOUT; break; }
            const int q = cand.i >> 1;
            const double dir = (cand.i & 1) ? -1.0 : 1.0;
            const int qlane = q & 31, qc = q >> 5;
            // ---- entering column: row i on lane i reads T[i][q]; its scalars come from the owner by shuffle ----
            double q_lo = 0.0, q_hi = 0.0, q_xn = 0.0, q_cost = 0.0;
            int q_state = 0;
#pragma unroll
            for (int c = 0; c < CPL; ++c)
                if (c == qc) { q_lo = clo[c]; q_hi = chi[c]; q_xn = cxn[c]; q_cost = ccost[c]; q_state = cstate[c]; }
            q_lo = __shfl_sync(0xffffffffu, q_lo, qlane);
            q_hi = __shfl_sync(0xffffffffu, q_hi, qlane);
            q_xn = __shfl_sync(0xffffffffu, q_xn, qlane);
            q_cost = __shfl_sync(0xffffffffu, q_cost, qlane);
            q_state = __shfl_sync(0xffffffffu, q_state, qlane);
            double d_q = 0.0;
#pragma unroll
            for (int c = 0; c < CPL; ++c) if (c == qc) d_q = d[c];
            d_q = __shfl_sync(0xffffffffu, d_q, qlane);
            const double cq = (lane < MR) ? Ts[lane * NS + q] : 0.0;
            if (lane < MR) colq[lane] = cq;
            // ---- ratio test: row i on lane i ---------------------------------------------------------
            double tloc = INFINITY, a = 0.0;
            int up = 0, kbas = -1;
            if (lane < m) {
                a = dir * cq;
                if (fabs(a) > TOL_PIVOT) {
                    kbas = basis[lane];
                    const double bi = beta[lane], l = blo[lane], u = bhi[lane];
                    double num = INFINITY;                 // one division per row: t = num / a
                    if (a > 0.0) {
                        if (bi > u + ptol(u)) { num = bi - u; up = 1; }
                        else if (bi >= l - ptol(l) && isfinite(l)) { num = fmax(bi - l, 0.0); up = 0; }
                    } else {
                        if (bi < l - ptol(l)) { num = bi - l; up = 0; }
                        else if (bi <= u + ptol(u) && isfinite(u)) { num = fmin(bi - u, 0.0); up = 1; }
                    }
                    if (num != INFINITY) tloc = num / a;
                }
            }
            const double tmin = warp_min_nonneg(tloc);
            const double tflip = (q_state == ST_FREE) ? INFINITY : q_hi - q_lo;
            if (tflip <= tmin) {
                if (!isfinite(tflip)) {
                    if (phase1) { status = ELP_STATUS_NUMFAILURE; break; }
                    status = ELP_STATUS_UNBOUNDED;
                    qfinal = q;
#pragma unroll
                    for (int c = 0; c < CPL; ++c)
                        if (c == qc && lane == qlane) cxn[c] = dir > 0 ? INFINITY : -INFINITY;
                    break;
                }
                if (lane < m) beta[lane] -= dir * tflip * cq;
#pragma unroll
                for (int c = 0; c < CPL; ++c) {
                    if (c == qc && lane == qlane) {
                        if (dir > 0) { cstate[c] = ST_UPPER; cxn[c] = chi[c]; }
                        else { cstate[c] = ST_LOWER; cxn[c] = clo[c]; }
                    }
                }
                ++pivots; degenerate_run = 0; bland = 0;
                __syncwarp();
                continue;
            }
            // ---- pass 2: among rows within a hair of tmin take the largest pivot (Bland: smallest basic id) ---
            const double window = tmin + 1e-12 * fmax(1.0, fabs(tmin));
            WVI rc{0.0, -1};
            if (kbas >= 0 && tloc <= window) { rc.v = fabs(a); rc.i = 2 * lane + up; }
            if (bland) rc.i = warp_best_bland(kbas, rc.i);
            else rc = warp_best_nonneg(rc);
            if (rc.i < 0) { status = ELP_STATUS_NUMFAILURE; break; }
            const int r = rc.i >> 1;
            const int to_upper = rc.i & 1;
            const double t = tmin;
            __syncwarp();                                  // colq is complete
            const double piv = colq[r];
            const int kl = basis[r];                       // leaving variable (a column id)
            const double kl_bound = to_upper ? bhi[r] : blo[r];
            if (lane < m) beta[lane] -= dir * t * cq;
            // pivot row of my columns: the dynamic row is just an address in shared memory
            double rr[CPL];
            const double* Tr = Tl + r * NS;
#pragma unroll
            for (int c = 0; c < CPL; ++c) rr[c] = Tr[32 * c] / piv;
            __syncwarp();                                  // everyone has read row r before it is rewritten
            // bookkeeping by the owners
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                const int col = lane + 32 * c;
                if (col == kl) { cstate[c] = to_upper ? ST_UPPER : ST_LOWER; cxn[c] = kl_bound; }
                if (col == q) {
                    cstate[c] = ST_BASIC;
                    rr[c] = 1.0;
                    beta[r] = q_xn + dir * t;
                    basis[r] = q; blo[r] = q_lo; bhi[r] = q_hi; bcost[r] = q_cost;
                }
            }
            // ---- rank-1 update of my columns:  T[i] -= colq[i] * rr for i != r, row r := rr.  Column q needs no
            // special case: its rr is exactly 1 and its entries ARE colq, so f - f*1 = 0 exactly. ----------------
#pragma unroll
            for (int i = 0; i < MR; ++i) {
                const double f = colq[i];
#pragma unroll
                for (int c = 0; c < CPL; ++c) Tl[i * NS + 32 * c] -= f * rr[c];
            }
            {
                double* Trw = Tl + r * NS;
#pragma unroll
                for (int c = 0; c < CPL; ++c) Trw[32 * c] = rr[c];
            }
            // objective row: the entering column's reduced cost becomes exactly 0 (its rr is 1)
#pragma unroll
            for (int c = 0; c < CPL; ++c) d[c] -= d_q * rr[c];
            if (++d_age >= 32) d_fresh_enough = false;
            ++pivots;
            if (t <= 1e-12) { if (++degenerate_run > 30) bland = 1; }
            else { degenerate_run = 0; bland = 0; }
            __syncwarp();
        }
        __syncwarp();

        // ---- write back -----------------------------------------------------------------------------
        double* xo = x_out + lp * (int64_t)n;
        double opart = 0.0;
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
            const int col = lane + 32 * c;
            if (col < n && cstate[c] != ST_BASIC) {
                xo[col] = cxn[c];
                opart += ccost[c] * ((col == qfinal) ? 0.0 : cxn[c]);
            }
        }
        if (lane < m) {
            const int k = basis[lane];
            if (k >= 0 && k < n) { xo[k] = beta[lane]; opart += bcost[lane] * beta[lane]; }
        }
        double obj = warp_sum(opart);
        if (status == ELP_STATUS_UNBOUNDED) obj = -INFINITY;
        if (lane == 0) {
            status_out[lp] = status;
            obj_out[lp] = maximize ? -obj : obj;
            if (pivots_out) pivots_out[lp] = pivots;
        }
        if (basis_out && lane < m) basis_out[lp * (int64_t)m + lane] = basis[lane];   // sensitivity ranging
        if (y_out) {
            // y_i = sum_k cost[basis[k]] * Tslack[k][i]: slack column n+i belongs to one lane
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                const int col = lane + 32 * c;
                if (col >= n && col < N) {
                    double s = 0.0;
#pragma unroll
                    for (int k = 0; k < MR; ++k) s += bcost[k] * Tl[k * NS + 32 * c];
                    y_out[lp * (int64_t)m + (col - n)] = maximize ? -s : s;
                }
            }
        }
        __syncwarp();
        // leave the tableau clean for the next LP: structural columns are overwritten by the copies / loads,
        // padding never changes, the slack block is rewritten at setup — nothing to do.
    }
}

// ------------------------------------------------------------------------------------------------
// Dense-tableau kernel for every shape the warp kernel does not take: one LP per C CTAs (C = 1, 2, 4, 8, 16).  With
// C = 1 one CTA holds the whole tableau in its shared memory; with C >= 2 the C CTAs form a thread-block cluster and
// the tableau is spread over its distributed shared memory.
//   column slices   CTA k owns the columns [k w, (k+1) w) of [A | I] for all m rows, and their lo, hi, cost, xn,
//                   state and pivot-row entries;
//   replicated rows every CTA keeps beta, basis, cb, colq and the bounds and cost of each row's basic variable;
//   per pivot       pricing over the own columns + an argmax of (value, index) over the CTAs (exchange 1: each CTA
//                   stores its candidate into every peer), then the owner of the entering column q stores colq and
//                   q's scalars into every peer (exchange 2); the ratio test runs redundantly on the replicated rows
//                   (same result everywhere, no exchange), the pivot row and the rank-1 update are local.
// Two barriers over the LP's CTAs per pivot, no global memory inside the loop.  With C = 1 those are block barriers
// and the exchanges are stores into the CTA's own shared memory: the kernel is launched without a cluster, so it pays
// neither the cluster barrier nor its MEMBAR.ALL.GPU.
// Determinism: every column's reduced cost, pivot-row entry and update is the same expression with the same
// sequential loop over i as oracle/simplex_ref.c; the argmax / argmin order (value, then smallest index) is total, so
// every C picks the same q and r.  Status, pivots, basis, x and y are therefore the same bytes for every C; the
// objective is one block sum per CTA, added in rank order, so it matches across C only to the last bits.
// ------------------------------------------------------------------------------------------------
constexpr int SC_THREADS = 256;
constexpr int SC_MAX_CTAS = 16;
constexpr size_t SC_SMEM_MAX = 227 * 1024;

// Per-CTA shared memory of simplex_kernel.  w = ceil((m + n) / C) rounded up to even (16-byte rows for the
// bulk copies).  Bytes = 8 m w (tableau slice) + 44 w (lo hi cost xn rowr, state) + 52 m (beta blo bhi bcost cb
// colq, basis; m rounded up to even / to 4) + 368 (reduction scratch, exchange slots, q's scalars, mbarrier).
struct SimplexLayout {
    int m, n, N, C, w;
    size_t off_T, off_beta, off_blo, off_bhi, off_bcost, off_cb, off_colq, off_lo, off_hi, off_cost, off_xn, off_rowr,
        off_redv, off_slotv, off_objv, off_q, off_bar, off_basis, off_state, off_redi, off_sloti, off_qstate, total;
    __host__ __device__ SimplexLayout(int m_, int n_, int C_) : m(m_), n(n_), N(m_ + n_), C(C_) {
        w = (((N + C - 1) / C) + 1) & ~1;
        auto up2 = [](size_t v) { return (v + 1) & ~(size_t)1; };
        size_t o = 0;
        off_T = o;     o += (size_t)m * w;
        off_beta = o;  o += up2(m);
        off_blo = o;   o += up2(m);
        off_bhi = o;   o += up2(m);
        off_bcost = o; o += up2(m);
        off_cb = o;    o += up2(m);
        off_colq = o;  o += up2(m);
        off_lo = o;    o += w;
        off_hi = o;    o += w;
        off_cost = o;  o += w;
        off_xn = o;    o += w;
        off_rowr = o;  o += w;
        off_redv = o;  o += 8;
        off_slotv = o; o += SC_MAX_CTAS;
        off_objv = o;  o += SC_MAX_CTAS;
        off_q = o;     o += 4;
        size_t bytes = o * sizeof(double);
        off_bar = bytes;    bytes += 16;
        off_basis = bytes;  bytes += (size_t)((m + 3) & ~3) * sizeof(int);
        off_state = bytes;  bytes += (size_t)((w + 3) & ~3) * sizeof(int);
        off_redi = bytes;   bytes += 8 * sizeof(int);
        off_sloti = bytes;  bytes += SC_MAX_CTAS * sizeof(int);
        off_qstate = bytes; bytes += 4 * sizeof(int);
        total = bytes;
    }
};

__device__ __forceinline__ double start_value(const double* lb, const double* ub, int j) {   // xn of a column at setup
    const double l = lb ? lb[j] : 0.0, u = ub ? ub[j] : INFINITY;
    return isfinite(l) ? l : (isfinite(u) ? u : 0.0);
}

// Barrier and peer address over the CTAs that hold one LP.  C = 1 runs without a cluster: a block barrier and the
// CTA's own shared memory.
__device__ __forceinline__ void lp_sync(int C) {
    if (C == 1) __syncthreads();
    else cooperative_groups::this_cluster().sync();
}
template <typename V>
__device__ __forceinline__ V* lp_peer(V* p, int k, int C) {
    return C == 1 ? p : cooperative_groups::this_cluster().map_shared_rank(p, (unsigned)k);
}

// CTAs per SM the 64-thread instance is compiled for: 12 hold it to 80 registers a thread (64 K / 768, rounded down to
// the allocation unit), so a batch of small tableaus (m + n <= 96, e.g. 33 x 10) keeps 12 LPs per SM instead of the 8
// that the 122 registers chosen otherwise allow.  0 leaves the other instances to the compiler (the same cap on the
// 128-thread instance was 4 % slower on 24 x 144 MILPs and 2 % faster at 90 x 120, so it is not applied).
constexpr int simplex_min_ctas(int threads) { return threads == 64 ? 12 : 0; }

template <int THREADS>
__global__ void __launch_bounds__(THREADS, simplex_min_ctas(THREADS))
simplex_kernel(int64_t B, int m, int n, int C, const double* __restrict__ Ag, const double* __restrict__ bg,
               const double* __restrict__ cg_, const double* __restrict__ lbg, const double* __restrict__ ubg,
               const int8_t* __restrict__ senseg, int maximize, int max_pivots, int shared_model,
               int32_t* __restrict__ status_out, double* __restrict__ obj_out, double* __restrict__ x_out,
               double* __restrict__ y_out, int32_t* __restrict__ pivots_out, int32_t* __restrict__ basis_out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int T = THREADS;
    const SimplexLayout lay(m, n, C);
    const int N = lay.N, w = lay.w;
    double* sd = reinterpret_cast<double*>(smem_raw);
    double* Tl = sd + lay.off_T;                 // [m][w]: my columns of [A | I]
    double* beta = sd + lay.off_beta;
    double* blo = sd + lay.off_blo;              // bounds and cost of row i's basic variable
    double* bhi = sd + lay.off_bhi;
    double* bcost = sd + lay.off_bcost;
    double* cb = sd + lay.off_cb;
    double* colq = sd + lay.off_colq;
    double* lo = sd + lay.off_lo;                // [w]: scalars of my columns
    double* hi = sd + lay.off_hi;
    double* cost = sd + lay.off_cost;
    double* xn = sd + lay.off_xn;
    double* rowr = sd + lay.off_rowr;
    double* red_v = sd + lay.off_redv;
    double* slot_v = sd + lay.off_slotv;         // exchange 1: one candidate per CTA
    double* obj_v = sd + lay.off_objv;           // objective partials (rank 0)
    double* qv = sd + lay.off_q;                 // exchange 2: lo, hi, xn, cost of the entering column
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + lay.off_bar);
    int* basis = reinterpret_cast<int*>(smem_raw + lay.off_basis);
    int* state = reinterpret_cast<int*>(smem_raw + lay.off_state);
    int* red_i = reinterpret_cast<int*>(smem_raw + lay.off_redi);
    int* slot_i = reinterpret_cast<int*>(smem_raw + lay.off_sloti);
    int* qstate = reinterpret_cast<int*>(smem_raw + lay.off_qstate);
    const int tid = threadIdx.x;
    const int rank = C == 1 ? 0 : (int)cooperative_groups::this_cluster().block_rank();
    const int j0 = rank * w;                                   // global id of my first column
    const int ns = min(max(n - j0, 0), w);                     // structural columns in my slice

    const int64_t lp = (int64_t)blockIdx.x / C;
    const int64_t mlp = shared_model ? 0 : lp;
    const double* A = Ag + mlp * (int64_t)m * n;
    const double* b = bg + mlp * (int64_t)m;
    const double* c = cg_ + mlp * (int64_t)n;
    const double* lb = lbg ? lbg + lp * (int64_t)n : nullptr;
    const double* ub = ubg ? ubg + lp * (int64_t)n : nullptr;
    const int8_t* sense = senseg ? senseg + mlp * (int64_t)m : nullptr;

    // ---- stage my slice: one bulk copy per row segment where alignment allows, cooperative loads otherwise -----
    const bool tA = m > 0 && ns > 0 && (ns % 2 == 0) && (n % 2 == 0) && ((((uintptr_t)A) & 15) == 0);
    if (tid == 0) { mbar_init(bar, 1); mbar_fence_init(); }
    __syncthreads();
    if (tA) {
        if (tid == 0) mbar_expect_tx(bar, (uint32_t)m * (uint32_t)ns * 8u);
        __syncthreads();
        for (int i = tid; i < m; i += T) tma_load_1d(Tl + (size_t)i * w, A + (size_t)i * n + j0, (uint32_t)ns * 8u, bar);
    } else {
        for (int e = tid; e < m * ns; e += T) { const int i = e / ns, jl = e - i * ns; Tl[i * w + jl] = A[(size_t)i * n + j0 + jl]; }
    }
    if (ns < w)      // slack columns (identity) and padding (zero)
        for (int e = tid; e < m * (w - ns); e += T) {
            const int i = e / (w - ns), jl = ns + (e - i * (w - ns)), j = j0 + jl;
            Tl[i * w + jl] = (j < N && j - n == i) ? 1.0 : 0.0;
        }
    for (int jl = tid; jl < w; jl += T) {
        const int j = j0 + jl;
        if (j < n) {
            const double l = lb ? lb[j] : 0.0, u = ub ? ub[j] : INFINITY;
            lo[jl] = l; hi[jl] = u;
            cost[jl] = maximize ? -c[j] : c[j];
            if (isfinite(l)) { state[jl] = ST_LOWER; xn[jl] = l; }
            else if (isfinite(u)) { state[jl] = ST_UPPER; xn[jl] = u; }
            else { state[jl] = ST_FREE; xn[jl] = 0.0; }
        } else if (j < N) {
            const int s = sense ? sense[j - n] : 0;
            lo[jl] = (s == ELP_GE) ? -INFINITY : 0.0;
            hi[jl] = (s == ELP_LE) ? INFINITY : 0.0;
            cost[jl] = 0.0; xn[jl] = 0.0; state[jl] = ST_BASIC;
        } else {
            lo[jl] = 0.0; hi[jl] = 0.0; cost[jl] = 0.0; xn[jl] = 0.0; state[jl] = ST_BASIC;
        }
        rowr[jl] = 0.0;
    }
    int bad = 0;
    for (int j = tid; j < n; j += T) {
        const double l = lb ? lb[j] : 0.0, u = ub ? ub[j] : INFINITY;
        if (l > u) bad = 1;
    }
    if (tA) mbar_wait(bar, 0);
    bad = __syncthreads_or(bad);
    // replicated rows; beta = b - A xN with one sequential loop over j.  One CTA reads A and xN from its own tableau
    // and columns; the CTAs of a cluster each read them from global memory, so the rows start identical in every CTA.
    for (int i = tid; i < m; i += T) {
        const int s = sense ? sense[i] : 0;
        blo[i] = (s == ELP_GE) ? -INFINITY : 0.0;
        bhi[i] = (s == ELP_LE) ? INFINITY : 0.0;
        bcost[i] = 0.0;
        basis[i] = n + i;
        double r = b[i];
        if (C == 1) {
            const double* Ti = Tl + (size_t)i * w;
            for (int j = 0; j < n; ++j) r -= Ti[j] * xn[j];
        } else {
            const double* Ai = A + (size_t)i * n;
            for (int j = 0; j < n; ++j) r -= Ai[j] * start_value(lb, ub, j);
        }
        beta[i] = r;
    }
    lp_sync(C);       // every CTA of the LP is running and staged before any peer store

    int status = ELP_STATUS_TIMEOUT, pivots = 0, degenerate_run = 0, bland = 0;
    int qfinal = -1;
    if (max_pivots <= 0) max_pivots = 50 * (m + n) + 1000;
    if (bad) status = ELP_STATUS_INFEASIBLE;

    while (!bad) {
        // ---- phase detection (replicated rows): phase 1 iff some basic variable is outside its bounds ----------
        int infeasible = 0;
        for (int i = tid; i < m; i += T) {
            const double bi = beta[i], l = blo[i], u = bhi[i];
            double g = 0.0;
            if (bi < l - ptol(l)) g = -1.0;
            else if (bi > u + ptol(u)) g = 1.0;
            cb[i] = g;
            infeasible |= (g != 0.0);
        }
        const bool phase1 = __syncthreads_or(infeasible);
        if (!phase1) for (int i = tid; i < m; i += T) cb[i] = bcost[i];
        __syncthreads();
        // ---- pricing over my columns, then the cluster argmax (exchange 1) ---------------------------------------
        ValIdx cand{0.0, -1};
        for (int jl = tid; jl < w; jl += T) {
            const int st = state[jl];
            if (st == ST_BASIC || !(lo[jl] < hi[jl])) continue;
            double d = phase1 ? 0.0 : cost[jl];
            for (int i = 0; i < m; ++i) d -= cb[i] * Tl[i * w + jl];
            int dd = 0;
            if ((st == ST_LOWER || st == ST_FREE) && d < -TOL_DUAL) dd = 1;
            else if ((st == ST_UPPER || st == ST_FREE) && d > TOL_DUAL) dd = -1;
            if (!dd) continue;
            const int j = j0 + jl;
            ValIdx me{bland ? -(double)j : fabs(d), 2 * j + (dd < 0 ? 1 : 0)};
            cand = better(cand, me);
        }
        cand = block_argmax<T>(cand, red_v, red_i);
        if (tid < C) {
            lp_peer(slot_v, tid, C)[rank] = cand.v;
            lp_peer(slot_i, tid, C)[rank] = cand.i;
        }
        lp_sync(C);
        cand = ValIdx{slot_v[0], slot_i[0]};
        for (int k = 1; k < C; ++k) cand = better(cand, ValIdx{slot_v[k], slot_i[k]});
        if (cand.i < 0) { status = phase1 ? ELP_STATUS_INFEASIBLE : ELP_STATUS_OPTIMAL; break; }
        if (pivots >= max_pivots) { status = ELP_STATUS_TIMEOUT; break; }
        const int q = cand.i >> 1;
        const double dir = (cand.i & 1) ? -1.0 : 1.0;
        const int qo = q / w, ql = q - qo * w;
        // ---- entering column: its owner stores colq and q's scalars into every CTA (exchange 2) ------------------
        if (rank == qo) {
            for (int k = 0; k < C; ++k) {
                double* dst = lp_peer(colq, k, C);
                for (int i = tid; i < m; i += T) dst[i] = Tl[i * w + ql];
            }
            if (tid < C) {
                double* dq = lp_peer(qv, tid, C);
                dq[0] = lo[ql]; dq[1] = hi[ql]; dq[2] = xn[ql]; dq[3] = cost[ql];
                lp_peer(qstate, tid, C)[0] = state[ql];
            }
        }
        lp_sync(C);
        const double q_lo = qv[0], q_hi = qv[1], q_xn = qv[2], q_cost = qv[3];
        const int q_state = qstate[0];
        // ---- ratio test, pass 1 (replicated) ----------------------------------------------------------------------
        double tloc = INFINITY;
        for (int i = tid; i < m; i += T) {
            const double a = dir * colq[i];
            if (fabs(a) <= TOL_PIVOT) continue;
            const double bi = beta[i], l = blo[i], u = bhi[i];
            double t = INFINITY;
            if (a > 0.0) {
                if (bi > u + ptol(u)) t = (bi - u) / a;
                else if (bi >= l - ptol(l)) { if (isfinite(l)) t = fmax(bi - l, 0.0) / a; }
            } else {
                if (bi < l - ptol(l)) t = (bi - l) / a;
                else if (bi <= u + ptol(u)) { if (isfinite(u)) t = fmin(bi - u, 0.0) / a; }
            }
            tloc = fmin(tloc, t);
        }
        ValIdx tm = block_argmax<T>(ValIdx{-tloc, tid}, red_v, red_i);
        const double tmin = -tm.v;
        double tflip = (q_state == ST_FREE) ? INFINITY : q_hi - q_lo;
        if (tflip <= tmin) {
            if (!isfinite(tflip)) {
                if (phase1) { status = ELP_STATUS_NUMFAILURE; break; }
                status = ELP_STATUS_UNBOUNDED;
                qfinal = q;
                __syncthreads();
                if (tid == 0 && rank == qo) xn[ql] = dir > 0 ? INFINITY : -INFINITY;
                break;
            }
            for (int i = tid; i < m; i += T) beta[i] -= dir * tflip * colq[i];
            __syncthreads();
            if (tid == 0 && rank == qo) {
                if (dir > 0) { state[ql] = ST_UPPER; xn[ql] = hi[ql]; }
                else { state[ql] = ST_LOWER; xn[ql] = lo[ql]; }
            }
            ++pivots; degenerate_run = 0; bland = 0;
            __syncthreads();
            continue;
        }
        // ---- pass 2: among rows within a hair of tmin take the largest pivot (Bland: smallest basic id) ----------
        const double window = tmin + 1e-12 * fmax(1.0, fabs(tmin));
        ValIdx rc{0.0, -1};
        for (int i = tid; i < m; i += T) {
            const double a = dir * colq[i];
            if (fabs(a) <= TOL_PIVOT) continue;
            const int k = basis[i];
            const double bi = beta[i], l = blo[i], u = bhi[i];
            double t = INFINITY; int up = 0;
            if (a > 0.0) {
                if (bi > u + ptol(u)) { t = (bi - u) / a; up = 1; }
                else if (bi >= l - ptol(l)) { if (isfinite(l)) { t = fmax(bi - l, 0.0) / a; up = 0; } }
            } else {
                if (bi < l - ptol(l)) { t = (bi - l) / a; up = 0; }
                else if (bi <= u + ptol(u)) { if (isfinite(u)) { t = fmin(bi - u, 0.0) / a; up = 1; } }
            }
            if (t > window) continue;
            ValIdx me{bland ? -(double)k : fabs(a), 2 * i + up};
            rc = better(rc, me);
        }
        rc = block_argmax<T>(rc, red_v, red_i);
        if (rc.i < 0) { status = ELP_STATUS_NUMFAILURE; break; }
        const int r = rc.i >> 1;
        const int to_upper = rc.i & 1;
        // ---- step + basis change --------------------------------------------------------------------------------
        const double t = tmin;
        const double piv = colq[r];
        for (int i = tid; i < m; i += T) beta[i] -= dir * t * colq[i];
        for (int jl = tid; jl < w; jl += T) rowr[jl] = Tl[r * w + jl] / piv;
        __syncthreads();
        if (tid == 0) {
            const int kl = basis[r];
            if (kl / w == rank) {
                const int l = kl - j0;
                if (to_upper) { state[l] = ST_UPPER; xn[l] = hi[l]; }
                else { state[l] = ST_LOWER; xn[l] = lo[l]; }
            }
            beta[r] = q_xn + dir * t;
            basis[r] = q; blo[r] = q_lo; bhi[r] = q_hi; bcost[r] = q_cost;
            if (rank == qo) { state[ql] = ST_BASIC; rowr[ql] = 1.0; }
        }
        __syncthreads();
        // ---- rank-1 update of my columns:  T -= colq * rowr  (row r := rowr) -------------------------------------
        for (int i = 0; i < m; ++i) {
            const double f = colq[i];
            if (i == r) {
                for (int jl = tid; jl < w; jl += T) Tl[i * w + jl] = rowr[jl];
            } else if (f != 0.0) {
                for (int jl = tid; jl < w; jl += T) {
                    double* e = &Tl[i * w + jl];
                    *e = (j0 + jl == q) ? 0.0 : *e - f * rowr[jl];      // the pivot column becomes a unit vector exactly
                }
            }
        }
        ++pivots;
        if (t <= 1e-12) { if (++degenerate_run > 30) bland = 1; }
        else { degenerate_run = 0; bland = 0; }
        __syncthreads();
    }
    __syncthreads();

    // ---- write back: owners write their non-basic columns and slack duals, rank 0 the replicated rows ----------
    double* xo = x_out + lp * (int64_t)n;
    for (int jl = tid; jl < ns; jl += T) if (state[jl] != ST_BASIC) xo[j0 + jl] = xn[jl];
    if (rank == 0) for (int i = tid; i < m; i += T) if (basis[i] < n) xo[basis[i]] = beta[i];
    double opart = 0.0;
    for (int jl = tid; jl < ns; jl += T) {
        if (state[jl] != ST_BASIC) opart += cost[jl] * ((j0 + jl == qfinal) ? 0.0 : xn[jl]);
    }
    if (rank == 0) for (int i = tid; i < m; i += T) if (basis[i] < n) opart += bcost[i] * beta[i];
    const double part = block_sum<T>(opart, red_v);
    if (tid == 0) lp_peer(obj_v, 0, C)[rank] = part;
    lp_sync(C);
    if (rank == 0) {
        if (tid == 0) {
            double obj = obj_v[0];      // C = 1: the block sum itself, a -0.0 included
            for (int k = 1; k < C; ++k) obj += obj_v[k];
            if (status == ELP_STATUS_UNBOUNDED) obj = -INFINITY;
            status_out[lp] = status;
            obj_out[lp] = maximize ? -obj : obj;
            if (pivots_out) pivots_out[lp] = pivots;
        }
        if (basis_out)
            for (int i = tid; i < m; i += T) basis_out[lp * (int64_t)m + i] = basis[i];
    }
    if (y_out) {     // y_i = sum_k cost[basis[k]] * T[k][n + i], by the owner of slack column n + i
        double* yo = y_out + lp * (int64_t)m;
        for (int jl = tid; jl < w; jl += T) {
            const int j = j0 + jl;
            if (j < n || j >= N) continue;
            double s = 0.0;
            for (int k = 0; k < m; ++k) s += bcost[k] * Tl[k * w + jl];
            yo[j - n] = maximize ? -s : s;
        }
    }
}

__global__ void k_densify(int m, int n, const int* __restrict__ ptr, const int* __restrict__ idx,
                          const double* __restrict__ val, double* __restrict__ A) {
    const int i = blockIdx.x;
    if (i >= m) return;
    for (int k = ptr[i] + threadIdx.x; k < ptr[i + 1]; k += blockDim.x) atomicAdd(&A[(size_t)i * n + idx[k]], val[k]);
}

// ELP_METHOD_AUTO's size rule: simplex when the dense tableau fits 200 KB.
// Stated on the former one-SM kernel's footprint, so that AUTO picks the same method for every shape as before.
bool simplex_auto_prefers(int m, int n) {
    auto up2 = [](size_t v) { return (v + 1) & ~(size_t)1; };
    auto up4 = [](size_t v) { return (v + 3) & ~(size_t)3; };
    const size_t N = (size_t)m + n;
    const size_t bytes = 8 * (up2((size_t)m * n) + up2((size_t)m * m) + 3 * up2(m) + 5 * up2(N) + 8) + 16 +
                         4 * (up4(m) + up4(N) + 8);
    return bytes <= 200 * 1024;
}

static int env_flag(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}

// Warp-per-LP path: returns false when the shape does not fit the register tableau (caller falls back).
template <int MR, int CPL>
static void simplex_warp_launch_inst(int64_t B, int m, int n, const double* A, const double* b, const double* c,
                                     const double* lb, const double* ub, const int8_t* sense, int maximize, int max_pivots,
                                     int32_t* status, double* obj, double* x, double* y, int32_t* pivots, cudaStream_t st,
                                     int shared_model, int32_t* basis) {
    auto kern = simplex_warp_kernel<MR, CPL>;
    const WarpSimplexLayout lay(MR, CPL);
    const size_t smem = (size_t)SW_WARPS * lay.total;
    ELP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    ELP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, SW_WARPS * 32, smem));
    occ = std::max(1, occ);
    auto al16 = [](const void* p) { return p == nullptr || (((uintptr_t)p) & 15) == 0; };
    const int use_tma = (n % 2 == 0) && al16(A) && env_flag("ELP_SIMPLEX_TMA", 1);   // 16-byte rows
    const int64_t want = (B + SW_WARPS - 1) / SW_WARPS;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)kNumSMs * occ));
    ELP_LAUNCH(kern, grid, SW_WARPS * 32, smem, st, B, m, n, A, b, c, lb, ub, sense, maximize, max_pivots, shared_model, use_tma,
               status, obj, x, y, pivots, basis);
}

static bool simplex_warp_launch(int64_t B, int m, int n, const double* A, const double* b, const double* c,
                                const double* lb, const double* ub, const int8_t* sense, int maximize, int max_pivots,
                                int32_t* status, double* obj, double* x, double* y, int32_t* pivots, cudaStream_t st,
                                int shared_model, int32_t* basis) {
    if (!env_flag("ELP_SIMPLEX_WARP", 1)) return false;
    const int N = m + n;
    if (m > 32 || N > 96) return false;
    const int mr = std::max(4, (m + 3) / 4 * 4), cpl = (N + 31) / 32;
    const size_t smem = (size_t)SW_WARPS * WarpSimplexLayout(mr, cpl).total;
    if (smem > 200 * 1024) return false;
#define ELP_SW(MR_, CPL_)                                                                                              \
    if (mr == MR_ && cpl == CPL_) {                                                                                    \
        simplex_warp_launch_inst<MR_, CPL_>(B, m, n, A, b, c, lb, ub, sense, maximize, max_pivots, status, obj, x, y, \
                                            pivots, st, shared_model, basis);                                          \
        return true;                                                                                                   \
    }
    ELP_SW(4, 1) ELP_SW(8, 1) ELP_SW(12, 1) ELP_SW(16, 1) ELP_SW(20, 1) ELP_SW(24, 1) ELP_SW(28, 1) ELP_SW(32, 1)
    ELP_SW(4, 2) ELP_SW(8, 2) ELP_SW(12, 2) ELP_SW(16, 2) ELP_SW(20, 2) ELP_SW(24, 2) ELP_SW(28, 2) ELP_SW(32, 2)
    ELP_SW(4, 3) ELP_SW(8, 3) ELP_SW(12, 3) ELP_SW(16, 3) ELP_SW(20, 3) ELP_SW(24, 3) ELP_SW(28, 3) ELP_SW(32, 3)
#undef ELP_SW
    return false;
}

// Can the device schedule one cluster of C CTAs with this much shared memory each?  C = 16 is a non-portable size.
static bool cluster_schedulable(int C, size_t smem) {
    if (smem > SC_SMEM_MAX) return false;
    const auto kern = simplex_kernel<SC_THREADS>;
    ELP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (C > 8) ELP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)C);
    cfg.blockDim = dim3(SC_THREADS);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int clusters = 0;
    if (cudaOccupancyMaxActiveClusters(&clusters, kern, &cfg) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return clusters >= 1;
}

// The one place that decides how many CTAs hold one LP's tableau: 1 (the warp kernel, else one CTA of simplex_kernel:
// one SM) or C (a cluster of simplex_kernel, the smallest C in {2, 4, 8, 16} that fits and can be scheduled).
// ELP_SIMPLEX_CLUSTER=C forces a cluster of C CTAs on any shape it can hold.  Throws when no kernel can take the shape.
int simplex_ctas(int m, int n) {
    const char* e = getenv("ELP_SIMPLEX_CLUSTER");
    const int forced = e ? atoi(e) : 0;
    if (forced == 2 || forced == 4 || forced == 8 || forced == 16) {
        if (cluster_schedulable(forced, SimplexLayout(m, n, forced).total)) return forced;
    }
    if (SimplexLayout(m, n, 1).total <= SC_SMEM_MAX) return 1;
    int largest = 0;
    for (int C = 2; C <= SC_MAX_CTAS; C *= 2) {
        if (!cluster_schedulable(C, std::min(SimplexLayout(m, n, C).total, SC_SMEM_MAX))) continue;
        largest = C;
        if (SimplexLayout(m, n, C).total <= SC_SMEM_MAX) return C;
    }
    int ncap = 0;          // structural columns the largest schedulable cluster holds at this row count
    if (largest) {
        int lo = 0, hi = 1 << 24;
        while (lo < hi) {
            const int mid = lo + (hi - lo + 1) / 2;
            if (SimplexLayout(m, mid, largest).total <= SC_SMEM_MAX) lo = mid;
            else hi = mid - 1;
        }
        ncap = lo;
    }
    throw Error(format("simplex: the dense tableau [A | I] of a %d x %d model (%lld doubles) exceeds the largest "
                       "thread-block cluster this device schedules (%d CTAs x 227 KB of shared memory: at %d rows it "
                       "holds at most %d columns)", m, n, (long long)m * (m + n), largest, m, ncap));
}

// all pointers are device pointers; returns the CTAs that held each tableau (simplex_ctas)
int simplex_batch_device(int64_t B, int m, int n, const double* A, const double* b, const double* c, const double* lb,
                         const double* ub, const int8_t* sense, int maximize, int max_pivots, int32_t* status,
                         double* obj, double* x, double* y, int32_t* pivots, cudaStream_t st, int shared_model,
                         int32_t* basis) {
    ELP_REQUIRE(n > 0 && m >= 0, "simplex: bad shape %d x %d", m, n);
    const int ctas = simplex_ctas(m, n);
    if (B <= 0) return ctas;
    ELP_REQUIRE(B * ctas < 0x7fffffffll, "simplex: batch too large");
    const size_t smem = SimplexLayout(m, n, ctas).total;
    if (ctas > 1) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(B * ctas));
        cfg.blockDim = dim3(SC_THREADS);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = (unsigned)ctas; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        g_launches.fetch_add(1, std::memory_order_relaxed);
        ELP_CUDA(cudaLaunchKernelEx(&cfg, simplex_kernel<SC_THREADS>, B, m, n, ctas, A, b, c, lb, ub, sense, maximize,
                                    max_pivots, shared_model, status, obj, x, y, pivots, basis));
        ELP_CUDA(cudaGetLastError());
        return ctas;
    }
    if (simplex_warp_launch(B, m, n, A, b, c, lb, ub, sense, maximize, max_pivots, status, obj, x, y, pivots, st, shared_model, basis)) return 1;
    // one CTA per LP, launched without a cluster: 32, 64 or 128 threads by the width m + n
    const int N = m + n, threads = N <= 32 ? 32 : (N <= 96 ? 64 : 128);
    const auto kern = threads == 32 ? simplex_kernel<32> : (threads == 64 ? simplex_kernel<64> : simplex_kernel<128>);
    ELP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ELP_LAUNCH(kern, (unsigned)B, threads, smem, st, B, m, n, 1, A, b, c, lb, ub, sense, maximize, max_pivots, shared_model,
               status, obj, x, y, pivots, basis);
    return 1;
}

void densify_device(int m, int n, const int* ptr, const int* idx, const double* val, double* A, cudaStream_t st) {
    ELP_CUDA(cudaMemsetAsync(A, 0, (size_t)std::max(m, 1) * n * sizeof(double), st));
    if (m > 0) ELP_LAUNCH(k_densify, m, 64, 0, st, m, n, ptr, idx, val, A);
}

}  // namespace elp
