/*
 * easylp_abi.h — C ABI of libeasylp_b200.so: the B200-native solve path behind EasyLP's R6 API.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  In the reference the boundary is the set of
 * lpSolveAPI R functions called from `$solve()` (/root/reference/R/class.R:260-278) plus the dense
 * R matrix algebra that `$con()` uses to build `constraint$mat` (/root/reference/R/class.R:189-220,
 * R/utils.R:95-106, R/methods.R:82-111,244-257).  Each entry point below names the reference
 * interface it replaces.  The R `.Call` glue that binds these lives in rpkg/src/r_glue.c; the ctypes
 * binding used by the tests lives in easylp_b200/_lib.py; INTEGRATION.md shows both.
 *
 * Conventions
 *   - plain C, POD arguments, caller-owned buffers, no exceptions cross the boundary;
 *   - every function returns 0 on success, nonzero on failure (then elp_last_error() has text);
 *   - indices are 0-based int32 (the R glue subtracts 1 from `ind`); doubles cross bit-for-bit;
 *   - +/-Inf bounds cross as IEEE infinities;
 *   - row sense codes: 0 "<=" (also "<"), 1 ">=" (also ">"), 2 "==" — the reference hands "<"/">"
 *     to lpSolveAPI::add.constraint, which treats them as "<="/">=" (R/class.R:271-274);
 *   - status codes are lp_solve's, exactly the keys of the switch at R/class.R:279-295:
 *     0 optimal, 2 unfeasible, 3 unbounded, 5 numerical failure, 7 timeout (iteration/time limit);
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with rc != 0.
 */
#ifndef EASYLP_ABI_H
#define EASYLP_ABI_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ELP_LE 0
#define ELP_GE 1
#define ELP_EQ 2

#define ELP_STATUS_OPTIMAL 0
#define ELP_STATUS_SUBOPTIMAL 1
#define ELP_STATUS_INFEASIBLE 2
#define ELP_STATUS_UNBOUNDED 3
#define ELP_STATUS_NUMFAILURE 5
#define ELP_STATUS_TIMEOUT 7

#define ELP_METHOD_AUTO 0    /* size rule: dense tableau fits 200 KB of one SM's shared memory -> simplex, else PDLP */
#define ELP_METHOD_SIMPLEX 1  /* dense tableau in one SM's shared memory, or beyond that spread over a thread-block
                                 cluster of 2-16 CTAs (about 420 k tableau entries m (m + n) at 16 CTAs, a few hundred
                                 rows); larger models are refused with an error naming the shape and the capacity */
#define ELP_METHOD_PDLP 2

/* How the plain PDHG iterations obtain g = A'y (pdlp.cu).
 *   GATHER  : a CSC (transposed) SpMV — deterministic, bit-reproducible run to run; the only mode when distributed.
 *   SCATTER : the CSR kernel that forms A.x-bar and the dual update also scatters val * y_new into g with fp64
 *             reductions (RED.ADD) while the row is still in shared memory, and the primal update becomes a gather-free
 *             elementwise pass.  One matrix stream per iteration instead of two; the summation order inside g is not
 *             fixed, so results agree with GATHER to rounding, not bit for bit.  Single GPU only.  Measured on C4
 *             (B200): 4037 vs 3745 iter/s — the reductions and the gathers share the L2 request rate, so the gain is small.
 *   AUTO    : GATHER (reproducible, and what north_star prescribes). */
#define ELP_TRANSPOSE_AUTO 0
#define ELP_TRANSPOSE_GATHER 1
#define ELP_TRANSPOSE_SCATTER 2

/* Options of a solve; mirrors the `...` that `$solve()` forwards to lpSolveAPI::lp.control()
 * (R/class.R:249-262): `timeout`, `epsilon`, `verbose` are mapped, the rest has no GPU meaning. */
typedef struct elp_options {
    double eps_rel;        /* PDLP relative KKT tolerance (default 1e-6; north_star) */
    double time_limit_s;   /* <=0: none. lp.control(timeout=) */
    int32_t max_iter;      /* PDLP iteration limit / simplex pivot limit (<=0: default) */
    int32_t check_every;   /* PDLP: iterations between termination/restart checks (<=0: default 64) */
    int32_t method;        /* ELP_METHOD_* */
    int32_t verbose;       /* lp.control(verbose=): 0 silent, >=1 progress lines to stderr */
    int32_t use_graph;     /* PDLP: replay the iteration chunk from a CUDA graph (default 1) */
    int32_t ruiz_iters;    /* <0: default 10 */
    int32_t transpose;     /* PDLP, how A'y is formed in the plain iterations: ELP_TRANSPOSE_* (default AUTO) */
    int32_t devices;       /* large-LP path: GPUs of this box to spread ONE solve over (0 or 1: the current device only;
                              N > 1: devices cur, cur+1, ... — row blocks of A, one worker thread per GPU inside this
                              call, see elp_solve_lp).  R: lp$solve(gpu.devices = N); default from env ELP_DEVICES */
} elp_options;

/* Per-solve statistics (SURVEY.md §5 "metrics"): returned to R as a list. */
typedef struct elp_stats {
    int32_t status;
    int32_t method_used;
    int32_t iterations;        /* PDHG iterations or simplex pivots (batch: total pivots) */
    int32_t restarts;
    double primal_obj;         /* in the problem's own sense, without objective_add */
    double dual_obj;
    double rel_primal_res;     /* ||Ax - proj(Ax)|| / (1 + ||b||) */
    double rel_dual_res;       /* ||r - proj(r)|| / (1 + ||c||) */
    double rel_gap;            /* |p - d| / (1 + |p| + |d|) */
    double setup_ms;           /* H2D + transpose + scaling + power iteration */
    double solve_ms;           /* device time of the iteration loop (CUDA events) */
    double total_ms;           /* host wall clock of the call */
    int64_t kernel_launches;   /* kernels launched by this call */
    int64_t h2d_bytes;
    int64_t d2h_bytes;
    double spmv_ms;            /* device time of the timed A.x / A'.y probe (elp_pdlp_probe_spmv) */
    int32_t limit_reached;     /* with status 7: 0 = only this call's max_new_iters ran out (call again), 1 = the iteration
                                  limit of the solve, 2 = its time limit (lp.control(timeout=)) — do not call again */
    int32_t simplex_ctas;      /* CTAs that held each simplex tableau: 0 PDLP ran, 1 one SM (a warp or one CTA), C a
                                  thread-block cluster of C CTAs (tableaus beyond one SM's shared memory) */
} elp_stats;

/* ---- housekeeping -------------------------------------------------------------------------- */
const char* elp_version(void);
int elp_last_error(char* buf, int32_t len);          /* copies the calling thread's last error text */
int elp_device_count(int32_t* count);
int elp_set_device(int32_t device);
int elp_default_options(elp_options* opt);
const char* elp_status_string(int32_t status);       /* the strings of R/class.R:279-295 */
int64_t elp_kernel_launches(void);                   /* process-wide counter of launched kernels */
int elp_release_workspace(void);                     /* frees the calling thread's cached device scratch (assembly) */

/* ---- (1) assembly: terms -> CSR ------------------------------------------------------------
 * Replaces the dense `constraint$mat` construction of `$con()`: rbind of evaluated atoms
 * (R/utils.R:95-106) whose entries were produced by dense adds in left-fold order
 * (R/methods.R:98-111, 244-257).  Input: T terms (row, col, val) in *emission order* (the order the
 * expression tree is folded in).  Output: canonical CSR = entries of the dense matrix that are != 0,
 * row-major, ascending column; duplicates of one (row, col) are summed strictly left-to-right in
 * emission order so the result is bit-identical to the reference's dense arithmetic.
 * row_ptr has m+1 entries; col_idx/vals must have room for n_terms entries; *nnz_out receives the count.
 * On the device: a stream that already is in (row, col) order — what `$con()` emits — takes two passes and no sort; any
 * other order is split into row buckets that one CTA each sorts and folds in shared memory; streams with a row too long
 * for a bucket fall back to a stable radix sort.  The three paths give the same bytes. */
int elp_assemble_csr(int64_t n_terms, const int32_t* term_row, const int32_t* term_col,
                     const double* term_val, int32_t m, int32_t n,
                     int32_t* row_ptr, int32_t* col_idx, double* vals, int64_t* nnz_out,
                     elp_stats* stats /* may be NULL */);

/* ---- (1b) lowered assembly: index-set descriptors expanded ON THE DEVICE (SURVEY §8f N2) ----------------------------
 * Replaces the interpreter loops of `for (v in seq) body` (R/utils.R:33-64: one `eval` per atom) and `sum_for`
 * (R/utils.R:391-411: one `eval` per grid row) for bodies that are affine in indexed variables: instead of T expanded
 * terms the host ships, per body term, a FAMILY descriptor — a loop nest (the `for` indices outermost first, then the
 * `sum_for` grid with its first name fastest, R/utils.R:402), a column-offset table per loop (the variable's
 * column-major ids, R/class.R:112-113) and a coefficient table over the loops the coefficient depends on.  One thread
 * per term decodes its position in the nest and writes (row, col, val, group); the stream then goes through the same
 * sort + ordered fold as elp_assemble_csr.
 * Fold order.  The reference folds each `sum_for` result on its own (`do.call(sum, ...)` = Reduce('+'),
 * R/methods.R:248-250) before the results of one atom are added (`e1 - e2`, R/methods.R:98-111) or scaled
 * (R/methods.R:82-97).  A GROUP is one such partial sum: inside a (row, col) the terms of a group are added left to
 * right in emission order, the group's sum is multiplied by its post-fold multipliers (one after the other), and the
 * group results are added left to right in group order.  Group 0 (explicit terms, no multipliers) reproduces
 * elp_assemble_csr.  Families of one (row, col) must be emitted in ascending group order. */
#define ELP_MAX_LOOPS 6
#define ELP_MAX_GROUP_MUL 4
typedef struct elp_term_family {
    int64_t count;                          /* terms emitted = product of the extents */
    int64_t out_offset;                     /* position of the family's first term in the lowered stream */
    int64_t coef_tab;                       /* offset of the coefficient table in dtab */
    int64_t col_tab[ELP_MAX_LOOPS];         /* per loop: offset in itab of its column-offset table, -1 = none */
    int64_t row_tab[ELP_MAX_LOOPS];         /* per loop: offset in itab of a row-offset table, -1 = use row_stride.  A ragged
                                               index set (`sum_for(a = out[[v]], ...)`) is one loop over the (v, a) pairs
                                               whose rows and columns both come from tables. */
    int64_t coef_stride[ELP_MAX_LOOPS];     /* per loop: stride in the coefficient table (0 = independent) */
    int32_t extent[ELP_MAX_LOOPS];          /* loops slowest first */
    int32_t row_stride[ELP_MAX_LOOPS];      /* per loop: contribution of one step to the row index */
    int32_t out_stride;                     /* distance in the stream between this family's terms of consecutive cells */
    int32_t group;                          /* fold group (index into `groups`; 0 = plain) */
    int32_t n_loops;
    int32_t row0;                           /* first row of the block */
    int32_t col0;                           /* column id of the variable's first entry plus the constant subscripts */
    int32_t reserved;
} elp_term_family;
typedef struct elp_fold_group {
    int64_t mul_tab[ELP_MAX_GROUP_MUL];     /* offset in dtab of multiplier k */
    int32_t mul_per_row[ELP_MAX_GROUP_MUL]; /* 1: one multiplier per row of the block (index row - row0), 0: a scalar */
    int32_t n_mul;                          /* post-fold multipliers, applied in this order */
    int32_t row0;
} elp_fold_group;
/* Explicit terms (may be none) + families -> canonical CSR.  col_idx/vals must have room for `capacity` entries
 * (n_terms + sum of family counts always suffices); fails if nnz exceeds it. */
int elp_assemble_lowered(int64_t n_terms, const int32_t* term_row, const int32_t* term_col, const double* term_val,
                         int32_t n_families, const elp_term_family* families,
                         int64_t n_itab, const int32_t* itab, int64_t n_dtab, const double* dtab,
                         int32_t n_groups, const elp_fold_group* groups,
                         int32_t m, int32_t n, int32_t* row_ptr, int32_t* col_idx, double* vals, int64_t capacity,
                         int64_t* nnz_out, elp_stats* stats /* may be NULL */);
/* The expanded term stream itself (tests: parity of the device expansion with the host's eager emission).
 * Arrays have room for the sum of the family counts. */
int elp_expand_terms(int32_t n_families, const elp_term_family* families, int64_t n_itab, const int32_t* itab,
                     int64_t n_dtab, const double* dtab, int32_t* row, int32_t* col, double* val, int32_t* group);

/* ---- (1c) device-resident model: the handle SURVEY 8b asks for (an R external pointer with a finalizer, treated as a
 * rebuildable cache).  elp_model_assemble = elp_assemble_lowered that KEEPS the canonical CSR in HBM; elp_model_solve =
 * elp_solve_lp on that CSR, so `$con()` ... `$solve()` moves the matrix over PCIe at most once (descriptors or terms
 * in, nothing out); elp_model_csr copies it back when the host wants `constraint$mat`. */
typedef struct elp_model elp_model;
int elp_model_assemble(int64_t n_terms, const int32_t* term_row, const int32_t* term_col, const double* term_val,
                       int32_t n_families, const elp_term_family* families,
                       int64_t n_itab, const int32_t* itab, int64_t n_dtab, const double* dtab,
                       int32_t n_groups, const elp_fold_group* groups,
                       int32_t m, int32_t n, elp_model** out, int64_t* nnz_out /* may be NULL */, elp_stats* stats /* may be NULL */);
int elp_model_dims(const elp_model* h, int32_t* m, int32_t* n, int64_t* nnz);
int elp_model_csr(const elp_model* h, int32_t* row_ptr /* m+1 */, int32_t* col_idx /* nnz */, double* vals /* nnz */);
int elp_model_solve(const elp_model* h, const int8_t* sense, const double* rhs, const double* c, int32_t maximize,
                    const double* lb, const double* ub, const elp_options* opt /* may be NULL */,
                    int32_t* status, double* objval, double* x /* n */, double* y /* m, may be NULL */, elp_stats* stats);
int elp_model_destroy(elp_model* h);

/* ---- (2) one LP: replaces make.lp/set.objfn/lp.control/set.bounds/add.constraint/solve/
 *      get.objective/get.variables  (R/class.R:260-278) ------------------------------------- */
int elp_solve_lp(int32_t m, int32_t n,
                 const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                 const int8_t* sense, const double* rhs,
                 const double* c, int32_t maximize,
                 const double* lb, const double* ub,
                 const elp_options* opt /* may be NULL */,
                 int32_t* status, double* objval, double* x /* n */, double* y /* m, may be NULL */,
                 elp_stats* stats /* may be NULL */);

/* ---- (2b) models with integer / binary variables: replaces `solve(prob)` after `set.type(prob, columns, "integer" |
 *      "binary")` (R/class.R:264-276), i.e. lp_solve's branch and bound.  is_integer[j] != 0 marks an integer column (a
 *      binary one is an integer column with bounds [0, 1], R/class.R:104-110).  The tree's open nodes share A, b, c and
 *      differ in their bounds: every frontier is ONE launch of the batched simplex kernel (csrc/mip.cu).  Status codes as
 *      lp_solve: 0 optimal, 2 unfeasible, 3 unbounded, 1 sub-optimal / 7 timeout when opt->max_iter (a NODE limit here) or
 *      opt->time_limit_s stops the search with / without an incumbent.  stats->restarts = nodes solved,
 *      stats->iterations = simplex pivots.  Models whose dense tableau does not fit one SM run on the cluster kernel
 *      (ELP_METHOD_SIMPLEX); beyond the largest cluster they are refused. */
int elp_solve_mip(int32_t m, int32_t n,
                  const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                  const int8_t* sense, const double* rhs,
                  const double* c, int32_t maximize,
                  const double* lb, const double* ub, const uint8_t* is_integer /* n */,
                  const elp_options* opt /* may be NULL */,
                  int32_t* status, double* objval, double* x /* n */, elp_stats* stats /* may be NULL */);

/* ---- (2c) sensitivity ranging: replaces lpSolveAPI::get.sensitivity.obj / get.sensitivity.rhs behind
 *      `$sensitivity_objective` and `$sensitivity_rhs` (R/class.R:613-646).  Solves the LP on the simplex path (ranging
 *      needs a basis; one SM, or a thread-block cluster for larger tableaus, as ELP_METHOD_SIMPLEX) and returns, per variable, the interval [obj_from, obj_till] of its cost over
 *      which the optimal basis stays optimal and, per constraint, the interval [rhs_from, rhs_till] of its right-hand
 *      side over which the basis stays feasible (the dual value `duals[i]` is valid there).  Infinite ends are IEEE
 *      infinities.  Textbook basis-invariance ranges; lp_solve's conventions at degenerate vertices are not pinned
 *      (csrc/sensitivity.cu). */
int elp_sensitivity(int32_t m, int32_t n,
                    const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                    const int8_t* sense, const double* rhs,
                    const double* c, int32_t maximize,
                    const double* lb, const double* ub,
                    const elp_options* opt /* may be NULL */,
                    int32_t* status, double* objval, double* x /* n */,
                    double* obj_from /* n */, double* obj_till /* n */,
                    double* rhs_from /* m */, double* rhs_till /* m */, double* duals /* m */);

/* ---- (3) a batch of small dense LPs (BASELINE config 3; additive entry point, SURVEY §0.5) ---
 * A is [B][m][n] row-major, b [B][m], c [B][n], lb/ub [B][n] (NULL => 0 / +Inf), sense [B][m]
 * (NULL => all "<=").  One LP per WARP with the tableau in shared memory (shapes with m > 32 or m + n > 96: one LP
 * per CTA; tableaus beyond one SM: one LP per thread-block cluster); outputs status[B], obj[B], x[B][n]. */
int elp_solve_batch(int64_t B, int32_t m, int32_t n,
                    const double* A, const double* b, const double* c,
                    const double* lb, const double* ub, const int8_t* sense, int32_t maximize,
                    const elp_options* opt, int32_t* status, double* obj, double* x,
                    elp_stats* stats);

/* Device-resident batch (bench `value`: inputs already in HBM when the timed region starts). */
typedef struct elp_batch elp_batch;
int elp_batch_create(int64_t B, int32_t m, int32_t n,
                     const double* A, const double* b, const double* c,
                     const double* lb, const double* ub, const int8_t* sense, int32_t maximize,
                     elp_batch** out);
int elp_batch_run(elp_batch* h, const elp_options* opt, elp_stats* stats);   /* solve in place, on device */
int elp_batch_fetch(elp_batch* h, int32_t* status, double* obj, double* x);
int elp_batch_destroy(elp_batch* h);

/* ---- (S4) post-solve feasibility re-check: replaces `mat %*% sol` + compare_tol
 *      (R/class.R:533-540, R/utils.R:167-171).  sense here keeps strictness: 0 <=, 1 >=, 2 ==,
 *      3 "<", 4 ">".  feasible[i] = 1/0. -------------------------------------------------------- */
int elp_spmv(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
             const double* x, double* out /* m */);
int elp_check_feasible(int32_t m, int32_t n, const int32_t* row_ptr, const int32_t* col_idx,
                       const double* vals, const double* x, const int8_t* sense, const double* rhs,
                       double tol, uint8_t* feasible /* m */);

/* ---- PDLP with device-resident state (bench + multi-GPU) -------------------------------------
 * elp_pdlp_create uploads the LP, builds the CSC copy, scales (Ruiz + Pock-Chambolle), estimates
 * ||A||_2.  elp_pdlp_run advances until convergence or `max_new_iters` more iterations.
 * With a communicator initialised (elp_comm_init) and dist != 0 the caller passes ITS row block:
 * rows [row_begin, row_begin + m_local) of the global matrix (column ids global, 0..n-1) and the FULL c, lb, ub.
 * The library keeps the row block for A.x-bar and builds, by one exchange among the ranks, the column block it
 * needs for A'.y; per iteration the ranks exchange their x-bar / y blocks over NVLink (peer stores from the kernel
 * epilogues, NCCL all-gather as fallback) and the scalar residuals travel in one allreduce (SURVEY §8e, DESIGN §5).
 * elp_pdlp_solution returns all n entries of x on every rank and the rank's own m_local entries of y. */
typedef struct elp_pdlp elp_pdlp;
int elp_pdlp_create(int32_t m_local, int32_t n,
                    const int32_t* row_ptr, const int32_t* col_idx, const double* vals,
                    const int8_t* sense, const double* rhs,
                    const double* c, int32_t maximize, const double* lb, const double* ub,
                    const elp_options* opt, int32_t dist, elp_pdlp** out, elp_stats* stats);
int elp_pdlp_run(elp_pdlp* h, int32_t max_new_iters, elp_stats* stats);
int elp_pdlp_reset(elp_pdlp* h);                                   /* back to the initial iterate */
int elp_pdlp_solution(elp_pdlp* h, double* x /* n */, double* y /* m_local, may be NULL */, double* objval);
int elp_pdlp_probe_spmv(elp_pdlp* h, int32_t reps, double* ms_csr, double* ms_csc);  /* times bare A.x and A'.y */
/* times the two fused iteration kernels alone (A'y + primal update; A.xbar + dual update); resets the iterate */
int elp_pdlp_probe_step(elp_pdlp* h, int32_t reps, double* ms_primal, double* ms_dual);
int elp_pdlp_transpose(elp_pdlp* h, int32_t* mode);   /* the ELP_TRANSPOSE_* the plain iterations of this handle use */
int elp_pdlp_destroy(elp_pdlp* h);
/* A PDLP handle on a device-resident model (elp_model_assemble): the CSR is copied device-to-device.  With
 * elp_pdlp_run(h, k) in a loop the caller regains control every k iterations — the R glue checks for user interrupts
 * there (SURVEY 8b) — and the result is the one elp_model_solve returns. */
int elp_model_pdlp_create(const elp_model* model, const int8_t* sense, const double* rhs, const double* c,
                          int32_t maximize, const double* lb, const double* ub, const elp_options* opt,
                          elp_pdlp** out, elp_stats* stats);

/* ---- multi-GPU plumbing for callers that run one process (or one host thread) per GPU.  The communicator belongs to the
 * CALLING THREAD; NCCL is resolved with dlopen at first use.  A caller that just wants one solve spread over the box sets
 * elp_options.devices instead and needs none of this. -------- */
#define ELP_UNIQUE_ID_BYTES 128
int elp_comm_unique_id(void* id /* ELP_UNIQUE_ID_BYTES */);
int elp_comm_init(int32_t nranks, int32_t rank, const void* id);
int elp_comm_size(int32_t* nranks, int32_t* rank);
int elp_comm_destroy(void);

#ifdef __cplusplus
}
#endif
#endif /* EASYLP_ABI_H */
